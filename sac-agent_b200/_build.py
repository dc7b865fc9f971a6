"""In-tree nvcc build of libboatenv.so (sm_100a only).

    python -m sac_agent_b200._build        # or __graft_entry__.build()

The shared library is written next to this file so that it travels with the source
tree to the GPU box; it is git-ignored (history stays source-only).
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libboatenv.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
          "-I", os.path.join(os.path.dirname(HERE), "include")]
# translation unit -> extra flags.  The fp64 validation kernels must keep the
# reference's unfused multiply/add rounding.
UNITS = {
    "step_f32.cu": [],
    "step_f64.cu": ["-fmad=false"],
    "abi.cu": [],
    "replay.cu": [],
    "toys.cu": ["-fmad=false"],
    "agent_ops.cu": [],
    "policy_mlp.cu": [],
    "record.cu": [],
    "rollout.cu": [],
    "learner.cu": [],
}


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libboatenv.so cannot be built (there is no CPU fallback)")
    return exe


def _deps_mtime() -> float:
    m = os.path.getmtime(os.path.join(os.path.dirname(HERE), "include", "boatenv.h"))
    for f in os.listdir(CSRC):
        if f.endswith((".cuh", ".h", ".inl")):
            m = max(m, os.path.getmtime(os.path.join(CSRC, f)))
    return m


def _compile(unit: str, flags, verbose: bool, obj_dir: str = OBJ, variant_flags=()) -> str:
    src = os.path.join(CSRC, unit)
    obj = os.path.join(obj_dir, unit.replace(".cu", ".o"))
    if os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(src), _deps_mtime()):
        return obj
    extra = os.environ.get("BOATENV_NVCC_FLAGS", "").split() + list(variant_flags)  # tuning experiments only
    cmd = [nvcc(), *ARCH, *COMMON, *flags, *extra, "-c", src, "-o", obj]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {unit}:\n{r.stdout}\n{r.stderr}")
    if verbose:
        sys.stderr.write(r.stderr)
    return obj


def build(force: bool = False, verbose: bool = False, variant: str = "", variant_flags=()) -> str:
    """Builds libboatenv.so.  ``variant`` (ablation experiments only, e.g. ("novote", ["-DBOAT_DEBUG_NO_REFILL_VOTE"]))
    builds libboatenv_<variant>.so with the extra nvcc flags; select it at run time with BOATENV_LIBRARY=<path>."""
    obj_dir = OBJ if not variant else os.path.join(CSRC, "_obj_" + variant)
    lib = LIB if not variant else os.path.join(HERE, f"libboatenv_{variant}.so")
    os.makedirs(obj_dir, exist_ok=True)
    if force:
        for f in os.listdir(obj_dir):
            os.remove(os.path.join(obj_dir, f))
    units = {u: fl for u, fl in UNITS.items() if os.path.exists(os.path.join(CSRC, u))}
    with cf.ThreadPoolExecutor(max_workers=len(units)) as ex:
        objs = list(ex.map(lambda kv: _compile(kv[0], kv[1], verbose, obj_dir, variant_flags), units.items()))
    if (not os.path.exists(lib)) or any(os.path.getmtime(o) > os.path.getmtime(lib) for o in objs):
        cmd = [nvcc(), *ARCH, "-shared", "-o", lib, *objs]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib


if __name__ == "__main__":
    if "--variant" in sys.argv:  # python -m sac_agent_b200._build --variant novote -DBOAT_DEBUG_NO_REFILL_VOTE
        i = sys.argv.index("--variant")
        print(build(variant=sys.argv[i + 1], variant_flags=[a for a in sys.argv[i + 2:] if a.startswith("-D")]))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
