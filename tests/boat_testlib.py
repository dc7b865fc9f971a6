"""Shared helpers of the test-suite (golden loading, the parity error metric, the replay ring's store counter, the host
reference of the device random streams)."""
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# observation normalisers of the reference (boat_env.py:310-321): the scale S_i of the
# error metric |a-b| / max(|b|, S_i) (SURVEY.md H6) -- applied to NORMALISED obs
# these scales are all 1; applied to raw quantities they are the spans below.
RAW_SCALES = dict(s_x=3900.0, v_x=5.0, a_x=0.025, s_y=800.0, v_y=2.0, a_y=0.37,
                  s_r=2 * np.pi, v_r=8.5e-3, a_r=1.4e-5, rudder=np.pi / 3, fuel=15000.0)


def load_golden(name):
    d = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    out = {k: d[k] for k in d.files}
    for k in ("config", "meta", "columns"):
        if k in out:
            out[k] = json.loads(str(out[k]))
    return out


AGENT_KEYS = ("learning_rate_alpha", "learning_rate_beta", "gamma", "tvn_parameter_modulation_tau", "reward_scale")


def reference_config_record():
    """The values of the reference's configs/original_config.yaml that tests/golden recorded (oracle/make_golden.py,
    make_agent_golden.py): the hot-path keys stored beside the reference roll-outs, which set
    base_settings.experiment per file (left out here), and the agent keys of the recorded SAC update."""
    cfgs = [load_golden(f"ref_rollout_exp{e}")["config"] for e in range(1, 7)]
    for e, cfg in enumerate(cfgs, 1):
        assert cfg["base_settings"].pop("experiment") == e
    assert all(cfg == cfgs[0] for cfg in cfgs)
    rec = np.load(os.path.join(GOLDEN, "agent_update.npz"))
    cfgs[0]["agent"] = {k: rec["meta/" + k].item() for k in AGENT_KEYS}
    return cfgs[0]


def set_mem_cntr(mem, value):
    """Moves the store counter of the ReplayBuffer `mem` (boatreplay_set_mem_cntr) without writing rows."""
    from sac_agent_b200 import _lib
    _lib.check(mem._L.boatreplay_set_mem_cntr(mem._h, int(value)), "boatreplay_set_mem_cntr")


def scaled_err(a, b, scale=1.0):
    """|a-b| / max(|b|, scale): the parity metric of SURVEY.md H6."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), scale)


# ---- the device random streams, restated on the host (DESIGN.md, "Random streams") ----------------------------------
_LO = np.uint64(0xFFFFFFFF)


def _u64(x):
    return np.asarray(x, dtype=np.uint64)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) over numpy arrays: the four counter words broadcast against each other, the
    key is two 32-bit integers.  Returns the four output words as uint64 arrays of 32-bit values (the 32 x 32-bit
    products are formed in uint64)."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(_u64(c) & _LO for c in (c0, c1, c2, c3)))
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    m0, m1, s = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2
        c0, c1, c2, c3 = (p1 >> s) ^ c1 ^ k0, p1 & _LO, (p0 >> s) ^ c3 ^ k1, p0 & _LO
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _LO, (k1 + np.uint64(0xBB67AE85)) & _LO
    return c0, c1, c2, c3


def _word(r, i):
    """Word i (0..3, an array) of the Philox blocks r."""
    return np.choose(_u64(i).astype(np.intp) & 3, r)


def acting_words(seed, rows, steps, a):
    """Words x, y of the acting-noise block of (handle row, step, action a): actor_normal_draw, csrc/actor_tc.cuh."""
    rows, steps, a = _u64(rows), _u64(steps), _u64(a)
    seed = int(seed)
    c3 = np.uint64(0xD0000000) | (a << np.uint64(16)) | ((steps >> np.uint64(32)) & np.uint64(0xFFFF))
    x, y, _, _ = philox4x32_10(rows, rows >> np.uint64(32), steps, c3, seed, seed >> 32)
    return x, y


def cospi(x):
    """cos(pi x) in float64 with the argument reduced exactly to the nearest multiple of 1/2 first, so that it is
    exactly 0 at odd multiples of 1/2, as cospif is (np.cos(2 np.pi * 0.75) is -1.8e-16)."""
    x = np.asarray(x, dtype=np.float64)
    n = np.rint(2.0 * x)
    r = np.pi * (x - 0.5 * n)   # |r| <= pi / 4
    return np.choose(n.astype(np.int64) & 3, [np.cos(r), -np.sin(r), -np.cos(r), np.sin(r)])


def acting_normal(seed, rows, steps, a):
    """The standard-normal acting draw of (handle row, step, action a): the uniforms formed in fp32 exactly as the
    kernel forms them, u = ((w >> 8) + 0.5) * 2^-24, then Box-Muller in float64."""
    x, y = acting_words(seed, rows, steps, a)
    u1, u2 = (((w >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24) for w in (x, y))
    return np.sqrt(-2.0 * np.log(u1.astype(np.float64))) * cospi(2.0 * u2.astype(np.float64))


def replay_indices(seed, counter, batch, max_mem):
    """The ring slots sample_buffer draws (replay_index, csrc/replay.cu): row b takes word b & 3 of the block
    (b >> 2, counter) and maps it to floor(w * max_mem / 2^32).  int64 [batch]."""
    assert 0 < max_mem < 2 ** 32
    counter, seed = int(counter), int(seed)
    blk = np.arange((batch + 3) // 4, dtype=np.uint64)
    r = philox4x32_10(blk, blk >> np.uint64(32), counter, 0xB0000000 | ((counter >> 32) & 0x0FFFFFFF), seed, seed >> 32)
    w = np.stack(r, axis=1).reshape(-1)[:batch]
    return ((w * np.uint64(max_mem)) >> np.uint64(32)).astype(np.int64)


def uniform_actions(seed, global_ids, step, scale, dtype):
    """The uniform(-1, 1) * scale action of each global env id at `step` (boat_fill_actions_kernel,
    csrc/aux_kernels.cuh): word g & 3 of the block (g >> 2, step), (w >> 8) * 2^-23 - 1 and the product with the
    scale rounded to fp32, all in fp32, then cast to `dtype`.  `scale` may be an array that broadcasts against the
    ids (several scales from one set of Philox blocks)."""
    g = _u64(global_ids)
    q, step, seed = g >> np.uint64(2), int(step), int(seed)
    r = philox4x32_10(q, q >> np.uint64(32), step, 0xA0000000 | ((step >> 32) & 0x0FFFFFFF), seed, seed >> 32)
    u = (_word(r, g) >> np.uint64(8)).astype(np.float32) * np.float32(2.0 ** -23) - np.float32(1.0)
    return (np.asarray(scale, dtype=np.float32) * u).astype(dtype)
