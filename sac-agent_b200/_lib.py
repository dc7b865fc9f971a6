"""ctypes binding of libboatenv.so (include/boatenv.h).  No torch types cross the ABI:
tensors are passed as ``data_ptr()`` integers, streams as ``cuda_stream`` integers.

Fails loudly: if the shared library has not been built (``__graft_entry__.build()`` /
``python -m sac_agent_b200._build``) every use raises -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

from .config import BoatEnvParams

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libboatenv.so"


class BoatEnvError(RuntimeError):
    def __init__(self, code: int, what: str = ""):
        self.code = code
        msg = _error_string(code)
        super().__init__(f"{what + ': ' if what else ''}{msg} (code {code})")


def library_path() -> str:
    """libboatenv.so next to this file; BOATENV_LIBRARY selects an ablation build (profiles/ experiments only)."""
    return os.environ.get("BOATENV_LIBRARY") or os.path.join(HERE, _LIB_NAME)


_lib = None

vp, i64, u64, i32, u32, dbl = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32, C.c_uint32, C.c_double
PP = C.POINTER(BoatEnvParams)


class RecordRing(C.Structure):
    """boatenv_record_ring: device column pointers [capacity][n_ids] of a recording ring."""
    _fields_ = [(name, vp) for name in ("s_x", "s_y", "v_x", "v_y", "s_r", "rudder_angle", "action", "reward",
                                        "term", "episode")] + [("capacity", i64)]

class SacMember(C.Structure):
    """boatagent_sac_member: one agent's arguments of boatagent_sac_update_members and its split calls."""
    _fields_ = [(name, vp) for name in ("state", "action", "reward", "new_state", "done", "eps", "max_action",
                                        "slots")] + [("n_slots", i32), ("gamma", C.c_float), ("reward_scale", C.c_float),
                                                     ("tau", C.c_float), ("adam_state", vp), ("losses", vp)]


class Sac2Member(C.Structure):
    """boatagent_sac2_member: one agent's arguments of boatagent_sac2_update_members."""
    _fields_ = [("base", SacMember), ("target_entropy", C.c_float)]


class SacPrioritizedMember(C.Structure):
    """boatagent_sac_prioritized_member: a SacMember with its rows' importance weights and TD-error output."""
    _fields_ = [("base", SacMember), ("weights", vp), ("td_out", vp)]


class Sac2PrioritizedMember(C.Structure):
    """boatagent_sac2_prioritized_member: a Sac2Member with its rows' importance weights and TD-error output."""
    _fields_ = [("base", Sac2Member), ("weights", vp), ("td_out", vp)]


class SampleMember(C.Structure):
    """boatreplay_sample_member: one ring's arguments of boatreplay_sample_members."""
    _fields_ = [("ring", vp), ("seed", u64), ("counter", u64)] + [(name, vp) for name in ("s_out", "a_out", "r_out",
                                                                                            "s2_out", "done_out")]


# name -> (restype, argtypes): one row per declaration in include/boatenv.h
SIGNATURES = {
    "boatenv_create": (C.c_int, [PP, i64, u64, i64, C.c_int, C.c_int, C.POINTER(vp)]),
    "boatenv_destroy": (C.c_int, [vp]),
    "boatenv_reset": (C.c_int, [vp, vp, vp, vp]),
    "boatenv_step": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, u32, vp]),
    "boatenv_step_k": (C.c_int, [vp, vp, i64, i32, vp, vp, vp, vp, vp, u32, vp]),
    "boatenv_step_host": (C.c_int, [vp, vp, vp, vp, vp, u32]),
    "boatenv_step_host_term": (C.c_int, [vp, vp, vp, vp, vp, vp, u32]),
    "boatenv_step_host_stream": (C.c_int, [vp, vp, vp, vp, vp, vp, u32, vp]),
    "boatenv_step_k_host": (C.c_int, [vp, vp, i32, vp, vp, vp, vp, vp, u32, vp]),
    "boatenv_get_field": (C.c_int, [vp, C.c_int, vp, vp]),
    "boatenv_set_field": (C.c_int, [vp, C.c_int, vp, vp]),
    "boatenv_env_state_host": (C.c_int, [vp, i64, C.POINTER(dbl)]),
    "boatenv_wind_table": (C.c_int, [vp, i64, vp, vp, vp]),
    "boatenv_record_rows": (C.c_int, [vp, vp, i64, vp, vp, vp, C.POINTER(RecordRing), i64, vp]),
    "boatenv_wind_length": (C.c_int, [vp]),
    "boatenv_set_episode_draws": (C.c_int, [vp, vp, vp, vp]),
    "boatenv_episode_draws_host": (C.c_int, [PP, u64, i64, u32, C.POINTER(i32), C.POINTER(dbl)]),
    "boatenv_episode_draws_batch_host": (C.c_int, [PP, u64, vp, i64, u32, i32, vp, vp]),
    "boatenv_state_bytes": (i64, [vp]),
    "boatenv_export_state": (C.c_int, [vp, vp, vp]),
    "boatenv_import_state": (C.c_int, [vp, vp, vp]),
    "boatenv_get_counters": (C.c_int, [vp, C.POINTER(dbl), vp]),
    "boatenv_reduce_counters": (C.c_int, [vp, vp, vp]),
    "boatenv_fill_uniform_actions": (C.c_int, [vp, u64, dbl, vp, vp]),
    "boatagent_gaussian_head_forward": (C.c_int, [vp, vp, vp, vp, i64, i32, vp, vp, vp]),
    "boatagent_gaussian_head_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, i64, i32, vp, vp, vp]),
    "boatagent_adam_polyak_step": (C.c_int, [vp, i32, C.c_float, C.c_float, C.c_float, C.c_float, vp, vp]),
    "boatagent_policy_act": (C.c_int, [vp, vp, vp, vp, u64, u64, i64, i32, i32, vp, vp]),
    "boatagent_rollout": (C.c_int, [vp, vp, vp, u64, u64, i32, u32, vp, vp, vp, vp, vp, vp]),
    "boatagent_collect": (C.c_int, [vp, vp, vp, vp, u64, u64, i32, C.c_int, vp, vp, vp, vp, vp]),
    "boatagent_collect_record": (C.c_int, [vp, vp, vp, vp, u64, u64, i32, C.c_int, vp, vp, vp, vp, vp, i64,
                                           C.POINTER(RecordRing), i64, vp]),
    "boatagent_sac_update_workspace_bytes": (i64, [i64]),
    "boatagent_sac_update": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, C.c_float, C.c_float, vp, i32, C.c_float,
                                       C.c_float, C.c_float, C.c_float, vp, vp, vp, i64, vp]),
    "boatagent_sac_gradients": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, C.c_float, C.c_float, vp, i32, C.c_float,
                                          vp, vp, i64, vp]),
    "boatagent_sac_update_members": (C.c_int, [C.POINTER(SacMember), i32, i64, C.c_float, C.c_float, C.c_float, vp,
                                               i64, vp]),
    "boatagent_sac_gradients_members": (C.c_int, [C.POINTER(SacMember), i32, i64, C.c_float, vp, i64, vp]),
    "boatagent_adam_polyak_members": (C.c_int, [C.POINTER(SacMember), i32, C.c_float, C.c_float, C.c_float, vp]),
    "boatagent_sac2_update_workspace_bytes": (i64, [i64]),
    "boatagent_sac2_update_members": (C.c_int, [C.POINTER(Sac2Member), i32, i64, C.c_float, C.c_float, C.c_float, vp,
                                                i64, vp]),
    "boatagent_sac_update_prioritized_members": (C.c_int, [C.POINTER(SacPrioritizedMember), i32, i64, C.c_float,
                                                           C.c_float, C.c_float, vp, i64, vp]),
    "boatagent_sac2_update_prioritized_members": (C.c_int, [C.POINTER(Sac2PrioritizedMember), i32, i64, C.c_float,
                                                            C.c_float, C.c_float, vp, i64, vp]),
    "boatreplay_sample_members": (C.c_int, [C.POINTER(SampleMember), i32, i64, vp]),
    "boatreplay_create": (C.c_int, [i64, i32, i32, C.c_int, C.c_int, C.POINTER(vp)]),
    "boatreplay_destroy": (C.c_int, [vp]),
    "boatreplay_store": (C.c_int, [vp, i64, vp, vp, vp, vp, vp, vp]),
    "boatreplay_sample": (C.c_int, [vp, i64, u64, u64, vp, vp, vp, vp, vp, vp, vp]),
    "boatreplay_gather": (C.c_int, [vp, i64, vp, vp, vp, vp, vp, vp, vp]),
    "boatreplay_mem_cntr": (i64, [vp]),
    "boatreplay_set_mem_cntr": (C.c_int, [vp, i64]),
    "boatreplay_mem_size": (i64, [vp]),
    "boatper_create": (C.c_int, [i64, C.c_int, C.POINTER(vp)]),
    "boatper_destroy": (C.c_int, [vp]),
    "boatper_fill_new": (C.c_int, [vp, i64, i64, vp]),
    "boatper_sample": (C.c_int, [vp, i64, u64, u64, dbl, vp, vp, vp]),
    "boatper_find": (C.c_int, [vp, i64, vp, vp, vp]),
    "boatper_update": (C.c_int, [vp, i64, vp, vp, dbl, dbl, vp]),
    "boatper_check": (C.c_int, [vp, vp]),
    "boatper_level_size": (i64, [vp, i32]),
    "boatper_filled": (i64, [vp]),
    "boatper_read": (C.c_int, [vp, i32, vp, vp]),
    "boatper_load": (C.c_int, [vp, vp, i64, vp, i64, vp]),
    "boatenv_step_store": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, C.c_int, u32, vp]),
    "boattoy_create": (C.c_int, [C.c_int, i64, C.POINTER(dbl), i32, dbl, u64, C.c_int, C.c_int, C.POINTER(vp)]),
    "boattoy_destroy": (C.c_int, [vp]),
    "boattoy_reset": (C.c_int, [vp, vp]),
    "boattoy_step": (C.c_int, [vp, i32, vp, vp, vp]),
    "boattoy_params_host": (C.c_int, [C.c_int, C.POINTER(dbl), i32, dbl, u64, i64, i64, vp]),
    "boatenv_version": (C.c_char_p, []),
    "boatenv_error_string": (C.c_char_p, [C.c_int]),
    "boatenv_kernel_launches": (i64, []),
}


def lib():
    """The loaded library; raises if it is missing (no fallback)."""
    global _lib
    if _lib is None:
        path = library_path()
        if not os.path.exists(path):
            raise ImportError(
                f"{path} is missing: build the CUDA extension first (python -c 'import "
                "__graft_entry__ as g; g.build()').  sac_agent_b200 has no CPU fallback.")
        L = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _error_string(code: int) -> str:
    try:
        return lib().boatenv_error_string(int(code)).decode()
    except Exception:  # pragma: no cover
        return "error"


def check(code: int, what: str = "") -> None:
    if code == 0:
        return
    # the reference raises ValueError for these two (wind.py:65-67, :73-75)
    if code in (-2, -3):
        raise ValueError(_error_string(code))
    raise BoatEnvError(code, what)
