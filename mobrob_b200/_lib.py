"""ctypes binding of libmobrob_b200.so (include/mobrob_b200.h).

There is no CPU fallback: importing this module without the built library, or calling
into it without a CUDA device, raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

from . import build as _build

_LIB = None

_P = c_void_p

_SIGNATURES = {
    "mr_version": (c_int, []),
    "mr_last_error": (c_char_p, []),
    "mr_launch_count": (c_uint64, []),
    "mr_env_create": (c_int, [c_int, c_int64, c_int, c_int, c_int, POINTER(c_void_p)]),
    "mr_env_destroy": (None, [_P]),
    "mr_env_obs_dim": (c_int, [_P]),
    "mr_env_state_dim": (c_int, [_P]),
    "mr_env_set_contacts": (c_int, [_P, c_int]),
    "mr_env_set_obs_flags": (c_int, [_P, ctypes.c_uint]),
    "mr_env_set_lidar": (c_int, [_P, c_int, c_double, c_double, c_int]),
    "mr_env_set_spaces": (c_int, [_P, _P, _P, _P]),
    "mr_env_seed": (c_int, [_P, _P, _P, _P, _P]),
    "mr_env_reset": (c_int, [_P, _P, c_int, _P, _P]),
    "mr_env_step": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mr_env_get_obs": (c_int, [_P, _P, _P]),
    "mr_env_get_state": (c_int, [_P, _P, _P]),
    "mr_env_set_state": (c_int, [_P, _P, _P]),
    "mr_env_get_pos": (c_int, [_P, _P, _P]),
    "mr_env_get_reset_counts": (c_int, [_P, _P, _P]),
    "mr_policy_forward": (c_int, [_P, c_int, _P, _P, _P, _P, _P, c_int64, _P]),
    "mr_gae": (c_int, [_P, _P, _P, _P, _P, c_double, c_double, _P, _P, c_int64, c_int64, _P]),
    "mr_ppo_num_params": (c_int, [c_int]),
    "mr_ppo_grad_stride": (c_int, [c_int]),
    "mr_ppo_max_parts": (c_int, []),
    "mr_ppo_epoch_scratch_floats": (c_int, [c_int]),
    "mr_ppo_adv_stats": (c_int, [_P, _P, c_int64, c_int64, c_int64, c_int64, _P, _P]),
    "mr_ppo_grad": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P, c_int64, _P, c_int64, c_int64,
                            c_float, c_float, c_float, c_int, c_float, _P, _P, _P, c_float, _P, _P]),
    "mr_ppo_train_epoch": (c_int, [_P, _P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, _P,
                                   c_int64, c_int64, c_float, c_float, c_float, c_int, c_float, c_float,
                                   c_float, c_float, c_float, _P, _P, _P, _P, c_float, c_float, _P, c_int64, _P]),
    "mr_ppo_train_summary": (c_int, [_P, c_int, _P, _P, c_int64, _P, _P, _P, _P, _P]),
    "mr_xchg_create": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_void_p), _P]),
    "mr_xchg_connect": (c_int, [_P, _P]),
    "mr_xchg_destroy": (None, [_P]),
    "mr_xchg_status": (c_int, [_P, POINTER(c_int)]),
    "mr_ppo_record_floats": (c_int, [c_int]),
    "mr_ppo_pack_samples": (c_int, [c_int, _P, _P, _P, _P, _P, _P, c_int64, _P, _P]),
    "mr_ppo_epoch_fused": (c_int, [_P, _P, _P, _P, c_int, _P, _P, _P, c_int64, c_int64, _P,
                                   c_int64, c_int64, c_float, c_float, c_float, c_int, c_float, c_float,
                                   c_float, c_float, c_float, _P, _P, _P, _P, c_float, c_float, _P, c_int64, _P]),
    "mr_rollout": (c_int, [_P, _P, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_uint64,
                           c_uint64, c_int64, c_double, _P, _P, _P, _P, _P, _P, c_int, _P]),
    "mr_rollout_unfused": (c_int, [_P, _P, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_uint64,
                                   c_uint64, c_int64, c_double, _P, _P, _P, _P, _P, _P, c_int, _P]),
    "mr_evaluate": (c_int, [_P, _P, c_int, c_int64, c_int64, c_uint64, c_uint64, c_int64, _P, _P, _P, _P, _P, _P,
                            _P]),
    "mr_device_permutations": (c_int, [c_uint64, _P, c_int, c_int64, _P, _P]),
    "mr_ppo_prepare_epochs": (c_int, [_P, _P, c_int, c_int64, c_int64, c_int64, c_int64, _P, _P, _P]),
    "mr_ppo_prepare_epochs_device": (c_int, [c_uint64, _P, c_int, _P, c_int64, c_int64, c_int64, c_int64, _P, _P, _P]),
    "mr_host_permutation": (c_int, [c_uint64, c_uint64, c_int64, _P]),
    "mr_adam_step": (c_int, [_P, _P, _P, _P, c_int, _P, c_float, c_float, c_float, c_float, c_float,
                             _P, c_float, _P, c_int64, _P]),
}


def exported_symbols():
    """Every symbol include/mobrob_b200.h declares (kept in sync by tests/test_abi.py)."""
    return sorted(_SIGNATURES)


def load():
    """dlopen the library and declare signatures.  A library older than its sources is rebuilt
    first when nvcc is on PATH (so tests and bench.py never run a stale .so after an edit of
    csrc/); without nvcc that is an error, not a silent stale run."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("MR_LIB_PATH")  # MR_LIB_PATH: debug variants (tools/trace_epoch.py), used as they are
    if path is None:
        path = _build.LIB_PATH
        if _build.needs_build():
            import shutil

            if shutil.which(os.environ.get("NVCC", "nvcc")):
                _build.build()
            elif os.path.exists(path):
                raise RuntimeError(f"{path} is older than mobrob_b200/csrc (or include/): rebuild it with "
                                   "`python -m mobrob_b200.build`; nvcc is not on PATH here.")
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: run `python -m mobrob_b200.build` (or __graft_entry__.build()). "
            "mobrob_b200 has no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


class MobrobError(RuntimeError):
    pass


def check(status: int):
    if status != 0:
        raise MobrobError(f"libmobrob_b200 error {status}: {load().mr_last_error().decode()}")


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array, None -> NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def launch_count() -> int:
    return int(load().mr_launch_count())
