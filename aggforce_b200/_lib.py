"""ctypes binding of ``libagf_b200.so`` (the C ABI declared in ``include/agf_b200.h``).

There is no CPU fallback: if the shared library is missing or a kernel fails, the call
raises.  Build the library with ``python -m aggforce_b200.csrc.build`` (or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

F32, F64 = 0, 1

_LIB: Optional[C.CDLL] = None
LIB_PATH = Path(os.environ.get("AGF_B200_LIB") or Path(__file__).resolve().parent / "csrc" / "libagf_b200.so")

_vp, _i32, _i64, _u64, _dbl, _flt = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double, C.c_float

# name -> argtypes; every function returns int status except the three noted below.
SIGNATURES = {
    "agf_gram_linear": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, _vp],
    "agf_gram_linear_ws": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, _vp, C.c_size_t, _vp],
    "agf_gram_linear_weighted": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp],
    "agf_gram_linear_ws_weighted": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, _vp, C.c_size_t, _vp, _vp],
    "agf_weighted_sumsq": [_vp, C.c_int, _i64, _i32, _vp, _vp, _vp],
    "agf_gram_linear_i8": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, C.c_uint32, _vp, _vp, C.c_size_t, _vp],
    "agf_gram_linear_i8t": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, _vp, C.c_size_t, _vp],
    "agf_symmetrize": [_vp, _i32, _vp],
    "agf_map_apply": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _i32, _vp, C.c_int, _vp, C.c_int, _dbl,
                      _vp, _vp],
    "agf_map_apply_ws": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _i32, _vp, C.c_int, _vp, C.c_int, _dbl,
                         _vp, _vp, C.c_size_t, _vp],
    "agf_map_apply_i8": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, _i32, _vp, C.c_int, _vp, C.c_int, _dbl, _vp, _vp,
                         C.c_size_t, _vp],
    "agf_map_apply_sparse": [_vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _i32, _vp, C.c_int, _vp, C.c_int, _dbl, _vp,
                             _vp],
    "agf_map_apply_slice": [_vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _vp, C.c_int, _vp, C.c_int, _dbl, _vp, _vp],
    "agf_pair_moments": [_vp, _vp, C.c_int, _i64, _i32, _i32, _vp, _i64, _vp, _vp, _vp],
    "agf_pair_first": [_vp, _vp, C.c_int, _i32, _i32, _vp, _i64, _vp, _vp],
    "agf_pair_select": [_vp, _dbl, _vp, _i32, _vp, _vp, C.c_int, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp],
    "agf_pair_screen": [_vp, _vp, C.c_int, _i64, _i32, _i32, _vp, _vp],
    "agf_gram_feat": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32, _dbl, _dbl,
                      _dbl, _vp, _vp],
    "agf_gram_feat_ws": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32, _dbl,
                         _dbl, _dbl, _vp, _vp, C.c_size_t, _vp],
    "agf_gram_feat_weighted": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32,
                               _dbl, _dbl, _dbl, _vp, _vp, _vp],
    "agf_gram_feat_ws_weighted": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32,
                                  _dbl, _dbl, _dbl, _vp, _vp, C.c_size_t, _vp, _vp],
    "agf_gram_feat_i8": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32, _dbl,
                         _dbl, _dbl, _vp, _vp, C.c_size_t, _vp],
    "agf_symmetrize_batch": [_vp, _i32, _i32, _vp],
    "agf_feat_rows": [_vp, C.c_int, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32,
                      _dbl, _dbl, _vp, _vp],
    "agf_feat_apply": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32, _dbl, _dbl,
                       _vp, _vp, C.c_int, _vp, _vp],
    "agf_gauss_augment": [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _dbl, _dbl, _vp, _u64,
                          C.c_uint32, _i64, _vp, _vp, _vp],
    "agf_gauss_field_moments": [_vp, _vp, C.c_int, _i64, _i32, _vp, _i32, _dbl, _vp, _vp],
    "agf_sq_gaussian_forces": [_vp, C.c_int, _i64, _i32, _dbl, _dbl, _vp, C.c_int, _vp],
    "agf_qp_equality_small": [_vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
    "agf_peer_exchange": [_vp, _i32, _i32, C.c_uint32, _i32, _vp, _vp, _i64, _i64, _vp, _vp],
    "agf_probe_dmma": [_i32, _vp, _vp, _vp],
    "agf_probe_read": [_vp, _i64, _vp, _vp],
    "agf_synth_frames": [_vp, _vp, _vp, _i32, _i64, _i64, _u64, _flt, _flt, _flt, _vp, _vp, _vp],
}
PLAIN = {"agf_version": (C.c_int, []), "agf_peer_buffer_bytes": (C.c_size_t, [_i64]), "agf_qp_equality_small_supported": (C.c_int, [_i32, _i32]), "agf_last_error": (C.c_char_p, []), "agf_device_sm_count": (C.c_int, []),
         "agf_gram_linear_workspace_bytes": (C.c_size_t, [_i32, _i32, _i64]),
         "agf_gram_linear_i8_workspace_bytes": (C.c_size_t, [_i32, _i32, _i64]),
         "agf_gram_linear_i8t_workspace_bytes": (C.c_size_t, [_i32, _i32, _i64]),
         "agf_map_apply_i8_workspace_bytes": (C.c_size_t, [_i32, _i32, _i32, _i64]),
         "agf_map_apply_workspace_bytes": (C.c_size_t, [C.c_int, _i32, _i32, _i32, _i32, _i64]),
         "agf_gram_feat_i8_workspace_bytes": (C.c_size_t, [_i32, _i32, _i32, _i32, _i64]),
         "agf_gram_feat_workspace_bytes": (C.c_size_t, [_i32, _i32, _i32, _i32, _i64])}


class AgfError(RuntimeError):
    """A libagf_b200 entry point returned a non-zero status."""


def exported_symbols() -> list:
    """Every symbol ``include/agf_b200.h`` declares (checked by the CPU test-suite)."""
    return sorted(list(SIGNATURES) + list(PLAIN))


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        if not LIB_PATH.exists():
            raise AgfError(
                f"{LIB_PATH} is missing: aggforce_b200 has no CPU fallback. Build it with "
                "`python -m aggforce_b200.csrc.build` (needs nvcc, targets sm_100a)."
            )
        handle = C.CDLL(str(LIB_PATH))
        for name, argtypes in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = C.c_int
        for name, (res, argtypes) in PLAIN.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = res
        _LIB = handle
    return _LIB


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().agf_last_error().decode(errors="replace")
        raise AgfError(f"{what} failed with status {status}: {msg}")


# --- launch accounting / per-kernel timing (used by bench.py; off by default)
LAUNCHES = {"count": 0}
_TIMING = {"on": False, "records": []}


def timing(enabled: bool) -> None:
    """Record a CUDA-event pair around every entry point (on the launching stream)."""
    _TIMING["on"] = enabled
    _TIMING["records"] = []


def timing_records():
    """[(entry point, milliseconds)] for the calls since ``timing(True)`` (synchronises)."""
    import torch

    torch.cuda.synchronize()
    return [(name, e0.elapsed_time(e1)) for name, e0, e1 in _TIMING["records"]]


def call(name: str, *args) -> None:
    LAUNCHES["count"] += 1
    if _TIMING["on"]:
        import torch

        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(getattr(lib(), name)(*args), name)
        e1.record()
        _TIMING["records"].append((name, e0, e1))
        return
    check(getattr(lib(), name)(*args), name)
