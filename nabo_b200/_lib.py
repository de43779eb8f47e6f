"""ctypes binding of libnabo_b200.so (the C ABI declared in include/nabo_b200.h).

The library is the product: there is no Python/CPU fallback.  ``lib()`` raises if
the shared object is missing and every compute wrapper raises ``RuntimeError`` with
the library's message on a non-zero status (SURVEY.md 8b: no exceptions cross the
C ABI; the host turns the int status into Python exceptions).
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, List

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NABO_B200_LIB") or os.path.join(HERE, "libnabo_b200.so")   # override: A/B builds (tools/)
HEADER = os.path.join(os.path.dirname(HERE), "include", "nabo_b200.h")

EUCLIDEAN, MOD_CANBERRA, COSINE, CORRELATION = 0, 1, 2, 3
METRICS = {"euclidean": EUCLIDEAN, "mod_canberra": MOD_CANBERRA, "cosine": COSINE, "correlation": CORRELATION}
MODE_EXACT, MODE_FAST = 0, 1

_p = C.c_void_p
_i = C.c_int
_d = C.c_double
_z = C.c_size_t


class PreparedDesc(C.Structure):
    """``nabo_prepared_ref``: host descriptor of a prepared reference (filled by ``nabo_ref_prepare``)."""
    _fields_ = [("magic", C.c_uint32), ("abi_version", _i), ("n_ref", _i), ("g", _i), ("metric", _i), ("plan", _i),
                ("r", _p), ("ldr", _i), ("ref_mask", _p), ("buffer", _p), ("buffer_bytes", _z), ("ops", _p * 3)]


_PD = C.POINTER(PreparedDesc)

# name -> (restype, argtypes); mirrors include/nabo_b200.h one to one
SIGNATURES: Dict[str, tuple] = {
    "nabo_abi_version": (_i, []),
    "nabo_last_error": (C.c_char_p, []),
    "nabo_device_check": (_i, [C.POINTER(_i)]),
    "nabo_euclidean_dist": (_i, [_p, _i, _p, _i, _p, _i, _i, _i, _i, _p]),
    "nabo_mod_canberra_dist": (_i, [_p, _i, _p, _i, _p, _i, _i, _i, _i, _d, _p]),
    "nabo_cosine_dist": (_i, [_p, _i, _p, _i, _p, _i, _i, _i, _i, _p]),
    "nabo_correlation_dist": (_i, [_p, _i, _p, _i, _p, _i, _i, _i, _i, _p]),
    "nabo_knn_workspace_bytes": (_z, [_i, _i, _i, _i, _i, _i]),
    "nabo_knn": (_i, [_p, _i, _p, _i, _i, _i, _i, _i, _i, _d, _p, _i, _i, _i, _p, _p, _p, _z,
                      C.POINTER(C.c_int64), _p]),
    "nabo_knn_candidates_width": (_i, [_i, _i]),
    "nabo_knn_candidates_workspace_bytes": (_z, [_i, _i, _i, _i, _i]),
    "nabo_knn_candidates": (_i, [_p, _i, _p, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p, _z, _p]),
    "nabo_rerank_exact": (_i, [_p, _i, _p, _i, _i, _i, _i, _i, _i, _d, _p, _i, _i, _p, _i, _p, _p, _p]),
    "nabo_merge_topk": (_i, [_p, _p, _i, _i, _i, _p, _p, _p]),
    "nabo_merge_topk_parts": (_i, [_i, _p, _p, _i, _i, _i, _p, _p, _p]),
    "nabo_knn_routed": (_i, [_p, _i, _p, _i, _i, _i, _i, _i, _i, _d, _p, _i, _i, _i, _i, _p, _p, _p, _p, _z,
                             C.POINTER(C.c_int64), _p]),
    "nabo_ref_prepared_bytes": (_z, [_i, _i, _i]),
    "nabo_ref_prepare": (_i, [_p, _i, _i, _i, _i, _p, _p, _z, _PD, _p]),
    "nabo_knn_prepared_workspace_bytes": (_z, [_i, _PD, _i, _d, _i]),
    "nabo_knn_prepared": (_i, [_p, _i, _i, _PD, _i, _d, _i, _i, _i, _p, _p, _p, _z, C.POINTER(C.c_int64), _p]),
    "nabo_knn_prepared_routed": (_i, [_p, _i, _i, _PD, _i, _d, _i, _i, _i, _i, _p, _p, _p, _p, _z,
                                      C.POINTER(C.c_int64), _p]),
    "nabo_score_accumulate": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, _p]),
    "nabo_scores_finalize": (_i, [_p, _i, _d, _d, C.c_longlong, _d, _p, _p]),
    "nabo_snn_weights": (_i, [_p, _i, _i, _p, _i, _i, _p, _p, _p, _p]),
    "nabo_scores_workspace_bytes": (_z, [_i, _i, _i]),
    "nabo_mapping_scores": (_i, [_p, _p, _p, _i, _i, _i, _p, _i, _d, _i, _d, _d, _p, _p, _z, _p]),
    "nabo_classify_targets": (_i, [_p, _p, _p, _i, _i, _p, _i, _d, _i, _d, _p, _p]),
    "nabo_specificity_workspace_bytes": (_z, [_i, _i]),
    "nabo_specificity_workspace_bytes_k": (_z, [_i, _i, _i]),
    "nabo_mapping_specificity": (_i, [_p, _p, _i, _p, _p, _i, _i, _p, _p, _p, _p, _z, _p]),
    "nabo_connected_components": (_i, [_p, _p, C.c_longlong, _i, _p, _p, _z, _p]),
    "nabo_sparse_row_stats": (_i, [_p, _p, _p, _i, _i, _p, _p, C.c_longlong, _i, _p, _p, _p, _p, _p, _p]),
    "nabo_scale_dense": (_i, [_p, _i, _i, _p, _i, _p, _p, _p, _p, _i, _p]),
    "nabo_project_dense": (_i, [_p, _i, _i, _p, _i, _p, _p, _p, _p, _p, _i, _p, _i, _p]),
    "nabo_project_dense_workspace_bytes": (_z, [_i, _i]),
    "nabo_project_dense_mma": (_i, [_p, _i, _i, _p, _i, _p, _p, _p, _p, _p, _i, _p, _i, _p, _z, _p]),
    "nabo_project_csr_workspace_bytes": (_z, [_i, _i]),
    "nabo_project_csr": (_i, [_p, _p, _p, _i, _p, _i, _i, _p, _p, _p, _p, _p, _i, _p, _i, _p, _z, _p]),
}

_LIB = None


def declared_symbols() -> List[str]:
    """Every function name include/nabo_b200.h declares (used by the CPU test that
    checks the library exports all of them)."""
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(nabo_[a-z0-9_]+)\s*\(", txt)))


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "nabo_b200: %s is missing. Build it with `python -m nabo_b200.build` "
                "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.nabo_abi_version() != 1:
            raise RuntimeError("nabo_b200: ABI version mismatch")
        _LIB = L
    return _LIB


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = lib().nabo_last_error().decode("utf-8", "replace")
        kind = "invalid argument" if status < 0 else "CUDA error %d" % status
        raise RuntimeError("nabo_b200 %s: %s (%s)" % (what, msg, kind))


_DEVICE_OK = False


def require_device() -> None:
    """Fail loudly unless a B200-class (sm_10x) device is current."""
    global _DEVICE_OK
    if _DEVICE_OK:
        return
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("nabo_b200: no CUDA device visible; this library has no CPU fallback")
    sm = _i(0)
    check(lib().nabo_device_check(C.byref(sm)), "device_check")
    _DEVICE_OK = True
