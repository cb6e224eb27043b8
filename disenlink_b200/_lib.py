"""ctypes binding of libdisenlink_b200.so (C ABI in include/disenlink_b200.h).

There is no CPU fallback: if the library is missing or a tensor is not on a CUDA device the call
raises.  The library is built in-tree by ``python -m disenlink_b200.build`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DL_LIB_PATH: load another build of the same library (A/B experiments with kernel variants)
LIB_PATH = os.environ.get("DL_LIB_PATH") or os.path.join(_HERE, "libdisenlink_b200.so")

DL_MAX_K = 32
DL_MAX_D = 256
DL_SEG = 512
DL_N_BUCKETS = 33
DL_HUB_BUCKET_END = 23

# dl_graph.flags (kernel-path switches for A/B runs and for testing the non-default paths)
DL_F_NO_STREAM, DL_F_NO_FL, DL_F_NO_FL_ATTN, DL_F_NO_PRESCALE = 1, 2, 4, 8
DL_F_NO_SJ, DL_F_NO_SR, DL_F_NO_XDOT, DL_F_NO_SYM = 16, 32, 64, 128
DL_F_NO_KEEPA = 256
_FLAG_NAMES = {"NO_STREAM": 1, "NO_FL": 2, "NO_FL_ATTN": 4, "NO_PRESCALE": 8, "NO_SJ": 16, "NO_SR": 32,
               "NO_XDOT": 64, "NO_SYM": 128, "NO_KEEPA": 256}
DL_EASYM, DL_EUNSUPPORTED = -4, -5


def default_flags() -> int:
    """Flags a new Graph starts with: 0, or the comma-separated names in DL_FLAGS (e.g.
    DL_FLAGS=NO_FL,NO_XDOT).  The environment is read here, on the host side; the library itself
    has no global state."""
    val = 0
    for name in filter(None, (x.strip().upper() for x in os.environ.get("DL_FLAGS", "").split(","))):
        if name not in _FLAG_NAMES:
            raise ValueError(f"DL_FLAGS: unknown flag {name!r} (known: {sorted(_FLAG_NAMES)})")
        val |= _FLAG_NAMES[name]
    return val

_c = ctypes
_vp = _c.c_void_p
_i64 = _c.c_int64
_int = _c.c_int
_f = _c.c_float
_sz = _c.c_size_t


class DlGraph(_c.Structure):
    """Mirror of ``struct dl_graph``."""
    _fields_ = [("N", _i64), ("nnz", _i64), ("rowptr", _vp), ("col", _vp), ("perm", _vp),
                ("n_hub", _i64), ("n_hub_items", _i64), ("hub_seg_ptr", _vp), ("item_hub", _vp),
                ("erow", _vp), ("row_base", _i64), ("flags", _c.c_uint32)]


class DlPushDesc(_c.Structure):
    """Mirror of ``struct dl_push_desc``."""
    _fields_ = [("dst", _vp), ("src_idx", _vp), ("dst_idx", _vp), ("mask", _vp), ("n", _i64)]


_GP = _c.POINTER(DlGraph)

# name -> (restype, argtypes); every symbol declared in include/disenlink_b200.h
SIGNATURES = {
    "dl_abi_version": (_int, []),
    "dl_error_string": (_c.c_char_p, [_int]),
    "dl_csr_build_workspace_bytes": (_sz, [_i64, _i64]),
    "dl_csr_build": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dl_csr_build_rect": (_int, [_vp, _vp, _i64, _i64, _i64, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dl_csr_from_dense": (_int, [_vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "dl_entry_rows": (_int, [_vp, _i64, _i64, _vp, _vp]),
    "dl_rev_index": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "dl_transpose_index_workspace_bytes": (_sz, [_i64, _i64]),
    "dl_transpose_index": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dl_degree_buckets_workspace_bytes": (_sz, [_i64]),
    "dl_degree_buckets": (_int, [_vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "dl_hub_items": (_int, [_vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "dl_hub_scratch_floats": (_sz, [_GP, _i64]),
    "dl_edge_attn_fwd": (_int, [_GP, _vp, _int, _int, _f, _vp, _vp, _vp, _vp, _vp]),
    "dl_sym_index_workspace_bytes": (_sz, [_i64, _i64]),
    "dl_sym_index": (_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dl_edge_attn_fwd_sym": (_int, [_GP, _GP, _vp, _vp, _int, _int, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dl_factor_spmm_fwd": (_int, [_GP, _vp, _vp, _vp, _vp, _int, _int, _f, _f, _vp, _vp, _vp, _i64, _vp, _vp]),
    "dl_factor_bwd": (_int, [_GP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _int, _int, _f, _f, _f, _vp, _vp, _vp, _vp]),
    "dl_factor_bwd_gather": (_int, [_GP, _vp, _vp, _vp, _vp, _vp, _int, _int, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dl_factor_bwd_edges_sym_supported": (_int, [_int, _int]),
    "dl_factor_bwd_edges_sym": (_int, [_GP, _GP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _int, _int, _f, _f, _int,
                                       _vp, _vp, _vp]),
    "dl_factor_bwd_edges": (_int, [_GP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _int, _int, _f, _f, _vp, _vp, _vp]),
    "dl_factor_bwd_directed": (_int, [_GP, _GP, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _f, _f, _f, _vp, _vp, _vp, _vp,
                                      _vp, _vp, _vp]),
    "dl_factor_bwd_directed_phase": (_int, [_GP, _GP, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _f, _f, _f, _i64, _i64,
                                            _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "dl_pair_score_fwd": (_int, [_vp, _vp, _i64, _vp, _vp, _i64, _int, _int, _f, _vp, _vp, _vp]),
    "dl_pair_incidence_workspace_bytes": (_sz, [_i64, _i64]),
    "dl_pair_incidence": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dl_pair_incidence_range": (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dl_pair_score_bwd": (_int, [_GP, _vp, _vp, _vp, _vp, _int, _int, _f, _vp, _vp, _vp, _vp]),
    "dl_allpairs_score_fwd": (_int, [_vp, _vp, _i64, _int, _int, _f, _vp, _vp]),
    "dl_allpairs_score_bwd": (_int, [_vp, _vp, _vp, _i64, _int, _int, _f, _vp, _vp, _vp]),
    "dl_dense_alpha0": (_int, [_vp, _i64, _int, _int, _f, _vp, _vp]),
    "dl_dense_att": (_int, [_GP, _vp, _vp, _vp, _int, _vp, _vp]),
    "dl_link_bce_workspace_bytes": (_i64, []),
    "dl_link_bce": (_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "dl_roc_auc_workspace_bytes": (_i64, [_i64]),
    "dl_roc_auc": (_int, [_vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "dl_link_bce_segments_workspace_bytes": (_i64, [_i64]),
    "dl_link_bce_segments": (_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp]),
    "dl_roc_auc_segments_workspace_bytes": (_i64, [_i64, _i64]),
    "dl_roc_auc_segments": (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp]),
    "dl_push_slice": (_int, [_vp, _vp, _int, _i64, _vp]),
    "dl_push_rows": (_int, [_vp, _i64, _int, _c.POINTER(DlPushDesc), _int, _vp]),
    "dl_push_entries": (_int, [_vp, _int, _c.POINTER(DlPushDesc), _int, _vp]),
    "dl_need_masks": (_int, [_GP, _vp, _vp, _int, _vp, _vp]),
    "dl_factor_spmm_fwd_push": (_int, [_GP, _vp, _vp, _vp, _vp, _int, _int, _f, _f, _vp, _vp, _vp, _vp, _int, _vp]),
    "dl_edge_attn_fwd_push": (_int, [_GP, _vp, _int, _int, _f, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "dl_factor_bwd_gather_push": (_int, [_GP, _vp, _vp, _vp, _vp, _vp, _int, _int, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "dl_pair_score_bwd_push": (_int, [_GP, _vp, _vp, _vp, _vp, _int, _int, _f, _vp, _vp, _vp, _vp, _int, _vp]),
    "dl_enable_peer_access": (_int, [_int]),
    "dl_ipc_open": (_int, [_vp, _vp]),
    "dl_ipc_close": (_int, [_vp]),
    "dl_structured_negative_sampling": (_int, [_GP, _vp, _i64, _i64, _c.c_uint64, _int, _vp, _vp, _vp]),
}

_lib = None
launches = 0  # kernels-launching C-ABI calls made through this binding (bench.py reports it)


def lib():
    """The loaded library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build the CUDA extension with "
                "`python -m disenlink_b200.build` (nvcc, sm_100a). There is no CPU fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class DlError(RuntimeError):
    def __init__(self, code: int, what: str):
        self.code = code
        msg = lib().dl_error_string(code)
        super().__init__(f"{what}: {msg.decode() if msg else code} (code {code})")


def check(code: int, what: str) -> None:
    global launches
    launches += 1
    if code != 0:
        raise DlError(code, what)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream_of(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} must be a CUDA tensor: disenlink_b200 runs only through its sm_100a CUDA "
            "kernels and has no CPU fallback")
