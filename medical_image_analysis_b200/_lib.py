"""ctypes binding of the C ABI in include/mia_selective_scan.h (libmia_scan.so).

There is deliberately NO fallback: if the CUDA library is missing or fails, every op raises.
"""
from __future__ import annotations

import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmia_scan.so")

MIA_F32, MIA_F16, MIA_BF16 = 0, 1, 2

_vp, _i32, _i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64


class MiaSSParams(ctypes.Structure):
    """Field-for-field mirror of ``struct mia_ss_params``."""
    _fields_ = (
        [(n, _i32) for n in ("batch", "dim", "seqlen", "dstate", "n_groups", "delta_dim", "itype", "otype",
                             "delta_softplus", "n_chunks")]
        + [(n, _vp) for n in ("u", "delta", "A", "B", "C", "D", "delta_bias", "z")]
        + [(n, _i64) for n in ("u_batch_stride", "u_d_stride", "delta_batch_stride", "delta_d_stride",
                               "A_d_stride", "A_dstate_stride", "B_batch_stride", "B_group_stride", "B_dstate_stride",
                               "C_batch_stride", "C_group_stride", "C_dstate_stride", "z_batch_stride", "z_d_stride")]
        + [(n, _vp) for n in ("out", "out_z", "x")]
        + [(n, _i64) for n in ("out_batch_stride", "out_d_stride", "out_z_batch_stride", "out_z_d_stride")]
        + [(n, _vp) for n in ("dout", "out_saved")]
        + [(n, _i64) for n in ("dout_batch_stride", "dout_d_stride", "out_saved_batch_stride", "out_saved_d_stride")]
        + [(n, _vp) for n in ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dz")]
        + [(n, _i64) for n in ("du_batch_stride", "du_d_stride", "ddelta_batch_stride", "ddelta_d_stride",
                               "dA_d_stride", "dA_dstate_stride", "dB_batch_stride", "dB_group_stride", "dB_dstate_stride",
                               "dC_batch_stride", "dC_group_stride", "dC_dstate_stride", "dz_batch_stride", "dz_d_stride")]
        + [("workspace", _vp), ("workspace_bytes", ctypes.c_size_t), ("hblk", _vp)]
    )


_lib = None


def lib() -> ctypes.CDLL:
    """Load libmia_scan.so (built in-tree by ``python -m medical_image_analysis_b200._build``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA library has not been built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` (or `python -m medical_image_analysis_b200._build`). "
                "There is no CPU / PyTorch fallback for the selective scan.")
        L = ctypes.CDLL(LIB_PATH)
        L.mia_abi_version.restype = ctypes.c_int
        L.mia_last_error.restype = ctypes.c_char_p
        L.mia_launch_count.restype = ctypes.c_uint64
        L.mia_ss_chunk_len.argtypes = [ctypes.c_int]
        L.mia_ss_chunk_len.restype = ctypes.c_int
        L.mia_ss_num_chunks.argtypes = [ctypes.c_int]
        L.mia_ss_num_chunks.restype = ctypes.c_int
        L.mia_selective_scan_fwd.argtypes = [ctypes.POINTER(MiaSSParams), _vp]
        L.mia_selective_scan_fwd.restype = ctypes.c_int
        L.mia_selective_scan_bwd.argtypes = [ctypes.POINTER(MiaSSParams), _vp]
        L.mia_selective_scan_bwd.restype = ctypes.c_int
        L.mia_selective_scan_bwd_workspace.argtypes = [ctypes.POINTER(MiaSSParams)]
        L.mia_selective_scan_bwd_workspace.restype = ctypes.c_size_t
        for fn in (L.mia_cross_scan, L.mia_cross_merge):
            fn.argtypes = [_vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]
            fn.restype = ctypes.c_int
        L.mia_cs_last_error.restype = ctypes.c_char_p
        L.mia_silu_gate.argtypes = [_vp, _vp, _vp, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, _vp]
        L.mia_silu_gate.restype = ctypes.c_int
        ll, ci = ctypes.c_longlong, ctypes.c_int
        L.mia_causal_conv1d_fwd.argtypes = [_vp, _vp, _vp, _vp, ci, ci, ci, ci, ci, ci, ll, ll, ll, ll, _vp]
        L.mia_causal_conv1d_fwd.restype = ci
        L.mia_causal_conv1d_bwd.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, ci, ci, ci, ci, ci, ci, ll, ll, ll, ll, ll, ll, _vp]
        L.mia_causal_conv1d_bwd.restype = ci
        L.mia_conv_last_error.restype = ctypes.c_char_p
        L.mia_dwconv2d_fwd.argtypes = [_vp, _vp, _vp, _vp, ci, ci, ci, ci, ci, ci, _vp]
        L.mia_dwconv2d_fwd.restype = ci
        L.mia_dwconv2d_bwd.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, ci, ci, ci, ci, ci, ci, _vp]
        L.mia_dwconv2d_bwd.restype = ci
        L.mia_dwconv2d_last_error.restype = ctypes.c_char_p
        L.mia_gemm_tn.argtypes = [_vp, _vp, _vp, _vp, ci, ci, ci, ll, ll, ll, ci, ci, ci, _vp]
        L.mia_gemm_tn.restype = ci
        L.mia_gemm.argtypes = [_vp, _vp, _vp, _vp, ci, ci, ci, ll, ll, ll, ci, ci, ci, ci, ci, _vp]
        L.mia_gemm.restype = ci
        L.mia_gemm_last_error.restype = ctypes.c_char_p
        L.mia_ss_block_state_floats.argtypes = [ctypes.POINTER(MiaSSParams)]
        L.mia_ss_block_state_floats.restype = ctypes.c_size_t
        L.mia_ss_fwd_writes_block_states.argtypes = [ctypes.POINTER(MiaSSParams)]
        L.mia_ss_fwd_writes_block_states.restype = ctypes.c_int
        L.mia_ss_describe_plan.argtypes = [ctypes.POINTER(MiaSSParams), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p,
                                           ctypes.c_size_t]
        L.mia_ss_describe_plan.restype = ctypes.c_int
        if L.mia_abi_version() != 2:
            raise RuntimeError(f"libmia_scan.so ABI version {L.mia_abi_version()} != 2: rebuild it")
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what}: {lib().mia_last_error().decode()} (code {rc})")


def launch_count() -> int:
    return int(lib().mia_launch_count())
