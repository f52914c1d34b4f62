"""ctypes binding of liblkg.so (include/lkg.h).  There is no fallback: a missing library, a missing
CUDA device or a non-sm_100 device raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "liblkg.so")

LKG_MAX_SEGMENTS = 4
LKG_SCALE_FLOATS = 8
ABI_VERSION = 8
SOLO_DEGREE, SEG_DEGREE, MAX_SEGS, SEG_STRIDE = 256, 512, 8, 576
ACT_NONE, ACT_LEAKY_RELU, ACT_TANH, ACT_ACCUMULATE = 0, 1, 2, 256
AGG_ONE_TERM, AGG_TWO_TERMS, AGG_BI, AGG_BI_Z = 0, 1, 2, 3     # lkg_agg_mode
L2_QUERY, L2_CANDIDATE = 0, 1                                  # lkg_l2_mode

i32, i64, f32p, vp = C.c_int32, C.c_int64, C.c_void_p, C.c_void_p


class LkgGraph(C.Structure):
    _fields_ = [("n_entities", i64), ("n_edges", i64), ("nnz", i64), ("n_relations", i32),
                ("row_begin", i64), ("row_end", i64), ("att_rowptr", vp), ("att_tail", vp), ("att_rel", vp), ("att_seg", vp),
                ("rowptr", vp), ("col", vp), ("row_order", vp), ("row_sched", vp), ("n_solo_rows", i64),
                ("n_sched", i64), ("seg_tickets", vp), ("seg_scratch", vp), ("seg_stride", i64)]


class LkgPlanes(C.Structure):
    _fields_ = [("n_segments", i32), ("ptr", vp * LKG_MAX_SEGMENTS), ("ld", i64 * LKG_MAX_SEGMENTS),
                ("plane_stride", i64 * LKG_MAX_SEGMENTS), ("k", i32 * LKG_MAX_SEGMENTS),
                ("scale", vp * LKG_MAX_SEGMENTS)]


# name -> (restype, argtypes); mirrors include/lkg.h one to one
SIGNATURES = {
    "lkg_abi_version": (C.c_int, []),
    "lkg_last_error": (C.c_char_p, []),
    "lkg_device_check": (C.c_int, [C.c_int]),
    "lkg_peer_push": (C.c_int, [vp, i64, C.POINTER(vp), i32, i32, vp]),
    "lkg_plan_workspace_bytes": (C.c_int, [i64, i64, C.POINTER(C.c_size_t)]),
    "lkg_plan_build": (C.c_int, [vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                 C.c_size_t, vp]),
    "lkg_segment_scatter_add": (C.c_int, [vp, vp, i64, vp, i64, vp]),
    "lkg_edge_fingerprint": (C.c_int, [vp, vp, vp, i64, vp, vp]),
    "lkg_laplacian_init": (C.c_int, [C.POINTER(LkgGraph), C.c_int, vp, vp, vp]),
    "lkg_attn_workspace_bytes": (C.c_int, [i32, i32, C.POINTER(C.c_size_t)]),
    "lkg_attn_update": (C.c_int, [C.POINTER(LkgGraph), vp, i64, vp, i64, i32, vp, vp, vp]),
    "lkg_attn_run_logits": (C.c_int, [vp, vp, i64, vp, vp, i64, i32, vp, i64, vp, vp]),
    "lkg_row_softmax": (C.c_int, [vp, i64, vp, vp]),
    "lkg_scale_from_data": (C.c_int, [vp, i64, vp, i64, i32, C.c_float, vp, vp]),
    "lkg_absmax_accumulate": (C.c_int, [vp, i64, vp, i64, i32, vp, vp]),
    "lkg_scale_finish": (C.c_int, [C.c_float, vp, vp]),
    "lkg_scale_from_bound": (C.c_int, [C.c_float, vp, vp, vp]),
    "lkg_split_planes": (C.c_int, [vp, i64, vp, i64, i32, vp, vp, i64, i64, vp]),
    "lkg_packed_weight_cols": (C.c_int, [C.POINTER(i32), i32, C.POINTER(i32)]),
    "lkg_pack_weight": (C.c_int, [vp, i64, i32, C.POINTER(i32), i32, C.POINTER(vp), vp, i64, vp, vp]),
    "lkg_gemm_set_cta_group": (C.c_int, [i32]),
    "lkg_linear_fwd": (C.c_int, [C.POINTER(LkgPlanes), i64, C.POINTER(LkgPlanes), i32, vp, i32, vp, i64, vp, i64,
                                 i64, vp, vp]),
    "lkg_linear_fwd_split": (C.c_int, [C.POINTER(LkgPlanes), i64, C.POINTER(LkgPlanes), i32, vp, i32, vp, i64, vp, i64, i32,
                                       vp, i64, i64, vp, vp]),
    "lkg_gate_fwd": (C.c_int, [C.POINTER(LkgPlanes), i64, C.POINTER(LkgPlanes), vp, i32, vp, i64, vp, i64, vp, i64,
                               i64, vp, vp, i64, vp]),
    "lkg_aggregate_supported": (C.c_int, [i32, i32, i32, C.POINTER(i32)]),
    "lkg_aggregate_workspace_bytes": (C.c_int, [C.POINTER(C.c_size_t)]),
    "lkg_aggregate_fwd": (C.c_int, [C.POINTER(LkgGraph), vp, vp, i64, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp,
                                    vp, vp, i64, vp, i64, vp, i64, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, vp]),
    "lkg_plan_transpose_workspace_bytes": (C.c_int, [i64, C.POINTER(C.c_size_t)]),
    "lkg_plan_transpose": (C.c_int, [C.POINTER(LkgGraph), vp, vp, vp, vp, C.c_size_t, vp]),
    "lkg_spmm_coo": (C.c_int, [vp, vp, vp, vp, i64, vp, i64, i32, vp, i64, vp]),
    "lkg_layer_bwd_rows": (C.c_int, [i64, i32, i32, vp, i64, vp, i64, vp, vp, i64, vp, i64, vp, vp, i64, vp, vp, vp, vp]),
    "lkg_bi_bwd_rows": (C.c_int, [i64, i32, i32, vp, i64, vp, vp, i64, vp, i64, vp, i64, vp, i64, i32, vp, i64, vp, vp]),
    "lkg_xt_y": (C.c_int, [vp, i64, vp, i64, i32, vp, i64, i32, i64, vp, i64, vp]),
    "lkg_xt_y_planes": (C.c_int, [C.POINTER(LkgPlanes), C.POINTER(LkgPlanes), i64, vp, i64, vp]),
    "lkg_colsum": (C.c_int, [vp, i64, i64, i32, vp, vp]),
    "lkg_gate_bwd": (C.c_int, [vp, i64, vp, i64, vp, i64, i64, i32, vp, i64, vp, i64, vp, vp]),
    "lkg_leaky_bwd": (C.c_int, [vp, i64, vp, i64, i64, i32, vp, i64, vp, vp]),
    "lkg_sample_batch": (C.c_int, [vp, vp, vp, vp, i64, vp, i64, i32, i32, C.c_uint64, i32, vp, vp, vp, vp, vp, vp]),
    "lkg_bpr_loss": (C.c_int, [vp, i64, i32, vp, vp, vp, i64, C.c_float, vp, vp, vp, i64, vp]),
    "lkg_transr_loss": (C.c_int, [vp, i64, i32, vp, i64, i32, vp, vp, vp, vp, vp, i64, C.c_float, vp, vp, vp, i64, vp, vp,
                                  vp]),
    "lkg_transe_loss": (C.c_int, [vp, i64, i32, vp, i64, vp, vp, vp, vp, i64, C.c_float, vp, vp, vp, i64, vp, vp]),
    "lkg_mlp_fc_fwd": (C.c_int, [vp, i64, vp, vp, i32, vp, vp, i64, i32, vp, i64, vp, i32, i32, vp, i64, vp, vp]),
    "lkg_bn_finalize": (C.c_int, [vp, i64, i32, vp, vp, C.c_float, C.c_float, vp, vp, i32, vp, vp, vp, vp, vp]),
    "lkg_mlp_fc_bwd_weight": (C.c_int, [vp, i64, vp, i64, vp, vp, i32, vp, vp, i64, i32, i32, vp, i64, vp, vp]),
    "lkg_mlp_fc_bwd_input": (C.c_int, [vp, i64, i64, i32, vp, i64, i32, vp, i64, vp, vp, i32, vp, i64, vp, vp, vp, vp]),
    "lkg_bn_relu_bwd": (C.c_int, [vp, i64, vp, i64, vp, vp, vp, vp, i64, i32, i32, vp, i64, vp, vp, vp]),
    "lkg_sigmoid_bwd": (C.c_int, [vp, vp, i64, vp, vp]),
    "lkg_score": (C.c_int, [C.POINTER(LkgPlanes), i64, C.POINTER(LkgPlanes), i64, vp, i64, vp, vp]),
    "lkg_minmax_reset": (C.c_int, [vp, vp]),
    "lkg_predict_threshold": (C.c_int, [vp, i64, i64, i64, vp, C.c_float, vp, i64, vp]),
    "lkg_topk_rows": (C.c_int, [vp, i64, i64, i64, i32, vp, vp, vp, vp, vp]),
    "lkg_shift_rows": (C.c_int, [vp, i64, vp, i64, i32, vp, vp, i64, vp]),
    "lkg_rank_prepare": (C.c_int, [vp, i64, vp, vp, i64, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp]),
    "lkg_score_rank": (C.c_int, [C.POINTER(LkgPlanes), i64, C.POINTER(LkgPlanes), i64, vp, vp, vp, vp, i32, vp]),
    "lkg_rank_finalize": (C.c_int, [vp, i64, vp, vp, i64, vp, vp, vp, vp, vp, vp, i32, i64, i64, i32, vp, vp]),
    "lkg_rank_filter": (C.c_int, [C.POINTER(LkgGraph), vp, vp, vp, vp, i64, vp, i64, i32, vp, vp, vp]),
    "lkg_rank_filter_scores": (C.c_int, [C.POINTER(LkgGraph), vp, vp, vp, vp, i64, vp, i64, i64, vp, vp]),
    "lkg_l2_rank_rows": (C.c_int, [vp, i64, vp, i64, i32, vp, i32, vp, vp, i64, vp]),
    "lkg_rank_prepare_l2": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, i64, i32, vp, vp, vp, vp, vp, vp]),
    "lkg_rank_finalize_l2": (C.c_int, [vp, i64, vp, i64, vp, vp, vp, vp, vp, i32, i64, i64, i32, vp, vp]),
    "lkg_rank_filter_l2": (C.c_int, [C.POINTER(LkgGraph), vp, vp, vp, vp, i64, vp, i64, vp, i64, i32, vp, vp, vp]),
    "lkg_topk_threshold_l2": (C.c_int, [vp, i64, i64, vp, i64, vp, i64, i64, i32, vp, vp, vp, i32, i32,
                                        C.POINTER(LkgGraph), vp, vp, vp, vp, vp, vp]),
    "lkg_topk_finalize_l2": (C.c_int, [vp, i64, i64, vp, i64, i64, i32, vp, vp, i32, i32, C.POINTER(LkgGraph), vp, vp,
                                       vp, vp, vp, vp]),
    "lkg_topk_threshold_dot": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, i64, i32, vp, vp, vp, vp, i32, i32,
                                         C.POINTER(LkgGraph), vp, vp, vp, vp, vp, vp]),
    "lkg_topk_finalize_dot": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, i64, i32, vp, vp, i32, i32, C.POINTER(LkgGraph),
                                        vp, vp, vp, vp, vp, vp]),
    "lkg_topk_merge": (C.c_int, [vp, vp, i32, i64, i32, vp, vp, vp]),
    "lkg_score_index": (C.c_int, [vp, i64, vp, i64, i32, vp, vp, i64, vp, vp, vp]),
    "lkg_score_topk_workspace_bytes": (C.c_int, [i64, i32, i32, C.POINTER(C.c_size_t)]),
    "lkg_score_topk": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, i64, i32, vp, vp, i64, i32, vp, i64, vp, i64, vp, vp,
                                 i32, i32, vp, vp, vp, vp]),
}

_lib: Optional[C.CDLL] = None
_checked_devices = set()


def load() -> C.CDLL:
    """Loads liblkg.so (built in-tree by ``python -m literalkg_b200.build``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m literalkg_b200.build` "
                "(literalkg_b200 has no CPU / PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.lkg_abi_version() != ABI_VERSION:
            raise RuntimeError("liblkg.so ABI version mismatch; rebuild with `python -m literalkg_b200.build`")
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().lkg_last_error().decode(errors="replace")
        raise RuntimeError(f"liblkg error {rc}: {msg}")


def require_cuda(t: torch.Tensor, what: str = "tensor") -> None:
    if not t.is_cuda:
        raise RuntimeError(f"literalkg_b200: {what} is on {t.device}; the path runs on CUDA sm_100 only "
                           "(no CPU fallback)")
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if idx not in _checked_devices:
        check(load().lkg_device_check(idx))
        _checked_devices.add(idx)


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def f32c(t: torch.Tensor) -> torch.Tensor:
    """fp32 + contiguous (no copy when already so)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class Planes:
    """Scaled fp16 hi/lo planes of an fp32 matrix: tensor [2, rows, ld] (ld % 8 == 0) with logical width k, plus
    the device scale record (float[8]: absmax, scale, 1/scale, scratch...) every kernel that touches them reads."""

    def __init__(self, rows: int, k: int, device, ld: Optional[int] = None, rec: Optional[torch.Tensor] = None):
        self.rows, self.k = int(rows), int(k)
        self.ld = int(ld) if ld is not None else (self.k + 7) // 8 * 8
        assert self.ld % 8 == 0 and self.ld >= self.k
        self.t = torch.empty((2, max(self.rows, 1), self.ld), dtype=torch.float16, device=device)
        self.rec = rec if rec is not None else torch.zeros(LKG_SCALE_FLOATS, dtype=torch.float32, device=device)

    @property
    def plane_stride(self) -> int:
        return self.t.stride(0)

    def ptr(self, col: int = 0) -> int:
        """Base address of a TMA-readable window: needs a 16-byte aligned column."""
        assert col % 8 == 0
        return self.t.data_ptr() + 2 * col

    def elem_ptr(self, col: int = 0) -> int:
        """Address of column ``col`` for kernels that write planes element-wise (no alignment needed)."""
        return self.t.data_ptr() + 2 * col

    def view(self, col: int, k: int, rec: Optional[torch.Tensor] = None) -> "PlanesView":
        return PlanesView(self, col, k, rec)

    def dequant(self) -> torch.Tensor:
        """fp32 reconstruction (hi + lo) / scale -- test / debugging helper (one host sync)."""
        return (self.t[0, :self.rows, :self.k].float() + self.t[1, :self.rows, :self.k].float()) * self.rec[2]


class PlanesView:
    """Column window [col, col + k) of a Planes buffer (col % 8 == 0) with its own scale record: the windows of
    the concat buffer (gate output | normalised layer outputs) have different magnitudes."""

    def __init__(self, base, col: int, k: int, rec: Optional[torch.Tensor] = None):
        self.base, self.col, self.k = base, int(col), int(k)
        self.rows, self.ld, self.plane_stride = base.rows, base.ld, base.plane_stride
        self.rec = rec if rec is not None else base.rec

    def ptr(self, col: int = 0) -> int:
        return self.base.ptr(self.col + col)

    def elem_ptr(self, col: int = 0) -> int:
        return self.base.elem_ptr(self.col + col)


def planes_operand(segments) -> LkgPlanes:
    op = LkgPlanes()
    op.n_segments = len(segments)
    for i, s in enumerate(segments):
        op.ptr[i] = s.ptr()
        op.ld[i] = s.ld
        op.plane_stride[i] = s.plane_stride
        op.k[i] = s.k
        op.scale[i] = s.rec.data_ptr()
    return op
