"""Thin functional wrappers over the C ABI (one per entry point of include/lkg.h).

All tensors must live on one sm_100 CUDA device; nothing here falls back to PyTorch math.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from .graph import GraphPlan


class Profile:
    """Optional per-entry-point CUDA-event timing + kernel-launch counting (used by bench.py).  Events are
    recorded on the current stream, which is the stream every kernel of this library is launched on."""

    def __init__(self, only=None):
        self.events = []          # (name, start_event, end_event)
        self.launches = 0
        self.only = only          # optional set of entry-point names to time (launches are always counted): two
                                  # event records per call are host time that a short multi-GPU pass cannot hide

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.events:
            tot, cnt = out.get(name, (0.0, 0))
            out[name] = (tot + a.elapsed_time(b), cnt + 1)
        return {k: {"ms_total": v[0], "calls": v[1], "ms_avg": v[0] / v[1]} for k, v in out.items()}


PROFILE: Optional[Profile] = None


class _dev_guard:
    """Sets the CUDA device of ``t`` for the call and, when profiling is on, brackets it with events."""

    def __init__(self, t: torch.Tensor, name: Optional[str] = None, kernels: int = 1):
        _lib.require_cuda(t)
        self.guard = torch.cuda.device(t.device)
        self.name, self.kernels = name, kernels

    def __enter__(self):
        self.guard.__enter__()
        self.timed = PROFILE is not None and bool(self.name) and (PROFILE.only is None or self.name in PROFILE.only)
        if self.timed:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()

    def __exit__(self, *exc):
        if self.timed:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            PROFILE.events.append((self.name, self.start, end))
        if PROFILE is not None and self.name:
            PROFILE.launches += self.kernels
        return self.guard.__exit__(*exc)


def attn_update(plan: GraphPlan, entity: torch.Tensor, relation: torch.Tensor,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A_in values after ``update_att`` (model.py:444-471), plan (coalesced) order."""
    entity, relation = _lib.f32c(entity), _lib.f32c(relation)
    if entity.shape[1] != relation.shape[1]:
        raise ValueError("update_att needs embed_dim == relation_dim (model.py:441 adds the two tables)")
    if out is None:
        out = torch.empty(max(plan.nnz, 1), dtype=torch.float32, device=entity.device)[:plan.nnz]
    with _dev_guard(entity, "attn_update", 2):
        _lib.check(_lib.load().lkg_attn_update(plan.byref(), entity.data_ptr(), entity.stride(0),
                                               relation.data_ptr(), relation.stride(0), entity.shape[1],
                                               out.data_ptr(), plan.attn_workspace(entity.shape[1]), _lib.stream()))
    return out


def attn_update_projected(plan: GraphPlan, entity: torch.Tensor, relation: torch.Tensor, w_rel: torch.Tensor,
                          out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A_in values of the relation-PROJECTED attention (north star (b); the formula commented out at model.py:436-439):
    v(h,r,t) = (e_t W_r) . tanh(e_h W_r + e_r), duplicate (h,t) logits summed, row softmax.  ``w_rel`` [R, D, D_rel].
    v = e_t . u_{h,r} with u_{h,r} = W_r tanh(W_r^T e_h + e_r): two chained tensor-core GEMMs per relation bucket over
    the (head, relation) runs of the plan, then one gather + dot per triple (csrc/attn.cu)."""
    entity, relation, w_rel = _lib.f32c(entity), _lib.f32c(relation), _lib.f32c(w_rel)
    n_rel, d, d_rel = w_rel.shape
    if entity.shape[1] != d or relation.shape[1] != d_rel or relation.shape[0] != n_rel:
        raise ValueError("w_rel must be [n_relations, embed_dim, relation_dim]")
    dev = entity.device
    runs = plan.runs()
    n_runs = runs["n_runs"]
    u_all = torch.empty((max(n_runs, 1), d), dtype=torch.float32, device=dev)        # bucket order
    unit = scale_from_bound(1.0, dev)
    for r in range(n_rel):
        lo, hi = runs["offsets"][r], runs["offsets"][r + 1]
        if hi == lo:
            continue
        heads = runs["run_head"][runs["order"][lo:hi]]
        hp = split_planes(entity, heads)                                              # gathered head rows as planes
        q = _lib.Planes(hi - lo, d_rel, dev, rec=unit)                                # |tanh| <= 1
        linear([hp], w_rel[r].t().contiguous(), relation[r], _lib.ACT_TANH, out_planes=q)      # tanh(e_h W_r + e_r)
        linear([q], w_rel[r].contiguous(), None, _lib.ACT_NONE, out=u_all[lo:hi])     # u = W_r q
    logits = torch.empty(max(plan.n_edges, 1), dtype=torch.float32, device=dev)
    with _dev_guard(entity, "attn_run_logits"):
        _lib.check(_lib.load().lkg_attn_run_logits(runs["run_ptr"].data_ptr(), runs["run_slot"].data_ptr(), n_runs,
                                                   plan.att_tail.data_ptr(), entity.data_ptr(), entity.stride(0), d,
                                                   u_all.data_ptr(), u_all.stride(0), logits.data_ptr(), _lib.stream()))
    if out is None:
        out = torch.empty(max(plan.nnz, 1), dtype=torch.float32, device=dev)[:plan.nnz]
    seg = (plan.att_seg & 0x7fffffff).contiguous()
    with _dev_guard(entity, "attn_merge_softmax", 2):
        lib = _lib.load()
        _lib.check(lib.lkg_segment_scatter_add(logits.data_ptr(), seg.data_ptr(), plan.n_edges, out.data_ptr(), plan.nnz,
                                               _lib.stream()))
        _lib.check(lib.lkg_row_softmax(plan.rowptr.data_ptr(), plan.n_entities, out.data_ptr(), _lib.stream()))
    return out


def scale_from_data(src: torch.Tensor, rows: Optional[torch.Tensor] = None, floor: float = 0.0,
                    rec: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Device scale record (float[8]) of max(|src[rows]|, floor); no host sync."""
    m = src.shape[0] if rows is None else rows.numel()
    if rec is None:
        rec = torch.empty(_lib.LKG_SCALE_FLOATS, dtype=torch.float32, device=src.device)
    with _dev_guard(src, "scale_from_data"):
        _lib.check(_lib.load().lkg_scale_from_data(src.data_ptr(), src.stride(0), _lib.ptr(rows), m, src.shape[1],
                                                   float(floor), rec.data_ptr(), _lib.stream()))
    return rec


def raw_record(device) -> torch.Tensor:
    """A zeroed scale record for the kernels that raise its absmax while they PRODUCE the data (``amax`` arguments of
    leaky_bwd / layer_bwd_rows / bi_bwd_rows / gate_bwd, or ``absmax_accumulate``); ``scale_finish`` completes it."""
    return torch.zeros(_lib.LKG_SCALE_FLOATS, dtype=torch.float32, device=device)


def absmax_accumulate(src: torch.Tensor, rec: torch.Tensor) -> torch.Tensor:
    """Raises the raw absmax of ``rec`` to cover ``src`` ([m, k] fp32, unit inner stride)."""
    _rowmajor(src)
    with _dev_guard(src, "scale_from_data"):
        _lib.check(_lib.load().lkg_absmax_accumulate(src.data_ptr(), src.stride(0), None, src.shape[0], src.shape[1],
                                                     rec.data_ptr(), _lib.stream()))
    return rec


def scale_finish(rec: torch.Tensor, floor: float = 0.0) -> torch.Tensor:
    with _dev_guard(rec, "scale_finish"):
        _lib.check(_lib.load().lkg_scale_finish(float(floor), rec.data_ptr(), _lib.stream()))
    return rec


def scale_from_bound(bound: float, device, other: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Scale record of max(bound, other.absmax) -- for planes whose magnitude is known a priori."""
    rec = torch.empty(_lib.LKG_SCALE_FLOATS, dtype=torch.float32, device=device)
    with _dev_guard(rec, "scale_from_bound"):
        _lib.check(_lib.load().lkg_scale_from_bound(float(bound), _lib.ptr(other), rec.data_ptr(), _lib.stream()))
    return rec


def split_planes(src: torch.Tensor, rows: Optional[torch.Tensor] = None, out=None, rec: Optional[torch.Tensor] = None):
    """fp32 [m, k] (unit inner stride; optional row gather) -> scaled fp16 hi/lo planes, pad columns zero filled.
    ``rec``: an existing scale record that bounds the data (default: measured from the data on device)."""
    if not (src.dtype == torch.float32 and src.stride(1) == 1):
        src = _lib.f32c(src)
    m = src.shape[0] if rows is None else rows.numel()
    k = src.shape[1]
    if rows is not None:
        rows = rows.to(device=src.device, dtype=torch.int64).contiguous()
    if out is None:
        out = _lib.Planes(m, k, src.device, rec=rec)
        if rec is None:
            scale_from_data(src, rows, rec=out.rec)
    elif rec is None:
        scale_from_data(src, rows, rec=out.rec)
    else:
        assert out.rec is rec
    with _dev_guard(src, "split_planes"):
        _lib.check(_lib.load().lkg_split_planes(src.data_ptr(), src.stride(0), _lib.ptr(rows), m, k, out.rec.data_ptr(),
                                                out.ptr(), out.ld, out.plane_stride, _lib.stream()))
    return out


def pack_weight(weight: torch.Tensor, segments: Sequence) -> _lib.Planes:
    """nn.Linear weight [n, sum(k)] -> packed planes: every K segment zero padded to a multiple of 64 and scaled
    against the scale record of the A segment it will meet (``segments``: the A operand's Planes / views)."""
    weight = _lib.f32c(weight)
    n = weight.shape[0]
    seg_k = [s.k for s in segments]
    if sum(seg_k) != weight.shape[1]:
        raise ValueError("segment widths do not add up to weight.shape[1]")
    arr = (C.c_int32 * len(seg_k))(*[int(x) for x in seg_k])
    recs = (C.c_void_p * len(seg_k))(*[s.rec.data_ptr() for s in segments])
    cols = C.c_int32(0)
    _lib.check(_lib.load().lkg_packed_weight_cols(arr, len(seg_k), C.byref(cols)))
    out = _lib.Planes(n, cols.value, weight.device, ld=cols.value)
    with _dev_guard(weight, "pack_weight", 3):
        _lib.check(_lib.load().lkg_pack_weight(weight.data_ptr(), weight.stride(0), n, arr, len(seg_k), recs, out.ptr(),
                                               out.plane_stride, out.rec.data_ptr(), _lib.stream()))
    return out


def _planes_out(out_planes):
    if out_planes is None:
        return None, 0, 0, None
    return out_planes.elem_ptr(), out_planes.ld, out_planes.plane_stride, out_planes.rec.data_ptr()


def linear(segments: Sequence, weight: torch.Tensor, bias: Optional[torch.Tensor], activation: int = _lib.ACT_NONE,
           out: Optional[torch.Tensor] = None, out_planes=None, out2: Optional[torch.Tensor] = None,
           split_col: int = 0) -> torch.Tensor:
    """out = act([seg0 | seg1 | ...] @ weight^T + bias) on the tensor cores.  ``segments``: Planes / PlanesView
    of the A operand; ``weight``: fp32 [out_features, sum(k)] (nn.Linear layout), packed per call.
    ``out_planes``: Planes whose scale record already bounds the result.  ``out2`` / ``split_col``: the result columns
    from ``split_col`` on are written to ``out2`` ([m, n - split_col] view) instead of ``out``."""
    wp = pack_weight(weight, segments)
    m, n = segments[0].rows, weight.shape[0]
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=weight.device)
    a, b = _lib.planes_operand(segments), _lib.planes_operand([wp])
    if activation & _lib.ACT_ACCUMULATE:
        assert out is not None
    if out2 is not None:
        assert out2.dtype == torch.float32 and out2.stride(1) == 1 and tuple(out2.shape) == (m, n - split_col)
    with _dev_guard(weight, f"linear_k{weight.shape[1]}_n{n}"):
        _lib.check(_lib.load().lkg_linear_fwd_split(C.byref(a), m, C.byref(b), n,
                                                    _lib.ptr(None if bias is None else _lib.f32c(bias)), activation,
                                                    out.data_ptr(), out.stride(0), _lib.ptr(out2),
                                                    0 if out2 is None else out2.stride(0), int(split_col),
                                                    *_planes_out(out_planes), _lib.stream()))
    return out


def gate(segments: Sequence, w_pair: torch.Tensor, bias_pair: torch.Tensor, x_ent: torch.Tensor,
         out: Optional[torch.Tensor] = None, out_planes=None, gz_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Literal gate (gate.py:22-28): out = (1 - z) * x_ent + z * tanh(g) with (g, z) interleaved in w_pair.
    ``out_planes``: its scale record must bound max(1, max|x_ent|) (see ``scale_from_bound``)."""
    wp = pack_weight(w_pair, segments)
    bias_pair = _lib.f32c(bias_pair)
    x_ent = x_ent if (x_ent.dtype == torch.float32 and x_ent.stride(1) == 1) else _lib.f32c(x_ent)
    m, dim = x_ent.shape
    if out is None:
        out = torch.empty((m, dim), dtype=torch.float32, device=x_ent.device)
    a, b = _lib.planes_operand(segments), _lib.planes_operand([wp])
    with _dev_guard(x_ent, "gate"):
        _lib.check(_lib.load().lkg_gate_fwd(C.byref(a), m, C.byref(b), bias_pair.data_ptr(), dim, x_ent.data_ptr(),
                                            x_ent.stride(0), out.data_ptr(), out.stride(0), *_planes_out(out_planes),
                                            _lib.ptr(gz_out), 0 if gz_out is None else gz_out.stride(0), _lib.stream()))
    return out


def aggregate_supported(d_in: int, d_out: int, mode: int) -> bool:
    """True iff ``aggregate`` runs (d_in, d_out) in ``mode`` (_lib.AGG_*) with aligned operands (host call)."""
    ok = C.c_int32(0)
    _lib.check(_lib.load().lkg_aggregate_supported(int(d_in), int(d_out), int(mode), C.byref(ok)))
    return bool(ok.value)


def aggregate(plan: GraphPlan, a_values: torch.Tensor, ego: torch.Tensor, d_out: int,
              pa: Optional[torch.Tensor], pb: torch.Tensor, p2: Optional[torch.Tensor],
              r1: Optional[torch.Tensor], r2: Optional[torch.Tensor],
              ln_weight: torch.Tensor, ln_bias: torch.Tensor, drop_mask: Optional[torch.Tensor],
              x_out: torch.Tensor, xn_out: Optional[torch.Tensor], xn_planes=None, local_row_base: int = 0,
              z: Optional[torch.Tensor] = None, o_out: Optional[torch.Tensor] = None,
              side_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One aggregator layer (lkg_aggregate_fwd).  r1 / r2: [N, d_out] views (any row stride) or [d_out] biases.
    With a row partition, r1 / r2 / drop_mask / xn_out / xn_planes hold the rows from ``local_row_base`` on.
    ``z`` (bi-interaction, wide rows): pre-projected sum term ego @ Pb, [N, d_out] view; then pa = pb = None."""
    assert ego.dtype == torch.float32 and ego.stride(1) == 1
    d_in = ego.shape[1]
    ld_r = 0
    for r in (r1, r2):
        if r is not None and r.dim() == 2:
            assert r.stride(1) == 1
            ld_r = r.stride(0)
    if r1 is not None and r2 is not None:
        assert (r1.dim() == r2.dim()) and (r1.dim() == 1 or r1.stride(0) == r2.stride(0))
    same = pa is not None and pa is pb
    pb_c = None if pb is None else _lib.f32c(pb)
    pa_c = pb_c if same else (None if pa is None else _lib.f32c(pa))
    if z is not None:
        assert z.dtype == torch.float32 and z.stride(1) == 1 and z.shape[1] == d_out and pa is None and pb is None
    p2_c = None if p2 is None else _lib.f32c(p2)
    with _dev_guard(ego, f"aggregate_d{d_in}"):
        _lib.check(_lib.load().lkg_aggregate_fwd(
            plan.byref(), _lib.ptr(a_values), ego.data_ptr(), ego.stride(0), d_in, d_out,
            _lib.ptr(pa_c), _lib.ptr(pb_c), _lib.ptr(p2_c), _lib.ptr(r1), _lib.ptr(r2), ld_r,
            _lib.f32c(ln_weight).data_ptr(), _lib.f32c(ln_bias).data_ptr(), _lib.ptr(drop_mask),
            x_out.data_ptr(), x_out.stride(0), _lib.ptr(xn_out), 0 if xn_out is None else xn_out.stride(0),
            *_planes_out(xn_planes), int(local_row_base), _lib.ptr(z), 0 if z is None else z.stride(0),
            _lib.ptr(o_out), 0 if o_out is None else o_out.stride(0),
            _lib.ptr(side_out), 0 if side_out is None else side_out.stride(0),
            plan.scratch(), _lib.stream()))
    return x_out


def score(emb: torch.Tensor, heads: torch.Tensor, tails: torch.Tensor,
          minmax: Optional[torch.Tensor] = None, rec: Optional[torch.Tensor] = None) -> torch.Tensor:
    """scores = emb[heads] @ emb[tails]^T (model.py:473-486); ``minmax``: opaque uint32[2] state."""
    assert emb.dtype == torch.float32 and emb.stride(1) == 1
    if rec is None:
        rec = scale_from_data(emb)                 # one record for both operands: they are rows of one matrix
    hp = split_planes(emb, heads, rec=rec)
    tp = split_planes(emb, tails, rec=rec)
    out = torch.empty((hp.rows, tp.rows), dtype=torch.float32, device=emb.device)
    if out.numel() == 0:
        return out
    a, b = _lib.planes_operand([hp]), _lib.planes_operand([tp])
    with _dev_guard(emb, "score", 1 if minmax is None else 2):
        lib = _lib.load()
        if minmax is not None:
            _lib.check(lib.lkg_minmax_reset(minmax.data_ptr(), _lib.stream()))
        _lib.check(lib.lkg_score(C.byref(a), hp.rows, C.byref(b), tp.rows, out.data_ptr(), out.stride(0),
                                 _lib.ptr(minmax), _lib.stream()))
    return out


def predict(emb: torch.Tensor, heads: torch.Tensor, tails: torch.Tensor, milestone: float) -> torch.Tensor:
    """(minmax-normalised scores > milestone).int() (model.py:488-491)."""
    mm = torch.empty(2, dtype=torch.int32, device=emb.device)
    s = score(emb, heads, tails, mm)
    pred = torch.empty(s.shape, dtype=torch.int32, device=emb.device)
    if s.numel():
        with _dev_guard(emb, "predict_threshold"):
            _lib.check(_lib.load().lkg_predict_threshold(s.data_ptr(), s.stride(0), s.shape[0], s.shape[1],
                                                         mm.data_ptr(), float(milestone), pred.data_ptr(),
                                                         pred.stride(0), _lib.stream()))
    return pred


def topk_rows(scores: torch.Tensor, k: int, target_cols: Optional[torch.Tensor] = None
              ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
    """Row-wise top-k (larger first, ties -> lower column) and optional rank of ``target_cols``."""
    assert scores.dtype == torch.float32 and scores.stride(1) == 1
    rows, cols = scores.shape
    vals = torch.empty((rows, k), dtype=torch.float32, device=scores.device)
    idx = torch.empty((rows, k), dtype=torch.int64, device=scores.device)
    ranks = None
    if target_cols is not None:
        target_cols = target_cols.to(device=scores.device, dtype=torch.int64).contiguous()
        ranks = torch.empty(rows, dtype=torch.int64, device=scores.device)
    with _dev_guard(scores, "topk_rows"):
        _lib.check(_lib.load().lkg_topk_rows(scores.data_ptr(), scores.stride(0), rows, cols, k, vals.data_ptr(),
                                             idx.data_ptr(), _lib.ptr(target_cols), _lib.ptr(ranks), _lib.stream()))
    return vals, idx, ranks


def topk_merge(vals: torch.Tensor, ids: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """vals / ids [parts, B, k] (per-rank survivors, ids = global positions, -1 pads) -> the k best per row."""
    parts, b, kk = vals.shape
    assert kk == k and ids.shape == vals.shape and vals.dtype == torch.float32 and ids.dtype == torch.int64
    vals, ids = vals.contiguous(), ids.contiguous()
    top_v = torch.empty((b, k), dtype=torch.float32, device=vals.device)
    top_i = torch.empty((b, k), dtype=torch.int64, device=vals.device)
    with _dev_guard(vals, "topk_merge"):
        _lib.check(_lib.load().lkg_topk_merge(vals.data_ptr(), ids.data_ptr(), parts, b, k, top_v.data_ptr(),
                                              top_i.data_ptr(), _lib.stream()))
    return top_v, top_i


# ---- fused all-entity scoring + top-k ---------------------------------------------------------------------
FUSED_TOPK_MIN_TAILS = 16384      # below this the score matrix is small: score() + topk_rows()
FUSED_TOPK_MAX_DIM = 256
FUSED_TOPK_CAP = 4096             # candidate slots per head (a head that overflows is re-scanned exactly)


def mean_row(emb: torch.Tensor, rows: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Mean of the rows ``emb[rows]`` (None: every row), fp32 [dim]: the centre of the rank GEMMs' candidates."""
    if rows is None:
        center = colsum(emb)
    else:                                        # a gathered candidate list: its own column sums
        center = torch.zeros(emb.shape[1], dtype=torch.float32, device=emb.device)
        for c0 in range(0, rows.numel(), 1 << 20):
            colsum(emb[rows[c0:c0 + (1 << 20)]], out=center)
    m = emb.shape[0] if rows is None else rows.numel()
    return (center / float(max(m, 1))).contiguous()


class ScoreIndex:
    """Scaled fp16 hi plane + norms of a set of rows of an embedding matrix (lkg_score_index).  The index of the
    candidate tails only depends on the embedding matrix: build it once and reuse it for every head batch."""

    def __init__(self, emb: torch.Tensor, rows: Optional[torch.Tensor], rec: Optional[torch.Tensor] = None):
        assert emb.dtype == torch.float32 and emb.stride(1) == 1
        self.emb, self.dim = emb, emb.shape[1]
        self.rows = None if rows is None else rows.to(device=emb.device, dtype=torch.int64).contiguous()
        self.m = emb.shape[0] if rows is None else self.rows.numel()
        self.rec = rec if rec is not None else scale_from_data(emb)
        self.ld = (self.dim + 7) // 8 * 8
        self.hi = torch.empty((max(self.m, 1), self.ld), dtype=torch.float16, device=emb.device)
        self.norms = torch.empty(max(self.m, 1), dtype=torch.float32, device=emb.device)
        self.max_norm = torch.empty(1, dtype=torch.float32, device=emb.device)
        with _dev_guard(emb, "score_index"):
            _lib.check(_lib.load().lkg_score_index(emb.data_ptr(), emb.stride(0), _lib.ptr(self.rows), self.m, self.dim,
                                                   self.rec.data_ptr(), self.hi.data_ptr(), self.ld,
                                                   self.norms.data_ptr(), self.max_norm.data_ptr(), _lib.stream()))


    def centered(self):
        """-> (center [dim], ScoreIndex of the rows minus their mean, its hi/lo planes): the operand of the rank GEMM.
        A common shift of the tails changes no head's ranking, and the error band of the GEMM is relative to
        max|t - center| instead of max|t| (model embeddings are tightly clustered).  Built on first use."""
        if getattr(self, "_centered", None) is None:
            center = mean_row(self.emb, self.rows)
            shifted = torch.empty((max(self.m, 1), self.dim), dtype=torch.float32, device=self.emb.device)[:self.m]
            with _dev_guard(self.emb, "shift_rows"):
                _lib.check(_lib.load().lkg_shift_rows(self.emb.data_ptr(), self.emb.stride(0), _lib.ptr(self.rows), self.m,
                                                      self.dim, center.data_ptr(), shifted.data_ptr(), shifted.stride(0),
                                                      _lib.stream()))
            ci = ScoreIndex(shifted, None)
            self._centered = (center.contiguous(), ci, split_planes(shifted, None, rec=ci.rec))
        return self._centered


def _count_band(lib, query_planes, cand_planes, n_cand: int, thr: torch.Tensor, cap: int):
    """lkg_score_rank of the query planes against ``n_cand`` candidate planes under the per-query thresholds ``thr``
    (fp32 [B, 2]) -> (counters int32 [2, B], band int32 [B, cap]): counters[0] = columns above thr[:, 1], counters[1] =
    columns at or above thr[:, 0] and not above thr[:, 1], listed in band (a count above ``cap``: the list overflowed)."""
    nq = thr.shape[0]
    counters = torch.zeros((2, nq), dtype=torch.int32, device=thr.device)
    band = torch.empty((nq, max(cap, 1)), dtype=torch.int32, device=thr.device)
    a, b = _lib.planes_operand([query_planes]), _lib.planes_operand([cand_planes])
    _lib.check(lib.lkg_score_rank(C.byref(a), nq, C.byref(b), n_cand, thr.data_ptr(), counters[0].data_ptr(),
                                  counters[1].data_ptr(), band.data_ptr(), cap, _lib.stream()))
    return counters, band


def _filter_ids(ranks: torch.Tensor, anchors, target_pos, relations, cand_map):
    """The query ids of a rank filter on the device of ``ranks``, one per rank: -> (anchors, target_pos, relations)."""
    assert ranks.dtype == torch.int64 and ranks.is_contiguous()
    dev = ranks.device
    anchors, tgt = _ids(anchors, dev), _ids(target_pos, dev)
    rels = None if relations is None else _ids(relations, dev)
    assert anchors.numel() == tgt.numel() == ranks.numel() and (rels is None or rels.numel() == ranks.numel())
    assert cand_map is None or (cand_map.dtype == torch.int32 and cand_map.is_contiguous())
    return anchors, tgt, rels


def _exclude_args(exclude, nq: int, n_cand: int, dev):
    """``exclude`` of the top-k calls, (known plan, anchors [nq], relations [nq] or None, candidate entity ids
    [n_cand] or None), or None -> (plan reference or None, anchors, relations, ids) on ``dev``."""
    if exclude is None:
        return None, None, None, None
    known, anchors, rels, cids = exclude
    anchors = _ids(anchors, dev)
    rels = None if rels is None else _ids(rels, dev)
    cids = None if cids is None else _ids(cids, dev)
    assert anchors.numel() == nq and (rels is None or rels.numel() == nq)
    assert cids is None or cids.numel() == n_cand
    return None if known is None else known.byref(), anchors, rels, cids


def score_rank(emb: torch.Tensor, heads: Optional[torch.Tensor], target_pos: torch.Tensor, tail_index: ScoreIndex,
               head_emb: Optional[torch.Tensor] = None, band_cap: int = 8192,
               tau_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Rank (0 = best) of tail position ``target_pos[i]`` for head i among the tails of ``tail_index`` under "larger
    exact score first, ties -> lower position", without the B x Nt score matrix (lkg_rank_prepare / lkg_score_rank /
    lkg_rank_finalize).  ``heads`` index ``head_emb`` (default ``emb``), None = every row.  ``tau_out`` (optional fp32
    [B]) receives the exact target scores the ranks were counted against (what ``filter_ranks`` compares with)."""
    ti = tail_index
    hsrc = emb if head_emb is None else head_emb
    assert hsrc.dtype == torch.float32 and hsrc.stride(1) == 1 and hsrc.shape[1] == emb.shape[1]
    hrows = None if heads is None else heads.to(device=emb.device, dtype=torch.int64).contiguous()
    hp = split_planes(hsrc, hrows)                       # own scale record: the two operands' factors multiply
    nh = hp.rows
    tgt = target_pos.to(device=emb.device, dtype=torch.int64).contiguous()
    assert tgt.numel() == nh
    ranks = torch.empty(nh, dtype=torch.int64, device=emb.device)
    if nh == 0:
        return ranks
    center, ci, tp = ti.centered()
    tau = torch.empty(nh, dtype=torch.float32, device=emb.device) if tau_out is None else tau_out
    assert tau.dtype == torch.float32 and tau.is_contiguous() and tau.numel() == nh
    thr = torch.empty((nh, 2), dtype=torch.float32, device=emb.device)
    with _dev_guard(emb, "score_rank", 3):
        lib = _lib.load()
        _lib.check(lib.lkg_rank_prepare(emb.data_ptr(), emb.stride(0), _lib.ptr(ti.rows), hsrc.data_ptr(), hsrc.stride(0),
                                        _lib.ptr(hrows), tgt.data_ptr(), nh, emb.shape[1], ci.max_norm.data_ptr(),
                                        ci.rec.data_ptr(), center.data_ptr(), tau.data_ptr(), thr.data_ptr(),
                                        _lib.stream()))
        counters, band = _count_band(lib, hp, tp, ti.m, thr, band_cap)
        _lib.check(lib.lkg_rank_finalize(emb.data_ptr(), emb.stride(0), _lib.ptr(ti.rows), hsrc.data_ptr(), hsrc.stride(0),
                                         _lib.ptr(hrows), tgt.data_ptr(), tau.data_ptr(), counters[0].data_ptr(),
                                         counters[1].data_ptr(), band.data_ptr(), band_cap, nh, ti.m, emb.shape[1],
                                         ranks.data_ptr(), _lib.stream()))
    return ranks


def filter_ranks(ranks: torch.Tensor, known: GraphPlan, heads: torch.Tensor, target_pos: torch.Tensor,
                 relations: Optional[torch.Tensor] = None, cand_map: Optional[torch.Tensor] = None,
                 emb: Optional[torch.Tensor] = None, tau: Optional[torch.Tensor] = None,
                 scores: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw ranks -> filtered ranks, in place: subtracts from ``ranks[i]`` the distinct known tails of query i that beat
    its target on the scores the raw rank was counted on (lkg_rank_filter / lkg_rank_filter_scores).  ``known``: plan of
    the known triples; ``relations`` (int64 [B] or None): filter by (head, relation), else by head; ``cand_map`` (int32
    [N] or None = identity): candidate position of every entity, -1 = not a candidate.  The scores are either
    ``emb`` + ``tau`` (after ``score_rank`` on ``emb``: the same exact re-score and target scores) or ``scores`` (the
    [B, Nc] matrix ``topk_rows`` ranked)."""
    heads, tgt, rels = _filter_ids(ranks, heads, target_pos, relations, cand_map)
    assert (scores is None) != (emb is None or tau is None), "give emb + tau (fused path) or scores (dense path)"
    with _dev_guard(ranks, "filter_ranks"):
        if scores is None:
            _rowmajor(emb)
            _lib.check(_lib.load().lkg_rank_filter(known.byref(), heads.data_ptr(), _lib.ptr(rels), _lib.ptr(cand_map),
                                                   tgt.data_ptr(), ranks.numel(), emb.data_ptr(), emb.stride(0),
                                                   emb.shape[1], tau.data_ptr(), ranks.data_ptr(), _lib.stream()))
        else:
            _rowmajor(scores)
            _lib.check(_lib.load().lkg_rank_filter_scores(known.byref(), heads.data_ptr(), _lib.ptr(rels),
                                                          _lib.ptr(cand_map), tgt.data_ptr(), ranks.numel(),
                                                          scores.data_ptr(), scores.stride(0), scores.shape[1],
                                                          ranks.data_ptr(), _lib.stream()))
    return ranks


# ---- distance rank: the triple score -|q - p_j|^2 (TransR / TransE) ------------------------------------------------
L2_RANK_MAX_DIM = 508              # the augmented GEMM width dim + 4 must stay <= 512


def l2_rank_rows(src: torch.Tensor, center: torch.Tensor, mode: int, stats: torch.Tensor,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Augmented operand of the distance rank GEMM (lkg_l2_rank_rows): ``mode`` _lib.L2_CANDIDATE writes
    [p - c, -|p - c|^2 / (2 alpha), 0, 0, 0] per row and fills ``stats`` (fp32 [2]); _lib.L2_QUERY writes
    [q - c, alpha, 0, 0, 0] with alpha taken from the candidates' ``stats``.  -> fp32 [m, dim + 4]."""
    _rowmajor(src)
    m, dim = src.shape
    if out is None:
        out = torch.empty((max(m, 1), dim + 4), dtype=torch.float32, device=src.device)[:m]
    with _dev_guard(src, "l2_rank_rows", 2 if mode == _lib.L2_CANDIDATE else 1):
        _lib.check(_lib.load().lkg_l2_rank_rows(src.data_ptr(), src.stride(0), None, m, dim, center.data_ptr(), int(mode),
                                                stats.data_ptr(), out.data_ptr(), out.stride(0), _lib.stream()))
    return out


class L2Index:
    """Candidate side of the distance rank: the candidates' rows p_j (fp32 [Nc, dim], dim % 4 == 0, e.g. the projected
    rows emb[cand] M_r zero padded to a multiple of 4 -- zero columns add nothing to a distance), their mean c (as
    ``ScoreIndex.centered`` takes it), and the hi/lo planes of the augmented rows [p_j - c, -|p_j - c|^2 / (2 alpha)].
    ``refill()`` rebuilds it in place after ``cand`` was overwritten (the next relation's projection): one relation's
    tables are alive at a time."""

    def __init__(self, cand: torch.Tensor):
        _rowmajor(cand)
        self.cand, (self.m, self.dim) = cand, cand.shape
        if self.dim % 4 or self.dim > L2_RANK_MAX_DIM:
            raise ValueError(f"the distance rank path needs a width that is a multiple of 4 and <= {L2_RANK_MAX_DIM}")
        dev = cand.device
        self.stats = torch.zeros(2, dtype=torch.float32, device=dev)
        self.aug = torch.empty((max(self.m, 1), self.dim + 4), dtype=torch.float32, device=dev)[:self.m]
        self.planes = _lib.Planes(self.m, self.dim + 4, dev)
        self.refill()

    def refill(self) -> "L2Index":
        self.center = mean_row(self.cand)
        l2_rank_rows(self.cand, self.center, _lib.L2_CANDIDATE, self.stats, out=self.aug)
        split_planes(self.aug, None, out=self.planes)
        return self


def score_rank_l2(index: L2Index, query: torch.Tensor, target_pos: torch.Tensor, band_cap: int = 8192,
                  tau_out: Optional[torch.Tensor] = None, stats: Optional[dict] = None) -> torch.Tensor:
    """Rank (0 = best) of candidate ``target_pos[i]`` for query row ``query[i]`` (fp32 [B, index.dim]) under "smaller
    exact distance first, ties -> lower position", d_j = |q_i - p_j|^2 in fp64 rounded once to fp32, without the B x Nc
    matrix (lkg_l2_rank_rows / lkg_rank_prepare_l2 / lkg_score_rank / lkg_rank_finalize_l2).  ``tau_out`` (fp32 [B])
    receives the exact target distances (what ``filter_ranks_l2`` compares with); ``stats`` (a dict) receives
    "band": int32 [B] columns inside each query's error band (above ``band_cap``: the query was re-scanned exactly)."""
    _rowmajor(query)
    nq, dev = query.shape[0], query.device
    assert query.shape[1] == index.dim
    tgt = target_pos.to(device=dev, dtype=torch.int64).contiguous()
    assert tgt.numel() == nq
    ranks = torch.empty(nq, dtype=torch.int64, device=dev)
    if nq == 0:
        return ranks
    aug = l2_rank_rows(query, index.center, _lib.L2_QUERY, index.stats)
    qp = split_planes(aug)                               # own scale record: the two operands' factors multiply
    tau = torch.empty(nq, dtype=torch.float32, device=dev) if tau_out is None else tau_out
    assert tau.dtype == torch.float32 and tau.is_contiguous() and tau.numel() == nq
    thr = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    with _dev_guard(query, "score_rank_l2", 3):
        lib = _lib.load()
        _lib.check(lib.lkg_rank_prepare_l2(index.cand.data_ptr(), index.cand.stride(0), query.data_ptr(), query.stride(0),
                                           aug.data_ptr(), aug.stride(0), tgt.data_ptr(), nq, index.dim,
                                           index.stats.data_ptr(), qp.rec.data_ptr(), index.planes.rec.data_ptr(),
                                           tau.data_ptr(), thr.data_ptr(), _lib.stream()))
        counters, band = _count_band(lib, qp, index.planes, index.m, thr, band_cap)
        _lib.check(lib.lkg_rank_finalize_l2(index.cand.data_ptr(), index.cand.stride(0), query.data_ptr(),
                                            query.stride(0), tgt.data_ptr(), tau.data_ptr(), counters[0].data_ptr(),
                                            counters[1].data_ptr(), band.data_ptr(), band_cap, nq, index.m, index.dim,
                                            ranks.data_ptr(), _lib.stream()))
    if stats is not None:
        stats["band"] = counters[1]
    return ranks


def filter_ranks_l2(ranks: torch.Tensor, known: GraphPlan, anchors: torch.Tensor, target_pos: torch.Tensor,
                    relations: Optional[torch.Tensor], cand_map: Optional[torch.Tensor], index: L2Index,
                    query: torch.Tensor, tau: torch.Tensor) -> torch.Tensor:
    """``filter_ranks`` after ``score_rank_l2`` (lkg_rank_filter_l2): query i's filter set is the run of
    (anchors[i], relations[i]) in ``known``; a member f is re-scored with the same exact distance between ``query[i]``
    and its candidate row ``index.cand[cand_map[f]]`` and compared with the same ``tau``."""
    anchors, tgt, rels = _filter_ids(ranks, anchors, target_pos, relations, cand_map)
    _rowmajor(query)
    with _dev_guard(ranks, "filter_ranks_l2"):
        _lib.check(_lib.load().lkg_rank_filter_l2(known.byref(), anchors.data_ptr(), _lib.ptr(rels), _lib.ptr(cand_map),
                                                  tgt.data_ptr(), ranks.numel(), index.cand.data_ptr(),
                                                  index.cand.stride(0), query.data_ptr(), query.stride(0), index.dim,
                                                  tau.data_ptr(), ranks.data_ptr(), _lib.stream()))
    return ranks


TOPK_L2_CAP = 8192                 # listed columns per query (a query that overflows is re-scanned exactly)
TOPK_L2_MAX_K = 1024


def topk_l2_samples(n_cand: int, k: int) -> int:
    """Default sample count S of the top-k threshold: about k n_cand / S ~ 4096 columns fall within the sampled k-th
    distance, plus the GEMM's error band.  Sampling costs S exact distances per query and finalize about as many
    listed re-scores plus their sort.  Chosen from a sweep at 1 M candidates on a B200 (DESIGN.md §6): half this S
    already lets lists overflow the default cap of 8192."""
    return min(n_cand, max(4096, -(-k * n_cand // 4096)))


def score_topk_l2(index: L2Index, query: torch.Tensor, k: int, exclude=None, cap: int = TOPK_L2_CAP,
                  n_sample: Optional[int] = None, stats: Optional[dict] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per query row ``query[i]`` (fp32 [B, index.dim]) the k candidates of ``index`` with the smallest exact distance
    d_j = |q_i - p_j|^2 (fp64, rounded once to fp32), ties -> lower position, without the B x Nc matrix
    (lkg_l2_rank_rows / lkg_topk_threshold_l2 / lkg_score_rank / lkg_topk_finalize_l2).  -> (dist fp32 [B, k]
    ascending, pos int64 [B, k] candidate positions), padded with +inf / -1 when fewer than k candidates remain.
    ``exclude`` = (known plan, anchors [B], relations [B] or None, candidate entity ids [Nc] or None = identity): query
    i leaves out the candidates whose entity is in the (anchors[i], relations[i]) run of the plan.  ``cap``: listed
    columns per query (2k <= cap <= 16384); ``n_sample``: samples of the threshold (default ``topk_l2_samples``);
    ``stats`` (a dict) receives "listed" (int32 [B], above ``cap``: re-scanned exactly) and "theta" (fp32 [B])."""
    _rowmajor(query)
    nq, dev = query.shape[0], query.device
    assert query.shape[1] == index.dim
    dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
    pos = torch.empty((nq, k), dtype=torch.int64, device=dev)
    if nq == 0:
        return dist, pos
    if n_sample is None:
        n_sample = topk_l2_samples(index.m, k)
    kb, anchors, rels, cids = _exclude_args(exclude, nq, index.m, dev)
    aug = l2_rank_rows(query, index.center, _lib.L2_QUERY, index.stats)
    qp = split_planes(aug)                               # own scale record: the two operands' factors multiply
    thr = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    theta = torch.empty(nq, dtype=torch.float32, device=dev)
    with _dev_guard(query, "score_topk_l2", 3):
        lib = _lib.load()
        _lib.check(lib.lkg_topk_threshold_l2(index.cand.data_ptr(), index.cand.stride(0), index.m, query.data_ptr(),
                                             query.stride(0), aug.data_ptr(), aug.stride(0), nq, index.dim,
                                             index.stats.data_ptr(), qp.rec.data_ptr(), index.planes.rec.data_ptr(),
                                             int(k), int(n_sample), kb, _lib.ptr(anchors), _lib.ptr(rels),
                                             _lib.ptr(cids), thr.data_ptr(), theta.data_ptr(), _lib.stream()))
        counters, band = _count_band(lib, qp, index.planes, index.m, thr, cap)
        _lib.check(lib.lkg_topk_finalize_l2(index.cand.data_ptr(), index.cand.stride(0), index.m, query.data_ptr(),
                                            query.stride(0), nq, index.dim, counters[1].data_ptr(), band.data_ptr(), cap,
                                            int(k), kb, _lib.ptr(anchors), _lib.ptr(rels), _lib.ptr(cids),
                                            dist.data_ptr(), pos.data_ptr(), _lib.stream()))
    if stats is not None:
        stats["listed"], stats["theta"] = counters[1], theta
    return dist, pos


TOPK_DOT_MAX_DIM = 512


def score_topk_dot(emb: torch.Tensor, anchors: torch.Tensor, k: int, index: ScoreIndex, exclude=None,
                   cap: int = TOPK_L2_CAP, n_sample: Optional[int] = None,
                   stats: Optional[dict] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per anchor row ``emb[anchors[i]]`` the k candidates of ``index`` (rows of ``index.emb``) with the largest exact
    dot product s_j = emb[a] . t_j (fp32 products summed in fp64, rounded once: the value ``score_topk`` returns), ties
    -> lower position, without the B x Nc matrix (lkg_topk_threshold_dot / lkg_score_rank / lkg_topk_finalize_dot on
    the centred candidate operand of ``index.centered()``).  Widths dim % 4 == 0 up to 512.  -> (scores fp32 [B, k]
    descending, pos int64 [B, k] candidate positions), padded with -inf / -1 when fewer than k candidates remain.
    ``exclude``, ``cap``, ``n_sample`` and ``stats`` as for ``score_topk_l2`` (the default sample count is
    ``topk_l2_samples``: a sweep under the dot score at 1 M candidates kept it, DESIGN.md §6)."""
    _rowmajor(emb)
    dev, dim = emb.device, emb.shape[1]
    assert index.dim == dim and index.emb.stride(1) == 1
    anchors = _ids(anchors, dev)
    nq = anchors.numel()
    vals = torch.empty((nq, k), dtype=torch.float32, device=dev)
    pos = torch.empty((nq, k), dtype=torch.int64, device=dev)
    if nq == 0:
        return vals, pos
    if n_sample is None:
        n_sample = topk_l2_samples(index.m, k)
    kb, ex_anchors, rels, cids = _exclude_args(exclude, nq, index.m, dev)
    center, ci, cp = index.centered()
    qp = split_planes(emb, anchors)                      # own scale record: the two operands' factors multiply
    thr = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    theta = torch.empty(nq, dtype=torch.float32, device=dev)
    src = index.emb
    with _dev_guard(emb, "score_topk_dot", 3):
        lib = _lib.load()
        _lib.check(lib.lkg_topk_threshold_dot(src.data_ptr(), src.stride(0), _lib.ptr(index.rows), index.m,
                                              emb.data_ptr(), emb.stride(0), anchors.data_ptr(), nq, dim,
                                              center.data_ptr(), ci.max_norm.data_ptr(), qp.rec.data_ptr(),
                                              ci.rec.data_ptr(), int(k), int(n_sample), kb, _lib.ptr(ex_anchors),
                                              _lib.ptr(rels), _lib.ptr(cids), thr.data_ptr(), theta.data_ptr(),
                                              _lib.stream()))
        counters, band = _count_band(lib, qp, cp, index.m, thr, cap)
        _lib.check(lib.lkg_topk_finalize_dot(src.data_ptr(), src.stride(0), _lib.ptr(index.rows), index.m,
                                             emb.data_ptr(), emb.stride(0), anchors.data_ptr(), nq, dim,
                                             counters[1].data_ptr(), band.data_ptr(), cap, int(k), kb,
                                             _lib.ptr(ex_anchors), _lib.ptr(rels), _lib.ptr(cids), vals.data_ptr(),
                                             pos.data_ptr(), _lib.stream()))
    if stats is not None:
        stats["listed"], stats["theta"] = counters[1], theta
    return vals, pos


def fused_topk_applicable(n_tails: int, dim: int, k: int) -> bool:
    """The fused path needs enough 128-tail tiles to bound the k-th best score from tile maxima."""
    return (dim <= FUSED_TOPK_MAX_DIM and dim % 4 == 0 and n_tails >= max(FUSED_TOPK_MIN_TAILS, 512 * k)
            and k <= 1024)


def score_topk(emb: torch.Tensor, heads: torch.Tensor, tails: Optional[torch.Tensor], k: int,
               tail_index: Optional[ScoreIndex] = None, cap: Optional[int] = None,
               sample_tiles: Optional[int] = None, theta: Optional[torch.Tensor] = None,
               head_emb: Optional[torch.Tensor] = None, stats: Optional[dict] = None
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per head the k best of ``tails`` (None = every row of emb) without materialising the score matrix.
    Returns (values [B, k] fp32, positions [B, k] int64 into the tail list).  ``theta`` (optional, [B] fp32): a known
    lower bound of every head's k-th best exact score; by default the kernels derive one from a strided sample.
    ``head_emb``: matrix the ``heads`` rows index (default ``emb``); its values must be bounded by the tail index's
    scale record (row partition: the record is built from the all-reduced absmax)."""
    assert emb.dtype == torch.float32 and emb.stride(1) == 1 and emb.shape[1] <= FUSED_TOPK_MAX_DIM
    if tail_index is None:
        tail_index = ScoreIndex(emb, tails)
    ti = tail_index
    hsrc = emb if head_emb is None else head_emb
    assert hsrc.dtype == torch.float32 and hsrc.stride(1) == 1 and hsrc.shape[1] == emb.shape[1]
    hi = ScoreIndex(hsrc, heads, rec=ti.rec)          # heads=None: every row of head_emb
    nh, nt = hi.m, ti.m
    vals = torch.empty((nh, k), dtype=torch.float32, device=emb.device)
    pos = torch.empty((nh, k), dtype=torch.int64, device=emb.device)
    if nh == 0:
        return vals, pos
    if cap is None:
        cap = FUSED_TOPK_CAP if k < 64 else 2 * FUSED_TOPK_CAP
    while cap < 2 * k:
        cap *= 2
    n_tiles = (nt + 127) // 128
    if sample_tiles is None:       # expected candidates per head ~ k * n_tiles / sample_tiles ~ max(250, 10 k)
        sample_tiles = min(n_tiles, 4096, max(2 * k, 64, k * n_tiles // max(250, 10 * k)))
    if theta is not None:
        theta = _lib.f32c(theta)
        sample_tiles = 0
    nbytes = C.c_size_t(0)
    _lib.check(_lib.load().lkg_score_topk_workspace_bytes(nh, cap, sample_tiles, C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=emb.device)
    with _dev_guard(emb, "score_topk", 5):
        _lib.check(_lib.load().lkg_score_topk(hi.hi.data_ptr(), hi.ld, hi.norms.data_ptr(), nh, ti.hi.data_ptr(), ti.ld,
                                              ti.max_norm.data_ptr(), nt, emb.shape[1], ti.rec.data_ptr(),
                                              _lib.ptr(theta), 1, sample_tiles, emb.data_ptr(), emb.stride(0),
                                              hsrc.data_ptr(), hsrc.stride(0),
                                              _lib.ptr(hi.rows), _lib.ptr(ti.rows), k, cap, vals.data_ptr(),
                                              pos.data_ptr(), ws.data_ptr(), _lib.stream()))
    if stats is not None and nh <= 256 * 148:   # diagnostics: candidates per head (counters [nh, streams] lead the ws)
        streams = min(148 // ((nh + 255) // 256), n_tiles)
        stats["candidates"] = ws[:4 * nh * streams].view(torch.int32).view(nh, streams).sum(1)
        stats["cap"], stats["cap_per_stream"], stats["sample_tiles"] = cap, cap // streams, sample_tiles
    return vals, pos


# ---- backward of the embedding pass (csrc/backward.cu) ------------------------------------------------------
def _rowmajor(t: torch.Tensor) -> torch.Tensor:
    assert t.dtype == torch.float32 and t.dim() == 2 and t.stride(1) == 1, "fp32 matrix with unit inner stride"
    return t


def spmm_t(plan: GraphPlan, a_values: torch.Tensor, x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out += A_in^T @ x  (backward of torch.sparse.mm(A_in, .), model.py:106)."""
    return spmm_coo(plan.transposed(), a_values, x, out)


def spmm_coo(coo, a_values: torch.Tensor, x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[seg] += a_values[perm] * x[src] over a COO list (seg, src, perm) sorted by seg (``GraphPlan.transposed``);
    perm None: ``a_values`` is already in list order."""
    t_tail, t_head, t_perm = coo
    _rowmajor(x); _rowmajor(out)
    with _dev_guard(x, f"spmm_t_d{x.shape[1]}"):
        _lib.check(_lib.load().lkg_spmm_coo(t_tail.data_ptr(), t_head.data_ptr(), _lib.ptr(t_perm), a_values.data_ptr(),
                                            t_tail.numel(), x.data_ptr(), x.stride(0), x.shape[1], out.data_ptr(),
                                            out.stride(0), _lib.stream()))
    return out


def layer_bwd_rows(y: torch.Tensor, o: torch.Tensor, has_o2: bool, mask: Optional[torch.Tensor],
                   dy_in: Optional[torch.Tensor], dyn: Optional[torch.Tensor], ln_weight: torch.Tensor,
                   d_o: torch.Tensor, dgb: torch.Tensor, amax: Optional[torch.Tensor] = None,
                   amax2: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``amax`` / ``amax2``: raw records (``raw_record``) raised to max|d_o|."""
    n, c = y.shape
    for t in (y, o, d_o):
        _rowmajor(t)
    with _dev_guard(y, "layer_bwd_rows"):
        _lib.check(_lib.load().lkg_layer_bwd_rows(
            n, c, int(has_o2), y.data_ptr(), y.stride(0), o.data_ptr(), o.stride(0), _lib.ptr(mask),
            _lib.ptr(dy_in), 0 if dy_in is None else _rowmajor(dy_in).stride(0),
            _lib.ptr(dyn), 0 if dyn is None else _rowmajor(dyn).stride(0),
            _lib.f32c(ln_weight).data_ptr(), d_o.data_ptr(), d_o.stride(0), dgb.data_ptr(), _lib.ptr(amax),
            _lib.ptr(amax2), _lib.stream()))
    return d_o


def bi_bwd_rows(d_o2: torch.Tensor, p2: torch.Tensor, x: torch.Tensor, side: torch.Tensor, w_out: torch.Tensor,
                dx: torch.Tensor, accumulate: bool, xs_out: Optional[torch.Tensor] = None,
                xs_amax: Optional[torch.Tensor] = None) -> None:
    n, d = x.shape
    c = d_o2.shape[1]
    for t in (d_o2, x, side, w_out, dx):
        _rowmajor(t)
    p2 = _lib.f32c(p2)
    assert tuple(p2.shape) == (d, c)
    with _dev_guard(x, f"bi_bwd_rows_d{d}"):
        _lib.check(_lib.load().lkg_bi_bwd_rows(n, d, c, d_o2.data_ptr(), d_o2.stride(0), p2.data_ptr(), x.data_ptr(),
                                               x.stride(0), side.data_ptr(), side.stride(0), w_out.data_ptr(),
                                               w_out.stride(0), dx.data_ptr(), dx.stride(0), int(accumulate),
                                               _lib.ptr(xs_out), 0 if xs_out is None else _rowmajor(xs_out).stride(0),
                                               _lib.ptr(xs_amax), _lib.stream()))


def xt_y(x: Optional[torch.Tensor], y: torch.Tensor, x2: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x^T @ y reduced over the rows (x None: column sums of y, shape [1, cy]); optional elementwise factor x2."""
    _rowmajor(y)
    n, cy = y.shape
    dx = 1 if x is None else _rowmajor(x).shape[1]
    if out is None:
        out = torch.zeros((dx, cy), dtype=torch.float32, device=y.device)
    with _dev_guard(y, f"xt_y_{dx}x{cy}"):
        _lib.check(_lib.load().lkg_xt_y(_lib.ptr(x), 0 if x is None else x.stride(0), _lib.ptr(x2),
                                        0 if x2 is None else _rowmajor(x2).stride(0), dx, y.data_ptr(), y.stride(0), cy, n,
                                        out.data_ptr(), out.stride(0), _lib.stream()))
    return out


def xt_y_planes(xp, yp, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x^T @ y over the rows on the tensor cores; xp / yp: Planes or PlanesView of [n, dx] and [n, cy]."""
    assert xp.rows == yp.rows
    if out is None:
        out = torch.zeros((xp.k, yp.k), dtype=torch.float32, device=xp.rec.device)
    assert out.dtype == torch.float32 and out.stride(1) == 1 and tuple(out.shape) == (xp.k, yp.k)
    a, b = _lib.planes_operand([xp]), _lib.planes_operand([yp])
    with _dev_guard(out, f"xt_y_tc_{xp.k}x{yp.k}"):
        _lib.check(_lib.load().lkg_xt_y_planes(C.byref(a), C.byref(b), xp.rows, out.data_ptr(), out.stride(0),
                                               _lib.stream()))
    return out


def colsum(y: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _rowmajor(y)
    if out is None:
        out = torch.zeros(y.shape[1], dtype=torch.float32, device=y.device)
    with _dev_guard(y, "colsum"):
        _lib.check(_lib.load().lkg_colsum(y.data_ptr(), y.stride(0), y.shape[0], y.shape[1], out.data_ptr(), _lib.stream()))
    return out


def gate_bwd(dh: torch.Tensor, gz: torch.Tensor, ent: torch.Tensor, d_pre: torch.Tensor, d_ent: torch.Tensor,
             pre_amax: Optional[torch.Tensor] = None) -> None:
    n, dim = dh.shape
    for t in (dh, gz, ent, d_pre, d_ent):
        _rowmajor(t)
    with _dev_guard(dh, "gate_bwd"):
        _lib.check(_lib.load().lkg_gate_bwd(dh.data_ptr(), dh.stride(0), gz.data_ptr(), gz.stride(0), ent.data_ptr(),
                                            ent.stride(0), n, dim, d_pre.data_ptr(), d_pre.stride(0), d_ent.data_ptr(),
                                            d_ent.stride(0), _lib.ptr(pre_amax), _lib.stream()))


def leaky_bwd(grad: torch.Tensor, out: torch.Tensor, d_pre: Optional[torch.Tensor] = None,
              amax: Optional[torch.Tensor] = None) -> torch.Tensor:
    n, c = out.shape
    grad = grad if (grad.dtype == torch.float32 and grad.stride(1) == 1) else _lib.f32c(grad)
    if d_pre is None:
        d_pre = torch.empty((n, c), dtype=torch.float32, device=out.device)
    with _dev_guard(out, "leaky_bwd"):
        _lib.check(_lib.load().lkg_leaky_bwd(grad.data_ptr(), grad.stride(0), out.data_ptr(), out.stride(0), n, c,
                                             d_pre.data_ptr(), d_pre.stride(0), _lib.ptr(amax), _lib.stream()))
    return d_pre


# ---- loss heads (csrc/loss.cu) ------------------------------------------------------------------------------------
def _ids(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.int64).contiguous()


def bpr_loss(emb: torch.Tensor, h, pos, neg, l2_lambda: float, loss: Optional[torch.Tensor],
             grad_scale: Optional[torch.Tensor] = None, d_emb: Optional[torch.Tensor] = None) -> None:
    _rowmajor(emb)
    h, pos, neg = (_ids(x, emb.device) for x in (h, pos, neg))
    with _dev_guard(emb, "bpr_loss"):
        _lib.check(_lib.load().lkg_bpr_loss(emb.data_ptr(), emb.stride(0), emb.shape[1], h.data_ptr(), pos.data_ptr(),
                                            neg.data_ptr(), h.numel(), float(l2_lambda), _lib.ptr(loss),
                                            _lib.ptr(grad_scale), _lib.ptr(d_emb),
                                            0 if d_emb is None else _rowmajor(d_emb).stride(0), _lib.stream()))


def transr_loss(emb: torch.Tensor, relation: torch.Tensor, trans_m: torch.Tensor, h, r, pos, neg, l2_lambda: float,
                loss: Optional[torch.Tensor], grad_scale: Optional[torch.Tensor] = None,
                d_emb: Optional[torch.Tensor] = None, d_relation: Optional[torch.Tensor] = None,
                d_trans_m: Optional[torch.Tensor] = None) -> None:
    _rowmajor(emb)
    relation, trans_m = _lib.f32c(relation), _lib.f32c(trans_m)
    assert trans_m.shape[1] == emb.shape[1] and trans_m.shape[2] == relation.shape[1]
    h, r, pos, neg = (_ids(x, emb.device) for x in (h, r, pos, neg))
    for t in (d_relation, d_trans_m):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous())
    with _dev_guard(emb, "transr_loss"):
        _lib.check(_lib.load().lkg_transr_loss(
            emb.data_ptr(), emb.stride(0), emb.shape[1], relation.data_ptr(), relation.stride(0), relation.shape[1],
            trans_m.data_ptr(), h.data_ptr(), r.data_ptr(), pos.data_ptr(), neg.data_ptr(), h.numel(), float(l2_lambda),
            _lib.ptr(loss), _lib.ptr(grad_scale), _lib.ptr(d_emb), 0 if d_emb is None else _rowmajor(d_emb).stride(0),
            _lib.ptr(d_relation), _lib.ptr(d_trans_m), _lib.stream()))


# ---- variant heads (csrc/mlp_head.cu): TransE loss and the `mlp` mode head --------------------------------------------
def transe_loss(emb: torch.Tensor, relation: torch.Tensor, h, r, pos, neg, l2_lambda: float,
                loss: Optional[torch.Tensor], grad_scale: Optional[torch.Tensor] = None,
                d_emb: Optional[torch.Tensor] = None, d_relation: Optional[torch.Tensor] = None) -> None:
    _rowmajor(emb)
    relation = _lib.f32c(relation)
    if relation.shape[1] != emb.shape[1]:
        raise ValueError("the TransE loss adds relation embeddings to rows of the final embeddings: relation_dim "
                         f"({relation.shape[1]}) must equal their width ({emb.shape[1]}) (model_bce.py:351-354)")
    h, r, pos, neg = (_ids(x, emb.device) for x in (h, r, pos, neg))
    assert d_relation is None or (d_relation.dtype == torch.float32 and d_relation.is_contiguous())
    with _dev_guard(emb, "transe_loss"):
        _lib.check(_lib.load().lkg_transe_loss(
            emb.data_ptr(), emb.stride(0), emb.shape[1], relation.data_ptr(), relation.stride(0), h.data_ptr(),
            r.data_ptr(), pos.data_ptr(), neg.data_ptr(), h.numel(), float(l2_lambda), _lib.ptr(loss),
            _lib.ptr(grad_scale), _lib.ptr(d_emb), 0 if d_emb is None else _rowmajor(d_emb).stride(0),
            _lib.ptr(d_relation), _lib.stream()))


ACT_FC_NONE, ACT_FC_RELU, ACT_FC_SIGMOID = 0, 1, 2


def mlp_fc_fwd(src: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], act: int, m: int,
               pair=None, affine=None, stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = act(input @ weight^T + bias) over ``m`` batch rows.  ``pair`` = (rows_a, rows_b): the input is
    [src[rows_a] | src[rows_b]]; ``affine`` = (scale, shift): the input is src * scale + shift (folded BatchNorm)."""
    _rowmajor(src)
    weight = _lib.f32c(weight)
    n, k = weight.shape
    out = torch.empty((m, n), dtype=torch.float32, device=src.device)
    ra = rb = sc = sh = None
    half = 0
    if pair is not None:
        ra, rb = pair
        half = src.shape[1]
        assert k == 2 * half
    if affine is not None:
        sc, sh = affine
    with _dev_guard(src, "mlp_fc_fwd"):
        _lib.check(_lib.load().lkg_mlp_fc_fwd(src.data_ptr(), src.stride(0), _lib.ptr(ra), _lib.ptr(rb), half, _lib.ptr(sc),
                                              _lib.ptr(sh), m, k, weight.data_ptr(), weight.stride(0),
                                              _lib.ptr(None if bias is None else _lib.f32c(bias)), n, act, out.data_ptr(),
                                              out.stride(0), _lib.ptr(stats), _lib.stream()))
    return out


def bn_finalize(stats: Optional[torch.Tensor], m: int, bn: "torch.nn.BatchNorm1d", training: bool):
    """-> (scale, shift, mean, rstd) of one BatchNorm1d; training updates the running buffers like torch."""
    n = bn.num_features
    dev = bn.weight.device
    scale, shift, mean, rstd = (torch.empty(n, dtype=torch.float32, device=dev) for _ in range(4))
    momentum = 0.1 if bn.momentum is None else float(bn.momentum)
    with _dev_guard(scale, "bn_finalize"):
        _lib.check(_lib.load().lkg_bn_finalize(_lib.ptr(stats), m, n, bn.weight.detach().data_ptr(),
                                               bn.bias.detach().data_ptr(), float(bn.eps), momentum,
                                               bn.running_mean.data_ptr(), bn.running_var.data_ptr(), int(training),
                                               scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                               _lib.stream()))
    if training and bn.num_batches_tracked is not None:
        bn.num_batches_tracked += 1
    return scale, shift, mean, rstd


def mlp_fc_bwd_weight(dz: torch.Tensor, src: torch.Tensor, k: int, pair=None, affine=None):
    """(dW [n, k], db [n]) of one fully-connected step; the input transform is recomputed like in the forward."""
    _rowmajor(dz); _rowmajor(src)
    m, n = dz.shape
    dw = torch.zeros((n, k), dtype=torch.float32, device=dz.device)
    db = torch.zeros(n, dtype=torch.float32, device=dz.device)
    ra = rb = sc = sh = None
    half = 0
    if pair is not None:
        ra, rb = pair
        half = src.shape[1]
    if affine is not None:
        sc, sh = affine
    with _dev_guard(dz, "mlp_fc_bwd_weight"):
        _lib.check(_lib.load().lkg_mlp_fc_bwd_weight(dz.data_ptr(), dz.stride(0), src.data_ptr(), src.stride(0),
                                                     _lib.ptr(ra), _lib.ptr(rb), half, _lib.ptr(sc), _lib.ptr(sh), m, k, n,
                                                     dw.data_ptr(), dw.stride(0), db.data_ptr(), _lib.stream()))
    return dw, db


def mlp_fc_bwd_input(dz: torch.Tensor, weight: torch.Tensor, dx: torch.Tensor, pair=None, bn=None) -> torch.Tensor:
    """dx = dz @ weight.  ``pair`` = (rows_a, rows_b): accumulated into the rows of ``dx`` (the embedding gradient);
    ``bn`` = (a, mean, rstd, stats): also accumulates the two column sums of the BatchNorm backward."""
    _rowmajor(dz); _rowmajor(dx)
    weight = _lib.f32c(weight)
    m, n = dz.shape
    k = weight.shape[1]
    ra = rb = a = mean = rstd = stats = None
    half = 0
    if pair is not None:
        ra, rb = pair
        half = dx.shape[1]
    if bn is not None:
        a, mean, rstd, stats = bn
    with _dev_guard(dz, "mlp_fc_bwd_input"):
        _lib.check(_lib.load().lkg_mlp_fc_bwd_input(dz.data_ptr(), dz.stride(0), m, n, weight.data_ptr(), weight.stride(0), k,
                                                    dx.data_ptr(), dx.stride(0), _lib.ptr(ra), _lib.ptr(rb), half,
                                                    _lib.ptr(a), 0 if a is None else a.stride(0), _lib.ptr(mean),
                                                    _lib.ptr(rstd), _lib.ptr(stats), _lib.stream()))
    return dx


def bn_relu_bwd(dy: torch.Tensor, a: torch.Tensor, mean, rstd, gamma, stats, training: bool):
    """-> (dz, dgamma, dbeta): BatchNorm (batch or running statistics) + ReLU backward."""
    m, k = dy.shape
    dz = torch.empty((m, k), dtype=torch.float32, device=dy.device)
    dgamma = torch.zeros(k, dtype=torch.float32, device=dy.device)
    dbeta = torch.zeros(k, dtype=torch.float32, device=dy.device)
    with _dev_guard(dy, "bn_relu_bwd"):
        _lib.check(_lib.load().lkg_bn_relu_bwd(dy.data_ptr(), dy.stride(0), a.data_ptr(), a.stride(0), mean.data_ptr(),
                                               rstd.data_ptr(), _lib.f32c(gamma).data_ptr(), stats.data_ptr(), m, k,
                                               int(training), dz.data_ptr(), dz.stride(0), dgamma.data_ptr(),
                                               dbeta.data_ptr(), _lib.stream()))
    return dz, dgamma, dbeta


def sigmoid_bwd(dy: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    dy, y = _lib.f32c(dy).reshape(-1), _lib.f32c(y).reshape(-1)
    dz = torch.empty_like(y)
    with _dev_guard(y, "sigmoid_bwd"):
        _lib.check(_lib.load().lkg_sigmoid_bwd(dy.data_ptr(), y.data_ptr(), y.numel(), dz.data_ptr(), _lib.stream()))
    return dz
