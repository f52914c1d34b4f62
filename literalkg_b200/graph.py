"""Device-resident CSR plan of the knowledge graph (lkg_graph in include/lkg.h).

Built once per edge list; the reference re-derives the same structure on every ``update_att`` call
inside ``torch.sparse.softmax`` (coalesce = sort + duplicate merge, model.py:466-470) and inside the
scipy Laplacian construction (dataloader.py:449-495).
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Optional

import torch

from . import _lib


def expand_schedule(sched: torch.Tensor, seg_degree: int = _lib.SEG_DEGREE, max_segs: int = _lib.MAX_SEGS,
                    solo_degree: int = _lib.SOLO_DEGREE):
    """``sched`` int32 [N, 8] = {row, att_lo, att_hi, agg_lo, agg_hi, 0, 0, 0} sorted by decreasing triple count ->
    (schedule with the leading rows of more than ``seg_degree`` triples cut into min(ceil(count / seg_degree),
    max_segs) records {row, att sub-range, agg sub-range, nseg, ticket, piece}, number of rows above ``solo_degree``,
    number of segmented rows).  The sub-ranges of a row partition its att range and its agg range exactly, in order;
    ticket = position of the row among the segmented rows.  Works on any device (tested on CPU)."""
    deg = (sched[:, 2] - sched[:, 1]).long()
    if sched.shape[0] == 0:
        return sched, 0, 0
    n_solo, n_heavy = (int(x) for x in torch.stack([(deg > solo_degree).sum(), (deg > seg_degree).sum()]).tolist())
    if n_heavy == 0:
        return sched, n_solo, 0
    dev = sched.device
    hv = sched[:n_heavy].long()
    nseg = torch.clamp((deg[:n_heavy] + seg_degree - 1) // seg_degree, max=max_segs)
    rid = torch.repeat_interleave(torch.arange(n_heavy, device=dev), nseg)              # = ticket of the row
    piece = torch.arange(rid.numel(), device=dev) - (torch.cumsum(nseg, 0) - nseg)[rid]
    ns = nseg[rid]

    def cut(lo, hi):
        ln = hi - lo
        return lo + ln * piece // ns, lo + ln * (piece + 1) // ns

    e0, e1 = cut(hv[rid, 1], hv[rid, 2])
    u0, u1 = cut(hv[rid, 3], hv[rid, 4])
    seg = torch.stack([hv[rid, 0], e0, e1, u0, u1, ns, rid, piece], dim=1).to(torch.int32)
    return torch.cat([seg, sched[n_heavy:]]).contiguous(), n_solo, n_heavy


class GraphPlan:
    """att order = kept triples sorted by (h, r, t); agg order = unique (h, t) pairs sorted by (h, t),
    i.e. the coalesced ``A_in`` of the reference.  ``file_seg[i]`` = pair index of input triple i."""

    def __init__(self, h: torch.Tensor, t: torch.Tensor, r: torch.Tensor, n_entities: int, n_relations: int,
                 relations: Optional[Iterable[int]] = None):
        _lib.require_cuda(h, "h_list")
        lib = _lib.load()
        dev = h.device
        h = h.to(torch.int64).contiguous()
        t = t.to(device=dev, dtype=torch.int64).contiguous()
        r = r.to(device=dev, dtype=torch.int64).contiguous()
        e = h.numel()
        if not (t.numel() == e and r.numel() == e):
            raise ValueError("h_list, t_list and r_list must have the same length")
        keep = None
        if relations is not None:
            rel = sorted({int(x) for x in relations})
            if rel != list(range(n_relations)):       # a relation list that omits ids drops their triples
                keep = torch.zeros(n_relations, dtype=torch.uint8)
                keep[[x for x in rel if 0 <= x < n_relations]] = 1
                keep = keep.to(dev)
        i32 = dict(dtype=torch.int32, device=dev)
        self.att_rowptr = torch.empty(n_entities + 1, **i32)
        self.rowptr = torch.empty(n_entities + 1, **i32)
        self.att_tail = torch.empty(max(e, 1), **i32)
        self.att_rel = torch.empty(max(e, 1), **i32)
        self.att_seg = torch.empty(max(e, 1), **i32)
        self.col = torch.empty(max(e, 1), **i32)
        self.row_order = torch.empty(n_entities, **i32)     # rows by decreasing triple count (LPT schedule)
        self.row_sched = torch.empty((n_entities, 8), **i32)   # the same order as {row, att range, agg range} records
        coo = torch.empty((2, max(e, 1)), dtype=torch.int64, device=dev)
        self.file_seg = torch.empty(max(e, 1), **i32)
        counts = torch.zeros(3, dtype=torch.int64, device=dev)
        nbytes = C.c_size_t(0)
        _lib.check(lib.lkg_plan_workspace_bytes(e, n_entities, C.byref(nbytes)))
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.lkg_plan_build(h.data_ptr(), t.data_ptr(), r.data_ptr(), e, n_entities, n_relations,
                                          _lib.ptr(keep), self.att_rowptr.data_ptr(), self.att_tail.data_ptr(),
                                          self.att_rel.data_ptr(), self.att_seg.data_ptr(), self.rowptr.data_ptr(),
                                          self.col.data_ptr(), self.row_order.data_ptr(), self.row_sched.data_ptr(),
                                          coo[0].data_ptr(), coo[1].data_ptr(),
                                          self.file_seg.data_ptr(), counts.data_ptr(), ws.data_ptr(), nbytes.value,
                                          _lib.stream()))
        kept, nnz, bad = counts.tolist()          # one host sync per plan build
        del ws
        if bad:
            raise ValueError(f"{bad} triples have entity / relation ids outside [0, n_entities) / [0, n_relations)")
        self.device = dev
        self.n_entities, self.n_relations = int(n_entities), int(n_relations)
        self.n_input, self.n_edges, self.nnz = e, int(kept), int(nnz)
        self.att_tail, self.att_rel, self.att_seg = (x[:self.n_edges] for x in (self.att_tail, self.att_rel, self.att_seg))
        self.col = self.col[:self.nnz]
        self.file_seg = self.file_seg[:e]
        self.indices = coo[:, :self.nnz]          # int64 [2, nnz]: A_in.coalesce().indices()
        self.c = _lib.LkgGraph(self.n_entities, self.n_edges, self.nnz, self.n_relations, 0, self.n_entities,
                               self.att_rowptr.data_ptr(), self.att_tail.data_ptr(), self.att_rel.data_ptr(),
                               self.att_seg.data_ptr(), self.rowptr.data_ptr(), self.col.data_ptr(),
                               self.row_order.data_ptr(), self.row_sched.data_ptr(), 0, 0, None, None, 0)
        self._row_deg = (self.row_sched[:, 2] - self.row_sched[:, 1])     # triples per row, row_order order
        self._seg_tickets = self._seg_scratch = None
        self._expand_schedule()
        self._part_order = self._part_sched = self._part_range = None
        self._scratch = torch.zeros(64, dtype=torch.int32, device=dev)   # dynamic row counter of the kernels
        self._attn_ws = None
        self._transposed = None
        self._transposed_part = None

    # -- constructors ---------------------------------------------------------------------------
    @classmethod
    def from_coo(cls, indices: torch.Tensor, n_entities: int) -> "GraphPlan":
        """Plan of an existing sparse matrix (e.g. ``A_in`` from the DataLoader or a checkpoint);
        every entry is treated as a triple of relation 0."""
        r = torch.zeros(indices.shape[1], dtype=torch.int64, device=indices.device)
        return cls(indices[0], indices[1], r, n_entities, 1)

    # -- helpers ------------------------------------------------------------------------------
    def _expand_schedule(self) -> None:
        """Rows are scheduled by decreasing triple count.  The leading rows longer than SEG_DEGREE are cut into
        up to MAX_SEGS pieces (records {row, att sub-range, agg sub-range, nseg, ticket, piece}) that different warps
        process; a row-long dependent chain in ONE warp is what bounds the kernels once the graph is split over
        several GPUs (a 4 096-triple row streams for ~0.7 ms).  Integer bookkeeping on the device, two scalar
        read-backs per plan build."""
        sched, n_solo, n_heavy = expand_schedule(self.row_sched)
        self._solo_full = n_solo
        self.c.n_solo_rows = self._solo_full
        self.c.n_sched = sched.shape[0]
        if n_heavy == 0:
            return
        self.row_sched = sched
        self._seg_tickets = torch.zeros(n_heavy, dtype=torch.int32, device=self.device)
        self._seg_scratch = torch.empty((n_heavy * _lib.MAX_SEGS, _lib.SEG_STRIDE), dtype=torch.float32, device=self.device)
        self.c.row_sched = self.row_sched.data_ptr()
        self.c.n_sched = self.row_sched.shape[0]
        self.c.seg_tickets = self._seg_tickets.data_ptr()
        self.c.seg_scratch = self._seg_scratch.data_ptr()
        self.c.seg_stride = _lib.SEG_STRIDE

    def byref(self):
        return C.byref(self.c)

    def set_row_range(self, begin: int, end: int) -> None:
        """Restrict the attention / aggregation kernels to head rows [begin, end) (multi-GPU row partition)."""
        if not (0 <= begin <= end <= self.n_entities):
            raise ValueError("bad row range")
        self.c.row_begin, self.c.row_end = int(begin), int(end)
        if begin == 0 and end == self.n_entities:
            self.c.row_order = self.row_order.data_ptr()
            self.c.row_sched = self.row_sched.data_ptr()
            self.c.n_sched = self.row_sched.shape[0]
            self.c.n_solo_rows = self._solo_full
            return
        if self._part_order is None or self._part_range != (begin, end):   # the partition's rows, heaviest first
            keep = (self.row_order >= begin) & (self.row_order < end)
            self._part_order = self.row_order[keep].contiguous()
            rows = self.row_sched[:, 0]
            self._part_sched = self.row_sched[(rows >= begin) & (rows < end)].contiguous()
            self._part_range = (begin, end)
            self._part_solo = int((self._row_deg[keep] > _lib.SOLO_DEGREE).sum().item())
        self.c.n_solo_rows = self._part_solo
        self.c.row_order = self._part_order.data_ptr()
        self.c.row_sched = self._part_sched.data_ptr()
        self.c.n_sched = self._part_sched.shape[0]

    @staticmethod
    def fingerprint(h: torch.Tensor, t: torch.Tensor, r: torch.Tensor):
        """Order-independent content fingerprint of a device edge list (one tiny kernel + one host sync)."""
        _lib.require_cuda(h, "h_list")
        fp = torch.empty(2, dtype=torch.int64, device=h.device)
        with torch.cuda.device(h.device):
            _lib.check(_lib.load().lkg_edge_fingerprint(h.data_ptr(), t.data_ptr(), r.data_ptr(), h.numel(),
                                                        fp.data_ptr(), _lib.stream()))
        return (h.numel(), *fp.tolist())

    def scratch(self) -> int:
        return self._scratch.data_ptr()

    def transposed(self, rows=None):
        """(t_tail, t_head, t_perm): the unique (h, t) pairs as a COO list sorted by (tail, head); t_perm = position of
        the pair in agg order.  What the backward of ``A_in @ x`` gathers over (built on first use, cached).
        ``rows`` = (begin, end): only the pairs whose HEAD lies in that range, heads renumbered from ``begin`` (the
        row partition: a rank reduces its own head rows into every tail row)."""
        if rows is not None:
            if self._transposed_part is None or self._transposed_part[0] != tuple(rows):
                t_tail, t_head, t_perm = self.transposed()
                keep = (t_head >= rows[0]) & (t_head < rows[1])           # order by (tail, head) is preserved
                self._transposed_part = (tuple(rows), (t_tail[keep].contiguous(),
                                                       (t_head[keep] - rows[0]).contiguous(), t_perm[keep].contiguous()))
            return self._transposed_part[1]
        if self._transposed is None:
            lib = _lib.load()
            i32 = dict(dtype=torch.int32, device=self.device)
            m = max(self.nnz, 1)
            t_tail, t_head, t_perm = torch.empty(m, **i32), torch.empty(m, **i32), torch.empty(m, **i32)
            nbytes = C.c_size_t(0)
            _lib.check(lib.lkg_plan_transpose_workspace_bytes(self.nnz, C.byref(nbytes)))
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(lib.lkg_plan_transpose(self.byref(), t_tail.data_ptr(), t_head.data_ptr(), t_perm.data_ptr(),
                                                  ws.data_ptr(), nbytes.value, _lib.stream()))
            self._transposed = tuple(x[:self.nnz] for x in (t_tail, t_head, t_perm))
        return self._transposed

    def reversed(self) -> "GraphPlan":
        """Plan of the swapped triples (t, h, r): the known set of head prediction (?, r, t), whose filter run is the
        heads h' of (h', r, t).  Built from this plan's own att arrays (its kept triples) on first use, cached."""
        if getattr(self, "_reversed", None) is None:
            counts = (self.att_rowptr[1:] - self.att_rowptr[:-1]).long()
            heads = torch.repeat_interleave(torch.arange(self.n_entities, device=self.device), counts)
            self._reversed = GraphPlan(self.att_tail, heads, self.att_rel, self.n_entities, self.n_relations)
        return self._reversed

    def runs(self):
        """The (head, relation) RUNS of the att order (triples sorted by (h, r, t)): what the relation-projected
        attention projects once each.  -> dict(run_ptr int32 [n_runs + 1], run_head int64 [n_runs], run_rel int64
        [n_runs], order int64 [n_runs] = run ids bucketed by relation (stable), run_slot int32 [n_runs] = position of
        a run in that bucket order, offsets = host list [R + 1] of the buckets).  Built on first use (integer
        bookkeeping with torch ops on the device, one read-back of R + 1 counts), cached with the plan."""
        if getattr(self, "_runs", None) is None:
            dev, e = self.device, self.n_edges
            counts = (self.att_rowptr[1:] - self.att_rowptr[:-1]).long()
            heads = torch.repeat_interleave(torch.arange(self.n_entities, device=dev), counts)
            rel = self.att_rel.long()
            new = torch.ones(e, dtype=torch.bool, device=dev)
            if e > 1:
                new[1:] = (heads[1:] != heads[:-1]) | (rel[1:] != rel[:-1])
            start = torch.nonzero(new).reshape(-1)
            n_runs = int(start.numel())
            run_ptr = torch.cat([start, torch.tensor([e], device=dev)]).to(torch.int32)
            run_head, run_rel = heads[start], rel[start]
            order = torch.sort(run_rel, stable=True).indices
            run_slot = torch.empty(n_runs, dtype=torch.int32, device=dev)
            run_slot[order] = torch.arange(n_runs, dtype=torch.int32, device=dev)
            offsets = [0] + torch.cumsum(torch.bincount(run_rel, minlength=self.n_relations), 0).tolist()
            self._runs = dict(run_ptr=run_ptr, run_head=run_head, run_rel=run_rel, order=order, run_slot=run_slot,
                              offsets=offsets, n_runs=n_runs)
        return self._runs

    def attn_workspace(self, dim: int) -> int:
        """Workspace of lkg_attn_update: row counter + the exp(2 e_r) table."""
        nbytes = C.c_size_t(0)
        _lib.check(_lib.load().lkg_attn_workspace_bytes(self.n_relations, int(dim), C.byref(nbytes)))
        if self._attn_ws is None or self._attn_ws.numel() < nbytes.value:
            self._attn_ws = torch.zeros(nbytes.value, dtype=torch.uint8, device=self.device)
        return self._attn_ws.data_ptr()

    def import_values(self, values: torch.Tensor) -> torch.Tensor:
        """Values given per INPUT entry -> plan (coalesced) order, duplicates summed."""
        values = _lib.f32c(values.to(self.device))
        out = torch.empty(max(self.nnz, 1), dtype=torch.float32, device=self.device)[:self.nnz]
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().lkg_segment_scatter_add(values.data_ptr(), self.file_seg.data_ptr(), self.n_input,
                                                           out.data_ptr(), self.nnz, _lib.stream()))
        return out

    def laplacian(self, laplacian_type: str = "random-walk") -> torch.Tensor:
        """Initial A_in values (dataloader.py:462-495), plan order, fp32."""
        if laplacian_type not in ("random-walk", "symmetric"):
            raise NotImplementedError(laplacian_type)
        out = torch.empty(max(self.nnz, 1), dtype=torch.float32, device=self.device)[:self.nnz]
        acc = torch.empty(max(self.nnz, 1), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().lkg_laplacian_init(self.byref(), int(laplacian_type == "symmetric"),
                                                      out.data_ptr(), acc.data_ptr(), _lib.stream()))
        return out

    def sparse(self, values: torch.Tensor) -> torch.Tensor:
        """Coalesced sparse COO view (shares ``values``) in the reference's A_in format."""
        return torch.sparse_coo_tensor(self.indices, values, (self.n_entities, self.n_entities), is_coalesced=True)
