"""Relation-aware top-k completion on the GPU (ops.score_topk_l2, LiteralKG.topk_triple) against the reference
restatement ``topk_of`` on the same fp32 rows, bit for bit (distance bits and positions), and its consistency with
LiteralKG.evaluate_ranking(score="triple"): entity ids[i, j] gets filtered rank j."""
import os
import socket
import tempfile

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import _parallel_worker as W
import _topk_oracle as T
from test_rank_triple_gpu import build_model, padded, project, triples, ulp_neighbour

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _inference_mode():
    with torch.no_grad():
        yield


def assert_same(got, want):
    """(dist, pos) pairs equal bit for bit."""
    gd, gp = (x.cpu() for x in got)
    wd, wp = (x.cpu() for x in want)
    assert torch.equal(gp, wp)
    assert torch.equal(gd.view(torch.int32), wd.view(torch.int32))


def clustered(n, d_s, nq, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.randn(1, d_s, generator=g, device="cuda") * 2.0
    cand = base + torch.nn.functional.leaky_relu(torch.randn(n, d_s, generator=g, device="cuda"), 0.05)
    query = base + torch.randn(nq, d_s, generator=g, device="cuda") * 0.8
    return cand, query


# ---- 1. ops level, bit exact -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
@pytest.mark.parametrize("d_s", [300, 256, 508, 64])
def test_ops_bit_exact(d_s, k):
    import literalkg_b200 as L
    from literalkg_b200 import ops
    n, nq = 40_000, 24
    cand, query = clustered(n, d_s, nq, seed=d_s + k)
    cand[500:510] = cand[7]                                    # exact duplicates: ties decided by position
    query[0] = cand[7] + 0.01
    # one-ulp neighbours and exact copies straddling the k-th distance of query 1
    d1 = T.dist_of(query[1:2], cand)[0]
    kth = int(torch.sort(d1, stable=True).indices[k - 1])
    spots = [p for p in range(1000, n, 997) if p != kth][:6]
    for p, sign in zip(spots[:4], (-1, +1, -1, +1)):
        cand[p] = ulp_neighbour(query[1], cand[kth], sign)
    cand[spots[4]] = cand[kth]
    cand[spots[5]] = cand[kth]
    d = T.dist_of(query, cand)
    assert int((d[1] == d[1, kth]).sum()) >= 3
    index = ops.L2Index(cand)
    st = {}
    got = ops.score_topk_l2(index, query, k, stats=st)
    assert_same(got, T.topk_rows_of(d, k))
    assert int((st["listed"] > ops.TOPK_L2_CAP).sum()) <= 1 and float(st["listed"].float().mean()) < 0.2 * n

    # a candidate subset with known triples excluded: the index holds cand[sub], exclusion by entity id
    g = torch.Generator().manual_seed(k)
    sub = torch.randperm(n, generator=g)[:30_000].cuda()
    anchors = torch.randint(0, n, (nq,), generator=g).cuda()
    rels = torch.randint(0, 2, (nq,), generator=g).cuda()
    near = torch.sort(d[:, sub], dim=1, stable=True).indices[:, :3 * k].cpu()      # the closest, by position
    kh, kr, kt = [], [], []
    for i in range(nq):
        ents = sub.cpu()[near[i, ::2]].tolist() + sub.cpu()[near[i, :4]].tolist()     # every other one, and duplicates
        ents += torch.randint(0, n, (20,), generator=g).tolist()                    # and arbitrary entities
        kh += [int(anchors[i])] * len(ents)
        kr += [int(rels[i])] * len(ents)
        kt += ents
    plan = L.GraphPlan(*(torch.tensor(x).cuda() for x in (kh, kt, kr)), n, 2)
    ds = T.dist_of(query, cand[sub])
    excl = T.excluded_positions(anchors.tolist(), rels.tolist(), sub.tolist(), triples(kh, kr, kt))
    got = ops.score_topk_l2(ops.L2Index(cand[sub].contiguous()), query, k, exclude=(plan, anchors, rels, sub))
    assert_same(got, T.topk_rows_of(ds, k, excl.cuda()))


# ---- 2. exclusion ------------------------------------------------------------------------------------------------------
def test_exclusion_hub_non_candidates_duplicates_and_padding():
    import literalkg_b200 as L
    from literalkg_b200 import ops
    n, nq, k, d_s = 40_000, 16, 50, 300
    cand, query = clustered(n, d_s, nq, seed=5)
    d = T.dist_of(query, cand)
    anchors = torch.arange(100, 100 + nq, device="cuda")
    rels = torch.zeros(nq, dtype=torch.int64, device="cuda")
    order = torch.sort(d[0], stable=True).indices
    kh, kr, kt = [], [], []
    hub = order[:2500].tolist()                                # query 0: the 2 500 closest candidates are known
    kt += hub + hub[:300]                                      # with duplicate triples
    kh += [100] * len(kt)
    kr += [0] * len(kt)
    sub = torch.arange(0, n, 2, device="cuda")                 # candidates: the even entities
    for i in range(1, nq):                                     # known tails, half of them not candidates
        near = torch.sort(d[i], stable=True).indices[:2 * k].tolist()
        kt += near
        kh += [100 + i] * len(near)
        kr += [0] * len(near)
    kt += [5, 5, 7]                                            # another relation's run: must not be used
    kh += [101] * 3
    kr += [1] * 3
    plan = L.GraphPlan(*(torch.tensor(x).cuda() for x in (kh, kt, kr)), n, 2)
    known = triples(kh, kr, kt)
    for cids in (None, sub):
        rows = cand if cids is None else cand[cids].contiguous()
        dd = d if cids is None else d[:, cids]
        ids = list(range(n)) if cids is None else cids.tolist()
        excl = T.excluded_positions(anchors.tolist(), rels.tolist(), ids, known)
        st = {}
        got = ops.score_topk_l2(ops.L2Index(rows), query, k, exclude=(plan, anchors, rels, cids), stats=st)
        assert_same(got, T.topk_rows_of(dd, k, excl.cuda()))
    # fewer than k candidates left: padding.  50 candidates, 45 of them known for the anchor
    small = torch.arange(50, device="cuda")
    plan_s = L.GraphPlan(torch.full((45,), 7, device="cuda"), torch.arange(45, device="cuda"),
                         torch.zeros(45, dtype=torch.int64, device="cuda"), n, 1)
    dist, pos = ops.score_topk_l2(ops.L2Index(cand[:50].contiguous()), query[:2], 10,
                                  exclude=(plan_s, torch.tensor([7, 8], device="cuda"), None, small))
    assert bool((pos[0, 5:] == -1).all()) and bool(torch.isinf(dist[0, 5:]).all())
    assert sorted(pos[0, :5].tolist()) == list(range(45, 50))
    assert bool((pos[1] >= 0).all())                                   # anchor 8 knows nothing


# ---- 3. forced paths ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 100])
def test_overflow_and_weak_threshold_give_the_same_result(k):
    import literalkg_b200 as L
    from literalkg_b200 import ops
    n, nq = 30_000, 12
    cand, query = clustered(n, 300, nq, seed=k)
    d = T.dist_of(query, cand)
    anchors = torch.arange(nq, device="cuda")
    near = torch.sort(d, dim=1, stable=True).indices[:, :k:3]
    kh = anchors[:, None].expand_as(near).reshape(-1)
    plan = L.GraphPlan(kh, near.reshape(-1).cuda(), torch.zeros_like(kh), n, 1)
    index = ops.L2Index(cand)
    for exclude in (None, (plan, anchors, None, None)):
        st_o, st_w = {}, {}
        ref = ops.score_topk_l2(index, query, k, exclude=exclude)
        over = ops.score_topk_l2(index, query, k, exclude=exclude, cap=2 * k, stats=st_o)
        weak = ops.score_topk_l2(index, query, k, exclude=exclude, n_sample=k, stats=st_w)
        assert bool((st_o["listed"] > 2 * k).all())                     # every query took the exact scan
        assert_same(over, ref)
        assert_same(weak, ref)
        assert bool((st_w["theta"] >= st_o["theta"]).all())             # k samples bound no better than the default
        excl = None
        if exclude is not None:
            excl = torch.zeros((nq, n), dtype=torch.bool, device="cuda")
            excl[kh, near.reshape(-1).cuda()] = True
        assert_same(ref, T.topk_rows_of(d, k, excl))


# ---- 4. consistency with evaluate_ranking ------------------------------------------------------------------------------
@pytest.mark.parametrize("with_known", [False, True])
@pytest.mark.parametrize("predict", ["tail", "head"])
@pytest.mark.parametrize("bce", [False, True])
def test_consistent_with_evaluate_ranking(bce, predict, with_known):
    m, known, _, (qh, qr, qt) = build_model(bce=bce)
    emb = m.gat_embeddings()
    anchors = qh if predict == "tail" else qt
    k, bs = 10, 48                                                      # several batches per relation
    kn = known if with_known else None
    cands = None
    if with_known:                                                      # a candidate subset, entity ids returned
        cands = torch.randperm(m.n_entities, generator=torch.Generator().manual_seed(4))[:3000].cuda()
    dist, ids = m.topk_triple(anchors, qr, k, known=kn, candidates=cands, predict=predict, batch_size=bs,
                              all_embed=emb)
    assert dist.shape == ids.shape == (anchors.numel(), k)
    assert bool((ids >= 0).all()) and bool((dist[:, 1:] >= dist[:, :-1]).all())
    if cands is not None:
        assert bool(torch.isin(ids, cands).all())
    for j in range(k):
        other = ids[:, j]
        h, t = (anchors, other) if predict == "tail" else (other, anchors)
        res = m.evaluate_ranking(h, t, qr, known=kn, candidates=cands, score="triple", predict=predict,
                                 batch_size=bs, all_embed=emb)
        assert torch.equal(res["ranks"].cpu(), torch.full((anchors.numel(),), j, dtype=torch.int64)), j
    if with_known:                                      # no known triple is returned
        got = {(a, r, e) for a, r, row in zip(anchors.tolist(), qr.tolist(), ids.tolist()) for e in row}
        kt = {(h, r, t) if predict == "tail" else (t, r, h) for h, r, t in _known_triples(known)}
        assert not (got & kt)


def _known_triples(plan):
    """(h, r, t) of a plan's att order (every triple, duplicates kept)."""
    rp = plan.att_rowptr.cpu()
    heads = torch.repeat_interleave(torch.arange(rp.numel() - 1), rp[1:] - rp[:-1])
    return set(zip(heads.tolist(), plan.att_rel.cpu().tolist(), plan.att_tail.cpu().tolist()))


# ---- 5. two ranks sharing cuda:0 over gloo -----------------------------------------------------------------------------
def _partitioned_worker(rank, world, port, out_dir):
    W._init(rank, world, port, "gloo")
    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    RowPartition = W.staged_partition_cls()
    m, known, _, (qh, qr, qt) = build_model(seed=3)
    qh, qr, qt = qh[:151], qr[:151], qt[:151]                           # not a multiple of the world size
    part = RowPartition(m.n_entities)
    m.set_partition(part)
    full = m.gat_embeddings()
    results = []
    for predict in ("tail", "head"):
        anchors = qh if predict == "tail" else qt
        dist, ids = m.topk_triple(anchors, qr, 20, known=known, batch_size=32, predict=predict)
        both = part.all_gather_stack(ids)
        assert torch.equal(both[0], both[1])
        results.append((anchors, dist, ids))
    m.set_partition(None)
    for predict, (anchors, dist, ids) in zip(("tail", "head"), results):
        one = m.topk_triple(anchors, qr, 20, known=known, batch_size=32, predict=predict, all_embed=full)
        assert torch.equal(one[1], ids) and torch.equal(one[0], dist)
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    torch.distributed.destroy_process_group()


def test_topk_triple_row_partitioned_two_ranks():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_partitioned_worker, args=(2, port, d), nprocs=2, join=True)
        assert sorted(os.listdir(d)) == ["ok0", "ok1"]


# ---- 6. scale ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 100])
def test_scale_bit_exact(k):
    from literalkg_b200 import ops
    n, width, d_s, nq = 262_144, 256, 300, 512
    g = torch.Generator(device="cuda").manual_seed(31)
    emb = torch.nn.functional.leaky_relu(torch.randn(n, width, generator=g, device="cuda"), 0.01) * 0.5
    w = torch.randn(width, d_s, generator=g, device="cuda") / width ** 0.5
    e_r = torch.randn(d_s, generator=g, device="cuda") * 0.5
    anchors = torch.randint(0, n, (nq,), generator=g, device="cuda")
    p = padded(project(emb, None, w))
    q = padded(project(emb, anchors, w, e_r))
    st = {}
    got = ops.score_topk_l2(ops.L2Index(p), q, k, stats=st)
    want_d, want_p = [], []
    for c0 in range(0, nq, 8):                                          # the restatement, chunked on the GPU
        dd, pp = T.topk_rows_of(T.dist_of(q[c0:c0 + 8], p), k)
        want_d.append(dd)
        want_p.append(pp)
    assert_same(got, (torch.cat(want_d), torch.cat(want_p)))
    assert int((st["listed"] > ops.TOPK_L2_CAP).sum()) == 0
