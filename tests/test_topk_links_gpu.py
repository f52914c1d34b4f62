"""Filtered top-k link prediction under the dot score on the GPU (ops.score_topk_dot, LiteralKG.topk_links) against the
reference restatement ``best_of`` on the same fp32 rows, bit for bit (score bits and positions / entity ids), its
agreement with ops.score_topk without exclusion, and its consistency with LiteralKG.evaluate_ranking(score="dot"):
entity ids[i, j] gets filtered rank j."""
import argparse
import os
import socket
import tempfile

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import _parallel_worker as W
import _topk_dot_oracle as T
import literalkg_oracle as O
from test_rank_filtered_gpu import build_model as dot_model
from test_rank_triple_cpu import _model
from test_rank_triple_gpu import build_model, triples

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _inference_mode():
    with torch.no_grad():
        yield


def assert_same(got, want):
    """(scores, pos) pairs equal bit for bit."""
    gv, gp = (x.cpu() for x in got)
    wv, wp = (x.cpu() for x in want)
    assert torch.equal(gp, wp)
    assert torch.equal(gv.view(torch.int32), wv.view(torch.int32))


def clustered(n, dim, nq, seed):
    """Embedding-like rows: a common offset (what the centring removes) plus a spread."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.randn(1, dim, generator=g, device="cuda")
    emb = base + torch.nn.functional.leaky_relu(torch.randn(n, dim, generator=g, device="cuda"), 0.05)
    return emb * 0.3, torch.randint(0, n, (nq,), generator=g, device="cuda")


def pad4(x):
    d4 = (x.shape[1] + 3) // 4 * 4
    out = torch.zeros((x.shape[0], d4), dtype=torch.float32, device=x.device)
    out[:, :x.shape[1]] = x
    return out


def dot_ulp_neighbour(q, t, sign):
    """A copy of row t whose fp32 dot product with q is one fp32 ulp above (sign +1) or below (-1) that of t: the
    coordinate k with the largest |q_k| is stepped through consecutive fp32 values, and the middle of the run of values
    that land on the neighbouring fp32 score is taken."""
    q64, t32 = q.double().cpu().numpy(), t.cpu().numpy().astype(np.float32)
    prod = q64 * t32.astype(np.float64)
    k = int(np.argmax(np.abs(q64)))
    rest = float(np.sum(np.delete(prod, k)))
    s0 = np.float32(rest + prod[k])
    goal = np.nextafter(s0, np.float32(np.inf if sign > 0 else -np.inf))
    up = np.sign(q64[k]) * sign                        # direction of t_k that moves the score the right way
    x = t32[k]
    hits = []
    for _ in range(200_000):
        x = np.nextafter(x, np.float32(np.inf if up > 0 else -np.inf))
        s = np.float32(rest + q64[k] * np.float64(x))
        if s == goal:
            hits.append(x)
        elif hits:
            break
    assert hits, "no fp32 neighbour found"
    out = t.clone()
    out[k] = float(hits[len(hits) // 2])
    return out


def gpu_model(bce=False):
    """A model whose only role is to host topk_links: every call below passes its embeddings (all_embed)."""
    return _model(bce=bce).cuda().eval()


# ---- 1. widths x k, bit exact ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
@pytest.mark.parametrize("dim", [64, 256, 396, 512, 298])
def test_bit_exact_sweep(dim, k):
    import literalkg_b200 as L
    from literalkg_b200 import ops
    n, nq = 40_000, 24
    emb, anchors = clustered(n, dim, nq, seed=dim + k)
    emb[500:510] = emb[7]                                      # exact duplicates: ties decided by position
    anchors[0] = 7                                             # the anchor scores its own duplicates
    # one-ulp neighbours and exact copies straddling the k-th score of query 1
    s1 = T.dot_of(emb[anchors[1:2]], emb)[0]
    kth = int(torch.sort(s1, descending=True, stable=True).indices[k - 1])
    spots = [p for p in range(1000, n, 997) if p not in (kth, int(anchors[1]))][:6]
    for p, sign in zip(spots[:4], (-1, +1, -1, +1)):
        emb[p] = dot_ulp_neighbour(emb[anchors[1]], emb[kth], sign)
    emb[spots[4]] = emb[kth]
    emb[spots[5]] = emb[kth]
    s = T.dot_of(emb[anchors], emb)
    assert int((s[1] == s[1, kth]).sum()) >= 3

    # ops level, every candidate (a width that is not a multiple of 4 padded by the caller)
    rows = emb if dim % 4 == 0 else pad4(emb)
    st = {}
    got = ops.score_topk_dot(rows, anchors, k, ops.ScoreIndex(rows, None), stats=st)
    assert_same(got, T.best_rows_of(s, k))
    assert int((st["listed"] > ops.TOPK_L2_CAP).sum()) <= 1 and float(st["listed"].float().mean()) < 0.2 * n

    # model level: a candidate subset, known triples excluded by entity id, with and without relations
    g = torch.Generator().manual_seed(k)
    sub = torch.randperm(n, generator=g)[:30_000].cuda()
    rels = torch.randint(0, 2, (nq,), generator=g).cuda()
    near = torch.sort(s[:, sub], dim=1, descending=True, stable=True).indices[:, :3 * k].cpu()
    kh, kr, kt = [], [], []
    for i in range(nq):
        ents = sub.cpu()[near[i, ::2]].tolist() + sub.cpu()[near[i, :4]].tolist()     # every other one, and duplicates
        ents += torch.randint(0, n, (20,), generator=g).tolist()                    # and arbitrary entities
        kh += [int(anchors[i])] * len(ents)
        kr += [int(rels[i])] * len(ents)
        kt += ents
    plan = L.GraphPlan(*(torch.tensor(x).cuda() for x in (kh, kt, kr)), n, 2)
    known = triples(kh, kr, kt)
    ss = s[:, sub]
    m = gpu_model()
    for with_rel in (True, False):
        if with_rel:
            excl = T.excluded_positions(anchors.tolist(), rels.tolist(), sub.tolist(), known)
        else:
            excl = T.excluded_any_relation(anchors.tolist(), sub.tolist(), known)
        want_v, want_p = T.best_rows_of(ss, k, excl.cuda())
        got_v, got_ids = m.topk_links(anchors, k, relations=rels if with_rel else None, known=plan, candidates=sub,
                                      all_embed=emb, batch_size=10)
        assert_same((got_v, got_ids), (want_v, torch.where(want_p >= 0, sub[want_p.clamp_min(0)], want_p)))


# ---- 2. exclusion ------------------------------------------------------------------------------------------------------
def test_exclusion_hub_non_candidates_duplicates_and_padding():
    import literalkg_b200 as L
    from literalkg_b200 import ops
    n, nq, k, dim = 40_000, 16, 50, 396
    emb, _ = clustered(n, dim, nq, seed=5)
    anchors = torch.arange(100, 100 + nq, device="cuda")
    s = T.dot_of(emb[anchors], emb)
    order = torch.sort(s[0], descending=True, stable=True).indices
    kh, kr, kt = [], [], []
    hub = order[:12_000].tolist()                              # anchor 100 knows its 12 000 best tails
    kt += hub + hub[:300]                                      # with duplicate triples
    kh += [100] * len(kt)
    kr += [0] * len(kt)
    sub = torch.arange(0, n, 2, device="cuda")                 # candidates: the even entities
    for i in range(1, nq):                                     # known tails, half of them not candidates
        near = torch.sort(s[i], descending=True, stable=True).indices[:2 * k].tolist()
        kt += near
        kh += [100 + i] * len(near)
        kr += [0] * len(near)
    kt += [5, 5, 7] + order[:k].tolist()                       # another relation's run
    kh += [101] * (3 + k)
    kr += [1] * (3 + k)
    plan = L.GraphPlan(*(torch.tensor(x).cuda() for x in (kh, kt, kr)), n, 2)
    known = triples(kh, kr, kt)
    assert int(plan.att_rowptr[101] - plan.att_rowptr[100]) > 10_000
    rels = torch.zeros(nq, dtype=torch.int64, device="cuda")
    for cids in (None, sub):
        ss = s if cids is None else s[:, cids]
        ids = list(range(n)) if cids is None else cids.tolist()
        index = ops.ScoreIndex(emb, cids)
        for r in (rels, None):
            if r is None:
                excl = T.excluded_any_relation(anchors.tolist(), ids, known)
            else:
                excl = T.excluded_positions(anchors.tolist(), r.tolist(), ids, known)
            st = {}
            got = ops.score_topk_dot(emb, anchors, k, index, exclude=(plan, anchors, r, cids), stats=st)
            assert_same(got, T.best_rows_of(ss, k, excl.cuda()))
    # fewer than k candidates left: padding.  50 candidates, 45 of them known for the anchor
    small = torch.arange(50, device="cuda")
    plan_s = L.GraphPlan(torch.full((45,), 7, device="cuda"), torch.arange(45, device="cuda"),
                         torch.zeros(45, dtype=torch.int64, device="cuda"), n, 1)
    vals, ids = gpu_model().topk_links(torch.tensor([7, 8], device="cuda"), 10, known=plan_s, candidates=small,
                                       all_embed=emb)
    assert bool((ids[0, 5:] == -1).all()) and bool((vals[0, 5:] == float("-inf")).all())
    assert sorted(ids[0, :5].tolist()) == list(range(45, 50))
    assert bool((ids[1] >= 0).all())                                   # anchor 8 knows nothing


# ---- 3. forced paths ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 100])
def test_overflow_and_weak_threshold_give_the_same_result(k):
    import literalkg_b200 as L
    from literalkg_b200 import ops
    n, nq = 30_000, 12
    emb, anchors = clustered(n, 396, nq, seed=k)
    s = T.dot_of(emb[anchors], emb)
    near = torch.sort(s, dim=1, descending=True, stable=True).indices[:, :k:3]
    kh = anchors[:, None].expand_as(near).reshape(-1)
    plan = L.GraphPlan(kh, near.reshape(-1).cuda(), torch.zeros_like(kh), n, 1)
    index = ops.ScoreIndex(emb, None)
    for exclude in (None, (plan, anchors, None, None)):
        st_o, st_w = {}, {}
        ref = ops.score_topk_dot(emb, anchors, k, index, exclude=exclude)
        over = ops.score_topk_dot(emb, anchors, k, index, exclude=exclude, cap=2 * k, stats=st_o)
        weak = ops.score_topk_dot(emb, anchors, k, index, exclude=exclude, n_sample=k, stats=st_w)
        assert bool((st_o["listed"] > 2 * k).all())                     # every query took the exact scan
        assert_same(over, ref)
        assert_same(weak, ref)
        assert bool((st_w["theta"] <= st_o["theta"]).all())             # k samples bound no better than the default
        excl = None
        if exclude is not None:
            excl = torch.zeros((nq, n), dtype=torch.bool, device="cuda")
            excl[torch.arange(nq, device="cuda")[:, None].expand_as(near).reshape(-1), near.reshape(-1)] = True
        assert_same(ref, T.best_rows_of(s, k, excl))


# ---- 4. agreement with the existing calls ------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 100])
def test_equals_score_topk_without_exclusion(k):
    from literalkg_b200 import ops
    n, nq = 60_000, 300
    emb, anchors = clustered(n, 256, nq, seed=11 + k)
    index = ops.ScoreIndex(emb, None)
    assert_same(ops.score_topk_dot(emb, anchors, k, index), ops.score_topk(emb, anchors, None, k, tail_index=index))
    cands = torch.randperm(n, generator=torch.Generator().manual_seed(k))[:40_000].cuda()
    sub = ops.ScoreIndex(emb, cands)
    assert_same(ops.score_topk_dot(emb, anchors, k, sub), ops.score_topk(emb, anchors, cands, k, tail_index=sub))


@pytest.mark.parametrize("with_rel", [False, True])
@pytest.mark.parametrize("predict", ["tail", "head"])
@pytest.mark.parametrize("bce", [False, True])
def test_consistent_with_evaluate_ranking(bce, predict, with_rel):
    from literalkg_b200 import ops
    m, known, triples_, (qh, qr, qt) = dot_model(bce=bce)
    emb = m.gat_embeddings()
    assert ops.fused_topk_applicable(m.n_entities, emb.shape[1], 1)    # evaluate_ranking takes its fused path
    anchors = qh if predict == "tail" else qt
    rels = qr if with_rel else None
    k = 10
    vals, ids = m.topk_links(anchors, k, relations=rels, known=known, predict=predict, batch_size=96, all_embed=emb)
    assert vals.shape == ids.shape == (anchors.numel(), k)
    assert bool((ids >= 0).all()) and bool((vals[:, 1:] <= vals[:, :-1]).all())
    for j in range(k):
        other = ids[:, j]
        h, t = (anchors, other) if predict == "tail" else (other, anchors)
        res = m.evaluate_ranking(h, t, rels, known=known, predict=predict, batch_size=128, all_embed=emb)
        assert torch.equal(res["ranks"].cpu(), torch.full((anchors.numel(),), j, dtype=torch.int64)), j
    # no known triple is returned
    got = {(a, r, e) for a, r, row in zip(anchors.tolist(), qr.tolist(), ids.tolist()) for e in row}
    kt = {(h, r, t) if predict == "tail" else (t, r, h) for h, r, t in triples_}
    if with_rel:
        assert not (got & kt)
    else:
        assert not ({(a, e) for a, _, e in got} & {(a, e) for a, _, e in kt})
    if not with_rel and predict == "tail":                             # raw: the ranks without known triples
        _, raw_ids = m.topk_links(anchors, k, all_embed=emb)
        for j in (0, k - 1):
            res = m.evaluate_ranking(anchors, raw_ids[:, j], all_embed=emb)
            assert torch.equal(res["ranks"].cpu(), torch.full((anchors.numel(),), j, dtype=torch.int64))


# ---- 5. the default width ----------------------------------------------------------------------------------------------
def test_default_width_model_level_and_errors():
    import literalkg_b200 as L
    n, n_rel = 6001, 4
    cfg = O.OracleConfig(n_conv_layers=3, mess_dropout=0.0, scale_gat_dim=None)
    kg = L.synthetic.make_kg(n, 40_000, n_rel, seed=2, max_out_degree=400)
    num, txt = L.synthetic.make_literals(n, seed=2)
    kt = L.KGTensors(kg.h, kg.t, kg.r, n_entities=n)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    torch.manual_seed(2)
    m = L.LiteralKG(args, n, n_rel, kt.A_in, num, txt).cuda().eval()
    with torch.no_grad():
        m.entity_embed.weight.mul_(30)
    known = L.GraphPlan(*(torch.from_numpy(x).cuda() for x in (kg.h, kg.t, kg.r)), n, n_rel)
    known_t = triples(kg.h, kg.r, kg.t)
    emb = m.gat_embeddings()
    assert emb.shape[1] == 396
    pick = np.random.default_rng(2).choice(kg.n_edges, 300, replace=False)
    qh, qr, qt = (torch.from_numpy(x[pick]).cuda() for x in (kg.h, kg.r, kg.t))
    for predict in ("tail", "head"):
        anchors = qh if predict == "tail" else qt
        vals, ids = m.topk_links(anchors, 20, relations=qr, known=known, predict=predict)   # its own embedding pass
        kn = known_t if predict == "tail" else [(t, r, h) for h, r, t in known_t]
        excl = T.excluded_positions(anchors.tolist(), qr.tolist(), list(range(n)), kn)
        assert_same((vals, ids), T.best_rows_of(T.dot_of(emb[anchors], emb), 20, excl.cuda()))
    # the refusals that need the model on its device
    a = qh[:4]
    with pytest.raises(ValueError, match="same length"):
        m.topk_links(a, 10, relations=qr[:3], known=known)
    with pytest.raises(ValueError, match="known plan has"):
        m.topk_links(a, 10, known=known, all_embed=emb[:-1])
    with pytest.raises(ValueError, match="no candidates"):
        m.topk_links(a, 10, candidates=[])
    with pytest.raises(ValueError, match="anchor ids outside"):
        m.topk_links(a + n, 10)
    with pytest.raises(ValueError, match="candidate ids outside"):
        m.topk_links(a, 10, candidates=[0, n])
    with pytest.raises(ValueError, match="duplicate candidate"):
        m.topk_links(a, 10, candidates=[0, 1, 0])
    with pytest.raises(ValueError, match="relation ids outside"):
        m.topk_links(a, 10, relations=qr[:4] + n_rel, known=known)


# ---- 6. two ranks sharing cuda:0 over gloo -----------------------------------------------------------------------------
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
    for predict, rels in (("tail", qr), ("head", None)):
        anchors = qh if predict == "tail" else qt
        vals, ids = m.topk_links(anchors, 20, relations=rels, known=known, batch_size=32, predict=predict)
        both = part.all_gather_stack(ids)
        assert torch.equal(both[0], both[1])
        results.append((anchors, rels, vals, ids))
    m.set_partition(None)
    for predict, (anchors, rels, vals, ids) in zip(("tail", "head"), results):
        one = m.topk_links(anchors, 20, relations=rels, known=known, batch_size=32, predict=predict, all_embed=full)
        assert torch.equal(one[1], ids) and torch.equal(one[0], vals)
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    torch.distributed.destroy_process_group()


def test_topk_links_row_partitioned_two_ranks():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_partitioned_worker, args=(2, port, d), nprocs=2, join=True)
        assert sorted(os.listdir(d)) == ["ok0", "ok1"]


# ---- 7. scale ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 100])
def test_scale_bit_exact(k):
    from literalkg_b200 import ops
    n, dim, nq = 262_144, 396, 512
    emb, anchors = clustered(n, dim, nq, seed=31)
    st = {}
    got = ops.score_topk_dot(emb, anchors, k, ops.ScoreIndex(emb, None), stats=st)
    want_v, want_p = [], []
    for c0 in range(0, nq, 8):                                          # the restatement, chunked on the GPU
        vv, pp = T.best_rows_of(T.dot_of(emb[anchors[c0:c0 + 8]], emb), k)
        want_v.append(vv)
        want_p.append(pp)
    assert_same(got, (torch.cat(want_v), torch.cat(want_p)))
    assert int((st["listed"] > ops.TOPK_L2_CAP).sum()) == 0
