"""Ranking by the triple score on the GPU (ops.L2Index / ops.score_rank_l2 / ops.filter_ranks_l2,
LiteralKG.evaluate_ranking(score="triple", predict=...), GraphPlan.reversed) against the reference restatement
``filtered_rank_of`` on s = -d.

The declared arithmetic: the projected rows q and p_j are the fp32 results of the projection GEMM, and d = |q - p_j|^2
is exact on them (fp64 differences and squares, one rounding to fp32).  So the ranks must equal the restatement on the
same fp32 tables bit for bit; against float64 projections they agree wherever the margin exceeds the projection
tolerance."""
import argparse
import os
import socket
import tempfile

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import _parallel_worker as W
import _rank_oracle as R
import literalkg_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _inference_mode():
    with torch.no_grad():
        yield


def neg_dist(query, cand):
    """-d with d = |q - p_j|^2: differences and squares in float64, summed, rounded once to fp32; [B, Nc] on the host
    (one query at a time on the device)."""
    cand = cand.double()
    return torch.stack([-((cand - q.double()) ** 2).sum(1).float() for q in query]).cpu()


def raw_rank(s, tpos):
    """#{ j : s_j > s_t or (s_j == s_t and j < t) } per row of s."""
    out = []
    for i, tp in enumerate(tpos.tolist()):
        row, st = s[i], s[i, tp]
        out.append(int(((row > st) | ((row == st) & (torch.arange(row.numel()) < tp))).sum()))
    return torch.tensor(out, dtype=torch.int64)


def triples(h, r, t):
    return list(zip(np.asarray(h).tolist(), np.asarray(r).tolist(), np.asarray(t).tolist()))


def project(emb, rows, w, bias=None):
    """The projection the triple score runs: emb[rows] @ w (+ bias) on the library's GEMM (fp32 out)."""
    from literalkg_b200 import ops
    return ops.linear([ops.split_planes(emb, rows)], w.t(), bias)


def padded(x):
    d4 = (x.shape[1] + 3) // 4 * 4
    if d4 == x.shape[1]:
        return x.contiguous()
    out = torch.zeros((x.shape[0], d4), dtype=torch.float32, device=x.device)
    out[:, :x.shape[1]] = x
    return out


# ---- 0. the reversed plan ----------------------------------------------------------------------------------------------
def test_reversed_plan_equals_the_plan_of_the_swapped_triples():
    import literalkg_b200 as L
    n = 5000
    kg = L.synthetic.make_kg(n, 40_000, 3, seed=4, max_out_degree=600)
    h, t, r = (torch.from_numpy(x).cuda() for x in (kg.h, kg.t, kg.r))
    plan = L.GraphPlan(h, t, r, n, 3)
    rev = plan.reversed()
    assert plan.reversed() is rev                                        # cached on the plan
    ref = L.GraphPlan(t, h, r, n, 3)
    for name in ("att_rowptr", "att_tail", "att_rel", "att_seg", "rowptr", "col", "indices"):
        assert torch.equal(getattr(rev, name), getattr(ref, name)), name
    assert (rev.n_edges, rev.nnz, rev.n_relations) == (ref.n_edges, ref.nnz, ref.n_relations)


# ---- 1. projection -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [256, 396])
@pytest.mark.parametrize("d_s", [300, 64])
def test_projection_against_float64(width, d_s):
    g = torch.Generator(device="cuda").manual_seed(width + d_s)
    emb = torch.randn(30_000, width, generator=g, device="cuda") * 0.3
    w = torch.randn(width, d_s, generator=g, device="cuda") / width ** 0.5
    e_r = torch.randn(d_s, generator=g, device="cuda")
    rows = torch.randint(0, 30_000, (3000,), generator=g, device="cuda")
    for bias, sel in ((None, None), (e_r, rows), (-e_r, rows)):
        got = project(emb, sel, w, bias)
        x = emb.double() if sel is None else emb[sel].double()
        ref = x @ w.double() + (0 if bias is None else bias.double())
        assert float((got.double() - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


# ---- 2. raw ranks, ops level -------------------------------------------------------------------------------------------
def ulp_neighbour(q, p, sign):
    """A copy of row p whose fp32 distance to q is one fp32 ulp above (sign +1) or below (-1) that of p: the coordinate
    k with the largest |q_k - p_k| is stepped through consecutive fp32 values away from / towards q_k, and the middle of
    the run of values that land on the neighbouring fp32 distance is taken."""
    q64, p32 = q.double().cpu().numpy(), p.cpu().numpy().astype(np.float32)
    diff = q64 - p32.astype(np.float64)
    k = int(np.argmax(np.abs(diff)))
    rest = float(np.sum(np.delete(diff, k) ** 2))
    d0 = np.float32(rest + diff[k] ** 2)
    goal = np.nextafter(d0, np.float32(np.inf if sign > 0 else -np.inf))
    away = np.sign(p32[k] - q64[k]) * sign            # direction of p_k that moves the distance the right way
    x = p32[k]
    hits = []
    for _ in range(200_000):
        x = np.nextafter(x, np.float32(np.inf if away > 0 else -np.inf))
        d = np.float32(rest + (q64[k] - np.float64(x)) ** 2)
        if d == goal:
            hits.append(x)
        elif hits:
            break
    assert hits, "no fp32 neighbour found"
    out = p.clone()
    out[k] = float(hits[len(hits) // 2])
    return out


@pytest.mark.parametrize("d_s", [300, 256, 508, 64])
def test_raw_ranks_bit_exact(d_s):
    from literalkg_b200 import ops
    n, nq = 40_000, 48
    g = torch.Generator(device="cuda").manual_seed(d_s)
    base = torch.randn(1, d_s, generator=g, device="cuda") * 2.0          # rows clustered off the origin
    cand = base + torch.nn.functional.leaky_relu(torch.randn(n, d_s, generator=g, device="cuda"), 0.05)
    query = base + torch.randn(nq, d_s, generator=g, device="cuda") * 0.8
    tpos = torch.randint(100, n - 100, (nq,), generator=g, device="cuda")
    cand[500:510] = cand[7]                                               # exact duplicates: ties decided by position
    tpos[0], tpos[1] = 505, 7
    # the target of queries 2 and 3 with one-ulp neighbours before and after it
    for i in (2, 3):
        t = int(tpos[i])
        for off, sign in ((-40, -1), (-30, +1), (30, -1), (40, +1)):
            cand[t + off] = ulp_neighbour(query[i], cand[t], sign)
        cand[t - 20] = cand[t]                                            # an exact tie before
        cand[t + 20] = cand[t]                                            # and after
    s = neg_dist(query, cand)
    for i in (2, 3):                                                      # the neighbours really are one ulp away
        t = int(tpos[i])
        st = s[i, t]
        for off, sign in ((-40, -1), (-30, +1), (30, -1), (40, +1)):
            assert s[i, t + off] == np.nextafter(st.numpy(), np.inf if sign < 0 else -np.inf)
    ref = raw_rank(s, tpos.cpu())
    index = ops.L2Index(cand)
    for band_cap in (8192, 1):                                            # 1: every query takes the exact scan
        tau, st = torch.empty(nq, dtype=torch.float32, device="cuda"), {}
        ranks = ops.score_rank_l2(index, query, tpos, band_cap=band_cap, tau_out=tau, stats=st)
        assert torch.equal(ranks.cpu(), ref), band_cap
        assert torch.equal(-tau.cpu(), s[torch.arange(nq), tpos.cpu()])   # tau = the exact target distance
        if band_cap == 1:                          # the target always lies in its own band; 2 and 3 overflow it
            assert bool((st["band"] >= 1).all()) and bool((st["band"][2:4] > 1).all())
    assert float(st["band"].float().mean()) < 0.01 * n                   # the band is narrow: the GEMM decides


# ---- 3. filtered ranks on the model's path, bit exact --------------------------------------------------------------------
def transr_model(n, n_rel, width, d_s, seed):
    """A TransR model whose triple-score parameters (gat_trans_M [R, width, d_s], relation_embed [R, d_s]) are seeded
    directly: evaluate_ranking is then called on given embeddings of that width."""
    import literalkg_b200 as L
    cfg = O.OracleConfig(n_conv_layers=1, mess_dropout=0.0, use_num_lit=False, use_txt_lit=False)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    m = L.LiteralKG(args, n, n_rel).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(seed)
    m.gat_trans_M = torch.nn.Parameter(torch.randn(n_rel, width, d_s, generator=g, device="cuda") / width ** 0.5)
    m.relation_embed = torch.nn.Embedding(n_rel, d_s).cuda()
    m.relation_embed.weight.copy_(torch.randn(n_rel, d_s, generator=g, device="cuda") * 0.5)
    return m


def filtered_case(n, seed):
    """Known triples with a hub (thousands of tails under one relation), duplicate triples, known tails that are not
    candidates; queries on the hub, the heaviest heads and random known triples (so the target itself is known)."""
    import literalkg_b200 as L
    kg = L.synthetic.make_kg(n, 4 * n, 2, seed=seed, max_out_degree=3000)
    rng = np.random.default_rng(seed)
    deg = np.bincount(kg.h, minlength=n)
    hub = int(deg.argmax())
    ex_t = [11, 12, 12, 13, 14, 15, 15, 15, 16, 17, 18, 19] + list(range(20, 2520))
    ex_h, ex_r = [hub] * len(ex_t), [0] * len(ex_t)
    h, r, t = (np.concatenate([a, b]) for a, b in ((kg.h, ex_h), (kg.r, ex_r), (kg.t, ex_t)))
    assert np.bincount(h * 2 + r, minlength=2 * n).max() > 2500
    pick = rng.choice(h.size, 150, replace=False)
    on_hub = np.nonzero((h == hub) & (r == 0))[0][:10]
    q = np.concatenate([on_hub, pick])
    plan = L.GraphPlan(*(torch.from_numpy(x).cuda() for x in (h, t, r)), n, 2)
    return plan, triples(h, r, t), [torch.from_numpy(x[q]).cuda() for x in (h, r, t)]


def mirror_tables(m, emb, anchors, rels, cands, sign):
    """The fp32 tables the model's path builds: per relation P_r = emb[cands] M_r and the queries of that relation
    projected together (one batch: batch_size covers them), so -d on them is what the ranks were counted on."""
    w = m.gat_trans_M.detach()
    e = m.relation_embed.weight.detach()
    s = torch.empty((anchors.numel(), cands.numel()), dtype=torch.float32)
    for r in torch.unique(rels).tolist():
        sel = torch.nonzero(rels == r).reshape(-1)
        p = padded(project(emb, cands, w[r]))
        q = padded(project(emb, anchors[sel], w[r], sign * e[r]))
        s[sel.cpu()] = neg_dist(q, p)
    return s


@pytest.mark.parametrize("n_cands", [None, 118])
@pytest.mark.parametrize("predict", ["tail", "head"])
def test_filtered_ranks_bit_exact(predict, n_cands):
    n, width, d_s = 40_000, 256, 300
    m = transr_model(n, 2, width, d_s, seed=11)
    plan, known, (qh, qr, qt) = filtered_case(n, seed=12)
    g = torch.Generator(device="cuda").manual_seed(13)
    emb = torch.nn.functional.leaky_relu(torch.randn(n, width, generator=g, device="cuda"), 0.01) * 0.5
    if n_cands is not None:                                            # 10 hub queries + 30 others
        qh, qr, qt = qh[:40], qr[:40], qt[:40]
    anchors, targets = (qh, qt) if predict == "tail" else (qt, qh)
    if n_cands is None:
        cands = torch.arange(n, device="cuda")
    else:          # the targets, some known tails of the hub, then other entities; not every known entity is a candidate
        must = torch.unique(torch.cat([targets, torch.arange(11, 16, device="cuda")]))
        rest = torch.randperm(n, generator=torch.Generator().manual_seed(1)).cuda()
        rest = rest[~torch.isin(rest, must)][:n_cands - must.numel()]
        cands = torch.cat([must, rest])[torch.randperm(n_cands, generator=torch.Generator().manual_seed(2)).cuda()]
    where = {int(c): p for p, c in enumerate(cands.tolist())}
    tpos = torch.tensor([where[int(x)] for x in targets.tolist()])
    s = mirror_tables(m, emb, anchors, qr, cands, 1.0 if predict == "tail" else -1.0)
    kn = known if predict == "tail" else [(t, r, h) for h, r, t in known]
    ref = R.filtered_rank_of(None, anchors.cpu(), cands.cpu(), tpos, kn, qr.cpu(), scores=s)
    kw = dict(all_embed=emb, score="triple", predict=predict, batch_size=4096,
              candidates=None if n_cands is None else cands)
    res = m.evaluate_ranking(qh, qt, qr, known=plan, **kw)
    raw = m.evaluate_ranking(qh, qt, qr, **kw)
    assert torch.equal(raw["ranks"].cpu(), raw_rank(s, tpos))
    assert torch.equal(res["ranks"].cpu(), ref)
    assert bool((res["ranks"] <= raw["ranks"]).all()) and bool((res["ranks"] < raw["ranks"]).any())


# ---- 4. the distance is the loss's -------------------------------------------------------------------------------------
@pytest.mark.parametrize("bce", [False, True])
def test_distance_equals_the_loss_term(bce):
    from literalkg_b200 import ops
    n, width, d_s = 20_000, 256, (256 if bce else 300)
    g = torch.Generator(device="cuda").manual_seed(21)
    emb = torch.randn(n, width, generator=g, device="cuda") * 0.4
    w = torch.randn(4, width, d_s, generator=g, device="cuda") / width ** 0.5
    e = torch.randn(4, d_s, generator=g, device="cuda") * 0.3
    h, r, t = (torch.randint(0, hi, (300,), generator=g, device="cuda") for hi in (n, 4, n))
    for rel in range(4):
        sel = torch.nonzero(r == rel).reshape(-1)
        if bce:
            p, q = emb, emb[h[sel]] + e[rel]
        else:
            p, q = project(emb, None, w[rel]), project(emb, h[sel], w[rel], e[rel])
        tau = torch.empty(sel.numel(), dtype=torch.float32, device="cuda")
        ops.score_rank_l2(ops.L2Index(padded(p)), padded(q), t[sel], tau_out=tau)
        # the per-triple term of oracle.triplet_loss / oracle.transe_loss, float64 on the same embeddings
        if bce:
            ref = ((emb[h[sel]].double() + e[rel].double() - emb[t[sel]].double()) ** 2).sum(1)
        else:
            wr = w[rel].double()
            ref = ((emb[h[sel]].double() @ wr + e[rel].double() - emb[t[sel]].double() @ wr) ** 2).sum(1)
        assert float(((tau.double() - ref).abs() / ref).max()) <= 1e-5


# ---- 5. model level ----------------------------------------------------------------------------------------------------
def build_model(n=6001, n_rel=4, seed=1, bce=False):
    import literalkg_b200 as L
    from literalkg_b200 import model_bce
    cfg = O.OracleConfig(n_conv_layers=1, mess_dropout=0.0, relation_dim=256 if bce else 300)
    kg = L.synthetic.make_kg(n, 40_000, n_rel, seed=seed, max_out_degree=400)
    num, txt = L.synthetic.make_literals(n, seed=seed)
    rng = np.random.default_rng(seed)
    test = np.zeros(kg.n_edges, dtype=bool)
    test[rng.choice(kg.n_edges, 200, replace=False)] = True
    kt = L.KGTensors(kg.h[~test], kg.t[~test], kg.r[~test], n_entities=n)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    torch.manual_seed(seed)
    m = (model_bce.LiteralKG if bce else L.LiteralKG)(args, n, n_rel, kt.A_in, num, txt).cuda().eval()
    with torch.no_grad():
        m.entity_embed.weight.mul_(30)
    known = L.GraphPlan(*(torch.from_numpy(x).cuda() for x in (kg.h, kg.t, kg.r)), n, n_rel)
    q = [torch.from_numpy(x[test]).cuda() for x in (kg.h, kg.r, kg.t)]
    return m, known, triples(kg.h, kg.r, kg.t), q


@pytest.mark.parametrize("predict", ["tail", "head"])
@pytest.mark.parametrize("bce", [False, True])
def test_evaluate_ranking_triple_model_level(bce, predict):
    m, known, triples_, (qh, qr, qt) = build_model(bce=bce)
    n = m.n_entities
    emb = m.gat_embeddings()
    anchors, targets = (qh, qt) if predict == "tail" else (qt, qh)
    sign = 1.0 if predict == "tail" else -1.0
    must = torch.unique(targets)[:100]
    rest = torch.arange(n, device="cuda")
    cands = torch.cat([must, rest[~torch.isin(rest, must)][:118 - must.numel()]])
    keep = torch.isin(targets, cands)
    qh, qr, qt, anchors, targets = qh[keep], qr[keep], qt[keep], anchors[keep], targets[keep]
    where = {int(c): p for p, c in enumerate(cands.tolist())}
    tpos = torch.tensor([where[int(x)] for x in targets.tolist()])
    # float64 restatement: q = emb[anchor] M_r + sign e_r, p_j = emb[j] M_r (TransE: M_r = I); and the same on the fp32
    # rows the call projects (each relation's queries in one batch: batch_size covers them)
    e64, e32 = m.relation_embed.weight.double(), m.relation_embed.weight.detach()
    s64 = torch.empty((anchors.numel(), cands.numel()), dtype=torch.float64)
    s32 = torch.empty((anchors.numel(), cands.numel()), dtype=torch.float32)
    for r in torch.unique(qr).tolist():
        sel = torch.nonzero(qr == r).reshape(-1)
        if bce:
            p64, q64 = emb[cands].double(), emb[anchors[sel]].double()
            p32, q32 = emb[cands], emb[anchors[sel]] + sign * e32[r]
        else:
            w = m.gat_trans_M[r].detach()
            p64, q64 = emb[cands].double() @ w.double(), emb[anchors[sel]].double() @ w.double()
            p32, q32 = padded(project(emb, cands, w)), padded(project(emb, anchors[sel], w, sign * e32[r]))
        q64 = q64 + sign * e64[r]
        s64[sel.cpu()] = torch.stack([-((p64 - q) ** 2).sum(1) for q in q64]).cpu()
        s32[sel.cpu()] = neg_dist(q32, p32)
    kn = triples_ if predict == "tail" else [(t, r, h) for h, r, t in triples_]
    res = m.evaluate_ranking(qh, qt, qr, known=known, candidates=cands, score="triple", predict=predict,
                             batch_size=4096)
    # bit exact on the rows the call projected
    assert torch.equal(res["ranks"].cpu(), R.filtered_rank_of(None, anchors.cpu(), cands.cpu(), tpos, kn, qr.cpu(),
                                                              scores=s32))
    # and the float64 order decides wherever the target's gap to its nearest competitor exceeds twice what the fp32
    # projection moved any distance of the query (the measured projection tolerance, plus one ulp of the target's)
    rows = torch.arange(s64.shape[0])
    st = s64[rows, tpos]
    tol = (s32.double() - s64).abs().max(1).values + st.abs() * 2.0 ** -23
    gap = (s64 - st[:, None]).abs()
    gap[rows, tpos] = float("inf")
    clear = gap.min(1).values > 2 * tol
    assert float(clear.double().mean()) > 0.8
    ref = R.filtered_rank_of(None, anchors.cpu(), cands.cpu(), tpos, kn, qr.cpu(), scores=s64)
    assert torch.equal(res["ranks"].cpu()[clear], ref[clear])
    want = R.ranking_metrics(res["ranks"].cpu().numpy())
    for key, v in want.items():
        assert res[key] == pytest.approx(v, rel=1e-12, abs=0), key
    # every entity a candidate: the metrics are those of the returned ranks, and filtering only lowers ranks
    full = m.evaluate_ranking(qh, qt, qr, known=known, score="triple", predict=predict)
    raw = m.evaluate_ranking(qh, qt, qr, score="triple", predict=predict)
    assert bool((full["ranks"] <= raw["ranks"]).all())
    for key, v in R.ranking_metrics(full["ranks"].cpu().numpy()).items():
        assert full[key] == pytest.approx(v, rel=1e-12, abs=0), key
    with pytest.raises(ValueError, match="of the model"):
        m.evaluate_ranking(qh, qt, qr + m.n_relations, score="triple")
    with pytest.raises(ValueError, match="of the model"):
        m.evaluate_ranking(qh, qt, qr - 1 - qr, known=known, score="triple", predict=predict)


# ---- 6. head prediction of the dot score -------------------------------------------------------------------------------
def test_dot_head_prediction_is_the_swapped_call():
    m, known, _, (qh, qr, qt) = build_model(seed=2)
    emb = m.gat_embeddings()
    for kw in (dict(relations=qr), dict()):
        head = m.evaluate_ranking(qh, qt, known=known, predict="head", all_embed=emb, **kw)
        swapped = m.evaluate_ranking(qt, qh, known=known.reversed(), all_embed=emb, **kw)
        assert torch.equal(head["ranks"], swapped["ranks"])
        assert all(head[k] == swapped[k] for k in ("mr", "mrr", "hits@1", "hits@3", "hits@10"))


# ---- 7. two ranks sharing cuda:0 over gloo -----------------------------------------------------------------------------
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
        res = m.evaluate_ranking(qh, qt, qr, known=known, batch_size=32, score="triple", predict=predict)
        both = part.all_gather_stack(res["ranks"])
        assert torch.equal(both[0], both[1])
        results.append(res)
    m.set_partition(None)
    for predict, res in zip(("tail", "head"), results):
        one = m.evaluate_ranking(qh, qt, qr, known=known, batch_size=32, all_embed=full, score="triple",
                                 predict=predict)
        assert torch.equal(one["ranks"], res["ranks"])
        assert all(one[k] == res[k] for k in ("mr", "mrr", "hits@1", "hits@3", "hits@10"))
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    torch.distributed.destroy_process_group()


def test_evaluate_ranking_triple_row_partitioned_two_ranks():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_partitioned_worker, args=(2, port, d), nprocs=2, join=True)
        assert sorted(os.listdir(d)) == ["ok0", "ok1"]
