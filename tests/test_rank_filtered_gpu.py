"""Filtered link-prediction ranks on the GPU (lkg_rank_filter / lkg_rank_filter_scores, ops.filter_ranks,
LiteralKG.evaluate_ranking) against the reference ``filtered_rank_of`` / ``ranking_metrics`` of tests/_rank_oracle.py.

Fused path: the raw rank of ops.score_rank and the filter re-score exactly (fp32 products summed in fp64, one rounding),
so the filtered ranks must equal the reference rule on float64 scores rounded once to fp32 -- bit exact.  Dense path: the
raw rank and the filter judge on the ops.score matrix, so the reference is applied to that same matrix."""
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


def exact_scores(emb, heads, cands):
    """float64 dot products rounded once to fp32 (the fused path's exact scores), on the host."""
    return (emb[heads].double() @ emb[cands].double().t()).float().cpu()


def triples(h, r, t):
    return list(zip(np.asarray(h).tolist(), np.asarray(r).tolist(), np.asarray(t).tolist()))


def make_case(n, dim, seed):
    """Embeddings with a tie group of identical rows, a synthetic known graph with hub heads (runs > 256 tails), extra
    known triples for the hub: members of the tie group, a duplicated triple, tails that are not candidates; a permuted
    candidate list without 40 entities; queries on the hub, the tie group, the heaviest heads and random known triples
    (every query's target is itself a known tail of its head)."""
    import literalkg_b200 as L
    g = torch.Generator(device="cuda").manual_seed(seed)
    emb = torch.nn.functional.leaky_relu(torch.randn(n, dim, generator=g, device="cuda"), 0.01) * 0.37
    emb[500:520] = emb[7]
    kg = L.synthetic.make_kg(n, 4 * n, 2, seed=seed, max_out_degree=700)
    rng = np.random.default_rng(seed)
    dropped = rng.choice(np.arange(1000, n), 40, replace=False)
    keep = np.ones(n, dtype=bool)
    keep[dropped] = False
    cands = torch.from_numpy(rng.permutation(np.nonzero(keep)[0])).cuda()
    deg = np.bincount(kg.h, minlength=n)
    hub = int(deg.argmax())
    ex_t = list(range(500, 512)) + [503, 503] + dropped[:5].tolist() + [515] + list(range(500, 520))
    ex_h = [hub] * 20 + [7] * 20
    ex_r = [0] * 40
    h = np.concatenate([kg.h, ex_h])
    r = np.concatenate([kg.r, ex_r])
    t = np.concatenate([kg.t, ex_t])
    run = np.bincount(h * 2 + r, minlength=2 * n).max()
    assert run > 256                                                   # some (h, r) run spans several warps' work
    qh, qr, qt = [hub, hub, 7, 7], [0, 1, 0, 0], [515, 515, 505, 519]
    for head in np.argsort(-deg)[:6]:                                  # the heaviest heads, one of their own tails
        i = int(np.nonzero((kg.h == head) & keep[kg.t])[0][0])
        qh.append(int(head)); qr.append(int(kg.r[i])); qt.append(int(kg.t[i]))
    for i in rng.choice(np.nonzero(keep[kg.t])[0], 150, replace=False):
        qh.append(int(kg.h[i])); qr.append(int(kg.r[i])); qt.append(int(kg.t[i]))
    plan = L.GraphPlan(*(torch.from_numpy(x).cuda() for x in (h, t, r)), n, 2)
    q = [torch.tensor(x, device="cuda") for x in (qh, qr, qt)]
    return emb, cands, plan, triples(h, r, t), q


def short_list(must, fill, size):
    """``size`` candidates: every id of ``must`` plus the first other ids of ``fill``, in a fixed permuted order."""
    base = torch.unique(must)
    out = torch.cat([base, fill[~torch.isin(fill, base)][:size - base.numel()]])
    assert out.numel() == size
    return out[torch.randperm(size, generator=torch.Generator().manual_seed(size)).cuda()]


def cand_map(cands, n):
    m = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    m[cands] = torch.arange(cands.numel(), dtype=torch.int32, device="cuda")
    return m


@pytest.mark.parametrize("n", [40_000, 70_001])
@pytest.mark.parametrize("dim", [256, 200, 64])
def test_fused_filter_bit_exact(n, dim):
    from literalkg_b200 import ops
    emb, cands, plan, known, (qh, qr, qt) = make_case(n, dim, seed=n + dim)
    cmap = cand_map(cands, n)
    tpos = cmap[qt].long()
    index = ops.ScoreIndex(emb, cands)
    s = exact_scores(emb, qh, cands)
    for rels in (qr, None):
        ref = R.filtered_rank_of(None, qh.cpu(), cands.cpu(), tpos.cpu(), known, None if rels is None else rels.cpu(),
                                 scores=s)
        for band_cap in (8192, 1):                                    # band_cap = 1: the exact-scan overflow path
            tau = torch.empty(qh.numel(), dtype=torch.float32, device="cuda")
            ranks = ops.score_rank(emb, qh, tpos, index, band_cap=band_cap, tau_out=tau)
            raw = ranks.clone()
            ops.filter_ranks(ranks, plan, qh, tpos, rels, cmap, emb=emb, tau=tau)
            assert torch.equal(ranks.cpu(), ref), (rels is None, band_cap)
            assert bool((ranks <= raw).all()) and bool((ranks < raw).any())
    # identity candidate list (no map): every entity
    index = ops.ScoreIndex(emb, None)
    tau = torch.empty(qh.numel(), dtype=torch.float32, device="cuda")
    ranks = ops.filter_ranks(ops.score_rank(emb, qh, qt, index, tau_out=tau), plan, qh, qt, qr, None, emb=emb, tau=tau)
    ref = R.filtered_rank_of(None, qh.cpu(), torch.arange(n), qt.cpu(), known, qr.cpu(),
                             scores=exact_scores(emb, qh, torch.arange(n, device="cuda")))
    assert torch.equal(ranks.cpu(), ref)


@pytest.mark.parametrize("dim,n_cands", [(396, None), (64, 118)])
def test_dense_filter_on_the_score_matrix(dim, n_cands):
    from literalkg_b200 import ops
    n = 40_000
    emb, cands, plan, known, (qh, qr, qt) = make_case(n, dim, seed=dim)
    if n_cands is not None:            # a short list: the targets of 40 queries, the tie group, then other entities
        qh, qr, qt = qh[:40], qr[:40], qt[:40]
        cands = short_list(torch.cat([qt, torch.arange(500, 520, device="cuda")]), cands, n_cands)
    cmap = cand_map(cands, n)
    tpos = cmap[qt].long()
    scores = ops.score(emb, qh, cands)
    for rels in (qr, None):
        ranks = ops.topk_rows(scores, 1, tpos)[2]
        raw = ranks.clone()
        ops.filter_ranks(ranks, plan, qh, tpos, rels, cmap, scores=scores)
        ref = R.filtered_rank_of(None, qh.cpu(), cands.cpu(), tpos.cpu(), known, None if rels is None else rels.cpu(),
                                 scores=scores.cpu())
        assert torch.equal(ranks.cpu(), ref)
        assert bool((ranks <= raw).all())


# ---- model level ---------------------------------------------------------------------------------------------------
def build_model(n=20_001, n_rel=4, seed=1, bce=False):
    """A model trained on nothing but built on a train split; the test split is 400 random triples; known = both."""
    import literalkg_b200 as L
    from literalkg_b200 import model_bce
    cfg = O.OracleConfig(n_conv_layers=1, mess_dropout=0.0)
    kg = L.synthetic.make_kg(n, 100_000, n_rel, seed=seed, max_out_degree=400)
    num, txt = L.synthetic.make_literals(n, seed=seed)
    rng = np.random.default_rng(seed)
    test = np.zeros(kg.n_edges, dtype=bool)
    test[rng.choice(kg.n_edges, 400, replace=False)] = True
    kt = L.KGTensors(kg.h[~test], kg.t[~test], kg.r[~test], n_entities=n)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    torch.manual_seed(0)
    m = (model_bce.LiteralKG if bce else L.LiteralKG)(args, n, n_rel, kt.A_in, num, txt).cuda().eval()
    with torch.no_grad():
        m.entity_embed.weight.mul_(30)
    known = L.GraphPlan(*(torch.from_numpy(x).cuda() for x in (kg.h, kg.t, kg.r)), n, n_rel)
    q = [torch.from_numpy(x[test]).cuda() for x in (kg.h, kg.r, kg.t)]
    return m, known, triples(kg.h, kg.r, kg.t), q


@pytest.mark.parametrize("bce", [False, True])
def test_evaluate_ranking_fused_path(bce):
    m, known, triples_, (qh, qr, qt) = build_model(bce=bce)
    n = m.n_entities
    emb = m.gat_embeddings()
    s = exact_scores(emb, qh, torch.arange(n, device="cuda"))
    raw = m.evaluate_ranking(qh, qt, batch_size=128)
    _, _, topk_ranks = m.topk(qh, torch.arange(n, device="cuda"), 10, target_tails=qt)
    assert torch.equal(raw["ranks"], topk_ranks)                     # known=None: the raw ranks of topk
    for rels in (qr, None):
        res = m.evaluate_ranking(qh, qt, rels, known=known, ks=(1, 3, 10, 100), batch_size=128)
        ref = R.filtered_rank_of(None, qh.cpu(), torch.arange(n), qt.cpu(), triples_,
                                 None if rels is None else rels.cpu(), scores=s)
        assert torch.equal(res["ranks"].cpu(), ref)
        assert bool((res["ranks"] <= raw["ranks"]).all()) and bool((res["ranks"] < raw["ranks"]).any())
        want = R.ranking_metrics(ref.numpy(), ks=(1, 3, 10, 100))
        assert res["n"] == qh.numel() and set(res) == set(want) | {"n", "ranks"}
        for key, v in want.items():
            assert isinstance(res[key], float) and res[key] == pytest.approx(v, rel=1e-12, abs=0), key


def test_evaluate_ranking_dense_path_and_errors():
    from literalkg_b200 import ops
    m, known, triples_, (qh, qr, qt) = build_model(seed=2)
    n = m.n_entities
    qh, qr, qt = qh[:50], qr[:50], qt[:50]
    cands = short_list(qt, torch.arange(n, device="cuda"), 118)
    emb = m.gat_embeddings()
    where = {int(c): p for p, c in enumerate(cands.tolist())}
    tpos = torch.tensor([where[int(t)] for t in qt.tolist()])
    scores = ops.score(emb, qh, cands).cpu()                         # what the dense path ranks on
    raw = m.evaluate_ranking(qh, qt, candidates=cands, batch_size=16)
    assert torch.equal(raw["ranks"].cpu(), R.filtered_rank_of(None, qh.cpu(), cands.cpu(), tpos, [], scores=scores))
    assert torch.equal(raw["ranks"], m.topk(qh, cands, 5, target_tails=tpos.cuda())[2])
    res = m.evaluate_ranking(qh, qt, qr, known=known, candidates=cands.tolist(), batch_size=16)
    ref = R.filtered_rank_of(None, qh.cpu(), cands.cpu(), tpos, triples_, qr.cpu(), scores=scores)
    assert torch.equal(res["ranks"].cpu(), ref)
    assert bool((res["ranks"] <= raw["ranks"]).all())
    # argument errors
    with pytest.raises(ValueError, match="not a candidate"):
        m.evaluate_ranking(qh, qt, candidates=cands[1:][cands[1:] != qt[0]])
    with pytest.raises(ValueError, match="duplicate"):
        m.evaluate_ranking(qh, qt, candidates=torch.cat([cands, cands[:1]]))
    with pytest.raises(ValueError, match="relation ids"):
        m.evaluate_ranking(qh, qt, qr + known.n_relations, known=known)
    with pytest.raises(ValueError, match="same length"):
        m.evaluate_ranking(qh, qt[:-1])
    with pytest.raises(ValueError, match="same length"):
        m.evaluate_ranking(qh, qt, qr[:-1], known=known)
    with pytest.raises(ValueError, match="outside"):
        m.evaluate_ranking(qh, qt + n)


# ---- two ranks sharing cuda:0 over gloo ------------------------------------------------------------------------------
def _partitioned_worker(rank, world, port, out_dir):
    W._init(rank, world, port, "gloo")
    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    RowPartition = W.staged_partition_cls()
    m, known, _, (qh, qr, qt) = build_model(seed=3)
    n = m.n_entities
    qh, qr, qt = qh[:301], qr[:301], qt[:301]                          # not a multiple of the world size
    part = RowPartition(n)
    m.set_partition(part)
    full = m.gat_embeddings()
    cands = torch.unique(torch.cat([qt, torch.arange(0, 1000, device="cuda")]))
    results = []
    for kw in (dict(relations=qr), dict(candidates=cands)):           # fused path (all entities); dense path
        res = m.evaluate_ranking(qh, qt, known=known, batch_size=64, **kw)       # a collective
        both = part.all_gather_stack(res["ranks"])
        assert torch.equal(both[0], both[1])
        mets = torch.tensor([res["mr"], res["mrr"], res["hits@1"], res["hits@10"]], dtype=torch.float64)
        allm = part.all_gather_stack(mets)
        assert torch.equal(allm[0], allm[1])
        results.append(res)
    m.set_partition(None)                                              # the same queries in one process
    for kw, res in zip((dict(relations=qr), dict(candidates=cands)), results):
        one = m.evaluate_ranking(qh, qt, known=known, batch_size=64, all_embed=full, **kw)
        assert torch.equal(one["ranks"], res["ranks"])
        assert all(one[k] == res[k] for k in ("mr", "mrr", "hits@1", "hits@3", "hits@10"))
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    torch.distributed.destroy_process_group()


def test_evaluate_ranking_row_partitioned_two_ranks():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_partitioned_worker, args=(2, port, d), nprocs=2, join=True)
        assert sorted(os.listdir(d)) == ["ok0", "ok1"]
