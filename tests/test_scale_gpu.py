"""CUDA path vs the CPU oracle on seeded synthetic graphs at sizes the oracle finishes in seconds, with the
reference's default dimensions (D = 300, C = 32, G = 256), plus size-independent properties."""
import argparse

import numpy as np
import pytest
import torch

import literalkg_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _inference_mode():
    """The parity tests exercise the inference path; with grad enabled gat_embeddings() takes the training path
    (same kernels + saved activations), which tests/test_backward_gpu.py covers."""
    with torch.no_grad():
        yield
REL = 1e-3


def rel_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def build(cfg, n, e, n_rel, seed=2022):
    import literalkg_b200 as L
    kg = L.synthetic.make_kg(n, e, n_rel, seed=seed, max_out_degree=300)
    num, txt = L.synthetic.make_literals(n, cfg.num_lit_dim, cfg.txt_lit_dim, seed=seed)
    p = O.init_params(cfg, n, n_rel, seed=seed)
    # larger-than-xavier embeddings so that tanh / softmax are exercised away from the linear regime
    p["entity_embed.weight"] = p["entity_embed.weight"] * 40
    p["relation_embed.weight"] = p["relation_embed.weight"] * 10
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    kt = L.KGTensors(kg.h, kg.t, kg.r, n_entities=n)
    m = L.LiteralKG(args, n, n_rel, kt.A_in, num if cfg.use_num_lit else None, txt if cfg.use_txt_lit else None)
    m.load_state_dict(p, strict=False)
    return kg, num, txt, p, kt, m.cuda().eval()


@pytest.mark.parametrize("agg,res", [("bi-interaction", True), ("gcn", True), ("graphsage", True),
                                     ("bi-interaction", False), ("graphsage", False)])
def test_default_dims_vs_oracle(agg, res):
    cfg = O.OracleConfig(aggregation_type=agg, use_residual=res, n_conv_layers=3, mess_dropout=0.0)
    n, e, n_rel = 6000, 60000, 16
    kg, num, txt, p, kt, m = build(cfg, n, e, n_rel)
    h, t, r = (torch.from_numpy(x) for x in (kg.h, kg.t, kg.r))
    # initial Laplacian: bit exact vs the scipy restatement
    li, lv = O.laplacian_A_in(kg.h, kg.t, kg.r, n)
    assert np.array_equal(kt.A_in.indices().cpu().numpy(), li)
    assert np.array_equal(kt.A_in.values().cpu().numpy(), lv)
    # attention update
    m(kt.h_list, kt.t_list, kt.r_list, kt.relations, device="cuda", mode="update_att")
    oi, ov = O.update_attention(p["entity_embed.weight"], p["relation_embed.weight"], h, t, r, kt.relations, n)
    a = m.A_in.data
    assert np.array_equal(a.indices().cpu().numpy(), oi.numpy())
    assert rel_err(a.values(), ov) < REL
    assert oi.shape[1] < kg.n_edges                       # the duplicate-merge path was exercised
    # full embedding pass: the yardstick is the oracle evaluated in FLOAT64 (two fp32 evaluations of the same formula
    # already differ by up to 5e-4 for graphsage + residual, so "within 1e-3 of an fp32 oracle" would not bound the
    # distance to the reference); the oracle's own fp32 evaluation is measured against it beside ours
    out = m.gat_embeddings()
    ref, st = O.gat_embeddings(p, cfg, oi, ov, num if cfg.use_num_lit else None, txt if cfg.use_txt_lit else None,
                               return_stages=True)
    p64 = O.cast_params(p, torch.float64)
    oi64, ov64 = O.update_attention(p64["entity_embed.weight"], p64["relation_embed.weight"], h, t, r, kt.relations, n)
    ref64 = O.gat_embeddings(p64, cfg, oi64, ov64, num.double() if cfg.use_num_lit else None,
                             txt.double() if cfg.use_txt_lit else None)
    e_cuda, e_fp32 = rel_err(out, ref64), rel_err(ref, ref64)
    big = ref64.abs() > 0.1 * ref64.abs().max()                 # element-wise on the top decade of magnitudes
    el_cuda = ((out.cpu().double() - ref64).abs()[big] / ref64.abs()[big]).max().item()
    el_fp32 = ((ref.double() - ref64).abs()[big] / ref64.abs()[big]).max().item()
    print(f"{agg} residual={res}: CUDA vs fp64 {e_cuda:.2e} (element-wise {el_cuda:.2e}); fp32 oracle vs fp64 {e_fp32:.2e} "
          f"(element-wise {el_fp32:.2e})")
    assert rel_err(a.values(), ov64) < REL
    assert e_cuda < REL and el_cuda < 5 * REL
    assert rel_err(out, ref) < REL
    # scoring + top-k against torch.topk of the oracle's calc_score (near-ties excluded by margin)
    heads = torch.arange(0, 64) * 7 % n
    tails = torch.arange(n)
    s = m.calc_score(heads.cuda(), tails.cuda())
    sref = O.calc_score(ref, heads, tails)
    assert rel_err(s, sref) < REL
    vals, pos, _ = m.topk(heads.cuda(), tails.cuda(), 10)
    tv, tp = torch.topk(sref, 11, dim=1)
    gap = (tv[:, :-1] - tv[:, 1:]).min(dim=1).values          # rows whose top-11 are separated by > 1e-4 rel
    clear = gap > 1e-4 * sref.abs().max()
    assert clear.sum() > 10
    assert torch.equal(pos.cpu()[clear], tp[:, :10][clear])


# widths other than the default reach other aggregation kernels: bi-interaction + residual takes layer 1's pre-projected
# z path only where that kernel runs (at 128 / 32 the one-slot stream instance; not at 128 / 48, 256 / 48 or 300 / 64:
# there the generic kernel combines side @ Pb), gcn / graphsage run layer 1 on the z table at d_out = 64 / 16
@pytest.mark.parametrize("agg,res,d,c", [("bi-interaction", True, 128, 32), ("bi-interaction", True, 128, 48),
                                         ("bi-interaction", True, 256, 48),
                                         ("bi-interaction", True, 300, 64), ("gcn", True, 300, 64),
                                         ("graphsage", True, 256, 16), ("bi-interaction", False, 300, 64)])
def test_other_dims_vs_oracle(agg, res, d, c):
    cfg = O.OracleConfig(aggregation_type=agg, use_residual=res, n_conv_layers=2, mess_dropout=0.0, embed_dim=d,
                         relation_dim=d, conv_dim=c)
    n, e, n_rel = 4000, 40000, 8
    kg, num, txt, p, kt, m = build(cfg, n, e, n_rel)
    h, t, r = (torch.from_numpy(x) for x in (kg.h, kg.t, kg.r))
    m(kt.h_list, kt.t_list, kt.r_list, kt.relations, device="cuda", mode="update_att")
    out = m.gat_embeddings()
    p64 = O.cast_params(p, torch.float64)
    oi64, ov64 = O.update_attention(p64["entity_embed.weight"], p64["relation_embed.weight"], h, t, r, kt.relations, n)
    assert np.array_equal(m.A_in.data.indices().cpu().numpy(), oi64.numpy())
    assert rel_err(m.A_in.data.values(), ov64) < REL
    ref64 = O.gat_embeddings(p64, cfg, oi64, ov64, num.double(), txt.double())
    big = ref64.abs() > 0.1 * ref64.abs().max()
    el = ((out.cpu().double() - ref64).abs()[big] / ref64.abs()[big]).max().item()
    print(f"{agg} residual={res} D={d} C={c}: CUDA vs fp64 {rel_err(out, ref64):.2e} (element-wise {el:.2e})")
    assert rel_err(out, ref64) < REL and el < 5 * REL


@pytest.mark.parametrize("agg", ["bi-interaction", "gcn"])
def test_heavy_rows_vs_oracle(agg):
    """Head rows with thousands of neighbours (longer than every per-warp staging limit: shared-memory logit slots,
    solo-scheduled rows of the narrow kernel, many ring refills) next to empty and single-neighbour rows."""
    import literalkg_b200 as L
    cfg = O.OracleConfig(aggregation_type=agg, use_residual=True, n_conv_layers=2, mess_dropout=0.0)
    n, n_rel = 5000, 6
    rng = np.random.default_rng(5)
    hubs = np.array([3, 77, 4100, 4999])
    h = np.concatenate([np.repeat(hubs, [3500, 2100, 700, 300]), rng.integers(0, n, 9000)])
    t = rng.integers(0, n, h.shape[0])
    r = rng.integers(0, n_rel, h.shape[0])
    r[:n_rel] = np.arange(n_rel)
    key = np.unique((h * n + t) * n_rel + r)
    rng.shuffle(key)
    h, t, r = key // (n * n_rel), (key // n_rel) % n, key % n_rel
    num, txt = L.synthetic.make_literals(n, seed=5)
    p = O.init_params(cfg, n, n_rel, seed=5)
    p["entity_embed.weight"] = p["entity_embed.weight"] * 40
    p["relation_embed.weight"] = p["relation_embed.weight"] * 10
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    kt = L.KGTensors(h, t, r, n_entities=n)
    m = L.LiteralKG(args, n, n_rel, kt.A_in, num, txt)
    m.load_state_dict(p, strict=False)
    m = m.cuda().eval()
    m(kt.h_list, kt.t_list, kt.r_list, kt.relations, device="cuda", mode="update_att")
    ht, tt, rt = (torch.from_numpy(x) for x in (h, t, r))
    oi, ov = O.update_attention(p["entity_embed.weight"], p["relation_embed.weight"], ht, tt, rt, kt.relations, n)
    a = m.A_in.data
    assert np.array_equal(a.indices().cpu().numpy(), oi.numpy())
    assert rel_err(a.values(), ov) < REL
    ref = O.gat_embeddings(p, cfg, oi, ov, num, txt)
    assert rel_err(m.gat_embeddings(), ref) < REL


def test_attention_properties_large():
    """Size-independent properties at a size the oracle is not run on: rows sum to 1, values in (0, 1],
    structure equals the sorted unique (h, t) list, result invariant to the input edge order."""
    import literalkg_b200 as L
    n, e, n_rel, d = 200_000, 3_000_000, 64, 300
    kg = L.synthetic.make_kg(n, e, n_rel, seed=7)
    g = torch.Generator().manual_seed(1)
    ent = (torch.randn(n, d, generator=g) * 0.3).cuda()
    rel = (torch.randn(n_rel, d, generator=g) * 0.3).cuda()
    h, t, r = (torch.from_numpy(x).cuda() for x in (kg.h, kg.t, kg.r))
    plan = L.GraphPlan(h, t, r, n, n_rel)
    vals = L.ops.attn_update(plan, ent, rel)
    key = np.unique(kg.h * n + kg.t)
    assert plan.nnz == len(key) and plan.n_edges == kg.n_edges
    idx = plan.indices.cpu().numpy()
    assert np.array_equal(idx[0] * n + idx[1], key)                         # sorted, unique, bit exact
    assert np.array_equal(plan.rowptr.cpu().numpy(), np.searchsorted(key // n, np.arange(n + 1)))
    rows = torch.zeros(n, device="cuda").index_add_(0, plan.indices[0], vals)
    live = torch.from_numpy(np.bincount(kg.h, minlength=n) > 0).cuda()
    assert torch.allclose(rows[live], torch.ones_like(rows[live]), atol=1e-5)
    assert (rows[~live] == 0).all() and (vals > 0).all() and (vals <= 1).all()
    perm = torch.randperm(kg.n_edges, generator=g).cuda()
    plan2 = L.GraphPlan(h[perm], t[perm], r[perm], n, n_rel)
    vals2 = L.ops.attn_update(plan2, ent, rel)
    assert torch.equal(plan2.indices, plan.indices)
    assert torch.allclose(vals2, vals, rtol=1e-5, atol=1e-9)
    # spot-check 2000 random pairs against the oracle formula evaluated on those heads' rows only
    pick = torch.from_numpy(np.random.default_rng(0).choice(n, 300, replace=False))
    sel = np.isin(kg.h, pick.numpy())
    oi, ov = O.update_attention(ent.cpu(), rel.cpu(), torch.from_numpy(kg.h[sel]), torch.from_numpy(kg.t[sel]),
                                torch.from_numpy(kg.r[sel]), list(range(n_rel)), n)
    dense_key = plan.indices[0].cpu() * n + plan.indices[1].cpu()
    where = torch.searchsorted(dense_key, oi[0] * n + oi[1])
    assert rel_err(vals.cpu()[where], ov) < REL
