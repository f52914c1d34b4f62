"""Cross-checks against the UNMODIFIED reference (the original NSLab-CUK/LiteralKG).  The live oracle comparison runs
on inputs that are not among the committed golden vectors, so it needs the reference classes and runs only where
LKG_REFERENCE names a checkout; the committed golden vectors (tests/test_oracle_golden.py) hold the reference's outputs
that every checkout is compared with.  The checkpoint test runs everywhere on the reference-written state dicts stored
in tests/golden; its last step, loading a drop-in checkpoint back into the reference classes, needs the checkout."""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

import literalkg_oracle as O
from _golden import CASES, Golden

REF = os.environ.get("LKG_REFERENCE", "")
HAVE_REF = bool(REF) and os.path.exists(os.path.join(REF, "model.py"))

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))


def close(a, b, rtol, atol=1e-7):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    assert a.shape == b.shape
    assert (a - b).abs().max().item() <= atol + rtol * b.abs().max().item(), (a - b).abs().max().item()


@pytest.mark.skipif(not HAVE_REF, reason="LKG_REFERENCE names no checkout of the original LiteralKG")
@pytest.mark.parametrize("agg,res,layers,seed", [("bi-interaction", True, 3, 101), ("gcn", False, 2, 102),
                                                 ("graphsage", True, 2, 103), ("bi-interaction", False, 1, 104)])
def test_oracle_matches_live_reference(agg, res, layers, seed):
    import make_golden as G
    ref_model, _ = G.import_reference()
    cfg = O.OracleConfig(aggregation_type=agg, use_residual=res, n_conv_layers=layers, mess_dropout=0.0,
                         embed_dim=20, relation_dim=20, scale_gat_dim=12, conv_dim=8, num_lit_dim=2, txt_lit_dim=6)
    n, n_rel = 83, 5
    torch.manual_seed(seed)
    h, t, r = G.make_kg(n, n_rel, 400, seed)
    rng = np.random.default_rng(seed)
    num = torch.from_numpy(rng.uniform(0, 1, (n, 2)).astype(np.float32)) * (torch.rand(n, 1) < 0.3)
    txt = torch.from_numpy(rng.normal(0, 0.3, (n, 6)).astype(np.float32)) * (torch.rand(n, 1) < 0.3)
    lap_idx, lap_val, relations = G.ref_laplacian(h, t, r, n, "random-walk")
    oi, ov = O.laplacian_A_in(h, t, r, n)
    assert np.array_equal(oi, lap_idx) and np.array_equal(ov, lap_val)            # bit exact
    a0 = torch.sparse_coo_tensor(torch.from_numpy(lap_idx), torch.from_numpy(lap_val), (n, n))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = ref_model.LiteralKG(G.namespace(cfg), n, n_rel, a0, num, txt).eval()
        with torch.no_grad():
            model.entity_embed.weight.mul_(8)
            model.relation_embed.weight.mul_(4)
        p = {k: v.detach().clone() for k, v in model.state_dict().items() if k != "A_in"}
        hl, tl, rl = (torch.from_numpy(x) for x in (h, t, r))
        model(hl, tl, rl, relations, device="cpu", mode="update_att")
        a = model.A_in.data.coalesce()
        idx, val = O.update_attention(p["entity_embed.weight"], p["relation_embed.weight"], hl, tl, rl, relations, n)
        assert torch.equal(idx, a.indices())
        close(val, a.values(), 2e-6)
        with torch.no_grad():
            ref_emb = model.gat_embeddings()
        emb = O.gat_embeddings(p, cfg, idx, val, num, txt)
        close(emb, ref_emb, 2e-5)
        heads, tails = torch.arange(0, 9), torch.arange(5, 40)
        with torch.no_grad():
            close(O.calc_score(emb, heads, tails), model.calc_score(heads, tails), 5e-5)
        bh, bp, bn = (torch.from_numpy(rng.integers(0, n, 31)) for _ in range(3))
        br = torch.from_numpy(rng.integers(0, n_rel, 31))
        pg = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in p.items()}
        for mode, ref_in, loss_fn in (
                ("pre_training", (bh, br, bp, bn), lambda e: O.triplet_loss(pg, e, cfg, bh, br, bp, bn)),
                ("fine_tuning", (bh, bp, bn), lambda e: O.prediction_loss(e, cfg, bh, bp, bn))):
            model.zero_grad()
            ref_loss = model(*ref_in, device="cpu", mode=mode)
            ref_loss.backward()
            for v in pg.values():
                v.grad = None
            loss = loss_fn(O.gat_embeddings(pg, cfg, idx, val, num, txt))
            loss.backward()
            assert abs(loss.item() - ref_loss.item()) <= 2e-5 * abs(ref_loss.item())
            for k, v in model.named_parameters():
                if k != "A_in" and v.grad is not None:
                    close(pg[k].grad, v.grad, 5e-4)


def test_reference_checkpoint_loads_into_the_drop_in(tmp_path):
    """SURVEY.md 8(f) rank 4: a checkpoint written by the reference (``torch.save(model.state_dict())``,
    utils/model_utils.py:19-38, sparse ``A_in`` inside) loads into the drop-in class key for key, and what the drop-in
    saves has the reference's keys, order, shapes and dtypes (and, with a reference checkout, loads back into it).
    Checkpoints: the reference's state dicts of every golden case with its Laplacian as ``A_in``.  Host-side only: no
    kernel runs."""
    import literalkg_b200 as L
    import make_golden as G
    ref_model = G.import_reference()[0] if HAVE_REF else None
    for case in CASES:
        g = Golden(case)
        a_ref = torch.sparse_coo_tensor(g.t("lap/idx"), g.t("lap/val"), (g.n, g.n)).coalesce()
        path = tmp_path / f"{case}.pth"
        torch.save({**g.sd, "A_in": a_ref}, path)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ours = L.LiteralKG(G.namespace(g.cfg), g.n, g.n_rel, None, g.num_lit, g.txt_lit)
            missing, unexpected = ours.load_state_dict(torch.load(path), strict=True)
            assert not missing and not unexpected, case
            sd = ours.state_dict()
            assert [k for k in sd if k != "A_in"] == list(g.sd), case          # the reference's key order
            for k, v in g.sd.items():
                assert sd[k].shape == v.shape and sd[k].dtype == v.dtype and torch.equal(sd[k], v), (case, k)
            a = sd["A_in"].coalesce()
            assert torch.equal(a.indices(), a_ref.indices()) and torch.equal(a.values(), a_ref.values()), case
            path2 = tmp_path / f"{case}_ours.pth"
            torch.save(sd, path2)
            back = torch.load(path2)
            assert list(back) == list(sd) and all(torch.equal(back[k], g.sd[k]) for k in g.sd), case
            if ref_model is not None:
                ref2 = ref_model.LiteralKG(G.namespace(g.cfg), g.n, g.n_rel, None, g.num_lit, g.txt_lit)
                ref2.load_state_dict(back)
                assert torch.equal(ref2.entity_embed.weight, g.sd["entity_embed.weight"]), case
