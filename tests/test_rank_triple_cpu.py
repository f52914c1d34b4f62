"""Ranking by the triple score (LiteralKG.evaluate_ranking(score="triple")) without a GPU: the reference restatement
(``filtered_rank_of`` on s = -d) on a hand-built 8-entity, 2-relation graph with hand-computed ranks, the argument
checks of the distance rank entry points (lkg_l2_rank_rows, lkg_rank_prepare_l2, lkg_rank_finalize_l2,
lkg_rank_filter_l2) and the model-level refusals that need no device."""
import argparse
import ctypes

import pytest
import torch

import _rank_oracle as R
import literalkg_oracle as O


def neg_dist(query, cand):
    """s = -d, d = |q - p_j|^2 summed in float64 and rounded once to fp32 (the declared arithmetic), [B, Nc]."""
    d = ((query.double()[:, None, :] - cand.double()[None, :, :]) ** 2).sum(-1)
    return -d.float()


# 1-wide embeddings x_j = j; TransR with scalar M_r: relation 0 (M = 1, e = 2), relation 1 (M = 2, e = -1)
X = torch.arange(8, dtype=torch.float64)[:, None]
M = {0: 1.0, 1: 2.0}
E = {0: 2.0, 1: -1.0}
KNOWN = [(1, 0, 2), (1, 0, 4), (1, 0, 4), (1, 1, 3), (6, 1, 5), (4, 1, 5), (4, 0, 5)]


def tail_rank(h, r, t, known=KNOWN, cands=range(8)):
    cands = list(cands)
    q = X[[h]] * M[r] + E[r]
    s = neg_dist(q, X[cands] * M[r])
    return R.filtered_rank_of(None, [h], cands, [cands.index(t)], known, [r], scores=s).tolist()[0]


def head_rank(h, r, t, known=KNOWN, cands=range(8)):
    """(?, r, t): query row x_t M_r - e_r against the candidates' x_j M_r; the filter keys are (t, r) of the swapped
    known triples."""
    cands = list(cands)
    q = X[[t]] * M[r] - E[r]
    s = neg_dist(q, X[cands] * M[r])
    swapped = [(tt, rr, hh) for hh, rr, tt in known]
    return R.filtered_rank_of(None, [t], cands, [cands.index(h)], swapped, [r], scores=s).tolist()[0]


def test_tail_prediction_hand_computed():
    # (1, 0, ?): q = 3, d_j = (3 - j)^2 = 9 4 1 0 1 4 9 16.  Target 4 (d = 1): 3 is closer, 2 ties before it -> raw 2;
    # F(1, 0) = {2, 4}: 2 beats it, 4 is the target -> 1
    assert tail_rank(1, 0, 4, known=[]) == 2
    assert tail_rank(1, 0, 4) == 1
    # target 2 (d = 1): only 3 is closer, 4 ties after it -> 1, and no member of F(1, 0) beats it
    assert tail_rank(1, 0, 2) == 1
    # candidates without 3: target 4 is beaten by the tie 2 placed before it -> raw 1, filtered 0; placed after it, 2
    # does not beat it -> 0
    assert tail_rank(1, 0, 4, known=[], cands=[7, 2, 4, 0]) == 1
    assert tail_rank(1, 0, 4, cands=[7, 2, 4, 0]) == 0
    assert tail_rank(1, 0, 4, known=[], cands=[7, 4, 2, 0]) == 0


def test_head_prediction_hand_computed():
    # (?, 1, 5): q' = 5 * 2 + 1 = 11, p_j = 2 j, d_j = (11 - 2 j)^2 = 121 81 49 25 9 1 1 9.  Target 4 (d = 9): 5 and 6
    # are closer, 7 ties after it -> raw 2; heads known for (?, 1, 5) are {6, 4}: 6 beats it -> 1
    assert head_rank(4, 1, 5, known=[]) == 2
    assert head_rank(4, 1, 5) == 1
    # target 6 (d = 1): 5 ties before it -> raw 1; 5 is not a known head of (?, 1, 5) -> 1
    assert head_rank(6, 1, 5) == 1
    # relation 0 keys another run: (?, 0, 5) knows head 4 only.  q' = 5 - 2 = 3, d_j = (3 - j)^2: target 4 -> raw 2
    # (3 closer, 2 ties before), the known head 4 is the target itself -> 2
    assert head_rank(4, 0, 5) == 2


def test_restatement_matches_the_loss_distance():
    # d of a triple equals the per-triple term of the TransR loss, sum((h M_r + e_r - t M_r)^2)
    g = torch.Generator().manual_seed(0)
    emb, w, rel = torch.randn(6, 5, generator=g), torch.randn(2, 5, 3, generator=g), torch.randn(2, 3, generator=g)
    h, r, t = 2, 1, 4
    d = -neg_dist((emb[[h]].double() @ w[r].double() + rel[r].double()).float(), (emb[[t]].double() @ w[r].double()).float())
    ref = ((emb[h].double() @ w[r].double() + rel[r].double() - emb[t].double() @ w[r].double()) ** 2).sum()
    assert float(d) == pytest.approx(float(ref), rel=1e-6)


# ---- the C ABI ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from literalkg_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


FAKE = 256                                   # never dereferenced: every call below stops at validation
ODD = 260                                    # not 16-byte aligned


def _refused(lib, rc, words):
    assert rc == -1, rc
    msg = lib.lkg_last_error().decode()
    assert any(w in msg for w in words), msg


def test_abi_version(lib):
    from literalkg_b200 import _lib
    assert lib.lkg_abi_version() == 9 == _lib.ABI_VERSION
    for name in ("lkg_l2_rank_rows", "lkg_rank_prepare_l2", "lkg_rank_finalize_l2", "lkg_rank_filter_l2"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)


def _rows(lib, src=FAKE, ld=300, m=10, dim=300, center=FAKE, mode=1, stats=FAKE, out=FAKE, ld_out=304):
    return lib.lkg_l2_rank_rows(src, ld, None, m, dim, center, mode, stats, out, ld_out, None)


def test_l2_rank_rows_refusals(lib):
    _refused(lib, _rows(lib, src=None), ["src is null"])
    _refused(lib, _rows(lib, center=None), ["center"])
    _refused(lib, _rows(lib, stats=None), ["stats"])
    _refused(lib, _rows(lib, out=None), ["out"])
    _refused(lib, _rows(lib, dim=512, ld=512, ld_out=516), ["dim"])          # augmented width 516 > 512
    _refused(lib, _rows(lib, dim=302, ld=304), ["dim"])                      # not a multiple of 4
    _refused(lib, _rows(lib, src=ODD), ["aligned"])
    _refused(lib, _rows(lib, ld=302), ["aligned"])
    _refused(lib, _rows(lib, center=ODD), ["center"])
    _refused(lib, _rows(lib, out=ODD), ["alignment"])
    _refused(lib, _rows(lib, ld_out=300), ["dim + 4"])
    _refused(lib, _rows(lib, m=-1), ["m)"])
    _refused(lib, _rows(lib, mode=5), ["mode"])
    assert _rows(lib, dim=508, ld=508, ld_out=512, mode=0, m=0) == 0          # the widest width, nothing to do


def _prep(lib, cand=FAKE, query=FAKE, aug=FAKE, ld_aug=304, tp=FAKE, n=4, dim=300, stats=FAKE, tau=FAKE, thr=FAKE):
    return lib.lkg_rank_prepare_l2(cand, 300, query, 300, aug, ld_aug, tp, n, dim, stats, FAKE, FAKE, tau, thr, None)


def test_rank_prepare_l2_refusals(lib):
    _refused(lib, _prep(lib, cand=None), ["cand is null"])
    _refused(lib, _prep(lib, query=None), ["query is null"])
    _refused(lib, _prep(lib, aug=None), ["query_aug"])
    _refused(lib, _prep(lib, aug=ODD), ["query_aug"])
    _refused(lib, _prep(lib, ld_aug=300), ["query_aug"])
    _refused(lib, _prep(lib, tp=None), ["bad rank arguments"])
    _refused(lib, _prep(lib, stats=None), ["bad rank arguments"])
    _refused(lib, _prep(lib, tau=None), ["bad rank arguments"])
    _refused(lib, _prep(lib, thr=None), ["bad rank arguments"])
    _refused(lib, _prep(lib, n=-1), ["bad rank arguments"])
    _refused(lib, _prep(lib, dim=516), ["dim"])
    _refused(lib, _prep(lib, dim=298), ["dim"])
    _refused(lib, _prep(lib, cand=ODD), ["aligned"])
    assert _prep(lib, n=0) == 0


def _fin(lib, cand=FAKE, query=FAKE, ld_query=300, band=FAKE, cap=64, n=4, n_cand=100, dim=300, ranks=FAKE):
    return lib.lkg_rank_finalize_l2(cand, 300, query, ld_query, FAKE, FAKE, FAKE, FAKE, band, cap, n, n_cand, dim,
                                    ranks, None)


def test_rank_finalize_l2_refusals(lib):
    _refused(lib, _fin(lib, cand=None), ["cand is null"])
    _refused(lib, _fin(lib, query=None), ["query is null"])
    _refused(lib, _fin(lib, band=None), ["bad rank arguments"])
    _refused(lib, _fin(lib, ranks=None), ["bad rank arguments"])
    _refused(lib, _fin(lib, cap=0), ["bad rank arguments"])
    _refused(lib, _fin(lib, n=-1), ["bad rank arguments"])
    _refused(lib, _fin(lib, n_cand=-1), ["bad rank arguments"])
    _refused(lib, _fin(lib, dim=520), ["dim"])
    _refused(lib, _fin(lib, dim=6), ["dim"])
    _refused(lib, _fin(lib, query=ODD), ["aligned"])
    _refused(lib, _fin(lib, ld_query=298), ["aligned"])
    assert _fin(lib, n=0) == 0


def test_rank_filter_l2_refusals(lib):
    from literalkg_b200 import _lib
    g = _lib.LkgGraph()
    g.n_entities = 8
    g.att_rowptr = g.att_tail = g.att_rel = g.rowptr = g.col = FAKE

    def call(known=ctypes.byref(g), anchors=FAKE, n=1, cand=FAKE, query=FAKE, dim=300, tau=FAKE):
        return lib.lkg_rank_filter_l2(known, anchors, None, None, FAKE, n, cand, 300, query, 300, dim, tau, FAKE, None)

    _refused(lib, call(known=None), ["known plan"])
    _refused(lib, call(anchors=None), ["bad filter arguments"])
    _refused(lib, call(n=-1), ["bad filter arguments"])
    _refused(lib, call(cand=None), ["cand is null"])
    _refused(lib, call(query=ODD), ["aligned"])
    _refused(lib, call(dim=512), ["dim"])
    _refused(lib, call(dim=30), ["dim"])
    _refused(lib, call(tau=None), ["bad filter arguments"])
    assert call(n=0) == 0


# ---- model-level refusals ------------------------------------------------------------------------------------------------
def _model(bce=False, **kw):
    import literalkg_b200 as L
    from literalkg_b200 import model_bce
    cfg = O.OracleConfig(n_conv_layers=1, **kw)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    cls = model_bce.LiteralKG if bce else L.LiteralKG
    return cls(args, 10, 2, None, torch.zeros(10, cfg.num_lit_dim), torch.zeros(10, cfg.txt_lit_dim))


def test_model_refusals_before_any_launch():
    m = _model()
    h, t = torch.tensor([0, 1]), torch.tensor([2, 3])
    with pytest.raises(ValueError, match="relation of every query"):
        m.evaluate_ranking(h, t, score="triple")
    with pytest.raises(ValueError, match="relation of every query"):
        _model(bce=True).evaluate_ranking(h, t, score="triple", predict="head")
    with pytest.raises(ValueError, match='score must be'):
        m.evaluate_ranking(h, t, score="transr")
    with pytest.raises(ValueError, match='predict must be'):
        m.evaluate_ranking(h, t, predict="both")
    wide = _model(relation_dim=512)
    with pytest.raises(ValueError, match="up to 508"):
        wide.evaluate_ranking(h, t, torch.tensor([0, 1]), score="triple")
