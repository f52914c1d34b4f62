"""Filtered top-k link prediction under the dot score (LiteralKG.topk_links) without a GPU: the reference restatement
``best_of`` on a hand-built 8-entity, 2-relation graph with hand-computed results (ties, exclusion with and without a
relation, duplicate triples, padding, candidate subsets, head prediction) and its consistency with the rank
restatement, the argument checks of lkg_topk_threshold_dot / lkg_topk_finalize_dot, and the model-level refusals that
need no device."""
import ctypes

import pytest
import torch

import _rank_oracle as R
import _topk_dot_oracle as T
from test_rank_triple_cpu import _model, _refused, FAKE, ODD

# 2-wide embeddings; anchor 2 = (1, 1) scores s_j = x_j0 + x_j1 = 1 1 2 2 2 2 -1 3
X = torch.tensor([[1, 0], [0, 1], [1, 1], [2, 0], [1, 1], [0, 2], [-1, 0], [2, 1]], dtype=torch.float32)
KNOWN = [(2, 0, 7), (2, 0, 3), (2, 0, 3), (2, 1, 4), (2, 1, 6), (5, 1, 2), (6, 0, 2), (3, 0, 0)]
INF = float("inf")


def links(a, k, r=None, known=KNOWN, cands=range(8), predict="tail"):
    """Anchor a -> (scores, entity ids): s_j = x_a . x_j, excluding the tails of (a, r or any, ?) (heads of (?, r, a)
    for head prediction) in known."""
    cands = list(cands)
    s = T.dot_of(X[[a]], X[cands])[0]
    if predict == "tail":
        keys = {t for h, rr, t in known if h == a and r in (None, rr)}
    else:
        keys = {h for h, rr, t in known if t == a and r in (None, rr)}
    vals, pos = T.best_of(s, k, {p for p, c in enumerate(cands) if c in keys})
    return vals.tolist(), [cands[p] if p >= 0 else -1 for p in pos.tolist()]


def test_tail_links_hand_computed():
    # raw: 7 (3), then the four-way tie 2 3 4 5 (2) by position, 0 1 (1), 6 (-1)
    assert links(2, 8, known=[]) == ([3, 2, 2, 2, 2, 1, 1, -1], [7, 2, 3, 4, 5, 0, 1, 6])
    # relation 0 keys {7, 3} (3 known twice: counted once); the anchor 2 itself is not known and stays
    assert links(2, 3, r=0) == ([2, 2, 2], [2, 4, 5])
    # relation 1 keys {4, 6}
    assert links(2, 4, r=1) == ([3, 2, 2, 2], [7, 2, 3, 5])
    # any relation: {7, 3, 4, 6} -> 4 left, then padding
    assert links(2, 6) == ([2, 2, 1, 1, -INF, -INF], [2, 5, 0, 1, -1, -1])
    # a candidate subset in another order: ties go by position in the list, not by entity id
    assert links(2, 3, known=[], cands=[5, 0, 4, 2]) == ([2, 2, 2], [5, 4, 2])
    # known entities outside the candidates are ignored
    assert links(2, 3, r=0, cands=[5, 0, 4, 2]) == ([2, 2, 2], [5, 4, 2])
    # every candidate known: nothing but padding
    assert links(2, 2, cands=[3, 7]) == ([-INF, -INF], [-1, -1])
    # anchor 3 = (2, 0) scores itself 4 and stays (it is not its own known tail); (3, 0, 0) leaves out 0
    assert links(3, 2, r=0) == ([4, 4], [3, 7])


def test_head_links_hand_computed():
    # (?, 0, 2): heads known {6}; (?, 1, 2): {5}; any relation: {5, 6}
    assert links(2, 8, r=0, predict="head") == ([3, 2, 2, 2, 2, 1, 1, -INF], [7, 2, 3, 4, 5, 0, 1, -1])
    assert links(2, 3, r=1, predict="head") == ([3, 2, 2], [7, 2, 3])
    assert links(2, 8, predict="head")[1] == [7, 2, 3, 4, 0, 1, -1, -1]
    # anchor 0 = (1, 0): s = 1 0 1 2 1 0 -1 2; (?, 0, 0) knows head 3, the best one
    assert links(0, 3, r=0, predict="head") == ([2, 1, 1], [7, 0, 2])


def test_rows_restatement_matches_best_of():
    g = torch.Generator().manual_seed(3)
    s = torch.randint(-3, 3, (5, 40), generator=g).float()           # many ties
    excl = torch.rand(5, 40, generator=g) < 0.3
    for k in (1, 7, 40):
        vals, pos = T.best_rows_of(s, k, excl)
        for i in range(5):
            want = T.best_of(s[i], k, set(torch.nonzero(excl[i]).reshape(-1).tolist()))
            assert torch.equal(vals[i], want[0]) and torch.equal(pos[i], want[1])


@pytest.mark.parametrize("r", [None, 0, 1])
def test_consistency_with_the_rank_restatement(r):
    """Entity ids[j] gets filtered rank j from the rank restatement, with the same known triples and relation."""
    for cands in (list(range(8)), [7, 4, 2, 0, 5]):
        for a in range(8):
            _, ids = links(a, 8, r=r, cands=cands)
            s = T.dot_of(X[[a]], X[cands])
            for j, e in enumerate(ids):
                if e < 0:
                    continue
                got = R.filtered_rank_of(None, [a], cands, [cands.index(e)], KNOWN, None if r is None else [r],
                                         scores=s)
                assert got.tolist() == [j]


def test_excluded_any_relation_restatement():
    ex = T.excluded_any_relation([2, 5], list(range(8)), KNOWN)
    assert torch.nonzero(ex[0]).reshape(-1).tolist() == [3, 4, 6, 7]
    assert torch.nonzero(ex[1]).reshape(-1).tolist() == [2]


# ---- the C ABI ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from literalkg_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _graph(att=FAKE):
    from literalkg_b200 import _lib
    g = _lib.LkgGraph()
    g.n_entities = 8
    g.att_rowptr, g.att_tail, g.att_rel, g.rowptr, g.col = att, FAKE, FAKE, FAKE, FAKE
    return g


def test_abi_entry_points(lib):
    from literalkg_b200 import _lib
    assert lib.lkg_abi_version() == 8 == _lib.ABI_VERSION
    for name in ("lkg_topk_threshold_dot", "lkg_topk_finalize_dot"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)


def test_topk_threshold_dot_refusals(lib):
    g, g_bad = _graph(), _graph(att=None)

    def call(cand=FAKE, ld_cand=396, n_cand=100, query=FAKE, ld_query=396, n=4, dim=396, center=FAKE, max_norm=FAKE,
             rec_q=FAKE, rec_c=FAKE, k=10, n_sample=50, known=None, anchors=None, thr=FAKE):
        return lib.lkg_topk_threshold_dot(cand, ld_cand, None, n_cand, query, ld_query, None, n, dim, center, max_norm,
                                          rec_q, rec_c, k, n_sample, known, anchors, None, None, thr, None, None)

    _refused(lib, call(cand=None), ["cand is null"])
    _refused(lib, call(cand=ODD), ["aligned"])
    _refused(lib, call(ld_cand=394), ["aligned"])
    _refused(lib, call(query=None), ["query is null"])
    _refused(lib, call(query=ODD), ["aligned"])
    _refused(lib, call(ld_query=392), ["aligned"])
    _refused(lib, call(center=None), ["center"])
    _refused(lib, call(center=ODD), ["center"])
    _refused(lib, call(max_norm=None), ["cand_max_norm"])
    _refused(lib, call(rec_q=None), ["rec_query"])
    _refused(lib, call(rec_c=None), ["rec_cand"])
    _refused(lib, call(thr=None), ["thr"])
    _refused(lib, call(dim=516, ld_cand=516, ld_query=516), ["dim"])
    _refused(lib, call(dim=298), ["dim"])                          # not a multiple of 4: the caller pads
    _refused(lib, call(dim=0), ["dim"])
    _refused(lib, call(n=-1), ["shape"])
    _refused(lib, call(n_cand=0), ["shape"])
    _refused(lib, call(k=0), ["k must be"])
    _refused(lib, call(k=1025), ["k must be"])
    _refused(lib, call(n_sample=0), ["n_sample"])
    _refused(lib, call(n_sample=101), ["n_sample"])
    _refused(lib, call(known=ctypes.byref(g_bad), anchors=FAKE), ["known plan"])
    _refused(lib, call(known=ctypes.byref(g)), ["anchors"])
    assert call(n=0, known=ctypes.byref(g), anchors=FAKE, k=1024, n_sample=100) == 0
    assert call(n=0, dim=512, ld_cand=512, ld_query=512, n_sample=1) == 0     # the widest width


def test_topk_finalize_dot_refusals(lib):
    g, g_bad = _graph(), _graph(att=None)

    def call(cand=FAKE, n_cand=100, query=FAKE, ld_query=396, n=4, dim=396, band_cnt=FAKE, band=FAKE, cap=64, k=10,
             known=None, anchors=None, score=FAKE, pos=FAKE):
        return lib.lkg_topk_finalize_dot(cand, 396, None, n_cand, query, ld_query, None, n, dim, band_cnt, band, cap, k,
                                         known, anchors, None, None, score, pos, None)

    _refused(lib, call(cand=None), ["cand is null"])
    _refused(lib, call(cand=ODD), ["aligned"])
    _refused(lib, call(query=None), ["query is null"])
    _refused(lib, call(ld_query=394), ["aligned"])
    _refused(lib, call(dim=516), ["dim"])
    _refused(lib, call(dim=30), ["dim"])
    _refused(lib, call(band_cnt=None), ["band_cnt"])
    _refused(lib, call(band=None), ["band"])
    _refused(lib, call(score=None), ["score"])
    _refused(lib, call(pos=None), ["pos"])
    _refused(lib, call(n=-1), ["shape"])
    _refused(lib, call(n_cand=0), ["shape"])
    _refused(lib, call(k=0), ["k must be"])
    _refused(lib, call(k=1025, cap=4096), ["k must be"])
    _refused(lib, call(cap=19), ["cap must be"])                  # < 2k
    _refused(lib, call(cap=16385), ["cap must be"])
    _refused(lib, call(known=ctypes.byref(g_bad), anchors=FAKE), ["known plan"])
    _refused(lib, call(known=ctypes.byref(g)), ["anchors"])
    assert call(n=0, known=ctypes.byref(g), anchors=FAKE, cap=20) == 0   # cap = 2k, any value in range
    assert call(n=0, k=1024, cap=16384) == 0


# ---- model-level refusals ------------------------------------------------------------------------------------------------
def test_model_refusals_before_any_launch():
    m = _model()
    a = torch.tensor([0, 1])
    emb = torch.zeros(10, 64)
    with pytest.raises(ValueError, match="predict must be"):
        m.topk_links(a, 10, predict="both", all_embed=emb)
    for k in (0, 1025, 2.5, True):
        with pytest.raises(ValueError, match="k must be"):
            m.topk_links(a, k, all_embed=emb)
    with pytest.raises(ValueError, match="pass the known triples"):
        m.topk_links(a, 10, relations=torch.tensor([0, 1]), all_embed=emb)
    with pytest.raises(ValueError, match="pass the known triples"):
        _model(bce=True).topk_links(a, 10, relations=[0, 1], predict="head", all_embed=emb)
    with pytest.raises(ValueError, match="up to 512"):
        m.topk_links(a, 10, all_embed=torch.zeros(10, 516))
