"""Relation-aware top-k completion (LiteralKG.topk_triple) without a GPU: the reference restatement ``topk_of`` on the
hand-built 8-entity, 2-relation graph of test_rank_triple_cpu.py with hand-computed results (ties, exclusion, padding,
candidate subsets, head prediction) and its consistency with the rank restatement, the argument checks of
lkg_topk_threshold_l2 / lkg_topk_finalize_l2, and the model-level refusals that need no device."""
import ctypes

import pytest
import torch

import _rank_oracle as R
import _topk_oracle as T
from test_rank_triple_cpu import E, KNOWN, M, X, _model, _refused, neg_dist, FAKE, ODD


def tail_topk(h, r, k, known=KNOWN, cands=range(8)):
    """(h, r, ?) -> (dist, entity ids): q = x_h M_r + e_r against x_j M_r, excluding { t : (h, r, t) in known }."""
    cands = list(cands)
    d = -neg_dist(X[[h]] * M[r] + E[r], X[cands] * M[r])[0]
    excl = {p for p, c in enumerate(cands) if (h, r, c) in set(known)}
    dist, pos = T.topk_of(d, k, excl)
    return dist.tolist(), [cands[p] if p >= 0 else -1 for p in pos.tolist()]


def head_topk(t, r, k, known=KNOWN, cands=range(8)):
    """(?, r, t): q' = x_t M_r - e_r, excluding { h : (h, r, t) in known }."""
    cands = list(cands)
    d = -neg_dist(X[[t]] * M[r] - E[r], X[cands] * M[r])[0]
    excl = {p for p, c in enumerate(cands) if (c, r, t) in set(known)}
    dist, pos = T.topk_of(d, k, excl)
    return dist.tolist(), [cands[p] if p >= 0 else -1 for p in pos.tolist()]


INF = float("inf")


def test_tail_topk_hand_computed():
    # (1, 0, ?): q = 3, d_j = (3 - j)^2 = 9 4 1 0 1 4 9 16.  Raw: 3, then the tie 2 / 4 by position
    assert tail_topk(1, 0, 3, known=[]) == ([0, 1, 1], [3, 2, 4])
    # known (1, 0, 2) and (1, 0, 4) (twice): both left out; the anchor 1 itself is not known and stays
    assert tail_topk(1, 0, 3) == ([0, 4, 4], [3, 1, 5])
    # k larger than what remains: 6 entities, then padding
    assert tail_topk(1, 0, 8) == ([0, 4, 4, 9, 9, 16, INF, INF], [3, 1, 5, 0, 6, 7, -1, -1])
    # a candidate subset in another order: ties go by position in the list, not by entity id
    assert tail_topk(1, 0, 2, known=[], cands=[7, 4, 2, 0]) == ([1, 1], [4, 2])
    assert tail_topk(1, 0, 3, cands=[7, 4, 2, 0]) == ([9, 16, INF], [0, 7, -1])
    # relation 1 keys another run: (1, 1, ?) knows 3 only.  q = 2 - 1 = 1, p_j = 2 j, d = 1 1 9 25 ...
    assert tail_topk(1, 1, 3) == ([1, 1, 9], [0, 1, 2])
    # every candidate known: nothing but padding
    assert tail_topk(1, 0, 2, cands=[2, 4]) == ([INF, INF], [-1, -1])


def test_head_topk_hand_computed():
    # (?, 1, 5): q' = 11, p_j = 2 j, d = 121 81 49 25 9 1 1 9.  Raw: 5 and 6 (tie by position), then 4 before 7
    assert head_topk(5, 1, 3, known=[]) == ([1, 1, 9], [5, 6, 4])
    # known heads of (?, 1, 5): 6 and 4 -> left out
    assert head_topk(5, 1, 3) == ([1, 9, 25], [5, 7, 3])
    # (?, 0, 5) knows head 4 only: q' = 3, d = (3 - j)^2
    assert head_topk(5, 0, 4) == ([0, 1, 4, 4], [3, 2, 1, 5])


def test_rows_restatement_matches_topk_of():
    g = torch.Generator().manual_seed(3)
    d = torch.randint(0, 6, (5, 40), generator=g).float()            # many ties
    excl = torch.rand(5, 40, generator=g) < 0.3
    for k in (1, 7, 40):
        dist, pos = T.topk_rows_of(d, k, excl)
        for i in range(5):
            want = T.topk_of(d[i], k, set(torch.nonzero(excl[i]).reshape(-1).tolist()))
            assert torch.equal(dist[i], want[0]) and torch.equal(pos[i], want[1])


@pytest.mark.parametrize("known", [[], KNOWN])
def test_consistency_with_the_rank_restatement(known):
    """Entity ids[j] gets filtered rank j (raw rank j without known triples) from the rank restatement."""
    for cands in (list(range(8)), [7, 4, 2, 0, 5]):
        for r in (0, 1):
            for a in range(8):
                _, ids = tail_topk(a, r, 8, known=known, cands=cands)
                s = neg_dist(X[[a]] * M[r] + E[r], X[cands] * M[r])
                for j, e in enumerate(ids):
                    if e < 0:
                        continue
                    got = R.filtered_rank_of(None, [a], cands, [cands.index(e)], known, [r], scores=s)
                    assert got.tolist() == [j]


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
    for name in ("lkg_topk_threshold_l2", "lkg_topk_finalize_l2"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)


def test_topk_threshold_l2_refusals(lib):
    g, g_bad = _graph(), _graph(att=None)

    def call(cand=FAKE, n_cand=100, query=FAKE, ld_query=300, aug=FAKE, ld_aug=304, n=4, dim=300, stats=FAKE,
             rec_q=FAKE, rec_c=FAKE, k=10, n_sample=50, known=None, anchors=None, thr=FAKE):
        return lib.lkg_topk_threshold_l2(cand, 300, n_cand, query, ld_query, aug, ld_aug, n, dim, stats, rec_q, rec_c, k,
                                         n_sample, known, anchors, None, None, thr, None, None)

    _refused(lib, call(cand=None), ["cand is null"])
    _refused(lib, call(query=None), ["query is null"])
    _refused(lib, call(query=ODD), ["aligned"])
    _refused(lib, call(ld_query=298), ["aligned"])
    _refused(lib, call(aug=None), ["query_aug"])
    _refused(lib, call(aug=ODD), ["query_aug"])
    _refused(lib, call(ld_aug=300), ["query_aug"])
    _refused(lib, call(stats=None), ["stats"])
    _refused(lib, call(rec_q=None), ["rec_query"])
    _refused(lib, call(rec_c=None), ["rec_cand"])
    _refused(lib, call(thr=None), ["thr"])
    _refused(lib, call(dim=512), ["dim"])                         # augmented width 516 > 512
    _refused(lib, call(dim=302), ["dim"])
    _refused(lib, call(n=-1), ["shape"])
    _refused(lib, call(n_cand=0), ["shape"])
    _refused(lib, call(k=0), ["k must be"])
    _refused(lib, call(k=1025), ["k must be"])
    _refused(lib, call(n_sample=0), ["n_sample"])
    _refused(lib, call(n_sample=101), ["n_sample"])
    _refused(lib, call(known=ctypes.byref(g_bad), anchors=FAKE), ["known plan"])
    _refused(lib, call(known=ctypes.byref(g)), ["anchors"])
    assert call(n=0, known=ctypes.byref(g), anchors=FAKE, k=1024, n_sample=100) == 0


def test_topk_finalize_l2_refusals(lib):
    g, g_bad = _graph(), _graph(att=None)

    def call(cand=FAKE, n_cand=100, query=FAKE, n=4, dim=300, band_cnt=FAKE, band=FAKE, cap=64, k=10, known=None,
             anchors=None, dist=FAKE, pos=FAKE):
        return lib.lkg_topk_finalize_l2(cand, 300, n_cand, query, 300, n, dim, band_cnt, band, cap, k, known, anchors,
                                        None, None, dist, pos, None)

    _refused(lib, call(cand=None), ["cand is null"])
    _refused(lib, call(cand=ODD), ["aligned"])
    _refused(lib, call(query=None), ["query is null"])
    _refused(lib, call(dim=516), ["dim"])
    _refused(lib, call(dim=30), ["dim"])
    _refused(lib, call(band_cnt=None), ["band_cnt"])
    _refused(lib, call(band=None), ["band"])
    _refused(lib, call(dist=None), ["dist"])
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
    a, r = torch.tensor([0, 1]), torch.tensor([0, 1])
    with pytest.raises(ValueError, match="relation of every query"):
        m.topk_triple(a, None, 10)
    with pytest.raises(ValueError, match="relation of every query"):
        _model(bce=True).topk_triple(a, None, 10, predict="head")
    with pytest.raises(ValueError, match="predict must be"):
        m.topk_triple(a, r, 10, predict="both")
    for k in (0, 1025, 2.5, True):
        with pytest.raises(ValueError, match="k must be"):
            m.topk_triple(a, r, k)
    with pytest.raises(ValueError, match="up to 508"):
        _model(relation_dim=512).topk_triple(a, r, 10)
