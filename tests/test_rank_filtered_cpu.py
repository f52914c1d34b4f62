"""Filtered link-prediction ranks without a GPU: the reference ``filtered_rank_of`` / ``ranking_metrics`` of
tests/_rank_oracle.py on a hand-built 8-entity graph with hand-computed answers, and the C ABI of the filter kernels
(declared, exported, bound, arguments checked before anything touches a device)."""
import ctypes

import pytest
import torch

import _rank_oracle as R

# 1-wide embeddings: s(h, j) = x_h * x_j, so for a positive head the order of the tails is the order of x
X = torch.tensor([[1.0], [5.0], [4.0], [4.0], [3.0], [2.0], [6.0], [0.5]], dtype=torch.float64)
ALL = list(range(8))
# head 0 knows: tail 1 twice (a duplicate triple), its own test target 4, tails 2 and 5 under relation 0; tail 6 under
# relation 1; tail 3 under relation 2.  Head 7 knows nothing.
KNOWN = [(0, 0, 1), (0, 0, 1), (0, 0, 4), (0, 0, 2), (0, 0, 5), (0, 1, 6), (0, 2, 3)]


def frank(heads, tails, rels=None, cands=ALL):
    where = {c: p for p, c in enumerate(cands)}
    tpos = torch.tensor([where[t] for t in tails])
    return R.filtered_rank_of(X, torch.tensor(heads), torch.tensor(cands), tpos, KNOWN, rels).tolist()


def test_filter_by_relation_duplicates_and_own_target():
    # (0, 0, 4): tails above 4 (score 3) are 6, 1, 2, 3 -> raw 4.  F = {1, 2, 4, 5}: 1 (known twice) and 2 beat it,
    # 4 is the target, 5 is below -> 2
    assert frank([0], [4], [0]) == [2]
    assert R.filtered_rank_of(X, torch.tensor([0]), torch.tensor(ALL), torch.tensor([4]), []).tolist() == [4]


def test_filter_by_head():
    # without a relation F = every tail of head 0 = {1, 2, 3, 4, 5, 6}: all four tails above 4 are known -> 0
    assert frank([0], [4]) == [0]
    # head 0's tails above 5 (score 2) are 6, 1, 2, 3, 4, all known -> 0; under relation 1 only 6 is removed -> 4
    assert frank([0, 0], [5, 5], [1, 1]) == [4, 4]
    assert frank([0], [5]) == [0]


def test_tie_with_a_filter_entry_on_both_sides():
    # tails 2 and 3 tie (score 4).  Target 3: 2 sits before it and beats it -> raw 3 (6, 1, 2), F(0, 0) removes 1, 2
    assert frank([0], [3], [0]) == [1]
    # target 2: the tied filter entry 3 sits after it and does not beat it -> raw 2 (6, 1); F(0, 2) = {3} removes none
    assert frank([0], [2], [2]) == [2]
    # by head: 1 and 6 are known and beat 2, 3 does not -> 0
    assert frank([0], [2]) == [0]
    # permuted candidates without 1: 3 now sits before 2 and beats it -> raw 2 (6, 3), F(0, 2) = {3} -> 1
    assert frank([0], [2], [2], cands=[7, 6, 3, 2, 4, 0]) == [1]


def test_known_tails_outside_the_candidates_are_ignored():
    # candidates lack 1 and 5: raw rank of 4 = #{6, 2, 3} = 3; F(0, 0) = {1, 2, 4, 5} -> only 2 is removed
    assert frank([0], [4], [0], cands=[7, 6, 2, 3, 4, 0]) == [2]


def test_empty_filter_run():
    # head 7 (x = 0.5 > 0, same order): target 5 (x = 2) is beaten by 6, 1, 2, 3, 4 and head 7 has no known tails
    assert frank([7], [5], [0]) == [5]
    assert frank([7], [5]) == [5]


def test_ranking_metrics_hand_computed():
    m = R.ranking_metrics([0, 1, 3, 9], ks=(1, 3, 10))
    assert m["mr"] == (1 + 2 + 4 + 10) / 4
    assert m["mrr"] == pytest.approx((1 + 1 / 2 + 1 / 4 + 1 / 10) / 4, rel=1e-15)
    assert (m["hits@1"], m["hits@3"], m["hits@10"]) == (0.25, 0.5, 1.0)


def test_filter_entry_points_are_bound_and_check_arguments():
    from literalkg_b200 import _lib, build
    build.build(verbose=False)
    lib = _lib.load()
    for name in ("lkg_rank_filter", "lkg_rank_filter_scores"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)
    fake = ctypes.c_void_p(256)                          # never dereferenced: every call below stops at validation
    g = _lib.LkgGraph()
    g.n_entities = 8
    g.att_rowptr = g.att_tail = g.att_rel = g.rowptr = g.col = fake.value
    assert lib.lkg_rank_filter(None, fake, None, None, fake, 1, fake, 4, 4, fake, fake, None) == -1
    assert b"known plan" in lib.lkg_last_error()
    assert lib.lkg_rank_filter(ctypes.byref(g), fake, None, None, fake, 1, fake, 4, 6, fake, fake, None) == -1
    assert b"dim" in lib.lkg_last_error()
    assert lib.lkg_rank_filter(ctypes.byref(g), fake, None, None, fake, 0, fake, 4, 4, fake, fake, None) == 0
    # a score matrix without a candidate map needs one column per entity
    assert lib.lkg_rank_filter_scores(ctypes.byref(g), fake, None, None, fake, 1, fake, 7, 7, fake, None) == -1
    assert b"candidate map" in lib.lkg_last_error()
    assert lib.lkg_rank_filter_scores(ctypes.byref(g), fake, None, None, fake, 0, fake, 8, 8, fake, None) == 0
