"""The target score tau of the fused dot rank comes from the same exact scorer as the re-scores it is compared with.

Both sums are fp64 sums of exact fp32 products, rounded once to fp32, but two summation orders can round to different
fp32 values when the score is small against the products (heavy cancellation: a target nearly orthogonal to its head).
If the target score were summed in another order than finalize re-scores the target's own column, the target could
beat itself by one ulp and every rank of such a query would come out one too high.  The pairs are mined on the host by
emulating two orders exactly (an fma of fp32 operands is the fp64 sum of the exact product, rounded once):
    lane order  8 lanes, lane q takes float4 q, q + 8, ...; xor-reduced over 4, 2, 1  (the exact scorer)
    warp order  32 lanes, lane l takes column l, l + 32, ...; xor-reduced over 16, 8, 4, 2, 1
and the GPU test ranks each mined target (where the lane order rounds above the warp order) among tails that all score
clearly lower: its rank must be 0, raw and filtered."""
import numpy as np
import pytest
import torch

DIM = 256


def _xor_reduce(parts, offsets):
    for o in offsets:
        parts = parts + parts[:, np.arange(parts.shape[1]) ^ o]
    return parts[:, 0]


def lane_order(h, t):
    """fp32 dot products of the rows of h and t in the exact scorer's order (8 lanes of float4)."""
    prod = h.astype(np.float64) * t.astype(np.float64)
    p4 = prod.reshape(len(h), -1, 4)                       # [pairs, float4 v, 4]
    acc = np.zeros((len(h), 8))
    for v in range(p4.shape[1]):
        for j in range(4):
            acc[:, v % 8] += p4[:, v, j]
    return _xor_reduce(acc, (4, 2, 1)).astype(np.float32)


def warp_order(h, t):
    """The same in a 32-lane scalar order."""
    prod = h.astype(np.float64) * t.astype(np.float64)
    acc = np.zeros((len(h), 32))
    for c in range(prod.shape[1]):
        acc[:, c % 32] += prod[:, c]
    return _xor_reduce(acc, (16, 8, 4, 2, 1)).astype(np.float32)


def mine_pairs(n_pairs=100000, seed=11, chunk=20000):
    """(h, t) fp32 rows, t = r - (1 - 1e-4) proj_h(r): the pairs whose lane-order score rounds above the warp order."""
    rng = np.random.default_rng(seed)
    hs, ts = [], []
    for _ in range(0, n_pairs, chunk):
        h = rng.standard_normal((chunk, DIM)).astype(np.float32)
        r = rng.standard_normal((chunk, DIM))
        hd = h.astype(np.float64)
        t = (r - (1 - 1e-4) * ((r * hd).sum(1) / (hd * hd).sum(1))[:, None] * hd).astype(np.float32)
        sel = lane_order(h, t) > warp_order(h, t)
        hs.append(h[sel])
        ts.append(t[sel])
    return np.concatenate(hs), np.concatenate(ts)


def test_summation_orders_disagree():
    """The premise of the GPU test: near-orthogonal targets on which the two orders round differently exist."""
    h, t = mine_pairs()
    assert len(h) >= 4, len(h)
    assert (lane_order(h, t) > warp_order(h, t)).all()


@pytest.mark.gpu
def test_target_never_beats_itself():
    import literalkg_b200 as L
    from literalkg_b200 import ops

    h, t = mine_pairs()
    n = 64
    g = torch.Generator().manual_seed(5)
    for i in range(min(len(h), 8)):
        hv, tv = torch.from_numpy(h[i]), torch.from_numpy(t[i])
        # entity 0 = the head, 1 = the target, the rest score about -|h|^2 (clearly below the target's ~0)
        emb = torch.empty((n, DIM))
        emb[0], emb[1] = hv, tv
        emb[2:] = -hv * (1 + torch.rand((n - 2, 1), generator=g)) + 0.01 * torch.randn((n - 2, DIM), generator=g)
        emb = emb.cuda()
        cand = torch.arange(1, n, device="cuda")                  # the head is not a candidate of itself
        cmap = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        cmap[cand] = torch.arange(n - 1, dtype=torch.int32, device="cuda")
        heads, tpos = torch.zeros(1, dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
        tau = torch.empty(1, dtype=torch.float32, device="cuda")
        ranks = ops.score_rank(emb, heads, tpos, ops.ScoreIndex(emb, cand), tau_out=tau)
        assert ranks.tolist() == [0], (i, ranks.tolist())
        assert tau.item() == lane_order(h[i:i + 1], t[i:i + 1])[0]
        # a known tail that scores lower than the target is not subtracted: the filtered rank stays 0
        known = L.GraphPlan(*(torch.tensor(x, device="cuda") for x in ([0, 0], [5, 1], [0, 0])), n, 1)
        ops.filter_ranks(ranks, known, heads, tpos, cand_map=cmap, emb=emb, tau=tau)
        assert ranks.tolist() == [0], (i, ranks.tolist())
