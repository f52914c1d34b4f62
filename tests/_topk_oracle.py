"""Reference restatement of relation-aware top-k completion (LiteralKG.topk_triple / ops.score_topk_l2), used by
tests/test_topk_triple_*.py: distances rounded once from float64, and per query the k candidates not excluded in
(distance, position) order, padded with +inf / -1."""
import torch


def dist_of(query, cand):
    """d = |q - p_j|^2 with differences and squares in float64, summed, rounded once to fp32; [B, Nc] on the device of
    the inputs, one query at a time."""
    cand = cand.double()
    return torch.stack([((cand - q.double()) ** 2).sum(1).float() for q in query])


def topk_of(d, k, excluded=()):
    """One query: ``d`` the distances of the candidates in position order, ``excluded`` a set of positions.
    -> (dist fp32 [k], pos int64 [k]): the k positions not excluded ordered by (d ascending, position ascending)."""
    d = [float(x) for x in d]
    keep = sorted((x, p) for p, x in enumerate(d) if p not in set(excluded))[:k]
    dist = [x for x, _ in keep] + [float("inf")] * (k - len(keep))
    pos = [p for _, p in keep] + [-1] * (k - len(keep))
    return torch.tensor(dist, dtype=torch.float32), torch.tensor(pos, dtype=torch.int64)


def topk_rows_of(d, k, excluded=None):
    """``topk_of`` for every row of ``d`` [B, Nc] (any device); ``excluded`` (bool [B, Nc] or None) marks the excluded
    positions.  A stable sort of each row's kept distances gives the (d, position) order."""
    b = d.shape[0]
    dist = torch.full((b, k), float("inf"), dtype=torch.float32, device=d.device)
    pos = torch.full((b, k), -1, dtype=torch.int64, device=d.device)
    for i in range(b):
        keep = torch.arange(d.shape[1], device=d.device) if excluded is None else torch.nonzero(~excluded[i]).reshape(-1)
        s = torch.sort(d[i, keep], stable=True)
        m = min(k, keep.numel())
        dist[i, :m] = s.values[:m]
        pos[i, :m] = keep[s.indices[:m]]
    return dist, pos


def excluded_positions(anchors, rels, cand_ids, known):
    """Per query the positions of the candidates whose entity is in { e : (anchor, rel, e) in known } (bool [B, Nc])."""
    by_key = {}
    for h, r, t in known:
        by_key.setdefault((int(h), int(r)), set()).add(int(t))
    cand_ids = [int(c) for c in cand_ids]
    out = torch.zeros((len(anchors), len(cand_ids)), dtype=torch.bool)
    for i, (a, r) in enumerate(zip(anchors, rels)):
        s = by_key.get((int(a), int(r)), set())
        out[i] = torch.tensor([c in s for c in cand_ids])
    return out
