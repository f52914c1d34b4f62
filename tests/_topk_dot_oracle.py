"""Reference restatement of filtered top-k link prediction under the dot score (LiteralKG.topk_links /
ops.score_topk_dot), used by tests/test_topk_links_*.py: dot products rounded once from float64, and per query the k
candidates not excluded in (score descending, position) order, padded with -inf / -1.  ``excluded_positions`` (the
(anchor, relation) filter set) is the one of the triple-score restatement."""
import torch

from _topk_oracle import excluded_positions  # noqa: F401 -- the relation-keyed filter set, shared


def dot_of(query, cand):
    """s = q . t_j with the fp32 products exact in float64, summed in float64, rounded once to fp32; [B, Nc] on the
    device of the inputs, one query at a time."""
    cand = cand.double()
    return torch.stack([(cand @ q.double()).float() for q in query])


def best_of(s, k, excluded=()):
    """``topk_of`` for a score where larger is better: the k positions not excluded ordered by (s descending, position
    ascending), padded with -inf / -1."""
    s = [float(x) for x in s]
    keep = sorted((-x, p) for p, x in enumerate(s) if p not in set(excluded))[:k]
    vals = [-x for x, _ in keep] + [float("-inf")] * (k - len(keep))
    pos = [p for _, p in keep] + [-1] * (k - len(keep))
    return torch.tensor(vals, dtype=torch.float32), torch.tensor(pos, dtype=torch.int64)


def best_rows_of(s, k, excluded=None):
    """``best_of`` for every row of ``s`` [B, Nc] (any device): a stable descending sort of each row's kept scores."""
    b = s.shape[0]
    vals = torch.full((b, k), float("-inf"), dtype=torch.float32, device=s.device)
    pos = torch.full((b, k), -1, dtype=torch.int64, device=s.device)
    for i in range(b):
        keep = torch.arange(s.shape[1], device=s.device) if excluded is None else torch.nonzero(~excluded[i]).reshape(-1)
        srt = torch.sort(s[i, keep], descending=True, stable=True)
        m = min(k, keep.numel())
        vals[i, :m] = srt.values[:m]
        pos[i, :m] = keep[srt.indices[:m]]
    return vals, pos


def excluded_any_relation(anchors, cand_ids, known):
    """Per query the positions of the candidates whose entity is in { e : (anchor, any r, e) in known } (bool [B, Nc])."""
    by_head = {}
    for h, _, t in known:
        by_head.setdefault(int(h), set()).add(int(t))
    cand_ids = [int(c) for c in cand_ids]
    out = torch.zeros((len(anchors), len(cand_ids)), dtype=torch.bool)
    for i, a in enumerate(anchors):
        s = by_head.get(int(a), set())
        out[i] = torch.tensor([c in s for c in cand_ids])
    return out
