"""Reference restatement of filtered link-prediction ranking (LiteralKG.evaluate_ranking), used by
tests/test_rank_filtered_*.py: the raw rank of ``literalkg_oracle.rank_of`` minus the known true tails that beat the
target, and the MR / MRR / Hits@k computed from the ranks."""
import numpy as np
import torch

import literalkg_oracle as O


def filtered_rank_of(all_embed, head_ids, tail_ids, target_pos, known, relations=None, scores=None):
    """Filtered rank: ``O.rank_of`` minus the filter tails that beat the target under the same rule on the same
    scores.  ``known``: (h, r, t) triples.  Query i's filter set is { t' : (h_i, r_i, t') in known } when ``relations``
    is given, else { t' : (h_i, any r, t') in known }; a tail counts once however often it is known, the target itself
    and tails outside ``tail_ids`` never.  ``scores``: the [B, Nt] matrix to rank on (default ``O.calc_score``)."""
    s = O.calc_score(all_embed, head_ids, tail_ids) if scores is None else scores
    head_ids, target_pos = [int(x) for x in head_ids], [int(x) for x in target_pos]
    where = {int(t): p for p, t in enumerate(tail_ids)}
    by_key = {}
    for h, r, t in known:
        by_key.setdefault((int(h), int(r)), set()).add(int(t))
        by_key.setdefault((int(h), None), set()).add(int(t))
    out = []
    for i, (h, tp) in enumerate(zip(head_ids, target_pos)):
        row = s[i]
        st = row[tp]
        rank = int(((row > st) | ((row == st) & (torch.arange(row.numel(), device=row.device) < tp))).sum())
        key = (h, None if relations is None else int(relations[i]))
        for f in by_key.get(key, ()):
            p = where.get(f)
            if p is not None and p != tp and (row[p] > st or (row[p] == st and p < tp)):
                rank -= 1
        out.append(rank)
    return torch.tensor(out, dtype=torch.int64)


def ranking_metrics(ranks, ks=(1, 3, 10)):
    """MR = mean(rank + 1), MRR = mean(1 / (rank + 1)), Hits@k = mean(rank < k) over 0-based ranks, in float64."""
    r = np.asarray(ranks, dtype=np.float64)
    out = {"mr": float(np.mean(r + 1.0)), "mrr": float(np.mean(1.0 / (r + 1.0)))}
    out.update({f"hits@{k}": float(np.mean(r < k)) for k in ks})
    return out
