"""Filtered link-prediction evaluation (LiteralKG.evaluate_ranking) on one GPU; prints one JSON line.

    python profiles/eval_ranking.py [--queries 65536] [--entities 1000000] [--edges 20000000] [--dim 256]

cfg 4 shape: every entity is a candidate (1 M), G = 256, batches of 2 048 queries, known set = a synthetic.make_kg
graph of 20 M triples, queries = 65 536 of its triples (so every target is a known tail and the filter has work).
Embeddings: leaky_relu(N(0, 1) + a shared offset) * 0.21 like the cfg 4 rank test (clustered rows, as trained
embeddings are).  Reported: queries/s of the whole call filtering by (head, relation) and by head (host clock around a
call that ends in its one host sync), CUDA-event milliseconds per batch of the fused rank (lkg_rank_prepare +
lkg_score_rank + lkg_rank_finalize) and of the filter kernel, and the dense path at T = 396 on 118 candidates.
Writes nothing to the tree."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch


def device_info():
    name, power = torch.cuda.get_device_name(0), None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return name, power


def embeddings(n, dim, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.randn(n, dim, generator=g, device="cuda") + 0.5 * torch.randn(1, dim, generator=g, device="cuda")
    return torch.nn.functional.leaky_relu(base, 0.01) * 0.21


def timed_call(model, emb, q, rels, known, batch, candidates=None):
    """queries/s of one evaluate_ranking call (after a warm-up call on the first two batches) and its result."""
    qh, qt = q
    kw = dict(known=known, all_embed=emb, batch_size=batch, candidates=candidates)
    model.evaluate_ranking(qh[:2 * batch], qt[:2 * batch], None if rels is None else rels[:2 * batch], **kw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = model.evaluate_ranking(qh, qt, rels, **kw)            # ends in the call's host sync
    dt = time.perf_counter() - t0
    return qh.numel() / dt, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=65536)
    ap.add_argument("--entities", type=int, default=1_000_000)
    ap.add_argument("--edges", type=int, default=20_000_000)
    ap.add_argument("--relations", type=int, default=64)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--batch", type=int, default=2048)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_ranking.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    import literalkg_b200 as L
    import literalkg_oracle as O
    from literalkg_b200 import ops
    name, power = device_info()
    n, dev = a.entities, torch.device("cuda:0")

    kg = L.synthetic.make_kg(n, a.edges, a.relations, seed=5)
    known = L.GraphPlan(*(torch.from_numpy(x).to(dev) for x in (kg.h, kg.t, kg.r)), n, a.relations)
    pick = np.random.default_rng(7).choice(kg.n_edges, a.queries, replace=False)
    qh, qr, qt = (torch.from_numpy(x[pick]).to(dev) for x in (kg.h, kg.r, kg.t))
    cfg = O.OracleConfig(n_conv_layers=1, use_num_lit=False, use_txt_lit=False, mess_dropout=0.0)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    model = L.LiteralKG(args, n, a.relations).to(dev).eval()  # only evaluate_ranking's host logic is used
    emb = embeddings(n, a.dim, seed=5)
    out = {"metric": "filtered link-prediction evaluation, queries/s", "device": name, "power_limit_w": power,
           "shape": {"candidates": n, "dim": a.dim, "queries": a.queries, "batch": a.batch,
                     "known_triples": kg.n_edges, "relations": a.relations},
           "path": "fused" if ops.fused_topk_applicable(n, a.dim, 1) else "dense"}
    for label, rels in (("by_relation", qr), ("by_head", None)):
        qps, res = timed_call(model, emb, (qh, qt), rels, known, a.batch)
        out[label] = {"queries_per_s": qps, "mrr": res["mrr"], "hits@10": res["hits@10"], "mr": res["mr"]}

    # per batch: the fused rank (prepare + counting GEMM + finalize) and the filter kernel, CUDA events
    index = ops.ScoreIndex(emb, None)
    index.centered()
    n_b = min(16, a.queries // a.batch)
    split = {}
    for label, rels in (("by_relation", qr), ("by_head", None)):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * n_b)]
        tau = torch.empty(a.batch, dtype=torch.float32, device=dev)
        for rep in range(2):                                     # the first pass warms up
            for i in range(n_b):
                b = slice(i * a.batch, (i + 1) * a.batch)
                ev[3 * i].record()
                r = ops.score_rank(emb, qh[b], qt[b], index, tau_out=tau)
                ev[3 * i + 1].record()
                ops.filter_ranks(r, known, qh[b], qt[b], None if rels is None else qr[b], None, emb=emb, tau=tau)
                ev[3 * i + 2].record()
        torch.cuda.synchronize()
        rank_ms = sum(ev[3 * i].elapsed_time(ev[3 * i + 1]) for i in range(n_b)) / n_b
        filt_ms = sum(ev[3 * i + 1].elapsed_time(ev[3 * i + 2]) for i in range(n_b)) / n_b
        split[label] = {"rank_ms_per_batch": rank_ms, "filter_ms_per_batch": filt_ms, "filter_over_rank": filt_ms / rank_ms}
    out["per_batch"] = split

    # dense path: T = 396 (scale_gat_dim None at the reference dims), 118 candidates = the most frequent tails
    del index, emb
    emb396 = embeddings(n, 396, seed=6)
    cands = torch.from_numpy(np.argsort(-np.bincount(kg.t, minlength=n))[:118].copy()).to(dev)
    sel = torch.isin(qt, cands)
    qps, res = timed_call(model, emb396, (qh[sel], qt[sel]), qr[sel], known, a.batch, candidates=cands)
    out["dense_t396_118_candidates"] = {"queries": int(sel.sum()), "queries_per_s": qps, "mrr": res["mrr"],
                                        "path": "fused" if ops.fused_topk_applicable(118, 396, 1) else "dense"}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
