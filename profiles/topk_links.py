"""Filtered top-k link prediction under the dot score (LiteralKG.topk_links) on one GPU; prints one JSON line.

    python profiles/topk_links.py [--queries 65536] [--entities 1000000] [--edges 20000000] [--relations 64]
                                  [--dims 256,396] [--batch 2048] [--ks 10,100] [--sample-scale 1]

Every entity is a candidate (1 M); the known set is the 20 M-triple synthetic.make_kg graph of topk_completion.py,
excluded by (anchor, relation) run; the queries are 65 536 of its triples, batches of 2 048.  Per width in --dims
and k in --ks, queries/s of the whole call (host clock around a call that ends in a device synchronise, after a
warm-up call) for tail and head prediction, and the baselines on the same anchors without exclusion: the fused
ops.score_topk where the width allows it (<= 256), else today's only route, ops.score + ops.topk_rows per batch
(the dense B x N matrix).  Per width and k, on 4 batches of tail queries: CUDA-kernel milliseconds per batch of the
threshold, the counting GEMM and the finalize kernel (torch.profiler, a run of its own), listed columns per query
(mean, max) and overflowed queries; --sample-scale f1,f2,.. repeats those for multiples of the default sample
count.  The card's name and power limit go in the same line.  Writes nothing to the tree."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "profiles")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

from eval_ranking import device_info, embeddings

KERNELS = {"threshold": "topk_threshold_kernel<0>", "gemm": "tc_gemm_kernel", "finalize": "topk_finalize_kernel<0>"}


def kernel_times(emb, index, batches, k, n_sample, cap, exclude_of):
    """Per-batch kernel ms (torch.profiler) and listing statistics of ops.score_topk_dot over the given batches."""
    from literalkg_b200 import ops
    for a, ex in zip(batches, exclude_of):                    # warm-up
        ops.score_topk_dot(emb, a, k, index, exclude=ex, n_sample=n_sample, cap=cap)
    torch.cuda.synchronize()
    listed = []
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for a, ex in zip(batches, exclude_of):
            st = {}
            ops.score_topk_dot(emb, a, k, index, exclude=ex, n_sample=n_sample, cap=cap, stats=st)
            listed.append(st["listed"])
        torch.cuda.synchronize()
    ms = {key: 0.0 for key in KERNELS}
    for ev in prof.key_averages():
        for key, name in KERNELS.items():
            if name in ev.key:
                ms[key] += ev.device_time_total / 1000.0
    nb = len(batches)
    listed = torch.cat(listed)
    out = {f"{key}_ms_per_batch": v / nb for key, v in ms.items()}
    out.update(n_sample=n_sample, cap=cap, listed_mean=float(listed.double().mean()), listed_max=int(listed.max()),
               overflow_queries=int((listed > cap).sum()))
    return out


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=65536)
    ap.add_argument("--entities", type=int, default=1_000_000)
    ap.add_argument("--edges", type=int, default=20_000_000)
    ap.add_argument("--relations", type=int, default=64)
    ap.add_argument("--dims", default="256,396")
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--ks", default="10,100")
    ap.add_argument("--sample-scale", default="1")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_links.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    import literalkg_b200 as L
    import literalkg_oracle as O
    from literalkg_b200 import ops
    name, power = device_info()
    n, dev = a.entities, torch.device("cuda:0")
    ks = [int(x) for x in a.ks.split(",")]

    kg = L.synthetic.make_kg(n, a.edges, a.relations, seed=5)
    known = L.GraphPlan(*(torch.from_numpy(x).to(dev) for x in (kg.h, kg.t, kg.r)), n, a.relations)
    pick = np.random.default_rng(7).choice(kg.n_edges, a.queries, replace=False)
    qh, qr, qt = (torch.from_numpy(x[pick]).to(dev) for x in (kg.h, kg.r, kg.t))
    cfg = O.OracleConfig(n_conv_layers=1, use_num_lit=False, use_txt_lit=False, mess_dropout=0.0)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    m = L.LiteralKG(args, 16, a.relations).to(dev).eval()     # hosts the call; the embeddings are passed in
    out = {"metric": "filtered top-k link prediction under the dot score, known triples excluded, queries/s",
           "device": name, "power_limit_w": power,
           "shape": {"candidates": n, "dims": a.dims, "queries": a.queries, "batch": a.batch,
                     "known_triples": kg.n_edges, "relations": a.relations}}
    warm = slice(0, 2 * a.batch)
    for dim in [int(x) for x in a.dims.split(",")]:
        emb = embeddings(n, dim, seed=5)
        res = out[f"dim{dim}"] = {}
        for k in ks:
            for predict in ("tail", "head"):
                anchors = qh if predict == "tail" else qt
                kw = dict(relations=qr, known=known, predict=predict, batch_size=a.batch, all_embed=emb)
                m.topk_links(anchors[warm], k, **{**kw, "relations": qr[warm]})
                dt, (vals, ids) = timed(lambda: m.topk_links(anchors, k, **kw))
                res[f"{predict}_k{k}"] = {"queries_per_s": a.queries / dt, "seconds": dt,
                                          "padded": int((ids < 0).sum()),
                                          "mean_best_score": float(vals[:, 0].double().mean())}
            # the baseline on the same anchors, without exclusion
            index = ops.ScoreIndex(emb, None)
            bs = [qh[b0:b0 + a.batch] for b0 in range(0, a.queries, a.batch)]
            if ops.fused_topk_applicable(n, dim, k):
                label = "baseline_score_topk_unfiltered"

                def base(batches):
                    return [ops.score_topk(emb, b, None, k, tail_index=index) for b in batches]
            else:
                label = "baseline_dense_score_topk_rows_unfiltered"
                rec = ops.scale_from_data(emb)
                cols = torch.arange(n, device=dev)

                def base(batches):
                    return [ops.topk_rows(ops.score(emb, b, cols, rec=rec), k)[:2] for b in batches]
            base(bs[:2])                                          # warm-up
            dt, _ = timed(lambda: base(bs))
            res[f"{label}_k{k}"] = {"queries_per_s": a.queries / dt, "seconds": dt}
            # kernels on 4 batches of tail queries
            nb = min(4, len(bs))
            exclude_of = [(known, b, qr[i * a.batch:(i + 1) * a.batch], None) for i, b in enumerate(bs[:nb])]
            for f in [float(x) for x in a.sample_scale.split(",")]:
                s = max(k, min(n, int(f * ops.topk_l2_samples(n, k))))
                key = f"kernels_k{k}" if f == 1 else f"kernels_k{k}_x{f:g}"
                res[key] = kernel_times(emb, index, bs[:nb], k, s, ops.TOPK_L2_CAP, exclude_of)
            del index
        del emb
        torch.cuda.empty_cache()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
