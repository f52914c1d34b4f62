"""Relation-aware top-k completion under the triple score (LiteralKG.topk_triple) on one GPU; prints one JSON line.

    python profiles/topk_completion.py [--queries 65536] [--entities 1000000] [--edges 20000000] [--dim 256]
                                       [--relation-dim 300] [--relations 64] [--batch 2048] [--ks 10,100]
                                       [--sample-scale 1]

The shape of eval_completion.py: every entity is a candidate (1 M), G = 256, relation_dim = 300, R = 64, the known set
a synthetic.make_kg graph of 20 M triples (left out of the results), queries = 65 536 of its triples, batches of 2 048.
Reported: queries/s of the whole call (host clock around a call that ends in a device synchronise, after a warm-up
call) for k in --ks, for TransR tail, TransR head and TransE tail prediction; for one relation (TransR tail) the
CUDA-kernel milliseconds per batch of the threshold, the counting GEMM and the finalize kernel (torch.profiler, a run
of its own), listed columns per query (mean, max), the overflowed queries and theta; with --sample-scale f1,f2,.. the
same per-batch numbers for those multiples of the default sample count.  Writes nothing to the tree."""
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

KERNELS = {"threshold": "topk_threshold_kernel<1>", "gemm": "tc_gemm_kernel", "finalize": "topk_finalize_kernel<1>"}


def one_relation(index, queries, k, n_sample, cap, exclude_of):
    """Per-batch kernel ms (torch.profiler) and listing statistics of ops.score_topk_l2 over the given batches."""
    from literalkg_b200 import ops
    for q, ex in zip(queries, exclude_of):                    # warm-up
        ops.score_topk_l2(index, q, k, exclude=ex, n_sample=n_sample, cap=cap)
    torch.cuda.synchronize()
    listed, theta = [], []
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for q, ex in zip(queries, exclude_of):
            st = {}
            ops.score_topk_l2(index, q, k, exclude=ex, n_sample=n_sample, cap=cap, stats=st)
            listed.append(st["listed"])
            theta.append(st["theta"])
        torch.cuda.synchronize()
    ms = {key: 0.0 for key in KERNELS}
    for ev in prof.key_averages():
        for key, name in KERNELS.items():
            if name in ev.key:
                ms[key] += ev.device_time_total / 1000.0
    nb = len(queries)
    listed = torch.cat(listed)
    out = {f"{key}_ms_per_batch": v / nb for key, v in ms.items()}
    out.update(n_sample=n_sample, cap=cap,
               listed_mean=float(listed.double().mean()), listed_max=int(listed.max()),
               overflow_queries=int((listed > cap).sum()), theta_mean=float(torch.cat(theta).double().mean()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=65536)
    ap.add_argument("--entities", type=int, default=1_000_000)
    ap.add_argument("--edges", type=int, default=20_000_000)
    ap.add_argument("--relations", type=int, default=64)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--relation-dim", type=int, default=300)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--ks", default="10,100")
    ap.add_argument("--sample-scale", default="1")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_completion.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    import literalkg_b200 as L
    import literalkg_oracle as O
    from literalkg_b200 import model_bce, ops
    name, power = device_info()
    n, dev = a.entities, torch.device("cuda:0")
    ks = [int(x) for x in a.ks.split(",")]

    kg = L.synthetic.make_kg(n, a.edges, a.relations, seed=5)
    known = L.GraphPlan(*(torch.from_numpy(x).to(dev) for x in (kg.h, kg.t, kg.r)), n, a.relations)
    pick = np.random.default_rng(7).choice(kg.n_edges, a.queries, replace=False)
    qh, qr, qt = (torch.from_numpy(x[pick]).to(dev) for x in (kg.h, kg.r, kg.t))
    emb = embeddings(n, a.dim, seed=5)

    def model(cls, relation_dim):
        cfg = O.OracleConfig(n_conv_layers=1, use_num_lit=False, use_txt_lit=False, mess_dropout=0.0,
                             scale_gat_dim=a.dim, relation_dim=relation_dim)
        args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
        return cls(args, n, a.relations).to(dev).eval()

    transr, transe = model(L.LiteralKG, a.relation_dim), model(model_bce.LiteralKG, a.dim)
    out = {"metric": "top-k KG completion under the triple score, known triples excluded, queries/s", "device": name,
           "power_limit_w": power,
           "shape": {"candidates": n, "dim": a.dim, "relation_dim": a.relation_dim, "queries": a.queries,
                     "batch": a.batch, "known_triples": kg.n_edges, "relations": a.relations}}
    kw = dict(known=known, all_embed=emb, batch_size=a.batch)
    warm = slice(0, 2 * a.batch)
    for k in ks:
        for label, m, predict in (("transr_tail", transr, "tail"), ("transr_head", transr, "head"),
                                  ("transe_tail", transe, "tail")):
            anchors = qh if predict == "tail" else qt
            m.topk_triple(anchors[warm], qr[warm], k, predict=predict, **kw)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dist, ids = m.topk_triple(anchors, qr, k, predict=predict, **kw)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out[f"{label}_k{k}"] = {"queries_per_s": a.queries / dt, "seconds": dt,
                                    "padded": int((ids < 0).sum()), "mean_best_distance": float(dist[:, 0].double().mean())}

    # one relation, TransR tail prediction: the candidate table and its index once, then per batch the three kernels
    r = int(torch.bincount(qr, minlength=a.relations).argmax())
    sel = torch.nonzero(qr == r).reshape(-1)
    w_r = transr.gat_trans_M[r].detach().t()
    e_r = transr.relation_embed.weight[r].detach().contiguous()
    table = torch.empty((n, a.relation_dim), dtype=torch.float32, device=dev)
    ops.linear([ops.split_planes(emb, None)], w_r, None, out=table)
    index = ops.L2Index(table)
    n_b = max(1, min(8, sel.numel() // a.batch))
    batches = [sel[i * a.batch:(i + 1) * a.batch] for i in range(n_b)]
    queries = [ops.linear([ops.split_planes(emb, qh[qs])], w_r, e_r) for qs in batches]
    exclude_of = [(known, qh[qs], qr[qs], None) for qs in batches]
    out["one_relation"] = {"relation": r, "queries": int(sel.numel()), "batches_timed": n_b,
                           "batch_queries": int(batches[0].numel())}
    for k in ks:
        for f in [float(x) for x in a.sample_scale.split(",")]:
            s = max(k, min(n, int(f * ops.topk_l2_samples(n, k))))
            key = f"k{k}" if f == 1 else f"k{k}_x{f:g}"
            out["one_relation"][key] = one_relation(index, queries, k, s, ops.TOPK_L2_CAP, exclude_of)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
