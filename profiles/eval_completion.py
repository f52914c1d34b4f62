"""Knowledge-graph completion under the triple score (LiteralKG.evaluate_ranking(score="triple")) on one GPU; prints one
JSON line.

    python profiles/eval_completion.py [--queries 65536] [--entities 1000000] [--edges 20000000] [--dim 256]
                                       [--relation-dim 300] [--relations 64] [--batch 2048]

cfg 4-like shape: every entity is a candidate (1 M), G = 256, relation_dim = 300, R = 64, known set = a
synthetic.make_kg graph of 20 M triples, queries = 65 536 of its triples (every target is a known tail, so the filter
has work), batches of 2 048.  Embeddings as in eval_ranking.py (clustered rows); gat_trans_M and relation_embed at the
model's xavier initialisation.  Reported: queries/s of the whole call (host clock around a call that ends in its host
sync) for TransR tail prediction, TransR head prediction and TransE tail prediction, with the dot path at the same shape
beside them; CUDA-event milliseconds for one relation's candidate projection + operand build, and per batch for the
rank (lkg_l2_rank_rows + prepare + counting GEMM + finalize) and the filter; the mean band columns per query and the
number of queries whose band overflowed (exact scan).  Writes nothing to the tree."""
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


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()                                               # ends in the call's host sync
    return time.perf_counter() - t0, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=65536)
    ap.add_argument("--entities", type=int, default=1_000_000)
    ap.add_argument("--edges", type=int, default=20_000_000)
    ap.add_argument("--relations", type=int, default=64)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--relation-dim", type=int, default=300)
    ap.add_argument("--batch", type=int, default=2048)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_completion.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    torch.set_grad_enabled(False)
    import literalkg_b200 as L
    import literalkg_oracle as O
    from literalkg_b200 import model_bce, ops
    name, power = device_info()
    n, dev = a.entities, torch.device("cuda:0")

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
    out = {"metric": "filtered KG completion under the triple score, queries/s", "device": name,
           "power_limit_w": power,
           "shape": {"candidates": n, "dim": a.dim, "relation_dim": a.relation_dim, "queries": a.queries,
                     "batch": a.batch, "known_triples": kg.n_edges, "relations": a.relations}}
    kw = dict(known=known, all_embed=emb, batch_size=a.batch)
    warm = slice(0, 2 * a.batch)
    for label, m, score, predict in (("transr_tail", transr, "triple", "tail"), ("transr_head", transr, "triple", "head"),
                                     ("transe_tail", transe, "triple", "tail"), ("dot_tail", transr, "dot", "tail")):
        m.evaluate_ranking(qh[warm], qt[warm], qr[warm], score=score, predict=predict, **kw)
        dt, res = timed(lambda: m.evaluate_ranking(qh, qt, qr, score=score, predict=predict, **kw))
        out[label] = {"queries_per_s": a.queries / dt, "seconds": dt, "mrr": res["mrr"], "mr": res["mr"],
                      "hits@10": res["hits@10"]}

    # one relation, TransR tail prediction: projection + operand build, then per batch the rank and the filter
    r = int(torch.bincount(qr, minlength=a.relations).argmax())
    sel = torch.nonzero(qr == r).reshape(-1)
    w_r = transr.gat_trans_M[r].detach().t()
    e_r = transr.relation_embed.weight[r].detach().contiguous()
    table = torch.empty((n, a.relation_dim), dtype=torch.float32, device=dev)
    cand_planes = ops.split_planes(emb, None)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    index = None
    for rep in range(3):
        ev[0].record()
        ops.linear([cand_planes], w_r, None, out=table)
        index = ops.L2Index(table) if index is None else index.refill()
        ev[1].record()
    torch.cuda.synchronize()
    build_ms = ev[0].elapsed_time(ev[1])
    n_b = max(1, min(8, sel.numel() // a.batch))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(3 * n_b)]
    bands = []
    for rep in range(2):                                      # the first pass warms up
        bands = []
        for i in range(n_b):
            qs = sel[i * a.batch:(i + 1) * a.batch]
            q = ops.linear([ops.split_planes(emb, qh[qs])], w_r, e_r)
            tau = torch.empty(qs.numel(), dtype=torch.float32, device=dev)
            st = {}
            evs[3 * i].record()
            rk = ops.score_rank_l2(index, q, qt[qs], tau_out=tau, stats=st)
            evs[3 * i + 1].record()
            ops.filter_ranks_l2(rk, known, qh[qs], qt[qs], qr[qs], None, index, q, tau)
            evs[3 * i + 2].record()
            bands.append(st["band"])
    torch.cuda.synchronize()
    band = torch.cat(bands)
    out["one_relation"] = {
        "relation": r, "queries": int(sel.numel()), "batches_timed": n_b, "batch_queries": int(min(a.batch, sel.numel())),
        "projection_and_operand_ms": build_ms,
        "rank_ms_per_batch": sum(evs[3 * i].elapsed_time(evs[3 * i + 1]) for i in range(n_b)) / n_b,
        "filter_ms_per_batch": sum(evs[3 * i + 1].elapsed_time(evs[3 * i + 2]) for i in range(n_b)) / n_b,
        "band_columns_mean": float(band.double().mean()), "band_columns_max": int(band.max()),
        "band_overflow_queries": int((band > 8192).sum()),
    }
    # the dot rank path at the same batch, for comparison (prepare + GEMM at K = 256 + finalize)
    sindex = ops.ScoreIndex(emb, None)
    sindex.centered()
    evd = [torch.cuda.Event(enable_timing=True) for _ in range(2 * n_b)]
    for rep in range(2):
        for i in range(n_b):
            qs = sel[i * a.batch:(i + 1) * a.batch]
            evd[2 * i].record()
            ops.score_rank(emb, qh[qs], qt[qs], sindex)
            evd[2 * i + 1].record()
    torch.cuda.synchronize()
    out["one_relation"]["dot_rank_ms_per_batch"] = sum(evd[2 * i].elapsed_time(evd[2 * i + 1]) for i in range(n_b)) / n_b
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
