#!/usr/bin/env python
"""Benchmark of the LiteralKG message-passing + scoring hot path on B200 (contract: see README / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole synthetic graph of BASELINE.json configs[2]
(N = 1 M entities, E = 20 M triples, R = 64 relations, D = 300, C = 32, L = 3 bi-interaction layers,
G = 256):  update_att (attention logits + duplicate merge + row softmax) followed by gat_embeddings
(literal gate, 3 aggregator layers, concat + linear_gat).  metric = triples (edges) processed per second.
`value`: inputs resident in HBM.  `e2e`: the same pass through the public API with the edge list uploaded from pinned
host memory for every step (double-buffered on a copy stream) and a slice of the result read back.
Also reported in the same JSON line: `roofline` of the dominant kernel (CUDA events on its stream inside the timed
region; ncu DRAM traffic from profiles/r01_traffic.json), `cpu_baseline` (the oracle port on the host cores, bounded
sample), the all-entity link-prediction scoring of configs[3] (2 048 heads x 1 M tails, fused top-10) and one
training step (fine-tuning loss, forward + backward to every parameter).  N > 1: head rows partitioned over the ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

METRIC = "edges/s, attention update + 3-layer bi-interaction aggregation pass"
UNIT = "edges/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--entities", type=int, default=1_000_000)
    ap.add_argument("--edges", type=int, default=20_000_000)
    ap.add_argument("--relations", type=int, default=64)
    ap.add_argument("--layers", type=int, default=3)
    ap.add_argument("--aggregator", default="bi-interaction")
    ap.add_argument("--score-heads", type=int, default=2048)
    ap.add_argument("--topk", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scoring", action="store_true")
    ap.add_argument("--no-training", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--config", default="3", choices=sorted(CONFIGS),
                    help="BASELINE.json workload: 3 = 1M / 20M bi-interaction (the metric's config, default); "
                         "5-gcn / 5-graphsage / 5-bi = 10M / 200M aggregator comparison; the per-stage extras "
                         "(scoring = cfg 4, training) ride along with cfg 3")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of what the last timed step computed (entity "
                         "embeddings and the attention matrix A_in) to DIR/<name>.npy, for comparing two builds; "
                         "with several ranks, rank 0 writes a sample of its own shard (its head rows), so compare "
                         "dumps taken with the same number of GPUs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    for k_, v_ in CONFIGS[a.config].items():
        setattr(a, k_, v_)
    return a


CONFIGS = {
    "3": {},
    "5-gcn": dict(entities=10_000_000, edges=200_000_000, aggregator="gcn", no_scoring=True, no_training=True),
    "5-graphsage": dict(entities=10_000_000, edges=200_000_000, aggregator="graphsage", no_scoring=True, no_training=True),
    "5-bi": dict(entities=10_000_000, edges=200_000_000, aggregator="bi-interaction", no_scoring=True, no_training=True),
}


def workload_name(a):
    return (f"cfg{a.config[0]}: synthetic power-law KG N={a.entities} E~{a.edges} R={a.relations}, D=300 C=32 L={a.layers} "
            f"{a.aggregator} + residual, G=256; update_att + gat_embeddings")


DTYPE = "f32 (GEMMs: fp16 hi/lo split operands, 3 tcgen05 products per k-step, fp32 TMEM accumulation: 2^-22)"


def oracle_config(a):
    import literalkg_oracle as O
    return O.OracleConfig(n_conv_layers=a.layers, aggregation_type=a.aggregator, mess_dropout=0.0)


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (pynvml; falls back to nvidia-smi polling)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.stop_flag = [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.thread = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                try:
                    bits = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, name in self.REASONS.items():
                    if bits & b and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def __enter__(self):
        if self.nv is not None:
            self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop_flag.set()
        if self.nv is not None:
            self.thread.join()

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path on a bounded sample of the same workload
# ------------------------------------------------------------------------------------------------
ENTITY_GAIN = 30.0     # the xavier-initialised entity table is ~3e-3: scaled up so that the attention logits spread
                       # (softmax far from uniform) in the parity leg; the timed legs do not care


def cpu_inputs(a, n, e, seed=2022):
    import literalkg_b200.synthetic as S
    import literalkg_oracle as O
    cfg = oracle_config(a)
    kg = S.make_kg(n, e, a.relations, seed=seed)
    num, txt = S.make_literals(n, seed=seed)
    p = O.init_params(cfg, n, a.relations, seed=seed)
    p["entity_embed.weight"] *= ENTITY_GAIN
    return cfg, kg, num, txt, p


def cpu_pass(a, n, e, seed=2022, repeats=1, warmup=0, inputs=None, dtype=torch.float32, keep=False):
    """The oracle port of the reference path (update_att + gat_embeddings) on the host cores.  Returns
    (n_edges, times) and, with ``keep``, the last pass's (indices, values, embeddings)."""
    import literalkg_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    cfg, kg, num, txt, p = inputs if inputs is not None else cpu_inputs(a, n, e, seed)
    if dtype != torch.float32:
        p, num, txt = O.cast_params(p, dtype), num.to(dtype), txt.to(dtype)
    h, t, r = (torch.from_numpy(x) for x in (kg.h, kg.t, kg.r))
    rels = list(range(a.relations))
    times, out = [], None
    with torch.no_grad():
        for i in range(warmup + repeats):
            t0 = time.perf_counter()
            idx, val = O.update_attention(p["entity_embed.weight"], p["relation_embed.weight"], h, t, r, rels, n)
            emb = O.gat_embeddings(p, cfg, idx, val, num, txt)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
            if keep:
                out = (idx, val, emb)
    return (kg.n_edges, times, out) if keep else (kg.n_edges, times)


def err_norm(x, ref):
    """max |x - ref| / max |ref| (the bound DESIGN.md states: 1e-3)."""
    return float((x.double() - ref.double()).abs().max() / ref.double().abs().max().clamp_min(1e-300))


def row_err_stats(x, ref, bound=1e-3):
    """Distribution over the entity rows of  max_j |x - ref| / max |ref|.  A handful of rows are ill conditioned in ANY
    fp32 evaluation (a LayerNorm over 32 channels whose inputs nearly cancel amplifies rounding by 10^3 - 10^4: the
    reference's own fp32 arithmetic is 1e-2 off float64 on its worst row of this graph), so the maximum alone says
    little; the quantiles and the number of rows over the bound are what the two fp32 evaluations are compared on."""
    ref = ref.double()
    d = (x.double() - ref).abs().max(dim=1).values / ref.abs().max().clamp_min(1e-300)
    ds = torch.sort(d).values
    q = lambda f: float(ds[min(len(ds) - 1, int(f * len(ds)))])
    return {"p50": q(0.5), "p99": q(0.99), "p999": q(0.999), "max": float(ds[-1]), "rows_over_bound": int((d > bound).sum()),
            "rows": int(len(ds))}


def parity_leg(a, dev, inputs, fp32_out):
    """Parity at bench scale: the CUDA path on the very graph / parameters the cpu_baseline leg just timed, against
    the oracle evaluated in float64 (the yardstick) -- with the oracle's own fp32 evaluation (= the reference's
    arithmetic) measured against the same yardstick beside it.  CSR structure bit exact; values to the bounds of
    DESIGN.md section 2."""
    import argparse as _ap
    import literalkg_b200 as L
    cfg, kg, num, txt, p = inputs
    n = kg.n_entities
    t0 = time.perf_counter()
    _, _, (idx64, val64, emb64) = cpu_pass(a, n, kg.n_edges, inputs=inputs, dtype=torch.float64, keep=True)
    t_f64 = time.perf_counter() - t0
    args = _ap.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    args.device = str(dev)
    m = L.LiteralKG(args, n, a.relations, None, num.to(dev), txt.to(dev))
    m.load_state_dict(p, strict=False)
    m = m.to(dev).eval()
    h, t, r = (torch.from_numpy(x).to(dev) for x in (kg.h, kg.t, kg.r))
    with torch.no_grad():
        m(h, t, r, list(range(a.relations)), device=dev, mode="update_att")
        emb = m.gat_embeddings().cpu()
    a_in = m.A_in.data
    csr_equal = bool(torch.equal(a_in.indices().cpu(), idx64))
    vals = a_in.values().cpu()
    idx32, val32, emb32 = fp32_out
    ours, floor = row_err_stats(emb, emb64), row_err_stats(emb32, emb64)
    out = {"graph": f"N={n} E={kg.n_edges} nnz={idx64.shape[1]} (the cpu_baseline sample), entity table x{ENTITY_GAIN:g}",
           "yardstick": "oracle evaluated in float64", "csr_equal": csr_equal,
           "attention_err": err_norm(vals, val64) if csr_equal else None,
           "attention_err_elementwise": float(((vals.double() - val64).abs() / val64).max()) if csr_equal else None,
           "embedding_row_err": ours, "fp32_oracle_embedding_row_err": floor,
           "fp32_oracle_attention_err": err_norm(val32, val64) if torch.equal(idx32, idx64) else None,
           "bound": 1e-3, "f64_oracle_s": round(t_f64, 1),
           "criterion": "CSR bit exact; attention < bound; 99.9 % of the embedding rows < bound; rows over it (ill "
                        "conditioned LayerNorm inputs, present in the reference's own fp32 arithmetic too) <= 1e-4 of "
                        "the rows"}
    out["ok"] = bool(csr_equal and out["attention_err"] < 1e-3 and ours["p999"] < 1e-3
                     and ours["rows_over_bound"] <= 1e-4 * ours["rows"])
    del m
    torch.cuda.empty_cache()
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # bounded sample: ~1e6 edges/s measured on the box's 16 host cores -> size the sample so that (K + W) steps
    # end within ~2 minutes
    steps = max(1, a.steps)
    budget_s = 120.0 / (steps + a.warmup)
    e = int(min(a.edges, max(50_000, budget_s * 1.0e6)))
    n = max(1000, int(a.entities * e / a.edges))
    n_edges, times = cpu_pass(a, n, e, repeats=steps, warmup=a.warmup)
    ms = 1e3 * float(np.mean(times))
    value = n_edges / (ms / 1e3)
    cores = torch.get_num_threads()
    sample = f"same generator scaled to N={n} E={n_edges} (reference temporaries at full size exceed a step budget)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
            "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a), "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(n, e, nnz, r, d, c, layers, bi=True):
    """Per-launch algorithmic bytes of the algorithm actually run (DESIGN.md section 5)."""
    att = e * (4 + 4 + 4 + 4 * d) + n * (4 * d + 8) + r * 4 * d + nnz * 4
    rterm = (2 if bi else 1) * 4 * c
    l1 = nnz * (4 + 4 + 4 * d) + n * (4 * d + 4 + rterm + 2 * 4 * c)
    lk = nnz * (4 + 4 + 4 * c) + n * (4 * c + 4 + rterm + 2 * 4 * c)
    return {"attn_update": att, f"aggregate_d{d}": l1, f"aggregate_d{c}": lk}


DUMP_EMBEDDING_BYTES = 32 << 20     # sampled embedding rows fill at most 32 MB
DUMP_ATTENTION_ENTRIES = 1 << 20    # sampled A_in entries: 4 MB of values + 16 MB of (head, tail) ids


def dump_outputs(out_dir, emb, a_in, row0):
    """Writes a seeded sample of one pass's outputs (at most ~52 MB) as float32 / float64 .npy files:
    embeddings [S, G] float32 (rows of gat_embeddings) with embedding_rows [S] (their entity ids), attention_values [M]
    float32 (A_in entries, coalesced order) with attention_indices [2, M] (their head and tail ids).  Ids are stored as
    float64, which holds them exactly.  The sample depends on the output shapes only, so two builds run with the same
    arguments are compared entry for entry.  Row partitioned, ``emb`` and ``a_in`` hold only this rank's head rows
    (``row0``: entity id of ``emb``'s first row), so the sample is of the shard and differs from a one-GPU dump."""
    os.makedirs(out_dir, exist_ok=True)
    rows, width = emb.shape
    pick = np.sort(np.random.default_rng(0).choice(rows, min(rows, DUMP_EMBEDDING_BYTES // (4 * width)), replace=False))
    nnz = a_in._nnz()
    apick = np.sort(np.random.default_rng(1).choice(nnz, min(nnz, DUMP_ATTENTION_ENTRIES), replace=False))
    pick, apick = (torch.from_numpy(x).to(emb.device) for x in (pick, apick))
    arrays = {"embeddings": emb[pick].float(), "embedding_rows": (pick + row0).double(),
              "attention_values": a_in._values()[apick].float(), "attention_indices": a_in._indices()[:, apick].double()}
    for name, x in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), x.cpu().numpy())


@torch.no_grad()
def run_ours(a):
    import torch.distributed as dist
    import literalkg_b200 as L
    from literalkg_b200 import ops
    import literalkg_oracle as O   # parameter shapes / init only (bench is allowed to use the oracle as checker)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # 128 MB all-gathers at 8 ranks: 0.30 ms with NCCL's default channel count, 0.21 ms with 32 (round-1 probe)
        os.environ.setdefault("NCCL_MIN_NCHANNELS", "32")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    cfg = oracle_config(a)
    n, n_rel = a.entities, a.relations
    kg = L.synthetic.make_kg(n, a.edges, n_rel)
    e = kg.n_edges
    num, txt = L.synthetic.make_literals(n, device=dev)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    args.device = str(dev)
    torch.manual_seed(2022)
    model = L.LiteralKG(args, n, n_rel, None, num, txt).to(dev).eval()
    rels = list(range(n_rel))
    part = None
    h_np, t_np, r_np = kg.h, kg.t, kg.r
    if world > 1:
        # head rows split over the ranks (SURVEY.md 8(e)), nnz-balanced contiguous ranges; the edge list is
        # pre-partitioned by head row (a rank uploads, sorts and keeps E / P triples), the raw parameter tables are
        # replicated, activations are exchanged per layer, embeddings stay sharded for the scoring
        from literalkg_b200.parallel import RowPartition
        part = RowPartition.balanced(n, kg.h)
        model.set_partition(part, local_edges=True)
        mine = (kg.h >= part.begin) & (kg.h < part.end)
        h_np, t_np, r_np = kg.h[mine], kg.t[mine], kg.r[mine]
    # pinned host copies of the (rank's) edge list, int32: the e2e arm uploads them every step like main.py:147-150
    h_pin, t_pin, r_pin = (torch.from_numpy(x.astype(np.int32)).pin_memory() for x in (h_np, t_np, r_np))
    h_dev, t_dev, r_dev = (x.to(dev) for x in (h_pin, t_pin, r_pin))

    def step():
        model(h_dev, t_dev, r_dev, rels, device=dev, mode="update_att")
        return model.gat_embeddings(gather=False)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sync()
    t_plan = time.perf_counter()
    emb = step()                    # first pass: builds the CSR plan of the edge list (radix sorts + emit kernels)
    sync()
    first_pass_ms = (time.perf_counter() - t_plan) * 1e3
    for _ in range(max(3, a.warmup)):
        emb = step()
    sync()
    nnz = model._agg_plan.nnz
    if world > 1:
        tn = torch.tensor([nnz], dtype=torch.int64, device=dev)
        dist.all_reduce(tn)
        nnz = int(tn.item())
    # timed region: the kernels the roofline is computed for are bracketed by CUDA events on their stream; every other
    # entry point is only counted (two event records per call are host time, which a 7 ms multi-GPU pass cannot hide).
    # The full per-call breakdown comes from two more passes after the timed region.
    roof_names = set(algorithmic_bytes(1, 1, 1, 1, cfg.embed_dim, cfg.conv_dim, 1))
    ops.PROFILE = ops.Profile(only=roof_names)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        sync()
        t_host = time.perf_counter()
        start.record()
        for _ in range(a.steps):
            emb = step()
        end.record()
        host_issue_ms = (time.perf_counter() - t_host) * 1e3 / a.steps     # time to enqueue a pass (no sync inside)
        sync()
    ms = start.elapsed_time(end) / a.steps
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, emb, model.A_in.data, 0 if part is None else part.begin)
    prof = ops.PROFILE
    kern = prof.summary()
    for v_ in kern.values():
        v_["passes"] = a.steps
    launches = prof.launches
    ops.PROFILE = ops.Profile()
    for _ in range(2):
        emb = step()
    sync()
    full = ops.PROFILE.summary()
    ops.PROFILE = None
    for k_, v_ in full.items():
        v_["passes"] = 2
        kern.setdefault(k_, v_)
    if world > 1:
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = tms.item()
    value = e / (ms / 1e3)

    # roofline of the dominant kernel
    ab = algorithmic_bytes(n, e, nnz, n_rel, cfg.embed_dim, cfg.conv_dim, cfg.n_conv_layers, a.aggregator == "bi-interaction")
    ab = {k_: v / world for k_, v in ab.items()}      # one launch covers this rank's 1 / world of the head rows
    dom = max((k for k in kern if k in ab), key=lambda k: kern[k]["ms_total"])
    achieved = ab[dom] / (kern[dom]["ms_avg"] / 1e3) / 1e9
    # ncu dram__bytes_read + write per launch of that kernel: measured per (config, GPU count) and committed under
    # profiles/ (ncu cannot run inside the timed bench); null when this configuration has no capture
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(f"cfg{a.config}/gpus{world}", {}).get(dom)
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": ab[dom], "kernel_ms_avg": kern[dom]["ms_avg"],
                "kernels": {k: {"ms_avg": round(v["ms_avg"], 4), "share": round(v["ms_total"] / v["passes"] / ms, 4),
                                **({"GBps": round(ab[k] / v["ms_avg"] / 1e6, 1)} if k in ab else {})}
                            for k, v in kern.items()},
                "host_issue_ms_per_step": host_issue_ms,
                "first_pass_ms_incl_plan_build": first_pass_ms}

    # e2e: public API with host buffers; H2D of the step's inputs and D2H of its result inside the timed region
    ids_pin = torch.arange(0, a.score_heads, dtype=torch.int64).pin_memory()
    out_pin = torch.empty((a.score_heads, emb.shape[1]), dtype=torch.float32).pin_memory()

    # Input pipeline: the step's edge list is uploaded from pinned memory on a copy stream into one of two device
    # buffers while the previous step computes (what a production loader does); every timed step still owns one full
    # H2D copy of its inputs and one D2H read of its result.
    copy_stream = torch.cuda.Stream(device=dev)
    slots = [tuple(torch.empty_like(x, device=dev) for x in (h_pin, t_pin, r_pin)) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    ids_dev = torch.empty(ids_pin.shape, dtype=torch.int64, device=dev)
    e_up = int(h_pin.numel())

    def upload(i):
        s_ = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s_])             # the step that last read this slot is done with it
            for dst, src in zip(slots[s_], (h_pin, t_pin, r_pin)):
                dst.copy_(src, non_blocking=True)
            ready[s_].record(copy_stream)

    def e2e_step(i):
        s_ = i % 2
        torch.cuda.current_stream().wait_event(ready[s_])
        upload(i + 1)                                        # next step's inputs travel while this one computes
        hd, td, rd = slots[s_]
        ids_dev.copy_(ids_pin, non_blocking=True)
        model(hd, td, rd, rels, device=dev, mode="update_att")
        consumed[s_].record()
        if part is None:
            res = model.get_final_embeddings(ids_dev)
        else:       # every rank reads back the first rows of its own shard
            res = model.gat_embeddings(gather=False)[:a.score_heads]
        out_pin[:res.shape[0]].copy_(res, non_blocking=True)

    for c_ in consumed:
        c_.record()
    upload(0)
    for i in range(2):
        e2e_step(i)
    sync()
    start.record()
    for i in range(2, 2 + a.steps):
        e2e_step(i)
    end.record()
    sync()
    e2e_ms = start.elapsed_time(end) / a.steps
    if world > 1:
        tms = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        e2e_ms = tms.item()
    e2e = {"value": e / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": int(3 * e_up * 4 + ids_pin.numel() * 8), "d2h_bytes_per_step": int(out_pin.numel() * 4),
           "input": ("int32 (h, t, r) lists" if world == 1 else
                     "this rank's head-row slice of the int32 (h, t, r) lists (bytes are per rank)")}

    scoring = None
    if not a.no_scoring:
        # cfg 4: head batches of 2 048 against all N tails, top-k fused into the scoring GEMM.  The timed region
        # builds the tail index once (it only depends on the embedding matrix) and scores `nb` head batches.
        nb = 8
        batches = [(torch.arange(0, a.score_heads, device=dev) * 487 + b * 7919) % n for b in range(nb)]

        def scoring_pass():
            out = None
            if part is None:
                ti = ops.ScoreIndex(emb, None)
                for hb in batches:
                    out = model.topk(hb, None, a.topk, all_embed=emb, tail_index=ti)
            else:   # tails sharded by row ownership, per-rank fused top-k, k-way merge
                ti = model.sharded_index(emb)
                out = model.topk_sharded(batches, a.topk, emb, tail_index=ti)   # one round of collectives for all
            return out

        for _ in range(2):
            scoring_pass()
        sync()
        ops.PROFILE = ops.Profile()
        ks = max(2, min(a.steps, 5))
        start.record()
        for _ in range(ks):
            scoring_pass()
        end.record()
        sync()
        sprof = ops.PROFILE.summary()
        ops.PROFILE = None
        sms = start.elapsed_time(end) / (ks * nb)
        if world > 1:
            tms = torch.tensor([sms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            sms = tms.item()
        flops = 2.0 * a.score_heads * n * emb.shape[1]
        tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0)) * world
        scoring = {"metric": f"triples/s, all-entity scoring {a.score_heads} heads x {n} tails, G={emb.shape[1]}, fused top-{a.topk}",
                   "value": a.score_heads * n / (sms / 1e3), "unit": "triples/s", "ms_per_batch": sms,
                   "batches_per_index_build": nb,
                   "tflops": flops / (sms / 1e3) / 1e12, "tensor_peak_tflops": tpeak,
                   "frac_of_tensor_peak": flops / (sms / 1e3) / 1e12 / tpeak,
                   "dtype": "f16 filter GEMM (1 product) + exact fp64-accumulated re-score of the candidates",
                   "calls": {k_: round(v["ms_avg"], 4) for k_, v in sprof.items()}}

    ranking = None
    if not a.no_scoring and part is None:
        # north star (d): rank of a given tail per head, fused -- the 3-product scoring GEMM with a counting epilogue +
        # exact re-score of the few columns inside the error band; no B x N score matrix.  Two target sets: the tail
        # that is 38th best for its head (what a link-prediction evaluation ranks: positives sit near the top; doubles
        # as an exactness check, every rank must come out as 37) and arbitrary tails (mid-ranked: the densest part of
        # the score distribution, the worst case for the band).
        ti = ops.ScoreIndex(emb, None)
        ti.centered()
        hb = batches[0]
        _, top_pos = ops.score_topk(emb, hb, None, 100, tail_index=ti)
        targets = {"top": top_pos[:, 37].contiguous(), "arbitrary": (hb * 31 + 17) % n}
        ranking = {"metric": f"triples/s, rank of a given tail per head, {a.score_heads} heads x {n} tails, fused (no score matrix)",
                   "unit": "triples/s"}
        for name, tgt in targets.items():
            for _ in range(2):
                ops.score_rank(emb, hb, tgt, ti)
            sync()
            start.record()
            for _ in range(3):
                ranks = ops.score_rank(emb, hb, tgt, ti)
            end.record()
            sync()
            rms = start.elapsed_time(end) / 3
            if name == "top":
                ranking.update(value=a.score_heads * n / (rms / 1e3), ms_per_batch=rms,
                               issued_tflops=3 * 2.0 * a.score_heads * n * emb.shape[1] / (rms / 1e3) / 1e12,
                               all_ranks_equal_37=bool((ranks == 37).all()))
            else:
                # checker: the first 32 heads against float64 scoring (exact products, fp64 sums, one rounding, ties by position)
                e64 = emb.double()
                s64 = (e64[hb[:32]] @ e64.t()).float()
                tg = torch.gather(s64, 1, tgt[:32].unsqueeze(1))
                posn = torch.arange(n, device=dev).unsqueeze(0)
                ref_rank = ((s64 > tg) | ((s64 == tg) & (posn < tgt[:32].unsqueeze(1)))).sum(1)
                ranking.update(arbitrary_targets_ms_per_batch=rms, arbitrary_targets_mean_rank=float(ranks.float().mean()),
                               arbitrary_first_32_heads_equal_float64_ranking=bool(torch.equal(ranks[:32], ref_rank)))
                del e64, s64
        ranking["frac_of_tensor_peak_issued"] = ranking["issued_tflops"] / float(peaks.get("bf16_tflops_sustained", 1400.0))

    projected = None
    if not a.no_scoring and part is None and a.entities <= 2_000_000:
        # north star (b), extension: relation-projected attention v = (e_t W_r) . tanh(e_h W_r + e_r) with an explicit
        # W [R, D, D]: two chained tensor-core GEMMs per relation bucket over the (head, relation) runs + one gather per triple
        gw = torch.Generator(device=dev).manual_seed(1)
        w_rel = torch.randn(n_rel, cfg.embed_dim, cfg.relation_dim, generator=gw, device=dev) / cfg.embed_dim ** 0.5
        keep_a = (model._agg_plan, model._agg_values, model.A_in.data)
        model(h_dev, t_dev, r_dev, rels, w_rel, device=dev, mode="update_att_projected")      # warm-up: run bookkeeping
        sync()
        ops.PROFILE = ops.Profile()
        start.record()
        for _ in range(2):
            model(h_dev, t_dev, r_dev, rels, w_rel, device=dev, mode="update_att_projected")
        end.record()
        sync()
        pprof = ops.PROFILE.summary()
        ops.PROFILE = None
        pms = start.elapsed_time(end) / 2
        n_runs = model._att_plan.runs()["n_runs"]
        gemm_ms = sum(v["ms_total"] for k_, v in pprof.items() if k_.startswith("linear_")) / 2
        pflops = 3 * 2 * 2.0 * n_runs * cfg.embed_dim * cfg.relation_dim                      # two GEMMs, three products
        projected = {"metric": "edges/s, relation-projected attention update (extension)", "value": e / (pms / 1e3),
                     "unit": UNIT, "ms_per_update": pms, "head_relation_runs": n_runs,
                     "gemm_ms": gemm_ms, "gemm_issued_tflops": pflops / (gemm_ms / 1e3) / 1e12 if gemm_ms else None,
                     "calls_ms_per_update": {k_: round(v["ms_total"] / 2, 3) for k_, v in
                                             sorted(pprof.items(), key=lambda kv: -kv[1]["ms_total"])}}
        model._agg_plan, model._agg_values = keep_a[0], keep_a[1]
        model.A_in.data = keep_a[2]
        model._a_in_epoch += 1
        del w_rel
        torch.cuda.empty_cache()

    training = None
    if not a.no_training:
        # one optimisation step's worth of kernels: fine-tuning (BPR) loss on the reference's effective minibatch of
        # 681 triples (SURVEY.md appendix A), full-graph forward with saved activations + backward to every parameter
        # (main.py:222-226: loss.backward()); reported next to the inference pass, not part of `value`
        with torch.enable_grad():
            model.train()
            for layer in model.aggregator_layers:
                layer.dropout = 0.1                      # argument.py default mess_dropout
            gen = torch.Generator(device=dev).manual_seed(0)
            bh, bp, bn = (torch.randint(0, n, (681,), device=dev, generator=gen) for _ in range(3))

            def train_step():
                for prm in model.parameters():
                    prm.grad = None
                loss = model(bh, bp, bn, device=dev, mode="fine_tuning")
                loss.backward()
                return loss

            for _ in range(2):
                train_step()
            sync()
            kt = max(2, min(a.steps, 5))
            start.record()
            for _ in range(kt):
                loss = train_step()
            end.record()
            sync()
            # per-entry-point breakdown from separate steps: two event records per call would otherwise sit inside the
            # timed region (~300 per step)
            ops.PROFILE = ops.Profile()
            for _ in range(kt):
                train_step()
            tprof = ops.PROFILE.summary()
            ops.PROFILE = None
            model.eval()
            for layer in model.aggregator_layers:
                layer.dropout = 0.0
        tms = start.elapsed_time(end) / kt
        if world > 1:
            tt = torch.tensor([tms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            tms = tt.item()
        training = {"metric": "edges/s, fine-tuning step (forward with saved activations + backward to all parameters, "
                              "batch 681, dropout 0.1)", "value": e / (tms / 1e3), "unit": UNIT, "ms_per_step": tms,
                    "loss": float(loss), "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9,
                    "calls_ms_per_step": {k_: round(v["ms_total"] / kt, 3) for k_, v in
                                          sorted(tprof.items(), key=lambda kv: -kv[1]["ms_total"])}}

    cpu_baseline = parity = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        ns, es = 500_000, 10_000_000                                # ~10 s of CPU work on 16 cores
        ns, es = min(ns, max(1000, n // 2)), min(es, max(20_000, a.edges // 2))
        inputs = cpu_inputs(a, ns, es)
        n_edges, times, fp32_out = cpu_pass(a, ns, es, repeats=1, warmup=0, inputs=inputs, keep=True)
        cpu_baseline = {"value": n_edges / times[0], "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"oracle port (fp32), same generator scaled to N={ns} E={n_edges}, one pass {times[0]:.1f} s"}
        if not a.no_parity:
            parity = parity_leg(a, dev, inputs, fp32_out)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE,
                "data": "synthetic", "impl": "ours",
                "config": {"workload": workload_name(a), "entities": n, "edges": e, "unique_pairs": nnz,
                           "relations": n_rel,
                           "parallelism": ("single GPU" if world == 1 else
                                           f"head rows split over {world} GPUs (nnz-balanced ranges, pre-partitioned edge "
                                           "list), per-layer exchange of the ego rows (symmetric-memory push over NVLink, "
                                           "NCCL fallback), tails sharded for scoring"),
                           "cache": "inputs (entity tables 1.2 GB each, 25 GB gathered per kernel) "
                           "are far larger than the 126 MB L2; no explicit flush"},
                "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity, "e2e": e2e, "gpu_launches": launches,
                "clocks": clocks.result(), "scoring": scoring, "ranking": ranking, "projected_attention": projected,
                "training": training}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    # The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner) write to fd 1 too, so the
    # process-level stdout is pointed at stderr for the whole run and the line goes to a private copy of the real one.
    global print
    real_stdout = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    builtin_print = print

    def print(*args, **kw):            # noqa: A001 -- the two run_* functions print exactly one line each
        kw["file"] = real_stdout
        builtin_print(*args, **kw)
        real_stdout.flush()

    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
