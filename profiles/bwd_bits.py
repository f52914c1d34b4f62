#!/usr/bin/env python
"""Bit identity of the backward kernels between two builds.

    python profiles/bwd_bits.py dump DIR [--root TREE]     # outputs of TREE's build (default: this tree) -> DIR
    python profiles/bwd_bits.py compare A B [A2]           # A, B: dumps of two builds; A2: a second run of A's build

`dump` runs lkg_layer_bwd_rows, lkg_gate_bwd and lkg_leaky_bwd on seeded inputs (aligned rows and rows placed one float
into wider buffers, with their scale records), and one fine-tuning step (forward with saved activations, backward to
every parameter) per aggregator on a seeded synthetic graph, and writes every output as int32 bit patterns: torch.equal
would take -0 and +0 for equal.  `compare` reports per output whether A and B are bit-equal.  The outputs that atomics
reduce in a varying order (dgamma / dbeta over many CTAs, every parameter gradient of the training step) are taken REPS
times per dump and differ between runs of one build; with A2 they are held to the spread of the A runs instead: the
median relative L2 distance of a B run to an A run at most twice the median distance between two A runs.
"""
import argparse
import hashlib
import itertools
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 100_000
REPS = 3


def placed(t, off):
    """t as a view `off` floats into a wider buffer (off = 0: t itself)."""
    import torch
    if not off:
        return t
    buf = torch.zeros(t.shape[0], t.shape[1] + off, device=t.device)
    buf[:, off:] = t
    return buf[:, off:]


def layer_cases(ops, out):
    import torch
    dev = "cuda"
    for c, off in ((10, 0), (32, 0), (50, 0), (64, 0), (32, 1), (48, 1)):
        g = torch.Generator(device=dev).manual_seed(c + 100 * off)
        o = torch.randn(N, 2 * c, generator=g, device=dev)
        y = torch.randn(N, c, generator=g, device=dev)
        mask = (torch.rand(N, c, generator=g, device=dev) < 0.8).float() / 0.8
        dy = torch.randn(N, c, generator=g, device=dev)
        dyn = torch.randn(N, c, generator=g, device=dev) * 1e-2
        lw = torch.rand(c, generator=g, device=dev) + 0.5
        vec = c % 4 == 0 and off == 0
        n_one = 8 * 32 // ((8 if c <= 32 else 16) if vec else 32)          # the rows one CTA of 8 warps covers
        negzero = dyn.clone()
        negzero[::7] = -0.0                                                # rows whose dyn is all -0.0
        for has_o2, use_mask, use_dy, use_dyn in itertools.product((0, 1), repeat=4):
            for n in (N, n_one):
                run_layer(ops, out, f"layer_c{c}_off{off}_o2{has_o2}_m{use_mask}_dy{use_dy}_dyn{use_dyn}_n{n}", n, c, off,
                          has_o2, o, y, mask if use_mask else None, dy if use_dy else None, dyn if use_dyn else None, lw)
        run_layer(ops, out, f"layer_c{c}_off{off}_negzero_dyn", N, c, off, 1, o, y, mask, None, negzero, lw)


def run_layer(ops, out, key, n, c, off, has_o2, o, y, mask, dy, dyn, lw):
    import torch
    nt = 2 if has_o2 else 1
    sl = lambda t: None if t is None else t[:n].contiguous()
    for r in range(REPS if n == N else 1):                            # dgb over many CTAs: atomics in varying order
        d_o = placed(torch.zeros(n, nt * c, device="cuda"), off)
        dgb = torch.zeros(2 * c, device="cuda")
        rec, rec2 = ops.raw_record("cuda"), ops.raw_record("cuda")
        ops.layer_bwd_rows(placed(y[:n], off), placed(o[:n, :nt * c].contiguous(), off), bool(has_o2), sl(mask), sl(dy),
                           sl(dyn), lw, d_o, dgb, amax=rec, amax2=rec2)
        out[f"{key}/dgb/r{r}"] = dgb
    out[key + "/d_o"], out[key + "/rec"], out[key + "/rec2"] = d_o, rec, rec2


def gate_leaky_cases(ops, out):
    import torch
    dev = "cuda"
    for dim, off in itertools.product((6, 300), (0, 1)):
        g = torch.Generator(device=dev).manual_seed(dim + off)
        dh = placed(torch.randn(N, dim, generator=g, device=dev), off)
        gz = placed(torch.rand(N, 2 * dim, generator=g, device=dev), 2 * off)        # (g, z) pairs stay 8-byte aligned
        ent = placed(torch.randn(N, dim, generator=g, device=dev), off)
        d_pre, d_ent = placed(torch.zeros(N, 2 * dim, device=dev), 2 * off), placed(torch.zeros(N, dim, device=dev), off)
        rec = ops.raw_record(dev)
        ops.gate_bwd(dh, gz, ent, d_pre, d_ent, pre_amax=rec)
        key = f"gate_dim{dim}_off{off}"
        out[key + "/d_pre"], out[key + "/d_ent"], out[key + "/rec"] = d_pre, d_ent, rec
    for c, off in itertools.product((10, 32, 256), (0, 1)):
        g = torch.Generator(device=dev).manual_seed(c + off)
        gr = placed(torch.randn(N, c, generator=g, device=dev), off)
        act = placed(torch.randn(N, c, generator=g, device=dev), off)
        d = placed(torch.zeros(N, c, device=dev), off)
        rec = ops.raw_record(dev)
        ops.leaky_bwd(gr, act, d_pre=d, amax=rec)
        key = f"leaky_c{c}_off{off}"
        out[key + "/d"], out[key + "/rec"] = d, rec


def training_cases(L, O, out, n=200_000, e=4_000_000, n_rel=16):
    import torch
    dev = torch.device("cuda:0")
    kg = L.synthetic.make_kg(n, e, n_rel, seed=5)
    num, txt = L.synthetic.make_literals(n, seed=5)
    kt = L.KGTensors(kg.h, kg.t, kg.r, n_entities=n, device=dev)
    for agg in ("bi-interaction", "gcn", "graphsage"):
        cfg = O.OracleConfig(n_conv_layers=3, aggregation_type=agg, mess_dropout=0.1)
        args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
        args.device = str(dev)
        torch.manual_seed(2022)
        model = L.LiteralKG(args, n, n_rel, kt.A_in, num, txt).to(dev).train()
        gen = torch.Generator(device=dev).manual_seed(0)
        bh, bp, bn = (torch.randint(0, n, (681,), device=dev, generator=gen) for _ in range(3))
        for r in range(REPS):
            for prm in model.parameters():
                prm.grad = None
            torch.manual_seed(7)                                               # dropout masks
            loss = model(bh, bp, bn, device=dev, mode="fine_tuning")
            loss.backward()
            out[f"train_{agg}/loss/r{r}"] = loss.detach().reshape(1)
            for k, prm in model.named_parameters():
                if prm.grad is not None and not prm.grad.is_sparse:
                    out[f"train_{agg}/grad/{k}/r{r}"] = prm.grad
        del model, loss
        torch.cuda.empty_cache()


ZERO = np.int32(-2 ** 31)                                       # the bits of -0.0
BIG = 1 << 22                                                   # words above which an output is kept as a fingerprint


def fingerprint(x):
    """Digests of the bits and of the bits with -0 read as +0, and every 16th row (for the size of a difference)."""
    return (hashlib.sha256(x.tobytes()).hexdigest(), hashlib.sha256(np.where(x == ZERO, 0, x).tobytes()).hexdigest(),
            x.reshape(x.shape[0], -1)[::16])


def dump(dst, root):
    for p in (root, os.path.join(root, "oracle")):
        sys.path.insert(0, p)
    import torch
    import literalkg_b200 as L
    import literalkg_oracle as O
    from literalkg_b200 import ops
    assert os.path.dirname(os.path.abspath(L.__file__)) == os.path.join(os.path.abspath(root), "literalkg_b200")
    out = {}
    layer_cases(ops, out)
    gate_leaky_cases(ops, out)
    training_cases(L, O, out)
    torch.cuda.synchronize()
    os.makedirs(dst, exist_ok=True)
    for k, t in out.items():
        x = t.detach().float().contiguous().cpu().numpy().view(np.int32)
        f = os.path.join(dst, k.replace("/", "__"))
        if x.size <= BIG:
            np.save(f + ".npy", x)
        else:
            sha, sha0, sample = fingerprint(x)
            np.save(f + ".sample.npy", sample)
            with open(f + ".sha", "w") as fh:
                fh.write(f"{sha} {sha0}\n")
    print(f"{len(out)} outputs from {os.path.abspath(root)} -> {dst}")


def load(d):
    """key -> runs, each (bits, None) for a full output or (every 16th row, (sha, sha0)) for a fingerprinted one"""
    out = {}
    for f in sorted(os.listdir(d)):
        path = os.path.join(d, f)
        if f.endswith(".sample.npy"):
            name, run = f[:-11], (np.load(path), tuple(open(path[:-11] + ".sha").read().split()))
        elif f.endswith(".npy"):
            name, run = f[:-4], (np.load(path), None)
        else:
            continue
        out.setdefault(re.sub(r"/r\d+$", "", name.replace("__", "/")), []).append(run)
    return out


def classify(x, y):
    """'equal', 'zero-sign' (only -0 against +0) or 'differs'"""
    (bx, hx), (by, hy) = x, y
    if hx is not None:
        return "equal" if hx[0] == hy[0] else ("zero-sign" if hx[1] == hy[1] else "differs")
    if np.array_equal(bx, by):
        return "equal"
    return "zero-sign" if np.array_equal(np.where(bx == ZERO, 0, bx), np.where(by == ZERO, 0, by)) else "differs"


def floats(x):
    return x[0].view(np.float32).astype(np.float64)


def max_rel(x, y):
    return np.abs(floats(x) - floats(y)).max() / max(np.abs(floats(x)).max(), 1e-30)


def rel_l2(x, y):
    return np.linalg.norm(floats(x) - floats(y)) / max(np.linalg.norm(floats(x)), 1e-30)


def compare(a_dir, b_dir, a2_dir=None):
    a, b = load(a_dir), load(b_dir)
    a2 = load(a2_dir) if a2_dir else {}
    assert a.keys() == b.keys(), sorted(set(a) ^ set(b))
    tally, ratios = {}, []
    for k in sorted(a):
        runs_a, runs_b = a[k] + a2.get(k, []), b[k]
        varies = any(classify(runs_a[0], x) != "equal" for x in runs_a[1:])
        note = ""
        if not varies:
            cats = {classify(runs_a[0], x) for x in runs_b}
            cat = "differs" if "differs" in cats else ("zero-sign" if "zero-sign" in cats else "equal")
            if cat == "zero-sign" and runs_a[0][1] is None:
                note = f"{int((runs_a[0][0] != runs_b[0][0]).sum())} words"
            if cat == "differs":
                cat, note = "DIFFERS", f"max rel {max(max_rel(runs_a[0], x) for x in runs_b):.3e}"
        else:
            spread = np.median([rel_l2(x, y) for x, y in itertools.combinations(runs_a, 2)])
            dist = np.median([rel_l2(x, y) for x in runs_a for y in runs_b])
            ratios.append(dist / spread)
            cat = "within spread" if dist <= 2 * spread else "OUTSIDE spread"
            note = f"rel L2 B-A {dist:.3e}, A-A {spread:.3e} ({len(runs_a)} A runs, {len(runs_b)} B runs)"
        tally[cat] = tally.get(cat, 0) + 1
        print(f"{k:70s} {cat:15s} {'varies run to run' if varies else '':18s} {note}")
    print("summary:", tally)
    if ratios:
        print(f"B-A / A-A distance ratio over the varying outputs: median {np.median(ratios):.2f}, max {max(ratios):.2f}")


def main():
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    d = sub.add_parser("dump")
    d.add_argument("dir")
    d.add_argument("--root", default=HERE)
    c = sub.add_parser("compare")
    c.add_argument("a")
    c.add_argument("b")
    c.add_argument("a2", nargs="?")
    args = ap.parse_args()
    if args.cmd == "dump":
        dump(args.dir, args.root)
    else:
        compare(args.a, args.b, args.a2)


if __name__ == "__main__":
    main()
