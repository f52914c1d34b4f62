"""lkg_aggregate_fwd, one case per kernel instance of its dispatcher, against a float64 restatement of the layer
(include/lkg.h, lkg_aggregate_fwd):

    side = A @ ego;  o1 = ego @ Pa + side @ Pb + r1  (kBiZ: o1 = r1 + A @ z);  o2 = (ego * side) @ P2 + r2
    emb = leaky(o1) (+ leaky(o2));  x = LayerNorm(emb) * mask;  xn = x / max(|x|, 1e-12)

Every case pins its instance (the kernel name, full template argument list, recorded by torch.profiler) and checks
x, xn, the saved [o1 | o2] and side element-wise against a bound built from the same computation on absolute values.
The graph has power-law rows, empty and one-neighbour rows, rows on both sides of the cooperative (96), solo (256) and
segmentation (512) thresholds, a hub cut into 8 pieces longer than 512 and a hub with 8 triples per (head, tail) pair."""
import re

import numpy as np
import pytest
import torch

import literalkg_oracle as O

pytestmark = pytest.mark.gpu

N, N_REL = 5000, 8
HUB, HUB2 = 17, 4321               # 4 600 distinct tails (8 pieces of 575); 1 200 triples over 150 tails (3 pieces)
EDGE_ROWS = {2000: 96, 2001: 97, 2002: 256, 2003: 257, 2004: 512, 2005: 513}
ONE_ROWS = range(3000, 3010)
PART = (1000, 4500)                # a row range with HUB2 and the threshold rows in it, HUB outside
U = 2.0 ** -24                     # fp32 unit roundoff
C_BOUND = 64                       # roundings per accumulated term the bound allows: covers the worst case of sums of
                                   # up to 64 terms; the 512-wide fp32 combines measure up to 0.45 of it on a B200,
                                   # a dropped hub neighbour over 1 000 times it
ONE, TWO, BI, BIZ = 0, 1, 2, 3


def make_edges(n, seed):
    rng = np.random.default_rng(seed)
    deg = np.minimum(rng.zipf(1.7, n) - 1, 80)                          # power law, ~45 % of the rows empty
    deg[[HUB, HUB2, *EDGE_ROWS, *ONE_ROWS]] = 0
    hs, ts, rs = [], [], []
    for row in np.nonzero(deg)[0]:
        hs.append(np.full(deg[row], row)); ts.append(rng.choice(n, deg[row], replace=False))
        rs.append(rng.integers(0, N_REL, deg[row]))
    for row, k in [(HUB, 4600), *EDGE_ROWS.items(), *((r, 1) for r in ONE_ROWS)]:
        hs.append(np.full(k, row)); ts.append(rng.choice(n, k, replace=False)); rs.append(np.zeros(k, np.int64))
    tails2 = rng.choice(n, 150, replace=False)
    hs.append(np.full(1200, HUB2)); ts.append(np.repeat(tails2, 8)); rs.append(np.tile(np.arange(8), 150))
    h, t, r = np.concatenate(hs), np.concatenate(ts), np.concatenate(rs)
    perm = rng.permutation(h.shape[0])
    return h[perm], t[perm], r[perm]


@pytest.fixture(scope="module")
def graph():
    import literalkg_b200 as L
    h, t, r = make_edges(N, 7)
    plan = L.GraphPlan(*(torch.from_numpy(x).cuda() for x in (h, t, r)), N, N_REL)
    idx = plan.indices.cpu()
    deg = torch.bincount(idx[0], minlength=N)
    rng = np.random.default_rng(8)
    a = rng.standard_normal(plan.nnz) * (0.5 + rng.random(plan.nnz)) / np.sqrt(deg[idx[0]].numpy())
    a = torch.from_numpy(a).float()
    sched = plan.row_sched.cpu()
    assert plan.nnz < plan.n_edges and (sched[:, 5] == 8).sum() == 8 and (sched[:, 5] == 3).sum() == 3
    assert int(deg[HUB2]) == 150 and (sched[sched[:, 0] == HUB, 4] - sched[sched[:, 0] == HUB, 3]).min() > 512
    # the sensitivity references: the largest-|A| neighbour of HUB dropped; HUB's second schedule piece dropped
    hub = sched[(sched[:, 0] == HUB)]
    lo, hi = int(hub[0, 3]), int(hub[-1, 4])
    drop_one = a.clone()
    drop_one[lo + int(a[lo:hi].abs().argmax())] = 0
    drop_seg = a.clone()
    drop_seg[int(hub[1, 3]):int(hub[1, 4])] = 0
    return dict(plan=plan, idx=idx, a=a, a_dev=a.cuda(), drop_one=drop_one, drop_seg=drop_seg)


def spmm(idx, a, x):
    return torch.zeros(N, x.shape[1], dtype=torch.float64).index_add_(0, idx[0], a.double()[:, None] * x[idx[1]])


def reference(g, a, inp):
    """float64 layer and the same layer on absolute values (the scale of every rounding the fp32 kernel makes)."""
    d = {k: (None if v is None else v.cpu().double()) for k, v in inp.items() if isinstance(v, torch.Tensor) or v is None}
    idx, mode = g["idx"], inp["mode"]
    ego, n_out = d["ego"], inp["d_out"]
    side, side_abs = spmm(idx, a, ego), spmm(idx, a.abs(), ego.abs())
    r1 = d["r1"] if d["r1"] is not None else torch.zeros(n_out, dtype=torch.float64)
    r2 = d["r2"] if d["r2"] is not None else torch.zeros(n_out, dtype=torch.float64)
    P = {k: d[k] for k in ("pa", "pb", "p2")}
    A = {k: (None if v is None else v.abs()) for k, v in P.items()}
    o2 = o2_abs = None
    if mode == BIZ:
        o1, o1_abs = r1 + spmm(idx, a, d["z"]), r1.abs() + spmm(idx, a.abs(), d["z"].abs())
    elif mode == TWO:
        o1 = ego @ P["pa"] + side @ P["pb"] + r1
        o1_abs = ego.abs() @ A["pa"] + side_abs @ A["pb"] + r1.abs()
    else:
        s = ego + side if P["pa"] is not None else side
        s_abs = ego.abs() + side_abs if P["pa"] is not None else side_abs
        o1, o1_abs = s @ P["pb"] + r1, s_abs @ A["pb"] + r1.abs()
    if mode in (BI, BIZ):
        o2 = (ego * side) @ P["p2"] + r2
        o2_abs = (ego.abs() * side_abs) @ A["p2"] + r2.abs()
    leaky = lambda v: torch.nn.functional.leaky_relu(v, O.LEAKY_SLOPE)
    emb = leaky(o1) + (leaky(o2) if o2 is not None else 0)
    eb = C_BOUND * U * (o1_abs + (o2_abs if o2 is not None else 0))          # |error of emb| (leaky is 1-Lipschitz)
    mean = emb.mean(1, keepdim=True)
    rstd = 1 / torch.sqrt(((emb - mean) ** 2).mean(1, keepdim=True) + O.LN_EPS)
    e_row = eb.max(1, keepdim=True).values
    assert (e_row * rstd).max() < 1e-2                  # every row far from a flat one: first-order bounds hold
    w, b = d["ln_w"], d["ln_b"]
    xl = (emb - mean) * rstd * w + b
    bx = 2 * w.abs() * rstd * (eb + e_row + (emb - mean).abs() * e_row * rstd) + C_BOUND * U * (xl.abs() + b.abs())
    if d["mask"] is not None:
        xl, bx = xl * d["mask"], bx * d["mask"].abs()
    nx = xl.norm(dim=1, keepdim=True).clamp_min(1e-12)
    xn = xl / nx
    bxn = (bx + xn.abs() * bx.norm(dim=1, keepdim=True)) / nx + C_BOUND * U * xn.abs()
    o = o1 if o2 is None else torch.cat([o1, o2], 1)
    bo = C_BOUND * U * (o1_abs if o2 is None else torch.cat([o1_abs, o2_abs], 1))
    return dict(x=(xl, bx), xn=(xn, bxn), o=(o, bo), side=(side, C_BOUND * U * side_abs))


def worst(ref, got, rows=slice(None)):
    """max over outputs and elements of |got - ref| / bound (NaN counts as infinitely wrong)."""
    out = 0.0
    for k, v in got.items():
        r, bd = (t[rows] for t in ref[k])
        q = (v.cpu().double() - r).abs() / bd.clamp_min(1e-30)
        out = max(out, torch.nan_to_num(q, nan=float("inf")).max().item())
    return out


def make_inputs(case, seed):
    """Device operands of one case, drawn on the host from ``seed``."""
    d_in, d_out, mode = case["d_in"], case["d_out"], case["mode"]
    gen = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=gen).cuda()
    inp = dict(mode=mode, d_out=d_out)
    ego = rn(N, d_in)
    inp["pb"] = None if mode == BIZ else rn(d_in, d_out) / d_in ** 0.5
    inp["pa"] = {TWO: rn(d_in, d_out) / d_in ** 0.5, ONE: inp["pb"] if case.get("sum_ego") else None,
                 BI: inp["pb"] if case.get("sum_ego") else None, BIZ: None}[mode]     # pa is pb: "ego + side"
    inp["p2"] = rn(d_in, d_out) / d_in ** 0.5 if mode in (BI, BIZ) else None
    nt = 2 if mode in (BI, BIZ) else 1
    if case.get("per_row", True):                        # r1 / r2 share one leading dimension: columns of one buffer
        r = rn(N, nt * d_out) * 0.5
        inp["r1"], inp["r2"] = r[:, :d_out], (r[:, d_out:] if nt == 2 else None)
    else:                                                 # ld_r = 0: broadcast biases
        inp["r1"], inp["r2"] = rn(d_out) * 0.5, (rn(d_out) * 0.5 if nt == 2 else None)
    inp["ln_w"], inp["ln_b"] = 1 + 0.2 * rn(d_out), 0.1 * rn(d_out)
    mask = None
    if case.get("mask"):
        mask = (torch.rand(N, d_out, generator=gen) < 0.8).float() / 0.8
        mask[:, 0] = 1 / 0.8
        mask = mask.cuda()
    inp["mask"] = mask
    inp["z"] = None
    if mode == BIZ:
        z = ego @ (rn(d_in, d_out) / d_in ** 0.5)
        if case.get("zcontig"):                            # [ego | z] rows back to back: one bulk copy per neighbour
            tab = torch.cat([ego, z], 1)
            ego, z = tab[:, :d_in], tab[:, d_in:]
        inp["z"] = z
    inp["ego"] = ego
    return inp


def run(plan, a_dev, inp, case, rows=(0, N), outputs=True, x_nan=False):
    import literalkg_b200 as L
    from literalkg_b200 import _lib
    rb, re_ = rows
    nl, d_in, d_out = re_ - rb, case["d_in"], case["d_out"]
    loc = lambda t: None if t is None else (t[rb:re_] if t.dim() == 2 else t)
    f32 = dict(dtype=torch.float32, device="cuda")
    if case.get("x_offset"):
        x_buf = torch.full((N, d_out + 4), float("nan"), **f32)
        x_out = x_buf[:, 1:1 + d_out]                     # rows 4 bytes off the 16-byte grid
    else:
        x_out = torch.full((N, d_out), float("nan"), **f32) if x_nan else torch.empty((N, d_out), **f32)
    nt = 2 if case["mode"] in (BI, BIZ) else 1
    res = dict(x=x_out)
    xn = o = side = planes = None
    if outputs:
        xn = torch.empty((nl, d_out), **f32)
        o = torch.empty((nl, (nt * d_out + 3) // 4 * 4), **f32)[:, :nt * d_out]     # rows 16-byte aligned
        side = torch.empty((nl, d_in), **f32)
        planes = _lib.Planes(nl, d_out, "cuda", rec=L.ops.scale_from_bound(1.0, "cuda"))
        res.update(xn=xn, o=o, side=side, planes=planes)
    plan.set_row_range(rb, re_)
    try:
        L.ops.aggregate(plan, a_dev, inp["ego"], d_out, inp["pa"], inp["pb"], inp["p2"], loc(inp["r1"]), loc(inp["r2"]),
                        inp["ln_w"], inp["ln_b"], loc(inp["mask"]), x_out, xn, planes, local_row_base=rb, z=inp["z"],
                        o_out=o, side_out=side)
    finally:
        plan.set_row_range(0, N)
    torch.cuda.synchronize()
    return res


def pinned_kernel(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {m.group(1) for e in prof.events() for m in [re.search(r"(aggregate_\w*kernel<[^>]*>)", e.name)] if m}
    return out, names


CASES = [
    ("16x16 one sum", dict(d_in=16, d_out=16, mode=ONE, sum_ego=True), "aggregate_narrow_kernel<4, 0, 1, 1, 1>"),
    ("16x16 one side", dict(d_in=16, d_out=16, mode=ONE, per_row=False), "aggregate_narrow_kernel<4, 0, 1, 1, 1>"),
    ("16x64 two", dict(d_in=16, d_out=64, mode=TWO, mask=True), "aggregate_narrow_kernel<4, 1, 4, 1, 1>"),
    ("16x44 bi", dict(d_in=16, d_out=44, mode=BI, sum_ego=True), "aggregate_narrow_kernel<4, 2, 3, 1, 1>"),
    ("32x32 bi", dict(d_in=32, d_out=32, mode=BI, sum_ego=True, mask=True), "aggregate_narrow_kernel<8, 2, 1, 2, 4>"),
    ("32x64 one", dict(d_in=32, d_out=64, mode=ONE, sum_ego=True, per_row=False), "aggregate_narrow_kernel<8, 0, 2, 1, 1>"),
    ("64x48 two", dict(d_in=64, d_out=48, mode=TWO), "aggregate_narrow_kernel<16, 1, 1, 2, 4>"),
    ("64x8 bi", dict(d_in=64, d_out=8, mode=BI, per_row=False, mask=True), "aggregate_narrow_kernel<16, 2, 1, 2, 4>"),
    ("12x8 bi", dict(d_in=12, d_out=8, mode=BI, sum_ego=True), "aggregate_kernel<1, 1, 2>"),
    ("48x40 two", dict(d_in=48, d_out=40, mode=TWO, mask=True), "aggregate_kernel<1, 2, 1>"),
    ("32x30 one", dict(d_in=32, d_out=30, mode=ONE, sum_ego=True), "aggregate_kernel<1, 1, 0>"),
    ("32x32 two x_out+1", dict(d_in=32, d_out=32, mode=TWO, x_offset=True), "aggregate_kernel<1, 1, 1>"),
    ("128x32 biz", dict(d_in=128, d_out=32, mode=BIZ, mask=True), "aggregate_stream_kernel<1, 1, 3>"),
    ("128x20 biz [ego|z]", dict(d_in=128, d_out=20, mode=BIZ, zcontig=True, per_row=False),
     "aggregate_stream_kernel<1, 1, 3>"),
    ("200x32 two", dict(d_in=200, d_out=32, mode=TWO, mask=True), "aggregate_stream_kernel<2, 1, 1>"),
    ("256x64 bi", dict(d_in=256, d_out=64, mode=BI), "aggregate_kernel<2, 2, 2>"),
    ("300x32 bi", dict(d_in=300, d_out=32, mode=BI, sum_ego=True), "aggregate_stream_kernel<3, 1, 2>"),
    ("300x32 biz [ego|z]", dict(d_in=300, d_out=32, mode=BIZ, zcontig=True, mask=True), "aggregate_stream_kernel<3, 1, 3>"),
    ("300x64 one", dict(d_in=300, d_out=64, mode=ONE, per_row=False), "aggregate_stream_kernel<3, 2, 0>"),
    ("300x48 biz", dict(d_in=300, d_out=48, mode=BIZ), "aggregate_stream_kernel<3, 2, 3>"),
    ("300x64 bi", dict(d_in=300, d_out=64, mode=BI, mask=True), "aggregate_kernel<3, 2, 2>"),
    ("512x32 one", dict(d_in=512, d_out=32, mode=ONE, sum_ego=True, mask=True), "aggregate_stream_kernel<4, 1, 0>"),
    ("512x32 bi", dict(d_in=512, d_out=32, mode=BI, per_row=False), "aggregate_kernel<4, 1, 2>"),
]


@pytest.mark.parametrize("name,case,kernel", CASES, ids=[c[0] for c in CASES])
def test_instance_vs_float64(graph, name, case, kernel):
    plan, a_dev = graph["plan"], graph["a_dev"]
    inp = make_inputs(case, seed=len(name) * 131 + case["d_in"] + case["d_out"])
    res, names = pinned_kernel(lambda: run(plan, a_dev, inp, case))
    print(f"{name}: {sorted(names)}")
    assert names == {kernel}, names

    ref = reference(graph, graph["a"], inp)
    got = {k: res[k] for k in ("x", "xn", "o", "side")}
    err = worst(ref, got)
    # the same bar must see a kernel that loses one neighbour of the hub, or one piece of its segmented schedule
    err_one = worst(reference(graph, graph["drop_one"], inp), got)
    err_seg = worst(reference(graph, graph["drop_seg"], inp), got)
    print(f"{name}: worst |err| / bound {err:.3g}; one hub neighbour dropped {err_one:.3g}, one piece dropped {err_seg:.3g}")
    assert err <= 1.0 and err_one >= 10 and err_seg >= 10

    # xn planes: bit exact split of the kernel's own xn with the record's scale
    s = res["planes"].rec[1]
    xs = res["xn"] * s
    hi = xs.half()
    lo = (xs - hi.float()).half()
    pl = res["planes"].t[:, :N, :case["d_out"]]
    assert torch.equal(pl[0].view(torch.int16), hi.view(torch.int16))
    assert torch.equal(pl[1].view(torch.int16), lo.view(torch.int16))

    # determinism, and the segment tickets are back at zero between launches
    if plan._seg_tickets is not None:
        assert (plan._seg_tickets == 0).all()
    again = run(plan, a_dev, inp, case)
    for k in ("x", "xn", "o", "side"):
        assert torch.equal(again[k], res[k]), k
    assert torch.equal(again["planes"].t[:, :, :case["d_out"]], res["planes"].t[:, :, :case["d_out"]])
    bare = run(plan, a_dev, inp, case, outputs=False)      # without the optional outputs: the same x
    assert torch.equal(bare["x"], res["x"])
    if plan._seg_tickets is not None:
        assert (plan._seg_tickets == 0).all()

    # row partition: local r1 / r2 / mask / xn / o / side / planes rows start at local_row_base, x_out is global
    rb, re_ = PART
    part = run(plan, a_dev, inp, case, rows=PART, x_nan=True)
    x = part["x"]
    assert torch.isnan(x[:rb]).all() and torch.isnan(x[re_:]).all()
    got = dict(x=x[rb:re_], xn=part["xn"], o=part["o"], side=part["side"])
    assert worst(ref, got, rows=slice(rb, re_)) <= 1.0
    if plan._seg_tickets is not None:
        assert (plan._seg_tickets == 0).all()


@pytest.mark.parametrize("n,edges", [(1, 0), (1, 1), (700, 0)])
@pytest.mark.parametrize("d_in,d_out,mode", [(16, 16, TWO), (12, 8, BI), (300, 32, BIZ), (200, 32, ONE)])
def test_tiny_and_empty_graphs(n, edges, d_in, d_out, mode):
    """nnz = 0 and a single row: every kernel family on a plan with nothing to gather (or one self loop)."""
    import literalkg_b200 as L
    h = torch.zeros(edges, dtype=torch.int64, device="cuda")
    plan = L.GraphPlan(h, h.clone(), h.clone(), n, 1)
    assert plan.nnz == edges
    gen = torch.Generator().manual_seed(n + edges + d_in)
    ego = torch.randn(n, d_in, generator=gen)
    a = torch.full((plan.nnz,), -0.75)
    pb = torch.randn(d_in, d_out, generator=gen) / d_in ** 0.5
    pa = torch.randn(d_in, d_out, generator=gen) / d_in ** 0.5 if mode == TWO else None
    p2 = torch.randn(d_in, d_out, generator=gen) / d_in ** 0.5 if mode in (BI, BIZ) else None
    r1, r2 = torch.randn(n, d_out, generator=gen), torch.randn(n, d_out, generator=gen)
    z = (ego @ pb) if mode == BIZ else None
    ln_w, ln_b = 1 + 0.2 * torch.randn(d_out, generator=gen), 0.1 * torch.randn(d_out, generator=gen)
    c = lambda t: None if t is None else t.cuda()
    x = torch.empty((n, d_out), device="cuda")
    o = torch.empty((n, (2 if p2 is not None else 1) * d_out), device="cuda")
    L.ops.aggregate(plan, a.cuda(), ego.cuda(), d_out, c(pa), None if mode == BIZ else pb.cuda(), c(p2), r1.cuda(),
                    c(r2) if p2 is not None else None, ln_w.cuda(), ln_b.cuda(), None, x, None, z=c(z), o_out=o)
    torch.cuda.synchronize()
    e, a64 = ego.double(), a.double()
    side = torch.zeros(n, d_in, dtype=torch.float64)
    if edges:
        side[0] = a64[0] * e[0]
    if mode == BIZ:
        zs = torch.zeros(n, d_out, dtype=torch.float64)
        if edges:
            zs[0] = a64[0] * z[0].double()
        o1 = r1.double() + zs
    elif mode == TWO:
        o1 = e @ pa.double() + side @ pb.double() + r1.double()
    else:
        o1 = side @ pb.double() + r1.double()
    leaky = lambda v: torch.nn.functional.leaky_relu(v, O.LEAKY_SLOPE)
    emb = leaky(o1)
    oo = o1
    if p2 is not None:
        o2 = (e * side) @ p2.double() + r2.double()
        emb, oo = emb + leaky(o2), torch.cat([o1, o2], 1)
    ref = torch.nn.functional.layer_norm(emb, (d_out,), ln_w.double(), ln_b.double(), O.LN_EPS)
    assert (x.cpu().double() - ref).abs().max().item() < 1e-4
    assert (o.cpu().double() - oo).abs().max().item() < 1e-4
