"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from the checkout of the original
NSLab-CUK/LiteralKG that LKG_REFERENCE names):

    LKG_REFERENCE=<checkout> python oracle/make_golden.py            # writes tests/golden/<case>.npz

Each file holds the inputs (config, state dict, literal tables, triples) and the reference's own
outputs for every stage of the hot path: initial Laplacian A_in (dataloader.py:449-495), attention
update (model.py:444-471), gate output, every aggregator layer, final embeddings
(model.py:298-314), scores / predictions (model.py:473-491), both losses and a few parameter
gradients (model.py:316-348, 364-428).  The oracle (oracle/literalkg_oracle.py) and the CUDA path
are both checked against these vectors.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("LKG_REFERENCE", "")
sys.path.insert(0, HERE)
from literalkg_oracle import OracleConfig  # noqa: E402


def import_reference():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import model as ref_model          # noqa
    import gate as ref_gate            # noqa
    return ref_model, ref_gate


def make_kg(n, n_rel, n_edges, seed, n_dup=6, n_isolated=5):
    """Small KG with (a) isolated entities (empty rows), (b) (h,t) pairs repeated under a second
    and third relation (duplicate-merge path), (c) a skewed head distribution."""
    rng = np.random.default_rng(seed)
    live = n - n_isolated
    w = 1.0 / np.arange(1, live + 1)
    w /= w.sum()
    h = rng.choice(live, size=n_edges, p=w)
    t = rng.integers(0, n, size=n_edges)
    r = rng.integers(0, n_rel, size=n_edges)
    r[:n_rel] = np.arange(n_rel)                      # every relation present
    # duplicates of (h,t) under other relations
    for i in range(n_dup):
        h = np.append(h, h[i]); t = np.append(t, t[i]); r = np.append(r, (r[i] + 1) % n_rel)
    h = np.append(h, h[0]); t = np.append(t, t[0]); r = np.append(r, (r[0] + 2) % n_rel)
    trip = np.unique(np.stack([h, r, t], 1), axis=0)
    rng.shuffle(trip)                                  # file order is arbitrary
    return trip[:, 0].astype(np.int64), trip[:, 2].astype(np.int64), trip[:, 1].astype(np.int64)


def namespace(cfg: OracleConfig):
    return argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})


def ref_laplacian(h, t, r, n, laplacian_type):
    """Calls the reference's own create_adjacency_dict / create_laplacian_dict / convert_coo2tensor
    on a stub object (SURVEY.md 8(c))."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import dataloader as ref_dl

    stub = ref_dl.DataLoader.__new__(ref_dl.DataLoader)
    stub.train_relation_dict = collections.defaultdict(list)
    for hh, tt, rr in zip(h.tolist(), t.tolist(), r.tolist()):
        stub.train_relation_dict[rr].append((hh, tt))
    stub.n_head_tail = n
    stub.laplacian_type = laplacian_type
    stub.create_adjacency_dict()
    stub.create_laplacian_dict()
    a = stub.A_in.coalesce()
    return a.indices().numpy(), a.values().numpy(), list(stub.laplacian_dict.keys())


def run_case(name, cfg: OracleConfig, n, n_rel, n_edges, seed, laplacian_type="random-walk",
             grad_numel_cap=None):
    ref_model, _ = import_reference()
    torch.manual_seed(seed)
    np.random.seed(seed)
    h, t, r = make_kg(n, n_rel, n_edges, seed)
    rng = np.random.default_rng(seed + 1)
    num_lit = torch.zeros(n, cfg.num_lit_dim)
    rows = rng.choice(n, size=n // 3, replace=False)
    num_lit[rows, rng.integers(0, cfg.num_lit_dim, size=len(rows))] = torch.from_numpy(
        rng.uniform(0.05, 1.0, size=len(rows)).astype(np.float32))
    txt_lit = torch.zeros(n, cfg.txt_lit_dim)
    rows = rng.choice(n, size=n // 4, replace=False)
    txt_lit[rows] = torch.from_numpy(rng.normal(0, 0.3, size=(len(rows), cfg.txt_lit_dim)).astype(np.float32))

    lap_idx, lap_val, relations = ref_laplacian(h, t, r, n, laplacian_type)
    a0 = torch.sparse_coo_tensor(torch.from_numpy(lap_idx), torch.from_numpy(lap_val), (n, n))

    args = namespace(cfg)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = ref_model.LiteralKG(args, n, n_rel, a0,
                                    num_lit if cfg.use_num_lit else None,
                                    txt_lit if cfg.use_txt_lit else None)
    # make embeddings less tiny than xavier at small n would already be; perturb biases / LN
    with torch.no_grad():
        for k, v in model.named_parameters():
            if k.endswith("gate_bias") or "layer_normalize" in k:
                v.add_(0.1 * torch.randn_like(v))
    model.eval()

    out = {"config": np.frombuffer(json.dumps({**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__},
                                               "n_entities": n, "n_relations": n_rel,
                                               "laplacian_type": laplacian_type}).encode(), dtype=np.uint8)}
    sd = {k: v for k, v in model.state_dict().items() if k != "A_in"}
    for k, v in sd.items():
        out["sd/" + k] = v.detach().numpy().copy()
    out["in/h"], out["in/t"], out["in/r"] = h, t, r
    out["in/relations"] = np.asarray(relations, dtype=np.int64)
    out["in/num_lit"], out["in/txt_lit"] = num_lit.numpy(), txt_lit.numpy()
    out["lap/idx"], out["lap/val"] = lap_idx, lap_val

    def stages(tag):
        with torch.no_grad():
            h0 = model.gate_embeddings()
            out[f"{tag}/gate"] = h0.numpy().copy()
            x, allv = h0, [h0]
            for k, layer in enumerate(model.aggregator_layers):
                x = layer(x, model.A_in, allv, model.lamda, model.alpha, k + 1)
                out[f"{tag}/layer{k}"] = x.numpy().copy()
            out[f"{tag}/final"] = model.gat_embeddings().numpy().copy()

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        stages("lap")                                  # forward with the initial Laplacian A_in
        hl, tl, rl = torch.from_numpy(h), torch.from_numpy(t), torch.from_numpy(r)
        model(hl, tl, rl, relations, device="cpu", mode="update_att")
        a = model.A_in.data.coalesce()
        out["att/idx"], out["att/val"] = a.indices().numpy().copy(), a.values().numpy().copy()
        stages("att")                                  # forward with the attention A_in

        heads = torch.from_numpy(rng.choice(n, size=min(9, n), replace=False).astype(np.int64))
        tails = torch.from_numpy(rng.choice(n, size=min(23, n), replace=False).astype(np.int64))
        out["score/heads"], out["score/tails"] = heads.numpy(), tails.numpy()
        with torch.no_grad():
            out["score/scores"] = model.calc_score(heads, tails).numpy().copy()
            out["score/predict"] = model(heads, tails, device="cpu", mode="predict").numpy().copy()

        b = 17
        bh = torch.from_numpy(rng.integers(0, n, size=b)); bp = torch.from_numpy(rng.integers(0, n, size=b))
        bn = torch.from_numpy(rng.integers(0, n, size=b)); br = torch.from_numpy(rng.integers(0, n_rel, size=b))
        out["loss/h"], out["loss/r"], out["loss/pos"], out["loss/neg"] = bh.numpy(), br.numpy(), bp.numpy(), bn.numpy()
        for mode, inp in (("pre_training", (bh, br, bp, bn)), ("fine_tuning", (bh, bp, bn))):
            model.zero_grad()
            loss = model(*inp, device="cpu", mode=mode)
            loss.backward()
            out[f"loss/{mode}"] = np.asarray(loss.item(), dtype=np.float64)
            for k, v in model.named_parameters():
                if v.grad is not None and k != "A_in" and (grad_numel_cap is None or v.numel() <= grad_numel_cap):
                    out[f"grad_{mode}/" + k] = v.grad.detach().numpy().copy()

    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, **out)
    print(f"{name}: N={n} E={len(h)} nnz={out['att/idx'].shape[1]} -> {os.path.getsize(path)/1e3:.0f} kB")


def run_head_case(name, cfg: OracleConfig, n, n_rel, n_edges, seed, variant):
    """The variant heads (SURVEY.md 8(f) rank 3) of the unmodified reference:
       variant 'bce'  model_bce.LiteralKG: TransE calc_triplet_loss, BPR loss, mode 'mlp' (constructor-built head);
       variant 'mlp'  model.LiteralKG + initialize_MLP(): mode 'mlp'.
    Stored: state dict (BatchNorm buffers included), A_in after update_att, final embeddings, the head's output in
    training mode (batch statistics; the updated running buffers) and in eval mode, nn.BCELoss against random labels
    and its gradients w.r.t. every parameter, and (bce) the TransE loss + gradients."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import importlib
    ref = importlib.import_module("model_bce" if variant == "bce" else "model")
    torch.manual_seed(seed)
    np.random.seed(seed)
    h, t, r = make_kg(n, n_rel, n_edges, seed)
    rng = np.random.default_rng(seed + 1)
    num_lit = torch.from_numpy(rng.uniform(0, 1, size=(n, cfg.num_lit_dim)).astype(np.float32))
    num_lit[rng.choice(n, n // 2, replace=False)] = 0
    txt_lit = torch.from_numpy(rng.normal(0, 0.3, size=(n, cfg.txt_lit_dim)).astype(np.float32))
    lap_idx, lap_val, relations = ref_laplacian(h, t, r, n, "random-walk")
    a0 = torch.sparse_coo_tensor(torch.from_numpy(lap_idx), torch.from_numpy(lap_val), (n, n))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = ref.LiteralKG(namespace(cfg), n, n_rel, a0, num_lit, txt_lit)
        if variant == "mlp":
            model.initialize_MLP()
        with torch.no_grad():
            model.entity_embed.weight.mul_(3.0)
            for k, v in model.named_parameters():
                if "norm" in k or k.endswith("gate_bias"):
                    v.add_(0.1 * torch.randn_like(v))
            for nm in ("norm1", "norm2"):                 # non-trivial running statistics for the eval-mode output
                getattr(model, nm).running_mean.add_(0.05 * torch.randn_like(getattr(model, nm).running_mean))
                getattr(model, nm).running_var.mul_(1.0 + 0.2 * torch.rand_like(getattr(model, nm).running_var))
        hl, tl, rl = torch.from_numpy(h), torch.from_numpy(t), torch.from_numpy(r)
        model(hl, tl, rl, relations, device="cpu", mode="update_att")
    out = {"config": np.frombuffer(json.dumps({**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__},
                                               "n_entities": n, "n_relations": n_rel,
                                               "laplacian_type": "random-walk"}).encode(), dtype=np.uint8)}
    for k, v in model.state_dict().items():
        if k != "A_in":
            out["sd/" + k] = v.detach().numpy().copy()
    a = model.A_in.data.coalesce()
    out["att/idx"], out["att/val"] = a.indices().numpy().copy(), a.values().numpy().copy()
    out["in/h"], out["in/t"], out["in/r"] = h, t, r
    out["in/relations"] = np.asarray(relations, dtype=np.int64)
    out["in/num_lit"], out["in/txt_lit"] = num_lit.numpy(), txt_lit.numpy()
    b = 37
    bh, bt = torch.from_numpy(rng.integers(0, n, size=b)), torch.from_numpy(rng.integers(0, n, size=b))
    labels = torch.from_numpy(rng.integers(0, 2, size=b).astype(np.float32))
    out["mlp/h"], out["mlp/t"], out["mlp/labels"] = bh.numpy(), bt.numpy(), labels.numpy()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.eval()
        with torch.no_grad():
            out["final"] = model.gat_embeddings().numpy().copy()
            out["mlp/eval_out"] = model(bh, bt, device="cpu", mode="mlp").numpy().copy()
        # training-mode output: batch statistics (dropout rate is 0 in these configs, so the trunk is deterministic)
        model.train()
        model.zero_grad()
        y = model(bh, bt, device="cpu", mode="mlp")
        loss = torch.nn.BCELoss()(y.reshape(-1), labels)          # main_finetuning_BCE.py:88,117-120
        loss.backward()
        out["mlp/train_out"] = y.detach().numpy().copy()
        out["mlp/bce_loss"] = np.asarray(loss.item(), dtype=np.float64)
        for k, v in model.named_parameters():
            if v.grad is not None and k != "A_in":
                out["grad_mlp/" + k] = v.grad.detach().numpy().copy()
        for nm in ("norm1", "norm2"):
            out[f"mlp/after/{nm}.running_mean"] = getattr(model, nm).running_mean.numpy().copy()
            out[f"mlp/after/{nm}.running_var"] = getattr(model, nm).running_var.numpy().copy()
        if variant == "bce":
            bp, bn = torch.from_numpy(rng.integers(0, n, size=b)), torch.from_numpy(rng.integers(0, n, size=b))
            br = torch.from_numpy(rng.integers(0, n_rel, size=b))
            out["loss/h"], out["loss/r"], out["loss/pos"], out["loss/neg"] = bh.numpy(), br.numpy(), bp.numpy(), bn.numpy()
            for mode, inp in (("pre_training", (bh, br, bp, bn)), ("fine_tuning", (bh, bp, bn))):
                model.zero_grad()
                loss = model(*inp, device="cpu", mode=mode)
                loss.backward()
                out[f"loss/{mode}"] = np.asarray(loss.item(), dtype=np.float64)
                for k, v in model.named_parameters():
                    if v.grad is not None and k != "A_in":
                        out[f"grad_{mode}/" + k] = v.grad.detach().numpy().copy()
    path = os.path.join(ROOT, "tests", "golden_heads", name + ".npz")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, **out)
    print(f"{name}: N={n} E={len(h)} -> {os.path.getsize(path)/1e3:.0f} kB")


def main_heads():
    # embed_dim == relation_dim (update_att adds the two tables) == scale_gat_dim (TransE adds relation rows to the
    # final embeddings, model_bce.py:351-354)
    small = dict(embed_dim=16, relation_dim=16, scale_gat_dim=16, num_lit_dim=2, txt_lit_dim=8, conv_dim=8,
                 n_conv_layers=2, mess_dropout=0.0)
    run_head_case("bce_small_bi", OracleConfig(aggregation_type="bi-interaction", **small), 57, 4, 240, 21, "bce")
    run_head_case("bce_small_gcn", OracleConfig(aggregation_type="gcn", use_residual=False, **small), 57, 4, 240, 22, "bce")
    run_head_case("mlp_small_sage", OracleConfig(aggregation_type="graphsage", **small), 57, 4, 240, 23, "mlp")


def main():
    if "--heads" in sys.argv:
        return main_heads()
    small = dict(embed_dim=12, relation_dim=12, scale_gat_dim=16, num_lit_dim=2, txt_lit_dim=8,
                 conv_dim=8, n_conv_layers=2, mess_dropout=0.0)
    for agg in ("bi-interaction", "gcn", "graphsage"):
        for res in (True, False):
            tag = {"bi-interaction": "bi", "gcn": "gcn", "graphsage": "sage"}[agg] + ("_res" if res else "_nores")
            run_case(f"small_{tag}", OracleConfig(aggregation_type=agg, use_residual=res, **small),
                     n=61, n_rel=4, n_edges=260, seed=11)
    # gate variants / no linear_gat / symmetric laplacian
    run_case("small_numonly", OracleConfig(use_txt_lit=False, **small), n=50, n_rel=3, n_edges=180, seed=12)
    run_case("small_txtonly", OracleConfig(use_num_lit=False, **small), n=50, n_rel=3, n_edges=180, seed=13)
    run_case("small_nolit_nogat", OracleConfig(use_num_lit=False, use_txt_lit=False,
                                               **{**small, "scale_gat_dim": None}),
             n=50, n_rel=3, n_edges=180, seed=14, laplacian_type="symmetric")
    # the reference's default dimensions (argument.py) on a tiny graph
    run_case("default_dims", OracleConfig(n_conv_layers=3, mess_dropout=0.0), n=40, n_rel=3, n_edges=150, seed=15,
             grad_numel_cap=16384)


if __name__ == "__main__":
    if not REF:
        sys.exit("set LKG_REFERENCE to a checkout of the original NSLab-CUK/LiteralKG")
    main()
