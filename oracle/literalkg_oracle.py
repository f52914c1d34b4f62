"""CPU oracle for the LiteralKG message-passing + scoring hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``literalkg_b200/`` may import this module; only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs use it, and there only as the checker / the timed CPU baseline -- never as the product.

It is a functional restatement (torch CPU + numpy + scipy, dtype-generic: fp32 or fp64) of the
reference's algorithm for the path named in BASELINE.json.  Every function cites the reference
``file:line`` it follows (paths relative to the upstream repository NSLab-CUK/LiteralKG).

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4).  This oracle is pinned
against the *reference itself*, imported unmodified in the build container by
``oracle/make_golden.py``; the resulting vectors live in ``tests/golden/*.npz`` and are checked by
``tests/test_oracle_golden.py`` (and, when ``LKG_REFERENCE`` names a checkout, against the live reference
classes in ``tests/test_oracle_vs_reference.py``).

Parameters are passed as a plain ``dict`` whose keys are the reference's ``state_dict`` names
(``entity_embed.weight``, ``aggregator_layers.0.linear1.weight``, ``emb_mul_lit.g.weight`` ...).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------
# configuration (mirrors the fields LiteralKG.__init__ reads from ``args``: model.py:172-204,263)
# ----------------------------------------------------------------------------------------------
@dataclass
class OracleConfig:
    embed_dim: int = 300
    relation_dim: int = 300
    scale_gat_dim: Optional[int] = 256
    num_lit_dim: int = 2
    txt_lit_dim: int = 300
    use_num_lit: bool = True
    use_txt_lit: bool = True
    aggregation_type: str = "bi-interaction"
    n_conv_layers: int = 8
    conv_dim: int = 32
    mess_dropout: float = 0.1
    use_residual: bool = True
    alpha: float = 0.1
    lamda: float = 0.5
    kg_l2loss_lambda: float = 1e-5
    fine_tuning_l2loss_lambda: float = 1e-5
    pre_training_neg_rate: int = 3
    fine_tuning_neg_rate: int = 3
    milestone_score: float = 0.5
    use_pretrain: int = 0
    device: str = "cpu"
    # only read by the (out-of-scope) gin branch of the reference constructor
    n_mlp_layers: int = 3
    mlp_hidden_dim: int = 64

    @property
    def conv_dims(self) -> List[int]:
        # model.py:193
        return [self.embed_dim] + [self.conv_dim] * self.n_conv_layers

    @property
    def total_conv_dim(self) -> int:
        # model.py:195
        return sum(self.conv_dims)


LEAKY_SLOPE = 0.01      # nn.LeakyReLU() default, model.py:29,223
LN_EPS = 1e-5           # nn.LayerNorm default, model.py:30
L2_EPS = 1e-12          # F.normalize default, model.py:305


# ----------------------------------------------------------------------------------------------
# graph tensors (dataloader.py)
# ----------------------------------------------------------------------------------------------
def parse_triples(text: str) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """``h r t`` lines, space separated, exact duplicate rows dropped keeping first occurrence and
    file order (dataloader.py:186-190 ``load_graph``; order consumed by ``construct_data``
    :395-403 to build h_list / t_list / r_list)."""
    rows = []
    seen = set()
    for line in text.splitlines():
        parts = line.split()
        if len(parts) != 3:
            continue
        key = (int(parts[0]), int(parts[1]), int(parts[2]))
        if key in seen:
            continue
        seen.add(key)
        rows.append(key)
    arr = np.asarray(rows, dtype=np.int64).reshape(-1, 3)
    return arr[:, 0].copy(), arr[:, 2].copy(), arr[:, 1].copy()   # h, t, r


def relation_order(r_list: np.ndarray) -> List[int]:
    """Insertion order of ``train_relation_dict`` (dataloader.py:393,403) == order of
    ``laplacian_dict.keys()`` that main.py:150 passes as ``relations``."""
    seen: Dict[int, None] = {}
    for r in r_list.tolist():
        if r not in seen:
            seen[r] = None
    return list(seen.keys())


def count_entities(h: np.ndarray, t: np.ndarray, lit_max_id: int = -1) -> int:
    """n_entities = max(max h + 1, max t + 1, literal max id + 1) (dataloader.py:405-418; the
    fine-tune file maxima the reference also folds in are supplied by the caller through
    ``lit_max_id`` when relevant)."""
    return int(max(h.max() + 1, t.max() + 1, lit_max_id + 1))


def laplacian_A_in(h: np.ndarray, t: np.ndarray, r: np.ndarray, n: int,
                   laplacian_type: str = "random-walk") -> Tuple[np.ndarray, np.ndarray]:
    """Initial attention matrix  A_in = sum_r norm(A_r)  (dataloader.py:449-495), float64 scipy
    arithmetic then fp32 cast (``convert_coo2tensor`` :440-447).

    Returns (indices int64 [2, nnz] sorted row-major / column ascending, values float32 [nnz]).
    """
    import scipy.sparse as sp

    total = None
    for rel in relation_order(r):
        m = r == rel
        adj = sp.coo_matrix((np.ones(int(m.sum())), (h[m], t[m])), shape=(n, n))      # :458
        rowsum = np.array(adj.sum(axis=1))
        with np.errstate(divide="ignore"):
            if laplacian_type == "random-walk":                                        # :473-481
                d = np.power(rowsum, -1.0).flatten()
                d[np.isinf(d)] = 0
                lap = sp.diags(d).dot(adj)
            elif laplacian_type == "symmetric":                                        # :463-471
                d = np.power(rowsum, -0.5).flatten()
                d[np.isinf(d)] = 0
                lap = sp.diags(d).dot(adj).dot(sp.diags(d))
            else:
                raise NotImplementedError(laplacian_type)
        lap = lap.tocoo()
        total = lap if total is None else total + lap                                  # :494
    coo = total.tocoo()
    # canonical (row, col) order so that indices can be compared bit-exactly
    order = np.lexsort((coo.col, coo.row))
    idx = np.vstack((coo.row[order], coo.col[order])).astype(np.int64)
    return idx, coo.data[order].astype(np.float32)


def numeric_literal_table(files_text: Sequence[str], n: int, numeric_dim: int) -> np.ndarray:
    """Numeric literal table (dataloader.py:111-137 + :426-431).  File *i* fills column *i* with
    ``(v + 1) / max(v)``; the first line (a count, no tab) is skipped by the ``len(data) > 1`` test.
    A later file overwrites the *whole row* of an entity that appeared in an earlier file, because
    the reference stores a fresh zero vector per (file, entity) (:129-133)."""
    table = np.zeros((n, numeric_dim), dtype=np.float32)
    for col, text in enumerate(files_text):
        vals: Dict[int, float] = {}
        vmax = 0.0
        for line in text.splitlines(keepends=False):
            parts = line.split("\t")
            if len(parts) > 1:
                v = float(parts[1].strip("\n"))
                vals[int(parts[0])] = v + 1
                vmax = max(vmax, v)
        for ent, v in vals.items():
            row = np.zeros(numeric_dim)
            if vmax != 0:
                row[col] = v / vmax
            table[ent] = row.astype(np.float32)
    return table


# ----------------------------------------------------------------------------------------------
# gate (gate.py)
# ----------------------------------------------------------------------------------------------
def gate_mul(p: Dict[str, torch.Tensor], prefix: str, x_ent, x_num, x_txt):
    """GateMul.forward (gate.py:22-28)."""
    x = torch.cat([x_ent, x_num, x_txt], dim=1)
    g = torch.tanh(F.linear(x, p[prefix + "g.weight"], p[prefix + "g.bias"]))
    z = torch.sigmoid(F.linear(x_ent, p[prefix + "gate_ent.weight"])
                      + F.linear(x_num, p[prefix + "gate_num_lit.weight"])
                      + F.linear(x_txt, p[prefix + "gate_txt_lit.weight"])
                      + p[prefix + "gate_bias"])
    return (1 - z) * x_ent + z * g


def gate_single(p: Dict[str, torch.Tensor], prefix: str, x_ent, x_lit):
    """Gate.forward (gate.py:45-51)."""
    x = torch.cat([x_ent, x_lit], dim=1)
    g = torch.tanh(F.linear(x, p[prefix + "g.weight"], p[prefix + "g.bias"]))
    z = torch.sigmoid(F.linear(x_ent, p[prefix + "gate_ent.weight"])
                      + F.linear(x_lit, p[prefix + "gate_lit.weight"])
                      + p[prefix + "gate_bias"])
    return (1 - z) * x_ent + z * g


def gate_embeddings(p, cfg: OracleConfig, num_lit, txt_lit):
    """LiteralKG.gate_embeddings (model.py:265-279)."""
    e = p["entity_embed.weight"]
    if cfg.use_num_lit and cfg.use_txt_lit:
        return gate_mul(p, "emb_mul_lit.", e, num_lit, txt_lit)
    if cfg.use_num_lit:
        return gate_single(p, "emb_num_lit.", e, num_lit)
    if cfg.use_txt_lit:
        return gate_single(p, "emb_txt_lit.", e, txt_lit)
    return e


# ----------------------------------------------------------------------------------------------
# aggregator (model.py:12-164)
# ----------------------------------------------------------------------------------------------
def _residual(p, pre: str, cfg: OracleConfig, hi, h0, layer_1based: int):
    """Aggregator.residual_connection (model.py:90-99).  Note ``(1 - beta) + beta * W`` adds the
    scalar to every element of W."""
    if not cfg.use_residual:
        return hi
    h0p = F.linear(h0, p[pre + "linear_h0.weight"], p[pre + "linear_h0.bias"])
    res = (1 - cfg.alpha) * hi + cfg.alpha * h0p
    beta = math.log(cfg.lamda / layer_1based + 1)
    ident = (1 - beta) + beta * p[pre + "weight"]
    return res @ ident


def spmm(indices: torch.Tensor, values: torch.Tensor, n: int, x: torch.Tensor) -> torch.Tensor:
    """side = A_in @ ego (model.py:106) with A given as coalesced COO (indices [2,nnz], values)."""
    out = torch.zeros((n, x.shape[1]), dtype=x.dtype)
    out.index_add_(0, indices[0], values.to(x.dtype).unsqueeze(1) * x[indices[1]])
    return out


def aggregator_forward(p, k: int, cfg: OracleConfig, ego, a_idx, a_val, h0):
    """Aggregator.forward in eval mode (model.py:101-164); ``k`` is the 0-based layer index, the
    reference passes ``l = k + 1`` (model.py:304).  gcn :108-111, graphsage :113-120,
    bi-interaction :122-130; LayerNorm :161 (dropout is identity in eval)."""
    pre = f"aggregator_layers.{k}."
    n = ego.shape[0]
    side = spmm(a_idx, a_val, n, ego)
    lin = lambda name, x: F.linear(x, p[pre + name + ".weight"], p[pre + name + ".bias"])
    act = lambda x: F.leaky_relu(x, LEAKY_SLOPE)
    t = cfg.aggregation_type
    if t == "gcn":
        emb = act(lin("linear", _residual(p, pre, cfg, ego + side, h0, k + 1)))
    elif t == "graphsage":
        hi = torch.cat([ego, side], dim=1)
        if cfg.use_residual:
            hi = _residual(p, pre, cfg, lin("linear_h", hi), h0, k + 1)
        emb = act(lin("linear", hi))
    elif t == "bi-interaction":
        s = act(lin("linear1", _residual(p, pre, cfg, ego + side, h0, k + 1)))
        b = act(lin("linear2", _residual(p, pre, cfg, ego * side, h0, k + 1)))
        emb = b + s
    else:
        raise NotImplementedError(t)
    c = emb.shape[1]
    return F.layer_norm(emb, (c,), p[pre + "layer_normalize.weight"],
                        p[pre + "layer_normalize.bias"], LN_EPS)


def gat_embeddings(p, cfg: OracleConfig, a_idx, a_val, num_lit=None, txt_lit=None,
                   return_stages: bool = False):
    """LiteralKG.gat_embeddings (model.py:298-314): gate -> L layers (each consumes the previous
    layer's *un-normalised* output, residual source = gate output) -> concat(h0, l2norm(x_1..L))
    -> LeakyReLU(linear_gat) (or the raw concat when scale_gat_dim is None)."""
    h0 = gate_embeddings(p, cfg, num_lit, txt_lit)
    stages = {"gate": h0}
    parts = [h0]
    x = h0
    for k in range(cfg.n_conv_layers):
        x = aggregator_forward(p, k, cfg, x, a_idx, a_val, h0)
        stages[f"layer{k}"] = x
        parts.append(F.normalize(x, p=2, dim=1, eps=L2_EPS))
    cat = torch.cat(parts, dim=1)
    stages["concat"] = cat
    if cfg.scale_gat_dim is not None:
        out = F.leaky_relu(F.linear(cat, p["linear_gat.weight"], p["linear_gat.bias"]), LEAKY_SLOPE)
    else:
        out = cat
    stages["final"] = out
    return (out, stages) if return_stages else out


# ----------------------------------------------------------------------------------------------
# attention update (model.py:430-471)
# ----------------------------------------------------------------------------------------------
def attention_logits(ent_w, rel_w, h, t, r):
    """Per-edge logit  v = sum_d e_t[d] * tanh(e_h[d] + e_r[d])  (model.py:441) on the RAW entity /
    relation tables (model.py:431-434)."""
    return torch.sum(ent_w[t] * torch.tanh(ent_w[h] + rel_w[r]), dim=1)


def update_attention(ent_w, rel_w, h, t, r, relations: Iterable[int], n: int):
    """LiteralKG.update_attention (model.py:444-471) with the reference's own op sequence: one
    pass per relation (``where`` + two gathers + tanh + row-sum), un-coalesced COO, then
    ``torch.sparse.softmax`` over dim 1, which coalesces (SUMS duplicate (h,t) logits) first.
    Edges whose relation is missing from ``relations`` vanish.  This is the routine bench.py
    times as the CPU baseline.  Returns coalesced (indices [2,nnz], values [nnz])."""
    rows, cols, vals = [], [], []
    for rel in relations:
        sel = torch.where(r == rel)
        bh, bt = h[sel], t[sel]
        rows.append(bh)
        cols.append(bt)
        vals.append(torch.sum(ent_w[bt] * torch.tanh(ent_w[bh] + rel_w[rel]), dim=1))
    idx = torch.stack([torch.cat(rows), torch.cat(cols)])
    a = torch.sparse_coo_tensor(idx, torch.cat(vals), (n, n))
    a = torch.sparse.softmax(a, dim=1).coalesce()
    return a.indices(), a.values()


def update_attention_projected(ent_w, rel_w, w_rel, h, t, r, relations: Iterable[int], n: int):
    """The relation-projected attention the reference keeps commented out (model.py:436-439), with the rest of
    update_attention (model.py:444-471) unchanged:  r_mul_h = h_embed @ W_r;  r_mul_t = t_embed @ W_r;
    v = sum(r_mul_t * tanh(r_mul_h + r_embed), dim=1).  ``w_rel`` [R, embed_dim, relation_dim]."""
    rows, cols, vals = [], [], []
    for rel in relations:
        sel = torch.where(r == rel)
        bh, bt = h[sel], t[sel]
        rows.append(bh)
        cols.append(bt)
        r_mul_h = ent_w[bh] @ w_rel[rel]
        r_mul_t = ent_w[bt] @ w_rel[rel]
        vals.append(torch.sum(r_mul_t * torch.tanh(r_mul_h + rel_w[rel]), dim=1))
    idx = torch.stack([torch.cat(rows), torch.cat(cols)])
    a = torch.sparse_coo_tensor(idx, torch.cat(vals), (n, n))
    a = torch.sparse.softmax(a, dim=1).coalesce()
    return a.indices(), a.values()


def update_attention_segments(ent_w, rel_w, h, t, r, relations: Iterable[int], n: int):
    """Independent numpy restatement of the same semantics (sort by (h,t), sum duplicate logits,
    max-subtracted softmax per head row) used to cross-check ``update_attention`` and to spell
    out the structure the CUDA kernel must reproduce bit-exactly (indices) / to tolerance (values)."""
    keep = np.isin(r.numpy(), np.asarray(list(relations), dtype=np.int64))
    hh, tt, rr = h.numpy()[keep], t.numpy()[keep], r.numpy()[keep]
    logits = attention_logits(ent_w, rel_w, torch.from_numpy(hh), torch.from_numpy(tt),
                              torch.from_numpy(rr)).numpy()
    order = np.lexsort((rr, tt, hh))
    hh, tt, logits = hh[order], tt[order], logits[order]
    new = np.ones(len(hh), dtype=bool)
    new[1:] = (hh[1:] != hh[:-1]) | (tt[1:] != tt[:-1])
    seg = np.cumsum(new) - 1
    nnz = int(seg[-1]) + 1 if len(seg) else 0
    summed = np.zeros(nnz, dtype=logits.dtype)
    np.add.at(summed, seg, logits)
    uh, ut = hh[new], tt[new]
    rowmax = np.full(n, -np.inf, dtype=logits.dtype)
    np.maximum.at(rowmax, uh, summed)
    ex = np.exp(summed - rowmax[uh])
    den = np.zeros(n, dtype=logits.dtype)
    np.add.at(den, uh, ex)
    vals = ex / den[uh]
    return torch.from_numpy(np.vstack((uh, ut))), torch.from_numpy(vals)


# ----------------------------------------------------------------------------------------------
# scoring / prediction (model.py:473-497) and the top-k extension
# ----------------------------------------------------------------------------------------------
def calc_score(all_embed, head_ids, tail_ids):
    """model.py:473-486 given the output of gat_embeddings()."""
    return all_embed[head_ids] @ all_embed[tail_ids].t()


def predict_links(all_embed, head_ids, tail_ids, milestone: float):
    """model.py:488-491: global min-max normalisation over the whole batch matrix, threshold,
    int32.  All-equal scores give NaN -> all zeros."""
    s = calc_score(all_embed, head_ids, tail_ids)
    s = (s - torch.min(s)) / (torch.max(s) - torch.min(s))
    return (s > milestone).int()


def topk_links(all_embed, head_ids, tail_ids, k: int):
    """Extension named by BASELINE.json (no counterpart in the reference, SURVEY.md fact 7):
    ``torch.topk`` of the reference's ``calc_score`` output.  Declared tie rule: larger score
    first, then lower tail position.  Returns (values [B,k], positions-in-tail_ids [B,k])."""
    s = calc_score(all_embed, head_ids, tail_ids)
    order = np.lexsort((np.broadcast_to(np.arange(s.shape[1]), s.shape), -s.numpy()), axis=1)
    pos = torch.from_numpy(np.ascontiguousarray(order[:, :k]))
    return torch.gather(s, 1, pos), pos


def rank_of(all_embed, head_ids, tail_ids, target_pos):
    """Rank (0 = best) of tail position ``target_pos[i]`` within row i under the same tie rule."""
    s = calc_score(all_embed, head_ids, tail_ids)
    tgt = s[torch.arange(s.shape[0]), target_pos].unsqueeze(1)
    pos = torch.arange(s.shape[1]).unsqueeze(0)
    better = (s > tgt) | ((s == tgt) & (pos < target_pos.unsqueeze(1)))
    return better.sum(dim=1)


# ----------------------------------------------------------------------------------------------
# losses (model.py:316-348, 364-428)
# ----------------------------------------------------------------------------------------------
def _l2_mean(x):
    # model.py:8-9
    return torch.mean(torch.sum(x * x, dim=1) / 2.0)


def prediction_loss(all_embed, cfg: OracleConfig, heads, pos, neg):
    """calculate_prediction_loss (model.py:316-348): BPR  -logsigmoid(h.t+ - h.t-)  + L2."""
    he, pe, ne = all_embed[heads], all_embed[pos], all_embed[neg]
    ps = torch.sum(he * pe, dim=1)
    ns = torch.sum(he * ne, dim=1)
    loss = torch.mean(-F.logsigmoid(ps - ns))
    return loss + cfg.fine_tuning_l2loss_lambda * (_l2_mean(he) + _l2_mean(pe) + _l2_mean(ne))


def triplet_loss(p, all_embed, cfg: OracleConfig, h, r, pos, neg):
    """calc_triplet_loss (model.py:364-428): TransR on the GAT embeddings with gat_trans_M[r]."""
    re = p["relation_embed.weight"][r]
    w = p["gat_trans_M"][r]
    proj = lambda ids: torch.bmm(all_embed[ids].unsqueeze(1), w).squeeze(1)
    hr, pr, nr = proj(h), proj(pos), proj(neg)
    ps = torch.sum((hr + re - pr) ** 2, dim=1)
    ns = torch.sum((hr + re - nr) ** 2, dim=1)
    loss = torch.mean(-F.logsigmoid(ns - ps))
    l2 = _l2_mean(hr) + _l2_mean(re) + _l2_mean(pr) + _l2_mean(nr)
    return loss + cfg.kg_l2loss_lambda * l2


# ----------------------------------------------------------------------------------------------
# variant heads: the `mlp` mode (model.py:499-519, model_bce.py:423-436) and the TransE loss of the
# BCE variant (model_bce.py:329-368)
# ----------------------------------------------------------------------------------------------
BN_EPS, BN_MOMENTUM = 1e-5, 0.1     # nn.BatchNorm1d defaults (model.py:501-503 passes none)


def batch_norm(p, pre: str, x, training: bool, update: bool = True):
    """nn.BatchNorm1d: batch mean / BIASED variance in training (running buffers updated with the UNBIASED one),
    running buffers in evaluation."""
    if training:
        mean, var = x.mean(0), x.var(0, unbiased=False)
        if update:
            p[pre + "running_mean"] = (1 - BN_MOMENTUM) * p[pre + "running_mean"] + BN_MOMENTUM * mean.detach()
            p[pre + "running_var"] = (1 - BN_MOMENTUM) * p[pre + "running_var"] + BN_MOMENTUM * x.var(0, unbiased=True).detach()
            p[pre + "num_batches_tracked"] = p[pre + "num_batches_tracked"] + 1
    else:
        mean, var = p[pre + "running_mean"], p[pre + "running_var"]
    return (x - mean) / torch.sqrt(var + BN_EPS) * p[pre + "weight"] + p[pre + "bias"]


def mlp_head(p, all_embed, head_ids, tail_ids, training: bool, update: bool = True):
    """train_MLP given gat_embeddings() (model.py:506-519): cat(head, tail) -> norm1(relu(fc1)) -> norm2(relu(fc2))
    -> sigmoid(fc3), [B, 1]."""
    x = torch.cat([all_embed[head_ids], all_embed[tail_ids]], dim=1)
    x = batch_norm(p, "norm1.", torch.relu(F.linear(x, p["fc1.weight"], p["fc1.bias"])), training, update)
    x = batch_norm(p, "norm2.", torch.relu(F.linear(x, p["fc2.weight"], p["fc2.bias"])), training, update)
    return torch.sigmoid(F.linear(x, p["fc3.weight"], p["fc3.bias"]))


def transe_loss(p, all_embed, cfg: OracleConfig, h, r, pos, neg):
    """calc_triplet_loss of model_bce.py:329-368: TransE on rows of the final embeddings."""
    re_ = p["relation_embed.weight"][r]
    he, pe, ne = all_embed[h], all_embed[pos], all_embed[neg]
    pos_s = torch.sum((he + re_ - pe) ** 2, dim=1)
    neg_s = torch.sum((he + re_ - ne) ** 2, dim=1)
    loss = torch.mean(-F.logsigmoid(neg_s - pos_s))
    l2 = _l2_mean(he) + _l2_mean(re_) + _l2_mean(pe) + _l2_mean(ne)
    return loss + cfg.kg_l2loss_lambda * l2


# ----------------------------------------------------------------------------------------------
# minibatch generators (dataloader.py:192-333)
# ----------------------------------------------------------------------------------------------
def build_kg_dict(h, t, r) -> Dict[int, List[Tuple[int, int]]]:
    """``train_kg_dict[h] -> [(t, r), ...]`` in file order (dataloader.py:395-403)."""
    d: Dict[int, List[Tuple[int, int]]] = {}
    for hh, tt, rr in zip(np.asarray(h).tolist(), np.asarray(t).tolist(), np.asarray(r).tolist()):
        d.setdefault(hh, []).append((tt, rr))
    return d


def generate_kg_batch(kg_dict, batch_size: int, neg_rate: int, training_tails: Sequence[int], rng):
    """``generate_kg_batch`` (dataloader.py:285-318) with ``sample_pos_triples_for_head`` (:254-271, one positive)
    and ``sample_neg_triples_for_head`` (:273-283).  ``rng``: a ``random.Random``.  (Upstream passes ``dict.keys()``
    to ``random.sample``, which Python >= 3.11 rejects; the list of keys is what it means.)"""
    exist_heads = list(kg_dict.keys())
    n = int(batch_size / neg_rate)
    heads = rng.sample(exist_heads, n) if n <= len(exist_heads) else [rng.choice(exist_heads) for _ in range(n)]
    out_h, out_r, out_p, out_n = [], [], [], []
    for hd in heads:
        pos = kg_dict[hd]
        tail, rel = pos[rng.randrange(len(pos))]
        negs: List[int] = []
        while len(negs) < neg_rate:
            cand = rng.choice(training_tails)
            if (cand, rel) not in pos and cand not in negs:
                negs.append(cand)
        out_h += [hd] * neg_rate                      # generate_batch_by_neg_rate (:320-333)
        out_r += [rel] * neg_rate
        out_p += [tail] * neg_rate
        out_n += negs
    return (np.asarray(out_h, dtype=np.int64), np.asarray(out_r, dtype=np.int64), np.asarray(out_p, dtype=np.int64),
            np.asarray(out_n, dtype=np.int64))


def generate_prediction_batch(head_dict, batch_size: int, neg_rate: int, tail_ids: Sequence[int], rng):
    """``generate_prediction_batch`` (dataloader.py:221-252): ``head_dict[h] -> [positive tails]``; negatives from
    ``prediction_tail_ids`` that are no positive of the head and not drawn before."""
    exist_heads = list(head_dict)
    tail_ids = list(tail_ids)
    n = int(batch_size / neg_rate)
    heads = rng.sample(exist_heads, n) if n <= len(exist_heads) else [rng.choice(exist_heads) for _ in range(n)]
    out_h, out_p, out_n = [], [], []
    for hd in heads:
        pos = head_dict[hd]
        tail = pos[rng.randrange(len(pos))]
        negs: List[int] = []
        while len(negs) < neg_rate:
            cand = rng.choice(tail_ids)
            if cand not in pos and cand not in negs:
                negs.append(cand)
        out_h += [hd] * neg_rate
        out_p += [tail] * neg_rate
        out_n += negs
    return (np.asarray(out_h, dtype=np.int64), np.asarray(out_p, dtype=np.int64), np.asarray(out_n, dtype=np.int64))


def check_batch_contract(kg_dict, heads, rels, pos, neg, neg_rate: int, candidates, distinct_heads: bool) -> None:
    """Asserts what the generators above guarantee for a batch (any random stream): heads / relations / positives
    repeated ``neg_rate`` times, every (h, r, t+) a triple of the graph, negatives from the candidate list, distinct
    per head and never a positive of the head under the drawn relation (``rels is None``: under any relation)."""
    heads, pos, neg = (np.asarray(x).reshape(-1, neg_rate) for x in (heads, pos, neg))
    assert (heads == heads[:, :1]).all() and (pos == pos[:, :1]).all()
    rr = None
    if rels is not None:
        rr = np.asarray(rels).reshape(-1, neg_rate)
        assert (rr == rr[:, :1]).all()
    if distinct_heads:
        assert len(set(heads[:, 0].tolist())) == heads.shape[0]
    cand = set(int(c) for c in candidates)
    for i in range(heads.shape[0]):
        hd = int(heads[i, 0])
        triples = kg_dict[hd]
        negs = [int(x) for x in neg[i]]
        assert len(set(negs)) == neg_rate and all(x in cand for x in negs)
        if rr is not None:
            rel = int(rr[i, 0])
            assert (int(pos[i, 0]), rel) in triples
            assert all((x, rel) not in triples for x in negs)
        else:
            tails = {tt for tt, _ in triples}
            assert int(pos[i, 0]) in tails and all(x not in tails for x in negs)


# ----------------------------------------------------------------------------------------------
# parameter initialisation with the reference's shapes (model.py:215-261, gate.py) -- used by
# bench.py / tests to create weights without importing the reference
# ----------------------------------------------------------------------------------------------
def init_params(cfg: OracleConfig, n_entities: int, n_relations: int, seed: int = 2022,
                dtype=torch.float32) -> Dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(seed)

    def xavier(*shape):
        # nn.init.xavier_uniform_ fan computation for 2-D / 3-D tensors
        recep = 1
        for s in shape[2:]:
            recep *= s
        fan_out, fan_in = shape[0] * recep, shape[1] * recep
        bound = math.sqrt(6.0 / (fan_in + fan_out))
        return ((torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * bound).to(dtype)

    def linear(prefix, out_f, in_f, bias=True, xav=True):
        if xav:
            p[prefix + ".weight"] = xavier(out_f, in_f)
        else:
            b = 1.0 / math.sqrt(in_f)
            p[prefix + ".weight"] = ((torch.rand((out_f, in_f), generator=g, dtype=torch.float64) * 2 - 1) * b).to(dtype)
        if bias:
            b = 1.0 / math.sqrt(in_f)
            p[prefix + ".bias"] = ((torch.rand((out_f,), generator=g, dtype=torch.float64) * 2 - 1) * b).to(dtype)

    p: Dict[str, torch.Tensor] = {}
    d, rd = cfg.embed_dim, cfg.relation_dim
    p["entity_embed.weight"] = xavier(n_entities, d)
    p["relation_embed.weight"] = xavier(n_relations, rd)
    if cfg.scale_gat_dim is not None:
        linear("linear_gat", cfg.scale_gat_dim, cfg.total_conv_dim)
        p["gat_trans_M"] = xavier(n_relations, cfg.scale_gat_dim, rd)
    else:
        p["gat_trans_M"] = xavier(n_relations, cfg.total_conv_dim, rd)
    if cfg.use_num_lit and cfg.use_txt_lit:
        pre = "emb_mul_lit"
        linear(pre + ".g", d, d + cfg.num_lit_dim + cfg.txt_lit_dim, xav=False)
        linear(pre + ".gate_ent", d, d, bias=False, xav=False)
        linear(pre + ".gate_num_lit", d, cfg.num_lit_dim, bias=False, xav=False)
        linear(pre + ".gate_txt_lit", d, cfg.txt_lit_dim, bias=False, xav=False)
        p[pre + ".gate_bias"] = torch.zeros(d, dtype=dtype)
    elif cfg.use_num_lit or cfg.use_txt_lit:
        pre = "emb_num_lit" if cfg.use_num_lit else "emb_txt_lit"
        lit = cfg.num_lit_dim if cfg.use_num_lit else cfg.txt_lit_dim
        linear(pre + ".g", d, d + lit, xav=False)
        linear(pre + ".gate_ent", d, d, bias=False, xav=False)
        linear(pre + ".gate_lit", d, lit, bias=False, xav=False)
        p[pre + ".gate_bias"] = torch.zeros(d, dtype=dtype)
    dims = cfg.conv_dims
    for k in range(cfg.n_conv_layers):
        pre = f"aggregator_layers.{k}"
        din, dout = dims[k], dims[k + 1]
        stdv = 1.0 / math.sqrt(dout)                                     # model.py:86-88
        p[pre + ".weight"] = ((torch.rand((din, din), generator=g, dtype=torch.float64) * 2 - 1) * stdv).to(dtype)
        if cfg.use_residual:
            linear(pre + ".linear_h0", din, d)
        p[pre + ".layer_normalize.weight"] = torch.ones(dout, dtype=dtype)
        p[pre + ".layer_normalize.bias"] = torch.zeros(dout, dtype=dtype)
        if cfg.aggregation_type == "gcn":
            linear(pre + ".linear", dout, din)
        elif cfg.aggregation_type == "graphsage":
            if cfg.use_residual:
                linear(pre + ".linear_h", din, 2 * din)
                linear(pre + ".linear", dout, din)
            else:
                linear(pre + ".linear", dout, 2 * din)
        elif cfg.aggregation_type == "bi-interaction":
            linear(pre + ".linear1", dout, din)
            linear(pre + ".linear2", dout, din)
        else:
            raise NotImplementedError(cfg.aggregation_type)
    return p


def cast_params(p: Dict[str, torch.Tensor], dtype) -> Dict[str, torch.Tensor]:
    return {k: (v.to(dtype) if v.is_floating_point() and not v.is_sparse else v) for k, v in p.items()}
