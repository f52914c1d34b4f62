"""B200-native drop-in for the reference's ``model.py`` (``Aggregator`` :12-164, ``LiteralKG`` :167-532).

Same class names, constructor signatures, ``forward(*input, device=, mode=)`` modes, public helpers,
attribute names and state-dict keys (SURVEY.md fact 9), so the reference's training / evaluation
scripts run unchanged.  What differs is the inside: every stage of the message-passing + scoring path
runs in the sm_100a kernels of liblkg.so (include/lkg.h); there is no PyTorch-math or CPU fallback.

Stage map (reference -> here)
    gate_embeddings   model.py:265-279 -> ops.gate        (one fused GEMM + tanh/sigmoid/mix epilogue)
    Aggregator        model.py:101-164 -> ops.aggregate   (CSR SpMM + folded combine + LayerNorm + L2 norm)
    cat + linear_gat  model.py:308-311 -> ops.linear      (the concat buffer is written in place by the layers)
    update_attention  model.py:444-471 -> ops.attn_update (logits + duplicate merge + row softmax, on device)
    calc_score        model.py:473-486 -> ops.score
    predict_links     model.py:488-491 -> ops.predict
"""
from __future__ import annotations

import math
from types import SimpleNamespace
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from .gate import Gate, GateMul
from .graph import GraphPlan


def _param_key(module: nn.Module):
    """Identity + in-place version of every parameter: cache key for tensors derived from the parameters only
    (folded matrices, stacked gate weights).  Optimizer steps and load_state_dict bump the versions."""
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


def _dense_param_key(module: nn.Module):
    """``_param_key`` without the sparse ``A_in`` entry of LiteralKG (a sparse tensor has no data pointer)."""
    return tuple((p.data_ptr(), p._version) for n_, p in module.named_parameters() if n_ != "A_in")


_EYE = {}


def _identity(n: int, device) -> torch.Tensor:
    key = (n, str(device))
    if key not in _EYE:
        _EYE[key] = torch.eye(n, dtype=torch.float32, device=device)
    return _EYE[key]


def _query_ids(x, dev) -> torch.Tensor:
    """Ids of a query call (any sequence or tensor) as a flat int64 tensor on ``dev``."""
    return torch.as_tensor(x).to(device=dev, dtype=torch.int64).reshape(-1)


def _outside(x: torch.Tensor, hi: int) -> torch.Tensor:
    """Device flag: some id of ``x`` lies outside [0, hi)."""
    return ((x < 0) | (x >= hi)).any()


def _candidate_ids(candidates, n: int, dev, bad: dict):
    """The candidate list of a query call: -> (cand int64 clamped to [0, n), n_cand, cmap int32 [n] = candidate position
    of every entity or -1), or (None, n, None) for every entity.  Adds the device flags "candidate ids outside
    [0, n_entities)" and "duplicate candidate ids" to ``bad``; they are raised after the call's one host read-back."""
    if candidates is None:
        return None, n, None
    cand = _query_ids(candidates, dev)
    n_cand = cand.numel()
    bad["candidate ids outside [0, n_entities)"] = _outside(cand, n)
    cand = cand.clamp(0, n - 1)
    pos = torch.arange(n_cand, dtype=torch.int32, device=dev)
    cmap = torch.full((n,), -1, dtype=torch.int32, device=dev)
    cmap[cand] = pos
    bad["duplicate candidate ids"] = (cmap[cand] != pos).any()
    return cand, n_cand, cmap


def _raise_flags(bad: dict, host: list) -> None:
    for msg, flag in zip(bad, host):
        if flag:
            raise ValueError(msg)


def _L2_loss_mean(x):
    return torch.mean(torch.sum(torch.pow(x, 2), dim=1, keepdim=False) / 2.)


class Aggregator(nn.Module):
    """One propagation layer (model.py:12-164): gcn / graphsage / bi-interaction, optional GCNII-style
    residual connection, LeakyReLU, LayerNorm, message dropout."""

    def __init__(self, in_dim, out_dim, dropout, aggregator_type, use_residual=False, args=None):
        super().__init__()
        self.in_dim, self.out_dim, self.dropout = in_dim, out_dim, dropout
        self.aggregator_type = aggregator_type
        self.use_residual = use_residual
        self.weight = nn.Parameter(torch.empty(in_dim, in_dim))
        if use_residual:
            self.linear_h0 = nn.Linear(args.embed_dim, in_dim)
            nn.init.xavier_uniform_(self.linear_h0.weight)
        self.reset_parameters()
        self.message_dropout = nn.Dropout(dropout)
        self.activation = nn.LeakyReLU()
        self.layer_normalize = nn.LayerNorm(out_dim)
        if aggregator_type == 'gcn':
            self.linear = nn.Linear(in_dim, out_dim)
            nn.init.xavier_uniform_(self.linear.weight)
        elif aggregator_type == 'graphsage':
            if use_residual:
                self.linear_h = nn.Linear(in_dim * 2, in_dim)
                nn.init.xavier_uniform_(self.linear_h.weight)
                self.linear = nn.Linear(in_dim, out_dim)
            else:
                self.linear = nn.Linear(in_dim * 2, out_dim)
            nn.init.xavier_uniform_(self.linear.weight)
        elif aggregator_type == 'bi-interaction':
            self.linear1 = nn.Linear(in_dim, out_dim)
            self.linear2 = nn.Linear(in_dim, out_dim)
            nn.init.xavier_uniform_(self.linear1.weight)
            nn.init.xavier_uniform_(self.linear2.weight)
        else:
            # 'gin' exists in the reference but is outside the accelerated path (SURVEY.md section 2, row 2)
            raise NotImplementedError(aggregator_type)
        self._plan_cache: Optional[Tuple[int, int, GraphPlan, torch.Tensor]] = None
        self._fold_cache = None

    def reset_parameters(self):
        stdv = 1. / math.sqrt(self.out_dim)
        self.weight.data.uniform_(-stdv, stdv)

    # ---- parameter folding (DESIGN.md section 4) -------------------------------------------------
    def folded(self, lamda: float, alpha: float, l: int, differentiable: bool = False
               ) -> Dict[str, Optional[torch.Tensor]]:
        """linear(residual(hi)) == hi @ P + h0 @ Q + c with  M = (1-b) + b*W,  b = ln(lamda/l + 1)
        (model.py:90-99): P = (1-a) M W_lin^T, Q = a W_h0^T M W_lin^T, c = a b_h0 M W_lin^T + b_lin.
        Formed in float64 from the live parameters, returned in fp32.  Keys: pa, pb, p2 ([d_in, d_out]),
        q1, q2 ([embed_dim, d_out] or None), c1, c2 ([d_out]).  ``differentiable``: build the fold under autograd
        (no cache) so that gradients w.r.t. P / Q / c flow on to the layer's parameters."""
        key = (float(lamda), float(alpha), int(l), _param_key(self))
        if not differentiable and self._fold_cache is not None and self._fold_cache[0] == key:
            return self._fold_cache[1]
        dd = torch.float64
        t = self.aggregator_type
        d = self.in_dim

        def lin(m):
            return m.weight.to(dd), m.bias.to(dd)

        out: Dict[str, Optional[torch.Tensor]] = dict(pa=None, pb=None, p2=None, q1=None, q2=None, c1=None, c2=None)
        if self.use_residual:
            beta = math.log(lamda / l + 1)
            m_id = (1 - beta) + beta * self.weight.to(dd)
            wh0, bh0 = lin(self.linear_h0)

            def fold(w_lin, b_lin):
                mw = m_id @ w_lin.t()                                  # [d, C]
                return (1 - alpha) * mw, alpha * (wh0.t() @ mw), alpha * (bh0 @ mw) + b_lin
        else:
            def fold(w_lin, b_lin):
                return w_lin.t(), None, b_lin

        if t == 'gcn':
            p, q, c = fold(*lin(self.linear))
            out.update(pa=p, pb=p, q1=q, c1=c)
        elif t == 'bi-interaction':
            p, q, c = fold(*lin(self.linear1))
            p2, q2, c2 = fold(*lin(self.linear2))
            out.update(pa=p, pb=p, p2=p2, q1=q, q2=q2, c1=c, c2=c2)
        else:  # graphsage
            if self.use_residual:
                wh, bh = lin(self.linear_h)
                p, q, c = fold(*lin(self.linear))
                out.update(pa=wh[:, :d].t() @ p, pb=wh[:, d:].t() @ p, q1=q, c1=bh @ p + c)
            else:
                w, b = lin(self.linear)
                out.update(pa=w[:, :d].t(), pb=w[:, d:].t(), c1=b)
        res = {}
        for k, v in out.items():
            res[k] = None if v is None else v.float().contiguous()
        if res["pa"] is not None and out["pa"] is out["pb"]:
            res["pa"] = res["pb"]                                      # keep identity: "sum" mode of the kernel
        if not differentiable:
            self._fold_cache = (key, res)   # derived from the parameters only: reused until one of them changes
        return res

    def _drop_mask(self, n: int, device) -> Optional[torch.Tensor]:
        if self.training and self.dropout > 0:
            keep = 1.0 - self.dropout
            return (torch.rand((n, self.out_dim), device=device) < keep).float() / keep
        return None

    def run(self, plan: GraphPlan, a_values: torch.Tensor, ego: torch.Tensor, f: Dict[str, Optional[torch.Tensor]],
            r1: Optional[torch.Tensor], r2: Optional[torch.Tensor], x_out: torch.Tensor,
            xn_out: Optional[torch.Tensor], fold_ego: bool = False, xn_planes=None, rows=None, z=None,
            saved: Optional[dict] = None) -> torch.Tensor:
        """``rows`` = (begin, end): the head rows this rank owns; r1 / r2 / xn_out / xn_planes then hold those rows
        only, ``ego`` and ``x_out`` stay indexed by the global row.  ``saved`` (training): receives the dropout
        mask, the pre-activations and (bi-interaction) side = A @ ego for the backward pass."""
        pa = None if fold_ego else f["pa"]
        rb, re = (0, ego.shape[0]) if rows is None else rows
        pb, p2 = f["pb"], f["p2"]
        mask = self._drop_mask(re - rb, ego.device)
        o_out = side_out = None
        if saved is not None:
            nt = 2 if p2 is not None else 1
            o_out = torch.empty((re - rb, nt * self.out_dim), dtype=torch.float32, device=ego.device)
            if p2 is not None:
                side_out = torch.empty((re - rb, ego.shape[1]), dtype=torch.float32, device=ego.device)
            saved.update(mask=mask, o=o_out, side=side_out)
        if z is not None:
            # the neighbour sum term arrives pre-projected (z = ego @ Pb, DESIGN.md section 4):
            #   bi-interaction: the wide kernel gathers z next to the ego rows and only combines the product term;
            #   gcn / graphsage: nothing but z is gathered -- the layer runs on the d_out-wide z table
            assert pa is None
            if p2 is None:
                ego, z, pb = z, None, _identity(self.out_dim, ego.device)
            else:
                pb = None
        return ops.aggregate(plan, a_values, ego, self.out_dim, pa, pb, p2, r1, r2,
                             self.layer_normalize.weight, self.layer_normalize.bias,
                             mask, x_out, xn_out, xn_planes, local_row_base=rb, z=z, o_out=o_out, side_out=side_out)

    def forward(self, ego_embeddings, A_in, all_layers, lamda, alpha, l):
        """Reference signature (model.py:101): ``A_in`` is a sparse COO tensor, ``all_layers[0]`` the gate
        output used by the residual connection, ``l`` the 1-based layer index."""
        from .autograd import require_no_grad
        require_no_grad(self, [ego_embeddings] + list(all_layers[:1]), "Aggregator")
        with torch.no_grad():
            ego = _lib.f32c(ego_embeddings)
            _lib.require_cuda(ego, "ego_embeddings")
            plan, vals = self._plan_for(A_in)
            f = self.folded(lamda, alpha, l)
            r1, r2 = f["c1"], f["c2"]
            if self.use_residual:
                h0 = _lib.f32c(all_layers[0])
                qs = [f["q1"]] + ([f["q2"]] if f["q2"] is not None else [])
                cs = [f["c1"]] + ([f["c2"]] if f["c2"] is not None else [])
                r = ops.linear([ops.split_planes(h0)], torch.cat(qs, dim=1).t().contiguous(), torch.cat(cs))
                r1 = r[:, :self.out_dim]
                r2 = r[:, self.out_dim:] if f["q2"] is not None else None
            x = torch.empty((ego.shape[0], self.out_dim), dtype=torch.float32, device=ego.device)
            return self.run(plan, vals, ego, f, r1, r2, x, None)

    def _plan_for(self, A_in: torch.Tensor) -> Tuple[GraphPlan, torch.Tensor]:
        key = (A_in._values().data_ptr(), A_in._nnz())
        if self._plan_cache is None or self._plan_cache[:2] != key:
            plan = GraphPlan.from_coo(A_in._indices(), A_in.shape[0])
            self._plan_cache = (*key, plan, plan.import_values(A_in._values()))
        return self._plan_cache[2], self._plan_cache[3]


class _GatEmbeddingsFn(torch.autograd.Function):
    """Full-graph embedding pass as one autograd node: forward = the inference kernels (+ saved activations),
    backward = csrc/backward.cu.  ``leaves`` only tie the node into the graph; values travel in ``pre``."""

    @staticmethod
    def forward(ctx, model, pre, *leaves):
        keep: dict = {}
        out = model._gat_embeddings_native(keep=keep, pre=pre)
        part = model._part if (model._part is not None and model._part.world > 1) else None
        if part is not None:
            # every rank evaluates the (replicated) loss on the full matrix: the gradient of that replica w.r.t. this
            # rank's rows is simply its row slice of d loss / d out
            full = torch.empty((part.padded, out.shape[1]), dtype=torch.float32, device=out.device)
            full[part.begin:part.end] = out
            out = part.all_gather_rows(full)[:model.n_entities]
        if getattr(model, "debug_keep_activations", False):      # tests: sign pattern of the LeakyReLU inputs
            model._debug_keep = keep
        ctx.model, ctx.pre, ctx.keep = model, pre, keep
        ctx.present = [t is not None for t in leaves]
        # the backward reads the live parameters (detached): remember their in-place versions so that an optimizer
        # step between this forward and its backward is an error, not a silently wrong gradient
        ctx.versions = _dense_param_key(model)
        return out

    @staticmethod
    def backward(ctx, g_out):
        if ctx.keep is None:
            raise RuntimeError("the saved activations of this gat_embeddings() pass were freed by its first backward; "
                               "run the forward again (retain_graph is not supported by the fused pass)")
        if _dense_param_key(ctx.model) != ctx.versions:
            raise RuntimeError("a parameter of the model was modified in place (optimizer step / load_state_dict) between "
                               "gat_embeddings() and its backward: the fused backward reads the live parameters")
        with torch.no_grad():
            grads = ctx.model._gat_backward(ctx.keep, ctx.pre, g_out)
        ctx.keep = None
        assert len(grads) == len(ctx.present)
        return (None, None, *[g if has else None for g, has in zip(grads, ctx.present)])


class _BprLossFn(torch.autograd.Function):
    """calculate_prediction_loss (model.py:316-348) as one kernel forward and one backward (csrc/loss.cu)."""

    @staticmethod
    def forward(ctx, emb, h, pos, neg, lam):
        emb = emb if (emb.dtype == torch.float32 and emb.stride(1) == 1) else _lib.f32c(emb)
        loss = torch.zeros((), dtype=torch.float32, device=emb.device)
        ops.bpr_loss(emb, h, pos, neg, lam, loss)
        ctx.save_for_backward(emb, h, pos, neg)
        ctx.lam = lam
        return loss

    @staticmethod
    def backward(ctx, g):
        emb, h, pos, neg = ctx.saved_tensors
        d_emb = torch.zeros_like(emb)
        ops.bpr_loss(emb, h, pos, neg, ctx.lam, None, grad_scale=g.float().contiguous(), d_emb=d_emb)
        return d_emb, None, None, None, None


class _TransRLossFn(torch.autograd.Function):
    """calc_triplet_loss (model.py:364-428): no [B, G, D] copy of W_r, gradients scattered by the kernel."""

    @staticmethod
    def forward(ctx, emb, rel, trans_m, h, r, pos, neg, lam):
        emb = emb if (emb.dtype == torch.float32 and emb.stride(1) == 1) else _lib.f32c(emb)
        loss = torch.zeros((), dtype=torch.float32, device=emb.device)
        ops.transr_loss(emb, rel, trans_m, h, r, pos, neg, lam, loss)
        ctx.save_for_backward(emb, rel, trans_m, h, r, pos, neg)
        ctx.lam = lam
        return loss

    @staticmethod
    def backward(ctx, g):
        emb, rel, trans_m, h, r, pos, neg = ctx.saved_tensors
        d_emb = torch.zeros_like(emb)
        d_rel = torch.zeros(rel.shape, dtype=torch.float32, device=emb.device)
        d_m = torch.zeros(trans_m.shape, dtype=torch.float32, device=emb.device)
        ops.transr_loss(emb, rel, trans_m, h, r, pos, neg, ctx.lam, None, grad_scale=g.float().contiguous(),
                        d_emb=d_emb, d_relation=d_rel, d_trans_m=d_m)
        return d_emb, d_rel, d_m, None, None, None, None, None


class _TransELossFn(torch.autograd.Function):
    """calc_triplet_loss of the BCE variant (model_bce.py:329-368): TransE on rows of the final embeddings."""

    @staticmethod
    def forward(ctx, emb, rel, h, r, pos, neg, lam):
        emb = emb if (emb.dtype == torch.float32 and emb.stride(1) == 1) else _lib.f32c(emb)
        loss = torch.zeros((), dtype=torch.float32, device=emb.device)
        ops.transe_loss(emb, rel, h, r, pos, neg, lam, loss)
        ctx.save_for_backward(emb, rel, h, r, pos, neg)
        ctx.lam = lam
        return loss

    @staticmethod
    def backward(ctx, g):
        emb, rel, h, r, pos, neg = ctx.saved_tensors
        d_emb = torch.zeros_like(emb)
        d_rel = torch.zeros(rel.shape, dtype=torch.float32, device=emb.device)
        ops.transe_loss(emb, rel, h, r, pos, neg, ctx.lam, None, grad_scale=g.float().contiguous(), d_emb=d_emb,
                        d_relation=d_rel)
        return d_emb, d_rel, None, None, None, None, None


class _MlpHeadFn(torch.autograd.Function):
    """train_MLP (model.py:506-519, model_bce.py:423-436) on one minibatch of (head, tail) pairs:
    sigmoid(fc3(norm2(relu(fc2(norm1(relu(fc1([emb[h] | emb[t]])))))))) as fused fully-connected steps
    (csrc/mlp_head.cu); the gathered [B, 2G] block and the BatchNorm outputs are never materialised."""

    @staticmethod
    def forward(ctx, owner, emb, h, t, w1, b1, g1, be1, w2, b2, g2, be2, w3, b3):
        emb = emb if (emb.dtype == torch.float32 and emb.stride(1) == 1) else _lib.f32c(emb)
        dev = emb.device
        h = h.to(device=dev, dtype=torch.int64).contiguous()
        t = t.to(device=dev, dtype=torch.int64).contiguous()
        m = h.numel()
        training = owner.norm1.training
        if training and m < 2:
            raise ValueError("Expected more than 1 value per channel when training (BatchNorm1d)")
        stats = (lambda n: torch.zeros(2 * n, dtype=torch.float64, device=dev)) if training else (lambda n: None)
        st1, st2 = stats(w1.shape[0]), stats(w2.shape[0])
        a1 = ops.mlp_fc_fwd(emb, w1, b1, ops.ACT_FC_RELU, m, pair=(h, t), stats=st1)
        sc1, sh1, mean1, rstd1 = ops.bn_finalize(st1, m, owner.norm1, training)
        a2 = ops.mlp_fc_fwd(a1, w2, b2, ops.ACT_FC_RELU, m, affine=(sc1, sh1), stats=st2)
        sc2, sh2, mean2, rstd2 = ops.bn_finalize(st2, m, owner.norm2, training)
        y = ops.mlp_fc_fwd(a2, w3, b3, ops.ACT_FC_SIGMOID, m, affine=(sc2, sh2))
        ctx.save_for_backward(emb, h, t, w1, w2, w3, g1, g2, a1, a2, y, sc1, sh1, mean1, rstd1, sc2, sh2, mean2, rstd2)
        ctx.training = training
        return y

    @staticmethod
    def backward(ctx, dy):
        (emb, h, t, w1, w2, w3, g1, g2, a1, a2, y, sc1, sh1, mean1, rstd1, sc2, sh2, mean2, rstd2) = ctx.saved_tensors
        dev, m, tr = emb.device, h.numel(), ctx.training
        f64 = lambda n: torch.zeros(2 * n, dtype=torch.float64, device=dev)
        dz3 = ops.sigmoid_bwd(dy, y).view(m, 1)
        dw3, db3 = ops.mlp_fc_bwd_weight(dz3, a2, w3.shape[1], affine=(sc2, sh2))
        s2 = f64(w2.shape[0])
        dy2 = ops.mlp_fc_bwd_input(dz3, w3, torch.empty((m, w2.shape[0]), dtype=torch.float32, device=dev),
                                   bn=(a2, mean2, rstd2, s2))
        dz2, dg2, dbe2 = ops.bn_relu_bwd(dy2, a2, mean2, rstd2, g2, s2, tr)
        dw2, db2 = ops.mlp_fc_bwd_weight(dz2, a1, w2.shape[1], affine=(sc1, sh1))
        s1 = f64(w1.shape[0])
        dy1 = ops.mlp_fc_bwd_input(dz2, w2, torch.empty((m, w1.shape[0]), dtype=torch.float32, device=dev),
                                   bn=(a1, mean1, rstd1, s1))
        dz1, dg1, dbe1 = ops.bn_relu_bwd(dy1, a1, mean1, rstd1, g1, s1, tr)
        dw1, db1 = ops.mlp_fc_bwd_weight(dz1, emb, w1.shape[1], pair=(h, t))
        d_emb = ops.mlp_fc_bwd_input(dz1, w1, torch.zeros_like(emb), pair=(h, t))
        return None, d_emb, None, None, dw1, db1, dg1, dbe1, dw2, db2, dg2, dbe2, dw3, db3


class LiteralKG(nn.Module):
    """model.py:167-532."""

    def __init__(self, args, n_entities, n_relations, A_in=None, numerical_literals=None, text_literals=None):
        super().__init__()
        self.use_pretrain = args.use_pretrain
        self.args = args
        self.device = args.device
        self.n_entities, self.n_relations = n_entities, n_relations
        self.embed_dim, self.relation_dim = args.embed_dim, args.relation_dim
        self.scale_gat_dim = args.scale_gat_dim
        self.use_residual, self.alpha, self.lamda = args.use_residual, args.alpha, args.lamda
        self.aggregation_type = args.aggregation_type
        self.n_layers = args.n_conv_layers
        self.conv_dim_list = [args.embed_dim] + [args.conv_dim] * self.n_layers
        self.total_conv_dim = sum(self.conv_dim_list)
        self.mess_dropout = [args.mess_dropout] * self.n_layers
        self.kg_l2loss_lambda = args.kg_l2loss_lambda
        self.prediction_l2loss_lambda = args.fine_tuning_l2loss_lambda
        self.pre_training_neg_rate = args.pre_training_neg_rate
        self.fine_tuning_neg_rate = args.fine_tuning_neg_rate
        self.n_num_lit, self.n_txt_lit = args.num_lit_dim, args.txt_lit_dim

        self.entity_embed = nn.Embedding(n_entities, self.embed_dim)
        self.relation_embed = nn.Embedding(n_relations, self.relation_dim)
        if self.scale_gat_dim is not None:
            self.linear_gat = nn.Linear(self.total_conv_dim, self.scale_gat_dim)
            self.gat_activation = nn.LeakyReLU()
            nn.init.xavier_uniform_(self.linear_gat.weight)
            self.gat_trans_M = nn.Parameter(torch.empty(n_relations, self.scale_gat_dim, self.relation_dim))
        else:
            self.gat_trans_M = nn.Parameter(torch.empty(n_relations, self.total_conv_dim, self.relation_dim))
        nn.init.xavier_uniform_(self.entity_embed.weight)
        nn.init.xavier_uniform_(self.relation_embed.weight)
        nn.init.xavier_uniform_(self.gat_trans_M)

        self.aggregator_layers = nn.ModuleList()
        # plain attributes, not buffers, exactly like the reference (model.py:241-242)
        self.numerical_literals_embed = numerical_literals
        self.text_literals_embed = text_literals
        if args.use_num_lit and args.use_txt_lit:
            self.emb_mul_lit = GateMul(self.embed_dim, self.n_num_lit, self.n_txt_lit)
        elif args.use_num_lit:
            self.emb_num_lit = Gate(self.embed_dim, self.n_num_lit)
        elif args.use_txt_lit:
            self.emb_txt_lit = Gate(self.embed_dim, self.n_txt_lit)
        for k in range(self.n_layers):
            self.aggregator_layers.append(
                Aggregator(self.conv_dim_list[k], self.conv_dim_list[k + 1], self.mess_dropout[k],
                           self.aggregation_type, self.use_residual, args))

        self.A_in = nn.Parameter(torch.sparse_coo_tensor(size=(n_entities, n_entities), dtype=torch.float32))
        if A_in is not None:
            self.A_in.data = A_in
        self.A_in.requires_grad = False
        self.milestone_score = args.milestone_score
        self._check_layer_shapes()

        # device-side plan state (not part of the state dict)
        self._agg_plan: Optional[GraphPlan] = None        # CSR of the current A_in
        self._agg_values: Optional[torch.Tensor] = None   # its values, plan order (shared with A_in.data)
        self._att_plan: Optional[GraphPlan] = None        # plan of the (h, t, r) lists given to update_att
        self._att_key = None
        self._att_ident = None
        self._att_refs = None
        self._lit_planes = None                           # fp16 hi/lo planes of the (constant) literal tables
        self._ent_planes = None                           # (key, planes) of entity_embed.weight, per parameter version
        self._unit_rec = None                             # scale record of planes bounded by 1 (normalised rows)
        self._h0q_cache = None                            # stacked h0 @ Q weight of all layers (parameter derived)
        self._part = None                                 # parallel.RowPartition when the path is row partitioned
        self._gate_prefetch = None                        # (key, gate stage) started by update_attention
        self._peer_x = None                               # parallel.PeerExchange: symmetric-memory exchange tables
        self.sync_attention = "lazy"                      # partitioned update_att: every rank fills its own rows of A_in;
                                                          # True = all-reduce at once, "lazy" = on state_dict() /
                                                          # complete_attention(), False = never
        self._a_in_pending = None
        self._local_edges = False                         # set_partition(local_edges=True)
        self.cache_embeddings = True                      # eval mode: keep gat_embeddings() until an input changes
        self._embed_cache = None
        self._a_in_epoch = 0
        self.prefetch_gate = True                         # partitioned update_att: start the next pass's gate stage
        self._lit_key = None

    # ---- helpers -------------------------------------------------------------------------------
    def _param_device(self) -> torch.device:
        dev = self.entity_embed.weight.device
        if dev.type != "cuda":
            raise RuntimeError("literalkg_b200.LiteralKG runs on CUDA sm_100 only: move the model with "
                               ".to('cuda') first (there is no CPU fallback)")
        return dev

    def _literal(self, name: str) -> torch.Tensor:
        t = getattr(self, name)
        if t is None:
            raise RuntimeError(f"{name} was not given to the constructor")
        dev = self._param_device()
        if t.device != dev or t.dtype != torch.float32 or not t.is_contiguous():
            t = t.to(device=dev, dtype=torch.float32).contiguous()
            setattr(self, name, t)           # the reference also caches the moved table (model.py:269-276)
        return t

    def _current_plan(self) -> Tuple[GraphPlan, torch.Tensor]:
        """CSR plan + values of whatever ``self.A_in`` currently holds (constructor argument, checkpoint,
        external assignment or our own update_att result)."""
        dev = self._param_device()
        a = self.A_in.data
        vals = a._values()
        if (self._agg_plan is not None and self._agg_values is not None and a.device == dev
                and vals.data_ptr() == self._agg_values.data_ptr() and a._nnz() == self._agg_plan.nnz):
            return self._agg_plan, self._agg_values
        a = a.to(dev)
        plan = GraphPlan.from_coo(a._indices(), self.n_entities)
        values = plan.import_values(a._values())
        self._agg_plan, self._agg_values = plan, values
        self._a_in_epoch += 1
        self.A_in.data = plan.sparse(values)              # same matrix, coalesced, values shared with the kernels
        return plan, values

    # ---- gate ------------------------------------------------------------------------------------
    def _literal_planes(self, tables, rows=None):
        """The literal tables are constants (plain attributes in the reference): their fp16 hi/lo planes for
        the gate GEMM are built once and reused, like the reference caches the ``.to(device)`` copy."""
        key = (tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in tables), rows)
        if self._lit_key != key:
            if rows is not None:
                tables = [t[rows[0]:rows[1]] for t in tables]
            src = tables[0] if len(tables) == 1 else torch.cat(list(tables), dim=1)
            self._lit_planes = ops.split_planes(src)
            self._lit_key = key
        return self._lit_planes

    def set_partition(self, part, local_edges: bool = False) -> None:
        """Row-partition the path over the ranks of ``part`` (``parallel.RowPartition``); None = single GPU.
        ``local_edges``: ``update_att`` will be given only the triples whose HEAD this rank owns (a pre-partitioned
        edge list: E / P triples to upload, sort and keep per rank instead of E); every kernel of the path only ever
        reads the rows of its own heads, so nothing else changes.  Not a collective: pending attention values of a
        previous partition must have been completed with ``complete_attention()`` (state_dict() checks)."""
        self._part = part
        self._local_edges = bool(local_edges) and part is not None and part.world > 1
        self._lit_key = None

    def _unit_record(self, dev) -> torch.Tensor:
        if self._unit_rec is None or self._unit_rec.device != dev:
            self._unit_rec = ops.scale_from_bound(1.0, dev)
        return self._unit_rec

    def _gate_module(self):
        """(gate module or None, its literal tables) for the configured literal kinds (model.py:265-279)."""
        if self.args.use_num_lit and self.args.use_txt_lit:
            return self.emb_mul_lit, (self._literal("numerical_literals_embed"), self._literal("text_literals_embed"))
        if self.args.use_num_lit:
            return self.emb_num_lit, (self._literal("numerical_literals_embed"),)
        if self.args.use_txt_lit:
            return self.emb_txt_lit, (self._literal("text_literals_embed"),)
        return None, ()

    def gate_embeddings(self, out: Optional[torch.Tensor] = None, planes_window=None, rows=None, packed=None,
                        gz_out=None):
        """model.py:265-279.  ``planes_window``: optional (Planes, col, k) column window that receives the scaled
        fp16 hi/lo copy of the result (A operand of the GEMMs that follow).  ``rows`` = (begin, end): only these
        entity rows (the gate is row local; used by the row partition).  ``packed`` / ``gz_out``: training path
        (interleaved weights built under autograd by the caller, saved activations for the backward)."""
        ent = self.entity_embed.weight
        dev = self._param_device()
        sl = slice(None) if rows is None else slice(rows[0], rows[1])
        with torch.no_grad():
            ent_rows = ent.detach()[sl]
            gate_mod, tables = self._gate_module()
            if gate_mod is not None:
                # operand preparation of a parameter: the fp16 hi/lo planes of the entity table are kept while the
                # table is unchanged (in-place version counter), like the planes of the constant literal tables
                pkey = (ent.data_ptr(), ent._version, rows)
                if self._ent_planes is None or self._ent_planes[0] != pkey:
                    self._ent_planes = (pkey, ops.split_planes(ent_rows))
                ent_planes = self._ent_planes[1]
                out_planes = None
                if planes_window is not None:
                    # |gate output| <= max(1, max|entity|): convex mix of the entity row and a tanh
                    base, col, k = planes_window
                    out_planes = base.view(col, k, rec=ops.scale_from_bound(1.0, dev, other=ent_planes.rec))
                lit_planes = self._literal_planes(tables, rows)
                if gz_out is not None:
                    self._gate_operands = (ent_planes, lit_planes)       # reused by the backward pass
                res = gate_mod(ent_rows, *[t[sl] for t in tables], out=out, out_planes=out_planes,
                               ent_planes=ent_planes, lit_planes=lit_planes, packed=packed, gz_out=gz_out)
                return (res, out_planes) if planes_window is not None else res
            if out is not None:
                out.copy_(ent_rows)
                if planes_window is not None:
                    base, col, k = planes_window
                    view = base.view(col, k, rec=torch.empty(_lib.LKG_SCALE_FLOATS, dtype=torch.float32, device=dev))
                    ops.split_planes(ent_rows, out=view)
                    return out, view
                return out
        return ent if rows is None else ent[sl]

    # ---- full-graph embedding pass -------------------------------------------------------------
    def gat_embeddings(self, gather: bool = True):
        """model.py:298-314.  Row partitioned: ``gather=False`` returns this rank's rows only (what the sharded
        scoring consumes); the default all-gathers the [N, G] result like the reference returns it."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return self._gat_embeddings_autograd()
        with torch.no_grad():
            # The reference recomputes the whole graph for every head batch of an evaluation (utils/model_utils.py:55-60
            # -> model.py:474).  In eval mode the result only depends on the parameters, the literal tables and A_in:
            # it is kept until one of them changes (in-place version counters; update_att bumps the A_in epoch).
            key = None
            if self.cache_embeddings and not self.training:
                self._gate_module()                # normalise the state the key is built from first: the literal tables
                self._current_plan()               # move to the device, A_in is re-expressed in plan order
                vals = self.A_in.data._values()
                key = (tuple((p.data_ptr(), p._version) for n_, p in self.named_parameters() if n_ != "A_in"),
                       tuple(None if t is None else (t.data_ptr(), t._version)
                             for t in (self.numerical_literals_embed, self.text_literals_embed)),
                       self._a_in_epoch, vals.data_ptr(), vals._version, id(self._part), bool(gather))
                if self._embed_cache is not None and self._embed_cache[0] == key:
                    return self._embed_cache[1]     # shared with every caller until an input changes: treat as read-only
            out = self._gat_embeddings_native()
            part = self._part
            if not (part is None or part.world == 1 or not gather):
                full = torch.empty((part.padded, out.shape[1]), dtype=torch.float32, device=out.device)
                full[part.begin:part.end] = out
                out = part.all_gather_rows(full)[:self.n_entities]
            self._embed_cache = None if key is None else (key, out)
            return out

    def _stack_q(self, folds):
        """The h0 @ Q GEMM of all layers as ONE stacked weight: rows = [layer 0: q1 + pa | q2 | layer 1: q1 | q2 ...
        | z columns = layer 0's pb].  Returns (wq [cols, embed_dim], cq [cols], offsets, zcol)."""
        qs, cs, off, offsets = [], [], 0, []
        for k, f in enumerate(folds):
            q1 = f["q1"] + f["pa"] if k == 0 else f["q1"]      # layer 0: ego == h0, fold ego @ Pa into h0 @ Q
            offsets.append(off)
            qs.append(q1); cs.append(f["c1"]); off += q1.shape[1]
            if f["q2"] is not None:
                qs.append(f["q2"]); cs.append(f["c2"]); off += f["q2"].shape[1]
        # layer 0 again: z = h0 @ Pb, the neighbour sum term projected BEFORE the aggregation
        # ((A h0) Pb == A (h0 Pb)): 32 more GEMM columns replace a 300 x 32 combine per row, and for
        # gcn / graphsage the 1 200-byte neighbour gather of layer 1 altogether
        zcol = off if self._layer1_z_path() else -1
        if zcol >= 0:
            qs.append(folds[0]["pb"]); cs.append(torch.zeros_like(folds[0]["c1"])); off += folds[0]["pb"].shape[1]
        return torch.cat(qs, dim=1).t().contiguous(), torch.cat(cs), offsets, zcol

    def _layer1_z_path(self) -> bool:
        """Layer 1 of a residual model with wide h0 gathers the pre-projected sum term z = h0 @ Pb.  gcn / graphsage
        then run on the d_out-wide z table (any width); bi-interaction needs the library's z mode at (embed_dim,
        conv_dim), which only the wide-row stream kernel has -- elsewhere layer 1 combines side @ Pb itself."""
        if not self.use_residual or self.n_layers == 0:
            return False
        d, c = self.embed_dim, self.aggregator_layers[0].out_dim
        if d < 128 or c % 4 != 0:
            return False
        return self.aggregation_type != 'bi-interaction' or ops.aggregate_supported(d, c, _lib.AGG_BI_Z)

    def _check_layer_shapes(self) -> None:
        """Refuses, at construction, widths the aggregation kernels do not run (instead of at the first forward)."""
        z1 = self._layer1_z_path()
        for k, layer in enumerate(self.aggregator_layers):
            if k == 0 and z1:
                continue                                  # supported by definition of the z path
            folded_ego = k == 0 and self.use_residual     # layer 1's ego @ Pa rides in the h0 @ Q GEMM
            if self.aggregation_type == 'bi-interaction':
                mode = _lib.AGG_BI
            elif self.aggregation_type == 'graphsage' and not folded_ego:
                mode = _lib.AGG_TWO_TERMS
            else:
                mode = _lib.AGG_ONE_TERM
            if not ops.aggregate_supported(layer.in_dim, layer.out_dim, mode):
                raise ValueError(
                    f"aggregator layer {k + 1} ({self.aggregation_type}, {layer.in_dim} -> {layer.out_dim}) is outside the "
                    "aggregation kernels: they need in_dim % 4 == 0, in_dim <= 512 and out_dim <= 64, and out_dim <= 60 "
                    "from in_dim 404 on where two combine matrices share the 227 KB of shared memory (include/lkg.h)")

    def _exchange_table(self, part, name: str, d: int, training: bool):
        """Symmetric-memory exchange table for the rows of one activation (``parallel.PeerTable``), or None: NCCL
        all-gather (no NCCL box / symmetric memory unavailable / training pass, whose saved activations must outlive
        the slot rotation)."""
        if part is None or training or not part.peer_tables_enabled():
            return None
        if self._peer_x is None or self._peer_x.part is not part:
            from .parallel import PeerExchange
            self._peer_x = PeerExchange(part, self._param_device())
        return self._peer_x.table(name, d)

    def _gather_rows(self, part, name: str, src_rows: torch.Tensor, training: bool) -> torch.Tensor:
        """Exchange of one row-partitioned activation: ``src_rows`` = this rank's rows [n_own, d] -> table [padded, d]
        (row index == entity id) holding every rank's rows, usable on the current stream."""
        tab = self._exchange_table(part, name, src_rows.shape[1], training)
        if tab is not None:
            table, handle = tab.begin()
            table[part.begin:part.end] = src_rows
            handle.start().wait()
            return table
        table = torch.empty((part.padded, src_rows.shape[1]), dtype=torch.float32, device=src_rows.device)
        table[part.begin:part.end] = src_rows
        return part.all_gather_rows(table)

    def _gate_stage_key(self, part):
        gate_mod, tables = self._gate_module()
        ent = self.entity_embed.weight
        return ((ent.data_ptr(), ent._version), None if gate_mod is None else _param_key(gate_mod),
                tuple((t.data_ptr(), t._version) for t in tables), None if part is None else (part.begin, part.end),
                tuple(_param_key(layer) for layer in self.aggregator_layers), float(self.lamda), float(self.alpha))

    def _combined_table(self, keep, pre) -> bool:
        """Inference pass of the bi-interaction model with the pre-projected sum term: the gate output h0 and
        z = h0 @ Pb live side by side in ONE table [rows, d + C] -- layer 1 fetches a neighbour's (h0 | z) row with one
        bulk copy, and the row partition exchanges one table instead of two."""
        return (keep is None and pre is None and self.scale_gat_dim is not None
                and self.aggregation_type == 'bi-interaction' and self._layer1_z_path())

    def _residual_gemm(self, h0_planes, folds, z_out=None):
        """h0 @ Q for all layers (+ layer 1's ego @ Pa and the z columns) as one GEMM -> (h0q, offsets, zoff).
        ``z_out``: [rows, C] view that receives the z columns instead of h0q (the [h0 | z] table)."""
        qkey = tuple(id(f) for f in folds)                 # the fold dicts are cached per parameter version
        if self._h0q_cache is None or self._h0q_cache[0] != qkey:
            self._h0q_cache = (qkey, *self._stack_q(folds), folds)
        _, wq, cq, offsets, zoff, _ = self._h0q_cache
        if z_out is not None and zoff > 0 and zoff % 4 == 0:
            return ops.linear([h0_planes], wq, cq, out2=z_out, split_col=zoff), offsets, zoff
        h0q = ops.linear([h0_planes], wq, cq)
        if z_out is not None:
            z_out.copy_(h0q[:, zoff:zoff + z_out.shape[1]])
        return h0q, offsets, zoff

    def _gate_stage(self, part, keep=None, pre=None) -> dict:
        """First stage of the embedding pass: buffers, the literal gate on this rank's rows and -- row partitioned,
        when layer 1 gathers raw h0 rows -- the all-gather of h0, started asynchronously.  It depends on the
        parameters only, not on A_in: ``update_attention`` runs it ahead of the attention kernel so that the
        all-gather (1.2 GB at N = 1 M) travels over NVLink while that kernel streams HBM."""
        dev = self._param_device()
        n, d, total = self.n_entities, self.embed_dim, self.total_conv_dim
        rb, re = (0, n) if part is None else (part.begin, part.end)
        rows = None if part is None else (rb, re)
        n_own, n_tab = re - rb, (n if part is None else part.padded)
        combined = self._combined_table(keep, pre)
        width = d + (self.aggregator_layers[0].out_dim if combined else 0)
        # concat buffer, this rank's rows (fp32 copy of what linear_gat reads as planes; not needed by the combined
        # inference layout, whose fp32 consumers are the gathers of layer 1 only)
        cat = None if combined else torch.empty((n_own, total), dtype=torch.float32, device=dev)
        gather_h0 = False
        if part is not None and self.n_layers > 0:
            gather_h0 = not self._layer1_z_path() or self.aggregation_type == 'bi-interaction'
        peer = None
        if combined:
            if part is None:
                h0_tab = torch.empty((n, width), dtype=torch.float32, device=dev)
            else:
                tab = self._exchange_table(part, "h0z", width, False)
                if tab is not None:
                    h0_tab, peer = tab.begin()
                else:
                    h0_tab = torch.empty((n_tab, width), dtype=torch.float32, device=dev)
            h0 = h0_tab[rb:re, :d]
        elif part is None:
            h0_tab = h0 = cat[:, :d]                      # gate output lives in the concat buffer
        else:
            tab = self._exchange_table(part, "h0", d, keep is not None) if gather_h0 else None
            if tab is not None:
                h0_tab, peer = tab.begin()                # symmetric-memory table: rows pushed by the copy engines
            else:
                h0_tab = torch.empty((n_tab, d), dtype=torch.float32, device=dev)   # row index == entity id
            h0 = h0_tab[rb:re]
        # scaled fp16 hi/lo planes of the concat buffer: A operand of the h0 @ Q and linear_gat tensor-core GEMMs.
        # Two K segments with their own scale records: the gate output and the L2-normalised layer outputs
        # (|x| <= 1); the second window starts on a 16-byte boundary.
        xcol = (d + 7) // 8 * 8
        cat_planes = _lib.Planes(n_own, xcol + (total - d), dev)
        gz = None
        if keep is not None and self._gate_module()[0] is not None:
            gz = torch.empty((n_own, 2 * d), dtype=torch.float32, device=dev)      # activated (g, z) pairs
        _, h0_planes = self.gate_embeddings(out=h0, planes_window=(cat_planes, 0, d), rows=rows,
                                            packed=None if pre is None else pre["packed"], gz_out=gz)
        extra = {}
        if combined:                                      # z = h0 @ Pb next to h0 (the residual GEMM only needs parameters)
            folds = [layer.folded(self.lamda, self.alpha, k + 1) for k, layer in enumerate(self.aggregator_layers)]
            # the z columns of the stacked GEMM land in the table directly (no copy between the two layouts)
            h0q, offsets, zoff = self._residual_gemm(h0_planes, folds, z_out=h0_tab[rb:re, d:])
            extra = dict(combined=True, folds=folds, h0q=h0q, offsets=offsets, zoff=zoff)
        work = None
        if gather_h0:
            work = peer.start() if peer is not None else part.all_gather_rows(h0_tab, async_op=True)
        return dict(cat=cat, h0_tab=h0_tab, h0=h0, cat_planes=cat_planes, h0_planes=h0_planes, xcol=xcol, gz=gz,
                    work=work, **extra)

    def _gat_embeddings_native(self, keep: Optional[dict] = None, pre: Optional[dict] = None) -> torch.Tensor:
        """``pre`` (training): {folds, wq, cq, offsets, zcol, packed} built under autograd by the caller (detached
        values are used here); ``keep`` then receives what the backward pass needs."""
        dev = self._param_device()
        plan, a_values = self._current_plan()
        n, d, total = self.n_entities, self.embed_dim, self.total_conv_dim
        part = self._part if (self._part is not None and self._part.world > 1) else None
        rb, re = (0, n) if part is None else (part.begin, part.end)
        rows = None if part is None else (rb, re)
        n_own, n_tab = re - rb, (n if part is None else part.padded)
        plan.set_row_range(rb, re)
        st = None
        if self._gate_prefetch is not None:
            key, st = self._gate_prefetch                  # gate output (and its all-gather) started by update_att
            self._gate_prefetch = None
            if keep is not None or pre is not None or key != self._gate_stage_key(part):
                if st["work"] is not None:
                    st["work"].wait()                      # stale: let the transfer finish, then drop it
                st = None
        if st is None:
            st = self._gate_stage(part, keep, pre)
        cat, h0_tab, h0, cat_planes, h0_planes, xcol, gz = (st[k_] for k_ in
                                                           ("cat", "h0_tab", "h0", "cat_planes", "h0_planes", "xcol", "gz"))
        xn_all = cat_planes.view(xcol, total - d, rec=self._unit_record(dev))
        h0q = None
        offsets: List[int] = []
        zoff = -1                                         # column of the pre-projected layer-1 sum term in h0q
        combined = bool(st.get("combined", False))
        if combined:
            folds, h0q, offsets, zoff = st["folds"], st["h0q"], st["offsets"], st["zoff"]
        elif pre is not None:
            folds, wq, cq, offsets, zoff = pre["folds"], pre["wq"], pre["cq"], pre["offsets"], pre["zcol"]
            if wq is not None:
                h0q = ops.linear([h0_planes], wq, cq)
        else:
            folds = [layer.folded(self.lamda, self.alpha, k + 1) for k, layer in enumerate(self.aggregator_layers)]
            if self.use_residual and self.n_layers > 0:
                h0q, offsets, zoff = self._residual_gemm(h0_planes, folds)     # this rank's rows

        c0 = self.aggregator_layers[0].out_dim if self.n_layers > 0 else 0
        z_tab = None
        if combined:
            z_tab = h0_tab[:, d:d + c0]                            # travels with h0: nothing to exchange
        elif zoff >= 0:
            if part is None:
                z_tab = h0q[:, zoff:zoff + c0]                     # [N, C] view, row index == entity id
            else:
                z_tab = self._gather_rows(part, "z", h0q[:, zoff:zoff + c0], keep is not None)
        if part is not None:
            if st["work"] is not None:
                st["work"].wait()                         # layer 1 gathers arbitrary neighbour rows of h0
            if self.scale_gat_dim is None:
                cat[:, :d] = h0

        x = h0_tab[:, :d] if combined else h0_tab
        col = d
        for k, (layer, f) in enumerate(zip(self.aggregator_layers, folds)):
            c = layer.out_dim
            if h0q is not None:
                r1 = h0q[:, offsets[k]:offsets[k] + c]
                r2 = h0q[:, offsets[k] + c:offsets[k] + 2 * c] if f["q2"] is not None else None
            else:
                r1, r2 = f["c1"], f["c2"]
            exchange = part is not None and k + 1 < self.n_layers     # the next layer reads every row of this one
            xtab = self._exchange_table(part, f"x{k}", c, keep is not None) if exchange else None
            if xtab is not None:
                x_out, xhandle = xtab.begin()             # the kernel writes this rank's rows straight into the table
            else:
                x_out = torch.empty((n_tab, c), dtype=torch.float32, device=dev)
            saved = None
            if keep is not None:
                saved = {}
                keep.setdefault("layers", []).append(saved)
                saved.update(x=x, y=x_out)
            layer.run(plan, a_values, x, f, r1, r2, x_out, None if cat is None else cat[:, col:col + c],
                      fold_ego=(h0q is not None and k == 0),
                      xn_planes=_lib.PlanesView(cat_planes, xcol + col - d, c, rec=xn_all.rec), rows=rows,
                      z=z_tab if k == 0 else None, saved=saved)
            if exchange:
                if xtab is not None:
                    xhandle.start().wait()
                else:
                    part.all_gather_rows(x_out)
            x = x_out
            col += c
        plan.set_row_range(0, n)
        if keep is not None:
            keep.update(cat=cat, h0=h0, gz=gz, plan=plan, a_values=a_values, h0_planes=h0_planes, xn_all=xn_all,
                        gate_operands=getattr(self, "_gate_operands", None))
            self._gate_operands = None
        if self.scale_gat_dim is not None:
            segs = [h0_planes] + ([xn_all] if total > d else [])
            out = ops.linear(segs, self.linear_gat.weight.detach(), self.linear_gat.bias.detach(), _lib.ACT_LEAKY_RELU)
            if keep is not None:
                keep["out"] = out
            return out
        return cat

    # ---- training path: the same forward kernels + the backward kernels of csrc/backward.cu ---------------------
    _FOLD_KEYS = ("pa", "pb", "p2", "c1", "c2")

    def _gat_embeddings_autograd(self) -> torch.Tensor:
        """gat_embeddings with gradient support (what pre_training / fine_tuning differentiate, model.py:298-314).
        The parameter folds (DESIGN.md section 4) and the interleaved gate weight are built under autograd from the
        live parameters, so the kernels only produce gradients w.r.t. the folded tensors and torch chains them on
        to linear / linear_h0 / weight / g / gate_* (tiny d x d matrix products)."""
        folds = [layer.folded(self.lamda, self.alpha, k + 1, differentiable=True)
                 for k, layer in enumerate(self.aggregator_layers)]
        wq = cq = None
        offsets, zcol = [], -1
        if self.use_residual and self.n_layers > 0:
            wq, cq, offsets, zcol = self._stack_q(folds)
        gate_mod, _ = self._gate_module()
        w_pair = b_pair = None
        if gate_mod is not None:
            w_pair, b_pair = gate_mod.pair()
        leaves: List[Optional[torch.Tensor]] = [self.entity_embed.weight, w_pair, b_pair, wq, cq]
        for k, (layer, f) in enumerate(zip(self.aggregator_layers, folds)):
            leaves += [f[key] for key in self._FOLD_KEYS]
            leaves += [layer.layer_normalize.weight, layer.layer_normalize.bias]
        if self.scale_gat_dim is not None:
            leaves += [self.linear_gat.weight, self.linear_gat.bias]
        det = lambda t: None if t is None else t.detach()
        pre = dict(folds=[{k_: det(v) for k_, v in f.items()} for f in folds], wq=det(wq), cq=det(cq),
                   offsets=offsets, zcol=zcol, packed=None if w_pair is None else (det(w_pair), det(b_pair)))
        for f, fd in zip(folds, pre["folds"]):
            if f["pa"] is not None and f["pa"] is f["pb"]:
                fd["pa"] = fd["pb"]                       # keep the identity the kernels dispatch on
        return _GatEmbeddingsFn.apply(self, pre, *leaves)

    def _gat_backward(self, keep: dict, pre: dict, g_out: torch.Tensor) -> List[Optional[torch.Tensor]]:
        """Gradients w.r.t. the leaves of ``_gat_embeddings_autograd`` (same order).

        Row partitioned: every rank differentiates its own head rows.  ``A^T x`` sums over ALL head rows, so each rank
        reduces its own rows' entries into a full-height partial and a reduce-scatter (the dual of the forward's
        all-gather) hands every rank the sum for its rows; parameter gradients are partial sums that one all-reduce
        completes, and the rows of d entity_embed are all-gathered (the table is replicated, like its optimizer)."""
        dev = g_out.device
        d, total = self.embed_dim, self.total_conv_dim
        L = self.n_layers
        part = self._part if (self._part is not None and self._part.world > 1) else None
        rb, re = (0, self.n_entities) if part is None else (part.begin, part.end)
        n = re - rb                                   # rows this rank differentiates
        plan, a_values = keep["plan"], keep["a_values"]
        own = (lambda t_: t_) if part is None else (lambda t_: t_[rb:re])
        if part is not None:
            g_out = g_out[rb:re]
        t_coo = plan.transposed() if part is None else plan.transposed(rows=(rb, re))
        # the values in the transposed list's order, gathered once: every A^T product below then streams them instead
        # of chasing the permutation (a random 4-byte read costs a 32-byte sector)
        a_values = a_values.index_select(0, t_coo[2])
        t_coo = (t_coo[0], t_coo[1], None)

        def spmm_t(x_rows, dst):
            """dst (this rank's rows) += (A^T x)[rows]; x_rows: this rank's head rows."""
            if part is None:
                return ops.spmm_coo(t_coo, a_values, x_rows, dst)
            full = torch.zeros((part.padded, x_rows.shape[1]), dtype=torch.float32, device=dev)
            ops.spmm_coo(t_coo, a_values, x_rows, full)
            dst += part.reduce_scatter_rows(full)[:n]
            return dst

        folds, wq, offsets, zcol = pre["folds"], pre["wq"], pre["offsets"], pre["zcol"]
        f32 = dict(dtype=torch.float32, device=dev)
        colsum = ops.colsum
        h0_planes = keep["h0_planes"]
        grads: List[Optional[torch.Tensor]] = []
        g_out = g_out if (g_out.dtype == torch.float32 and g_out.stride(1) == 1) else _lib.f32c(g_out)
        # scale records of the gradient matrices: raised by the kernels that write them, no absmax pass re-reads them
        recs = torch.zeros((2 * L + 3, _lib.LKG_SCALE_FLOATS), **dict(dtype=torch.float32, device=dev))
        dpre_rec, pre_rec, dmat_rec = recs[0], recs[1], recs[2]

        # ---- linear_gat + LeakyReLU (model.py:311) ----
        g_wg = g_bg = None
        if self.scale_gat_dim is not None:
            dpre = ops.leaky_bwd(g_out, keep["out"], amax=dpre_rec)
            dpre_pl = ops.split_planes(dpre, rec=ops.scale_finish(dpre_rec))
            g_wg = torch.zeros_like(self.linear_gat.weight)                     # [G, T] = dpre^T [h0 | xn_1 | ...]
            ops.xt_y_planes(dpre_pl, h0_planes, out=g_wg[:, :d])
            if total > d:
                ops.xt_y_planes(dpre_pl, keep["xn_all"], out=g_wg[:, d:])
            g_bg = colsum(dpre)
            dcat = ops.linear([dpre_pl], self.linear_gat.weight.detach().t().contiguous(), None)
            del dpre, dpre_pl
        else:
            dcat = g_out.clone()
        # accumulates every contribution to d loss / d h0 in place (a strided view when its rows stay 16-byte aligned)
        dh0 = dcat[:, :d] if dcat.stride(0) % 4 == 0 else dcat[:, :d].contiguous()
        h0 = keep["h0"]

        # ---- aggregator layers, last to first (model.py:101-164) ----
        residual = wq is not None
        dmat = None
        if residual:
            dmat = torch.empty((n, wq.shape[0]), **f32)        # [dO of every layer | t1 of layer 0]: d (h0 @ Q)
        layer_grads = [None] * L
        dy_in = None
        col = d + sum(layer.out_dim for layer in self.aggregator_layers)
        for k in reversed(range(L)):
            layer, f, sv = self.aggregator_layers[k], folds[k], keep["layers"][k]
            c, dk = layer.out_dim, layer.in_dim
            col -= c
            x_k, y_k = own(sv["x"]), own(sv["y"])
            has_o2 = f["p2"] is not None
            nt = 2 if has_o2 else 1
            d_o = dmat[:, offsets[k]:offsets[k] + nt * c] if residual else torch.empty((n, nt * c), **f32)
            dgb = torch.zeros(2 * c, **f32)
            do_rec, xs_rec = recs[3 + 2 * k], recs[4 + 2 * k]
            ops.layer_bwd_rows(y_k, sv["o"], has_o2, sv["mask"], dy_in, dcat[:, col:col + c],
                               layer.layer_normalize.weight.detach(), d_o, dgb, amax=do_rec,
                               amax2=dmat_rec if residual else None)
            ops.scale_finish(do_rec)                           # bounds do1 and do2 alike
            do1 = d_o[:, :c]
            do2 = d_o[:, c:] if has_o2 else None
            fold_ego = residual and k == 0                     # ego @ Pa lives inside h0 @ Q
            z_path = fold_ego and zcol >= 0                    # ... and so does the projected sum term
            t1 = dmat[:, zcol:zcol + c] if z_path else torch.empty((n, c), **f32)
            t1.zero_()
            spmm_t(do1, t1)                                    # A^T do1: (A x) Pb backward without the wide gather
            if z_path:
                ops.absmax_accumulate(t1, dmat_rec)
            g = dict.fromkeys(self._FOLD_KEYS)
            use_pa = f["pa"] is not None and not fold_ego
            use_pb = not z_path
            do1_pl = ops.split_planes(do1, rec=do_rec) if use_pa else None
            t1_pl = ops.split_planes(t1) if use_pb else None
            if use_pa or use_pb:
                xk_pl = h0_planes if k == 0 else ops.split_planes(x_k)
            if use_pa:
                g["pa"] = ops.xt_y_planes(xk_pl, do1_pl)
            if use_pb:
                g["pb"] = ops.xt_y_planes(xk_pl, t1_pl)        # (A x)^T do1 == x^T (A^T do1)
            if not residual:
                g["c1"] = colsum(do1)
                if has_o2:
                    g["c2"] = colsum(do2)
            # d loss / d x_k = do1 Pa^T + t1 Pb^T + (do2 P2^T) * side + A^T ((do2 P2^T) * x_k)
            dx = dh0 if k == 0 else torch.empty((n, dk), **f32)
            acc = _lib.ACT_ACCUMULATE if k == 0 else _lib.ACT_NONE
            segs, ws = [], []
            if use_pa:
                segs.append(do1_pl); ws.append(f["pa"])
            if use_pb:
                segs.append(t1_pl); ws.append(f["pb"])
            if segs:
                ops.linear(segs, torch.cat(ws, dim=1).contiguous(), None, acc, out=dx)
            if has_o2:
                wbuf, xs = torch.empty((n, dk), **f32), torch.empty((n, dk), **f32)
                ops.bi_bwd_rows(do2, f["p2"], x_k, sv["side"], wbuf, dx, accumulate=True, xs_out=xs, xs_amax=xs_rec)
                spmm_t(wbuf, dx)
                g["p2"] = ops.xt_y_planes(ops.split_planes(xs, rec=ops.scale_finish(xs_rec)),
                                          ops.split_planes(do2, rec=do_rec))               # (x * side)^T do2
                del wbuf, xs
            layer_grads[k] = (g, dgb[:c], dgb[c:])
            dy_in = dx
        g_wq = g_cq = None
        if residual:
            dmat_pl = ops.split_planes(dmat, rec=ops.scale_finish(dmat_rec))
            g_wq = ops.xt_y_planes(dmat_pl, h0_planes)                          # [cols, embed_dim]
            g_cq = colsum(dmat)
            ops.linear([dmat_pl], wq.t().contiguous(), None, _lib.ACT_ACCUMULATE, out=dh0)
            del dmat_pl

        # ---- literal gate (gate.py:22-28) ----
        gate_mod, tables = self._gate_module()
        g_wpair = g_bpair = None
        if gate_mod is not None:
            ent = own(self.entity_embed.weight.detach())
            w_pair = pre["packed"][0]
            d_pre = torch.empty((n, 2 * d), **f32)
            g_ent = torch.empty((n, d), **f32)
            ops.gate_bwd(dh0, keep["gz"], ent, d_pre, g_ent, pre_amax=pre_rec)
            d_pre_pl = ops.split_planes(d_pre, rec=ops.scale_finish(pre_rec))
            ops.linear([d_pre_pl], w_pair[:, :d].t().contiguous(), None, _lib.ACT_ACCUMULATE, out=g_ent)
            g_wpair = torch.zeros_like(w_pair)                  # [2 dim, dim + literals] = d_pre^T [ent | literals]
            ent_planes, lit_planes = keep["gate_operands"]
            ops.xt_y_planes(d_pre_pl, ent_planes, out=g_wpair[:, :d])
            ops.xt_y_planes(d_pre_pl, lit_planes, out=g_wpair[:, d:])
            g_bpair = colsum(d_pre)
            del d_pre_pl
        else:
            g_ent = dh0.contiguous()

        grads += [g_ent, g_wpair, g_bpair, g_wq, g_cq]
        for g, g_lw, g_lb in layer_grads:
            grads += [g[key] for key in self._FOLD_KEYS] + [g_lw, g_lb]
        if self.scale_gat_dim is not None:
            grads += [g_wg, g_bg]
        if part is not None:
            full = torch.zeros((part.padded, d), **f32)
            full[rb:re] = g_ent
            grads[0] = part.all_gather_rows(full)[:self.n_entities]
            small = [g_ for g_ in grads[1:] if g_ is not None]                # partial sums over this rank's rows
            flat = torch.cat([g_.reshape(-1) for g_ in small])
            part.all_reduce(flat)
            off = 0
            for g_ in small:
                g_.copy_(flat[off:off + g_.numel()].view(g_.shape))
                off += g_.numel()
        return grads

    # ---- losses ----------------------------------------------------------------------------------
    def calculate_prediction_loss(self, head_ids, tail_pos_ids, tail_neg_ids):
        """model.py:316-348 (BPR on the final embeddings)."""
        self.gat_embed = self.gat_embeddings()
        return self.prediction_loss_from(self.gat_embed, head_ids, tail_pos_ids, tail_neg_ids)

    def calc_triplet_loss(self, h, r, pos_t, neg_t):
        """model.py:364-428 (TransR on the GAT embeddings)."""
        self.gat_embed = self.gat_embeddings()
        return self.triplet_loss_from(self.gat_embed, h, r, pos_t, neg_t)

    # The reference recomputes (and differentiates) the whole graph for every minibatch (main.py:112-124, 213-226).
    # The two helpers below take the embedding matrix as an argument, so ONE ``gat_embeddings()`` -- one forward and,
    # after summing the losses, one backward pass over the graph -- can serve several minibatches: gradient
    # accumulation over those batches at fixed parameters (SURVEY.md 8(f) rank 2; an explicit choice of the caller,
    # not the reference's one-update-per-batch schedule).
    def prediction_loss_from(self, all_embed, head_ids, tail_pos_ids, tail_neg_ids):
        """BPR loss (model.py:316-348) of one minibatch on a given embedding matrix."""
        return _BprLossFn.apply(all_embed, head_ids, tail_pos_ids, tail_neg_ids, float(self.prediction_l2loss_lambda))

    def triplet_loss_from(self, all_embed, h, r, pos_t, neg_t):
        """TransR loss (model.py:364-428) of one minibatch on a given embedding matrix."""
        return _TransRLossFn.apply(all_embed, self.relation_embed.weight, self.gat_trans_M, h, r, pos_t, neg_t,
                                   float(self.kg_l2loss_lambda))

    # ---- attention update ------------------------------------------------------------------------
    def update_attention(self, h_list, t_list, r_list, relations):
        """model.py:444-471.  Entirely on device: no host round trip, no per-relation Python loop."""
        plan = self._edge_plan(h_list, t_list, r_list, relations)
        return self._apply_attention(plan, None)

    def update_attention_projected(self, h_list, t_list, r_list, relations, w_rel):
        """Extension (BASELINE.json north star (b)): the relation-PROJECTED attention the reference keeps commented
        out (model.py:436-439), v = (e_t W_r) . tanh(e_h W_r + e_r) with an explicit ``w_rel`` [R, embed_dim,
        relation_dim]; same duplicate merge, row softmax and ``A_in`` side effect as ``update_att``."""
        if self._part is not None and self._part.world > 1:
            raise NotImplementedError("the projected attention extension runs on one GPU")
        plan = self._edge_plan(h_list, t_list, r_list, relations)
        return self._apply_attention(plan, w_rel)

    def _edge_plan(self, h_list, t_list, r_list, relations) -> GraphPlan:
        dev = self._param_device()
        # the CSR plan only depends on the edge list.  The very same tensors (address, length, in-place version) as
        # last time need no look at all; otherwise an unchanged list is recognised by content (one small kernel + a
        # scalar read-back), not by address.  int32 / host lists are accepted (converted on the device).
        rels = tuple(int(x) for x in relations)
        ident = (tuple((x.data_ptr(), x.numel(), x._version, x.dtype, str(x.device)) for x in (h_list, t_list, r_list)),
                 rels)
        if self._att_plan is None or self._att_ident != ident:
            i64 = dict(device=dev, dtype=torch.int64, non_blocking=True)
            h, t, r = h_list.to(**i64).contiguous(), t_list.to(**i64).contiguous(), r_list.to(**i64).contiguous()
            key = (GraphPlan.fingerprint(h, t, r), rels)
            if self._att_plan is None or self._att_key != key:
                self._att_plan = GraphPlan(h, t, r, self.n_entities, self.n_relations, relations)
                self._att_key = key
            self._att_ident = ident
            self._att_refs = (h_list, t_list, r_list)   # keeps the addresses from being reused by other tensors
        return self._att_plan

    def _apply_attention(self, plan: GraphPlan, w_rel) -> None:
        dev = self._param_device()
        part = self._part if (self._part is not None and self._part.world > 1) else None
        with torch.no_grad():
            if w_rel is not None:
                values = ops.attn_update_projected(plan, self.entity_embed.weight.detach(),
                                                   self.relation_embed.weight.detach(), w_rel.detach().to(dev))
            elif part is None:
                values = ops.attn_update(plan, self.entity_embed.weight.detach(), self.relation_embed.weight.detach())
            else:   # rows are independent: every rank fills the values of its own head rows
                if self.prefetch_gate:
                    self._gate_prefetch = (self._gate_stage_key(part), self._gate_stage(part))
                plan.set_row_range(part.begin, part.end)
                values = torch.zeros(max(plan.nnz, 1), dtype=torch.float32, device=dev)[:plan.nnz]
                ops.attn_update(plan, self.entity_embed.weight.detach(), self.relation_embed.weight.detach(), out=values)
                plan.set_row_range(0, self.n_entities)
                self._a_in_pending = None
                if self._local_edges:             # A_in of this rank = its own head rows only
                    self._a_in_pending = ("local", plan, values)
                elif self.sync_attention is True:   # complete A_in on every rank; the layers only need own rows
                    part.all_reduce(values)
                elif self.sync_attention == "lazy":
                    self._a_in_pending = ("rows", plan, values)
                elif part.world > 1:
                    self._a_in_pending = ("never", plan, values)
        self._agg_plan, self._agg_values = plan, values
        self._a_in_epoch += 1
        self.A_in.data = plan.sparse(values)

    def complete_attention(self) -> None:
        """Row partitioned: after ``update_att`` every rank holds the attention values of its own head rows (all the
        embedding pass reads).  This completes ``A_in`` to the full matrix of the reference on every rank -- needed
        for checkpoints, not for the pass.  COLLECTIVE: call it on all ranks (``state_dict()`` refuses to run while it
        is pending instead of hiding a collective inside a call that is usually made by rank 0 alone).
        Replicated edge list: the other ranks' values are summed in (x + 0 is exact).  ``local_edges``: the per-rank
        COO blocks (disjoint, ascending head ranges) are all-gathered and concatenated in rank order, which is the
        coalesced order of the full matrix."""
        pend, part = self._a_in_pending, self._part
        if pend is None or part is None or part.world == 1:
            self._a_in_pending = None
            return
        kind, plan, values = pend
        if kind == "local":
            dev = values.device
            counts = part.all_gather_stack(torch.tensor([plan.nnz], dtype=torch.int64, device=dev)).view(-1).tolist()
            width = max(max(counts), 1)
            pad_i = torch.zeros((2, width), dtype=torch.int64, device=dev)
            pad_v = torch.zeros(width, dtype=torch.float32, device=dev)
            pad_i[:, :plan.nnz] = plan.indices
            pad_v[:plan.nnz] = values
            all_i, all_v = part.all_gather_stack(pad_i), part.all_gather_stack(pad_v)
            idx = torch.cat([all_i[r][:, :c] for r, c in enumerate(counts)], dim=1)
            val = torch.cat([all_v[r][:c] for r, c in enumerate(counts)])
            self.A_in.data = torch.sparse_coo_tensor(idx, val, (self.n_entities, self.n_entities), is_coalesced=True)
            self._agg_plan = self._agg_values = None          # rebuilt from the full matrix when next needed
            self._a_in_epoch += 1
        else:
            part.all_reduce(values)
        self._a_in_pending = None

    def state_dict(self, *args, **kwargs):
        if self._a_in_pending is not None and self._part is not None and self._part.world > 1:
            raise RuntimeError(
                "A_in holds only this rank's head rows after a row-partitioned update_att: call "
                "model.complete_attention() on ALL ranks (it is a collective) before state_dict() / torch.save")
        return super().state_dict(*args, **kwargs)

    # ---- scoring -----------------------------------------------------------------------------------
    def calc_score(self, head_ids, tail_ids):
        """model.py:473-486."""
        with torch.no_grad():
            all_embed = self.gat_embeddings()
            return ops.score(all_embed, head_ids, tail_ids)

    def predict_links(self, head_ids, tail_ids):
        """model.py:488-491."""
        with torch.no_grad():
            all_embed = self.gat_embeddings()
            return ops.predict(all_embed, head_ids, tail_ids, self.milestone_score)

    def topk(self, head_ids, tail_ids, k, target_tails=None, all_embed=None, tail_index=None):
        """Extension (BASELINE.json north star; no reference counterpart): per head the k best tails among
        ``tail_ids`` (larger score first, ties -> lower position), as (values, positions, ranks-of-targets).
        Large candidate sets go through the fused scoring + top-k kernels (no B x Nt score matrix);
        ``tail_index`` (``ops.ScoreIndex`` of the tails) can be reused across head batches."""
        if all_embed is None:
            with torch.no_grad():
                all_embed = self.gat_embeddings()
        n_tails = tail_index.m if tail_index is not None else len(tail_ids)
        if ops.fused_topk_applicable(n_tails, all_embed.shape[1], k):
            if tail_index is None:
                tail_index = ops.ScoreIndex(all_embed, tail_ids)
            vals, pos = ops.score_topk(all_embed, head_ids, tail_ids, k, tail_index=tail_index)
            # ranks of the given target positions: the scoring GEMM again with a counting epilogue + exact re-score of
            # the few columns inside the error band -- no B x Nt matrix either
            ranks = None if target_tails is None else ops.score_rank(all_embed, head_ids, target_tails, tail_index)
            return vals, pos, ranks
        scores = ops.score(all_embed, head_ids, tail_ids)
        return ops.topk_rows(scores, k, target_tails)

    def evaluate_ranking(self, heads, tails, relations=None, known=None, candidates=None, ks=(1, 3, 10),
                         batch_size=2048, all_embed=None, score="dot", predict="tail"):
        """Filtered link-prediction evaluation (extension: the MR / MRR / Hits@k protocol; the reference only has its
        threshold metrics).  Query i is (heads[i], relations[i] or any relation, target tails[i]).  Its raw rank is the
        rank of ``topk``: #{ j in candidates : s_j > s_t, or s_j == s_t and pos(j) < pos(t) }, 0 = best, with
        s_j = emb[h] . emb[j] (``calc_score``; the relation only selects the filter set) and ``candidates`` a list of
        entity ids (None = every entity).  The filtered rank subtracts the members of
            F(i) = { t' : (h, r, t') in known }   with a relation,   { t' : (h, any r, t') in known }   without,
        that beat the target under the same rule on the same scores; a tail is counted once however often it is known,
        the target itself and non-candidates never.  ``known``: ``GraphPlan`` of the known true triples (e.g. train +
        valid + test over the same entity ids), None = raw ranks.  Head prediction (?, r, t): the score is symmetric, so
        it is this call with heads and tails swapped and ``known`` built from the swapped triples.

        Returns {"mr": mean(rank + 1), "mrr": mean(1 / (rank + 1)), "hits@k": mean(rank < k) for k in ``ks`` (float64,
        as Python floats), "n": number of queries, "ranks": the filtered ranks, int64 [Q] on the device}.  One embedding
        pass (or the given ``all_embed``), one tail index for all batches of ``batch_size`` queries, the fused / dense
        path choice of ``topk``, and ONE host sync, which also carries the argument checks: ids outside
        [0, n_entities), a target that is not a candidate, duplicate candidates and relation ids outside the plan's
        range raise ValueError after it (the kernels only ever see clamped ids).
        Row partitioned (``set_partition``, world > 1) this is a collective: every rank ranks a contiguous slice of the
        queries on the gathered embeddings, the slices are all-gathered, and every rank returns the same result.

        ``predict="head"``: query i is (?, relations[i], tails[i]) with target heads[i]; the candidates are ranked as
        heads and the filter set is { h' : (h', r, t) in known } (``known.reversed()``).  Ranks stay in input order.
        ``score="triple"``: rank by the model's own triple score s(h, r, t) = -d(h, r, t) instead of the dot product,
        d = |emb[h] M_r + e_r - emb[t] M_r|^2 (TransR, the distance ``calc_triplet_loss`` trains; ``model_bce``: TransE,
        M_r = I), e_r = relation_embed.weight[r]; for head prediction the query row is emb[t] M_r - e_r.  The projected
        rows are the fp32 results of the projection GEMM; d is exact on them (differences and squares in fp64, one
        rounding to fp32) and the ranks are bit exact w.r.t. that rule.  ``relations`` are required (ids of the model's
        relations); the scoring width (``relation_dim``) must be <= 508.  The queries are ranked relation by relation
        (one host read-back of the per-relation counts, which also carries the argument checks, before the first
        launch)."""
        if score not in ("dot", "triple"):
            raise ValueError('score must be "dot" or "triple"')
        triple = score == "triple"
        if relations is not None and known is None and not triple:
            raise ValueError("relations only select the filter set: pass the known triples as well")
        with torch.no_grad():
            qs = self._queries(predict, heads, relations, known, candidates, all_embed, targets=tails, triple=triple)
            bad, sl = qs.bad, slice(qs.lo, qs.hi)
            if triple:
                counts = torch.bincount(qs.rels[sl], minlength=self.n_relations)
                host = torch.cat([torch.stack(list(bad.values())).long(), counts]).tolist()
                _raise_flags(bad, host)
                ranks = self._rank_triple(qs.emb, qs.anchors[sl], qs.tpos[sl], qs.rels[sl], host[len(bad):], qs.known,
                                          qs.cmap, qs.cand, qs.n_cand, batch_size, 1.0 if predict == "tail" else -1.0)
            else:
                ranks = self._rank_queries(qs.emb, qs.anchors[sl], qs.tpos[sl], None if qs.rels is None else qs.rels[sl],
                                           qs.known, qs.cmap, qs.cand, qs.n_cand, batch_size)
            q = qs.q
            if qs.world > 1:
                padded = torch.zeros(qs.per, dtype=torch.int64, device=ranks.device)
                padded[:qs.hi - qs.lo] = ranks
                ranks = qs.part.all_gather_stack(padded).reshape(-1)[:q]

            r1 = ranks.double() + 1.0
            ks = [int(k) for k in ks]
            metrics = [r1.mean(), (1.0 / r1).mean()] + [(ranks < k).double().mean() for k in ks]
            host = torch.cat([torch.stack(metrics), torch.stack(list(bad.values())).double()]).tolist()
            _raise_flags(bad, host[len(metrics):])
            out = {"mr": host[0], "mrr": host[1]}
            out.update({f"hits@{k}": v for k, v in zip(ks, host[2:len(metrics)])})
            out.update(n=q, ranks=ranks)
            return out

    def topk_triple(self, anchors, relations, k, known=None, candidates=None, predict="tail", batch_size=2048,
                    all_embed=None):
        """Knowledge-graph completion under the model's own triple score: per query the k most likely tails of
        (anchors[i], relations[i], ?) (``predict="tail"``) or heads of (?, relations[i], anchors[i]) (``"head"``),
        leaving out the triples already known.  The distance is the one of ``evaluate_ranking(score="triple")``:
        d_j = |q - emb[j] M_r|^2 with q = emb[a] M_r + e_r for tails and emb[a] M_r - e_r for heads (``model_bce``:
        TransE, M_r = I), exact on the fp32 projected rows (fp64 differences and squares, one rounding).  Excluded:
        { t' : (a, r, t') in known } for tails, { h' : (h', r, a) in known } for heads (``known.reversed()``); the anchor
        itself only if it is known.  ``candidates``: entity ids (None = every entity).

        Returns (dist fp32 [Q, k], ids int64 [Q, k] entity ids): per query the k non-excluded candidates ordered by
        (d ascending, candidate position ascending), padded with +inf / -1 when fewer than k remain.  With the same
        queries, ``batch_size`` and ``known``, ``evaluate_ranking(score="triple")`` gives entity ids[i, j] the filtered
        rank j (the raw rank j with ``known=None``): both calls project the queries in the same batches.  1 <= k <= 1024,
        relations are required, widths up to 508; the argument checks ride on one host read-back before the first
        launch.  Row partitioned (``set_partition``, world > 1) this is a collective: every rank completes a contiguous
        slice of the queries and every rank returns the whole result."""
        with torch.no_grad():
            qs = self._queries(predict, anchors, relations, known, candidates, all_embed, k=k, triple=True)
            k, sl = int(k), slice(qs.lo, qs.hi)
            counts = torch.bincount(qs.rels[sl], minlength=self.n_relations)
            host = torch.cat([torch.stack(list(qs.bad.values())).long(), counts]).tolist()
            _raise_flags(qs.bad, host)
            mine, a_sl, r_sl = qs.hi - qs.lo, qs.anchors[sl], qs.rels[sl]
            dist = torch.empty((mine, k), dtype=torch.float32, device=a_sl.device)
            pos = torch.empty((mine, k), dtype=torch.int64, device=a_sl.device)
            for b, index, qrows in self._triple_batches(qs.emb, a_sl, r_sl, host[len(qs.bad):], qs.cand, qs.n_cand,
                                                        batch_size, 1.0 if predict == "tail" else -1.0):
                exclude = None if qs.known is None else (qs.known, a_sl[b], r_sl[b], qs.cand)
                dist[b], pos[b] = ops.score_topk_l2(index, qrows, k, exclude=exclude)
            return self._gather_topk(dist, pos, qs.cand, qs.q, qs.per, float("inf"))

    def topk_links(self, anchors, k, relations=None, known=None, candidates=None, predict="tail", batch_size=2048,
                   all_embed=None):
        """Link prediction under the fine-tuned dot score s(a, j) = emb[a] . emb[j] (``calc_score``): per anchor the k
        most likely new tails (``predict="tail"``) or heads (``"head"``; the score is symmetric, so only the excluded
        set changes), leaving out the links already known.  s_j is the exact dot product ``score_topk`` returns and
        the fused ``evaluate_ranking(score="dot")`` compares (fp32 products summed in fp64, rounded once).  Excluded:
        { t' : (a, relations[i], t') in known } with relations, { t' : (a, any r, t') in known } without -- the filter
        set of ``evaluate_ranking``; for heads the same sets of ``known.reversed()``.  Duplicate triples count once,
        non-candidates are ignored, the anchor itself is excluded only if it is known.  ``candidates``: entity ids
        (None = every entity).

        Returns (scores fp32 [Q, k], ids int64 [Q, k] entity ids): per query the k non-excluded candidates ordered by
        (s descending, candidate position ascending), padded with -inf / -1 when fewer than k remain.  With the same
        ``known`` and ``relations``, ``evaluate_ranking`` gives entity ids[i, j] the filtered rank j wherever it takes
        its fused path.  1 <= k <= 1024; embedding widths up to 512 (a width that is not a multiple of 4 is zero padded
        once per call).  One embedding pass (or the given ``all_embed``), one candidate index for all batches of
        ``batch_size`` queries, no B x N score matrix at any width; the argument checks ride on one host read-back
        before the first launch.  Row partitioned (``set_partition``, world > 1) this is a collective: every rank
        completes a contiguous slice of the queries and every rank returns the whole result."""
        if relations is not None and known is None:
            raise ValueError("relations only select the excluded set: pass the known triples as well")

        def check_width(emb):
            if emb.shape[1] > ops.TOPK_DOT_MAX_DIM:
                raise ValueError(f"the dot top-k supports widths up to {ops.TOPK_DOT_MAX_DIM} (got {emb.shape[1]})")

        with torch.no_grad():
            qs = self._queries(predict, anchors, relations, known, candidates, all_embed, k=k, check_width=check_width)
            k, all_embed, n, dev = int(k), qs.emb, qs.emb.shape[0], qs.emb.device
            _raise_flags(qs.bad, torch.stack(list(qs.bad.values())).tolist())
            if all_embed.shape[1] % 4:           # zero columns add nothing to a dot product
                padded = torch.zeros((n, (all_embed.shape[1] + 3) // 4 * 4), dtype=torch.float32, device=dev)
                padded[:, :all_embed.shape[1]] = all_embed
                all_embed = padded
            index = ops.ScoreIndex(all_embed, qs.cand)
            mine, a_sl = qs.hi - qs.lo, qs.anchors[qs.lo:qs.hi]
            r_sl = None if qs.rels is None else qs.rels[qs.lo:qs.hi]
            vals = torch.empty((mine, k), dtype=torch.float32, device=dev)
            pos = torch.empty((mine, k), dtype=torch.int64, device=dev)
            for b0 in range(0, mine, batch_size):
                b = slice(b0, b0 + batch_size)
                exclude = None if qs.known is None else (qs.known, a_sl[b], None if r_sl is None else r_sl[b], qs.cand)
                vals[b], pos[b] = ops.score_topk_dot(all_embed, a_sl[b], k, index, exclude=exclude)
            return self._gather_topk(vals, pos, qs.cand, qs.q, qs.per, float("-inf"))

    def _queries(self, predict, anchors, relations, known, candidates, all_embed, targets=None, k=None, triple=False,
                 check_width=None):
        """The argument checks and query preparation of ``evaluate_ranking`` (``targets`` = its tails), ``topk_triple``
        (``triple``) and ``topk_links`` (``check_width``, called on the embeddings), in the order that keeps every
        refusal before the first launch.  Head prediction swaps anchors and targets and reverses ``known``.  The embedding
        pass runs unless ``all_embed`` is given.  Ids outside their range are clamped and recorded in ``bad`` (message ->
        device flag) for the caller's one host read-back.  -> a namespace of: emb (fp32 contiguous), anchors, tpos
        (target positions among the candidates; None without targets), rels (None without relations), known, cand,
        n_cand, cmap, bad, q and the row partition's slice part, world, per, lo, hi (``_query_slice``)."""
        if predict not in ("tail", "head"):
            raise ValueError('predict must be "tail" or "head"')
        if k is not None and (isinstance(k, bool) or int(k) != k or not 1 <= k <= ops.TOPK_L2_MAX_K):
            raise ValueError(f"k must be an integer in [1, {ops.TOPK_L2_MAX_K}], got {k}")
        if triple:
            if relations is None:
                raise ValueError("the triple score needs the relation of every query")
            d_s = self.relation_embed.weight.shape[1]
            if d_s > ops.L2_RANK_MAX_DIM:
                raise ValueError(f"the triple score supports widths up to {ops.L2_RANK_MAX_DIM} (relation_dim {d_s})")
        if check_width is not None and all_embed is not None:
            check_width(all_embed)
        if predict == "head":
            if targets is not None:
                anchors, targets = targets, anchors
            known = None if known is None else known.reversed()
        dev = self._param_device()
        if all_embed is None:
            all_embed = self.gat_embeddings()
            if check_width is not None:
                check_width(all_embed)
        all_embed = _lib.f32c(all_embed)
        n, dim = all_embed.shape

        anchors = _query_ids(anchors, dev)
        q = anchors.numel()
        tpos = None if targets is None else _query_ids(targets, dev)
        rels = None if relations is None else _query_ids(relations, dev)
        if (tpos is not None and tpos.numel() != q) or (rels is not None and rels.numel() != q):
            raise ValueError("heads, tails and relations must have the same length" if targets is not None else
                             "anchors and relations must have the same length")
        if triple and self._triple_projection() is None and dim != self.relation_embed.weight.shape[1]:
            raise ValueError(f"the TransE score adds relation embeddings ({self.relation_embed.weight.shape[1]} wide) "
                             f"to rows of the embeddings ({dim} wide)")
        if known is not None and known.n_entities != n:
            raise ValueError(f"the known plan has {known.n_entities} entities, the embeddings {n}")
        if candidates is not None and len(candidates) == 0 and (q or targets is None):
            raise ValueError("no candidates")

        if tpos is None:
            bad = {"anchor ids outside [0, n_entities)": _outside(anchors, n)}
        else:
            bad = {"head or tail ids outside [0, n_entities)": _outside(anchors, n) | _outside(tpos, n)}
            tpos = tpos.clamp(0, n - 1)
        anchors = anchors.clamp(0, n - 1)
        cand, n_cand, cmap = _candidate_ids(candidates, n, dev, bad)
        if tpos is not None and candidates is not None:
            tpos = cmap[tpos].long()
            bad["a target tail is not a candidate"] = (tpos < 0).any()
            tpos = tpos.clamp_min(0)
        if triple:                   # the relation selects M_r and e_r, not only a filter run
            bad[f"relation ids outside [0, {self.n_relations}) of the model"] = _outside(rels, self.n_relations)
            rels = rels.clamp(0, self.n_relations - 1)
        if rels is not None and known is not None:
            bad[f"relation ids outside [0, {known.n_relations})"] = _outside(rels, known.n_relations)
            rels = rels.clamp(0, known.n_relations - 1)
        part, world, per, lo, hi = self._query_slice(q)
        return SimpleNamespace(emb=all_embed, anchors=anchors, tpos=tpos, rels=rels, known=known, cand=cand,
                               n_cand=n_cand, cmap=cmap, bad=bad, q=q, part=part, world=world, per=per, lo=lo, hi=hi)

    def _query_slice(self, q: int):
        """The queries a rank answers in a row-partitioned collective: -> (part, world, per, lo, hi), a contiguous
        slice [lo, hi) of ``per`` = ceil(q / world) queries (world 1: all of them)."""
        part = self._part
        world = 1 if part is None else part.world
        per = max(1, (q + world - 1) // world)
        lo = 0 if world == 1 else min(q, part.rank * per)
        hi = q if world == 1 else min(q, lo + per)
        return part, world, per, lo, hi

    def _gather_topk(self, vals, pos, cand, q, per, pad):
        """Candidate positions -> entity ids (-1 pads stay), then, row partitioned, the [per, k] slices of every rank
        all-gathered (padded with ``pad`` / -1) into the whole [q, k] result."""
        ent = pos if cand is None else torch.where(pos >= 0, cand[pos.clamp_min(0)], pos)
        part = self._part
        if part is not None and part.world > 1:
            k, mine = vals.shape[1], vals.shape[0]
            pv = torch.full((per, k), pad, dtype=torch.float32, device=vals.device)
            pi = torch.full((per, k), -1, dtype=torch.int64, device=vals.device)
            pv[:mine], pi[:mine] = vals, ent
            vals = part.all_gather_stack(pv).reshape(-1, k)[:q]
            ent = part.all_gather_stack(pi).reshape(-1, k)[:q]
        return vals, ent

    @staticmethod
    def _rank_queries(all_embed, heads, tpos, rels, known, cmap, cand, n_cand, batch_size):
        """Filtered ranks of the queries (heads, target positions, relations or None) against the candidates ``cand``
        (entity ids or None = every entity; ``cmap`` their position map), ``batch_size`` queries at a time."""
        m = heads.numel()
        ranks = torch.empty(m, dtype=torch.int64, device=heads.device)
        if ops.fused_topk_applicable(n_cand, all_embed.shape[1], 1):
            index = ops.ScoreIndex(all_embed, cand)
            tau = torch.empty(m, dtype=torch.float32, device=heads.device)
            for b0 in range(0, m, batch_size):
                b = slice(b0, b0 + batch_size)
                r = ops.score_rank(all_embed, heads[b], tpos[b], index, tau_out=tau[b])
                if known is not None:
                    ops.filter_ranks(r, known, heads[b], tpos[b], None if rels is None else rels[b], cmap,
                                     emb=all_embed, tau=tau[b])
                ranks[b] = r
            return ranks
        # dense path: the raw rank comes from the score matrix, so the filter judges on that matrix too (the second
        # instance of the filter kernel reads s from it; masking the matrix would cost a write of every filter entry
        # and make -inf targets ambiguous).  Matrices of at most 2 GB per chunk of queries.
        rec = ops.scale_from_data(all_embed)
        cols = torch.arange(n_cand, device=heads.device) if cand is None else cand
        step = max(1, min(batch_size, (1 << 29) // max(n_cand, 1)))
        for b0 in range(0, m, step):
            b = slice(b0, b0 + step)
            scores = ops.score(all_embed, heads[b], cols, rec=rec)
            r = ops.topk_rows(scores, 1, tpos[b])[2]
            if known is not None:
                ops.filter_ranks(r, known, heads[b], tpos[b], None if rels is None else rels[b], cmap, scores=scores)
            ranks[b] = r
        return ranks

    def _triple_projection(self):
        """M_r of the triple score: TransR's ``gat_trans_M`` [R, embed width, relation_dim]; None = TransE (identity)."""
        return self.gat_trans_M

    def _rank_triple(self, all_embed, anchors, tpos, rels, counts, known, cmap, cand, n_cand, batch_size, sign):
        """Filtered ranks under the triple score, batch by batch of ``_triple_batches``: each batch is ranked and
        filtered on its projected query rows."""
        ranks = torch.empty(anchors.numel(), dtype=torch.int64, device=anchors.device)
        for qs, index, q in self._triple_batches(all_embed, anchors, rels, counts, cand, n_cand, batch_size, sign):
            tau = torch.empty(qs.numel(), dtype=torch.float32, device=anchors.device)
            rk = ops.score_rank_l2(index, q, tpos[qs], tau_out=tau)
            if known is not None:
                ops.filter_ranks_l2(rk, known, anchors[qs], tpos[qs], rels[qs], cmap, index, q, tau)
            ranks[qs] = rk
        return ranks

    def _triple_batches(self, all_embed, anchors, rels, counts, cand, n_cand, batch_size, sign):
        """The per-relation loop of the triple score, shared by ``evaluate_ranking`` and ``topk_triple`` so that both
        see bit-identical rows: the queries (anchor rows, relations; ``counts`` = host list of queries per relation)
        are taken relation by relation in stable order.  Per relation the candidate rows are projected once
        (P_r = emb[cand] M_r, the projection GEMM) and indexed (``ops.L2Index``, buffers reused), then each batch of
        ``batch_size`` queries is projected (emb[anchor] M_r + sign * e_r; the projection's scale record comes from the
        batch, so the batching is part of the rows).  Yields (query indices, index, query rows [len, d4]); the index
        and the rows are valid until the next step."""
        dev = anchors.device
        proj = self._triple_projection()
        rel_w = _lib.f32c(self.relation_embed.weight.detach())
        d_s = rel_w.shape[1]
        d4 = (d_s + 3) // 4 * 4                  # zero columns up to a multiple of 4 add nothing to a distance
        order = torch.sort(rels, stable=True).indices
        qbuf = torch.zeros((max(1, min(batch_size, anchors.numel())), d4), dtype=torch.float32, device=dev)
        if proj is None:                         # TransE: the candidate rows are the embeddings, for every relation
            if cand is None and d4 == d_s:
                table = all_embed
            else:
                table = torch.zeros((max(n_cand, 1), d4), dtype=torch.float32, device=dev)[:n_cand]
                table[:, :d_s] = all_embed if cand is None else all_embed[cand]
            index, cand_planes = ops.L2Index(table), None
        else:
            table = torch.zeros((max(n_cand, 1), d4), dtype=torch.float32, device=dev)[:n_cand]
            index, cand_planes = None, ops.split_planes(all_embed, cand)
        off = 0
        for r, c in enumerate(counts):
            if c == 0:
                continue
            sel, off = order[off:off + c], off + c
            if proj is not None:
                w_r = proj[r].detach().t()
                ops.linear([cand_planes], w_r, None, out=table[:, :d_s])
                index = ops.L2Index(table) if index is None else index.refill()
            bias = rel_w[r] * sign
            for b0 in range(0, c, batch_size):
                qs = sel[b0:b0 + batch_size]
                q = qbuf[:qs.numel()]
                if proj is None:
                    q[:, :d_s] = all_embed[anchors[qs]] + bias
                else:
                    ops.linear([ops.split_planes(all_embed, anchors[qs])], w_r, bias, out=q[:, :d_s])
                yield qs, index, q

    def topk_sharded(self, head_ids, k, local_embed, tail_index=None):
        """Row-partitioned all-entity top-k: every rank scores the heads against the entities it owns
        (``local_embed`` = ``gat_embeddings(gather=False)``) and the per-rank survivors are merged.  Returns
        (values, entity ids) [B, k], identical on every rank.  ``head_ids`` may be a LIST of head batches: the
        collectives (head rows, survivors) then run once for all of them and a list of results is returned."""
        part = self._part
        assert part is not None, "topk_sharded needs set_partition()"
        many = isinstance(head_ids, (list, tuple))
        batches = list(head_ids) if many else [head_ids]
        dev = local_embed.device
        sizes = [int(hb.numel()) for hb in batches]
        heads = torch.cat([hb.to(device=dev, dtype=torch.int64).reshape(-1) for hb in batches])
        # head rows from their owners: a zero-padded [B, G] block summed over the ranks (x + 0 is exact)
        mine = (heads >= part.begin) & (heads < part.end)
        hmat = torch.zeros((heads.numel(), local_embed.shape[1]), dtype=torch.float32, device=dev)
        hmat[mine] = local_embed[heads[mine] - part.begin]
        part.all_reduce(hmat)
        if tail_index is None:
            tail_index = self.sharded_index(local_embed)
        # every head of every batch in ONE scoring call (the per-call sampling / threshold / finalize launches and the
        # resident head blocks are amortised over all of them), then one exchange of the survivors and one merge
        if ops.fused_topk_applicable(tail_index.m, local_embed.shape[1], k):
            vals, pos = ops.score_topk(local_embed, None, None, k, tail_index=tail_index, head_emb=hmat)
        else:               # small shards: score matrix + row top-k, 2 048 heads at a time
            both = torch.cat([local_embed, hmat])
            tails_all = torch.arange(local_embed.shape[0], device=dev)
            chunks = []
            for c0 in range(0, hmat.shape[0], 2048):
                rows = torch.arange(c0, min(c0 + 2048, hmat.shape[0]), device=dev) + local_embed.shape[0]
                chunks.append(ops.topk_rows(ops.score(both, rows, tails_all, rec=tail_index.rec), k)[:2])
            vals, pos = torch.cat([c[0] for c in chunks]), torch.cat([c[1] for c in chunks])
        ids = torch.where(pos >= 0, pos + part.begin, pos)
        all_v, all_i = part.all_gather_stack(vals), part.all_gather_stack(ids)
        if part.world * k <= 1024:
            top_v, top_i = ops.topk_merge(all_v, all_i, k)
        else:
            from .parallel import merge_topk
            top_v, top_i = merge_topk(all_v, all_i, k, lambda sc, kk: ops.topk_rows(sc, kk)[:2])
        if not many:
            return top_v, top_i
        return list(zip(torch.split(top_v, sizes), torch.split(top_i, sizes)))

    def sharded_index(self, local_embed):
        """Tail index of this rank's rows with a scale record that bounds EVERY rank's embeddings (the head rows
        come from other ranks): the absmax is all-reduced before the power-of-two scale is derived."""
        part = self._part
        rec = ops.scale_from_data(local_embed)
        part.all_reduce(rec[0:1], op=torch.distributed.ReduceOp.MAX)
        rec = ops.scale_from_bound(0.0, local_embed.device, other=rec)
        return ops.ScoreIndex(local_embed, None, rec=rec)

    def get_final_embeddings(self, entity_ids):
        """model.py:493-497."""
        with torch.no_grad():
            return self.gat_embeddings()[entity_ids]

    # ---- `mlp` mode: the BCE fine-tuning head (model.py:499-519) ------------------------------------------------
    def initialize_MLP(self):
        """model.py:499-504: fc1 / norm1 / fc2 / norm2 / fc3 (same attribute names = same state-dict keys)."""
        width = self.scale_gat_dim if self.scale_gat_dim is not None else self.total_conv_dim
        if self.scale_gat_dim is None:
            raise TypeError("initialize_MLP needs scale_gat_dim (the reference multiplies it by 2, model.py:500)")
        self.fc1 = nn.Linear(width * 2, 128)
        self.norm1 = nn.BatchNorm1d(128)
        self.fc2 = nn.Linear(128, 64)
        self.norm2 = nn.BatchNorm1d(64)
        self.fc3 = nn.Linear(64, 1)
        dev = self.entity_embed.weight.device
        for mod in (self.fc1, self.norm1, self.fc2, self.norm2, self.fc3):
            mod.to(dev)

    def mlp_scores_from(self, all_embed, head_ids, tail_ids):
        """The head of ``train_MLP`` on a given embedding matrix -> [B, 1] probabilities."""
        if not hasattr(self, "fc1"):
            raise AttributeError("call initialize_MLP() first (model.py:499)")
        return _MlpHeadFn.apply(self, all_embed, head_ids, tail_ids, self.fc1.weight, self.fc1.bias,
                                self.norm1.weight, self.norm1.bias, self.fc2.weight, self.fc2.bias,
                                self.norm2.weight, self.norm2.bias, self.fc3.weight, self.fc3.bias)

    def train_MLP(self, head_ids, tail_ids):
        """model.py:506-519."""
        self.gat_embed = self.gat_embeddings()
        return self.mlp_scores_from(self.gat_embed, head_ids, tail_ids)

    def forward(self, *input, device, mode):
        """model.py:521-532."""
        self.device = device
        if mode == 'fine_tuning':
            return self.calculate_prediction_loss(*input)
        if mode == 'pre_training':
            return self.calc_triplet_loss(*input)
        if mode == 'update_att':
            return self.update_attention(*input)
        if mode == 'update_att_projected':               # extension, see update_attention_projected
            return self.update_attention_projected(*input)
        if mode == 'predict':
            return self.predict_links(*input)
        if mode == 'mlp':
            return self.train_MLP(*input)
        raise NotImplementedError(f"unknown mode {mode!r}")
