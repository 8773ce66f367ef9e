"""Drop-in ``InfluentialNet`` / ``IRSNN`` (reference: model/influentialRS.py:22-216, :219-470).

Same class names, constructor arguments (the argparse Namespace read at :36-47), method signatures,
return types and ``state_dict`` keys/shapes as the reference, so pipeline.py / main.py can import
these instead (INTEGRATION.md).  The arithmetic runs in libirs_b200.so:

  inference (d=128, ffn=256): embedding gather+PE (K1) -> first in_proj written as attention operand images (tcgen05)
  -> per layer [persistent tcgen05 PIM attention (K3) -> fused decoder-chain kernel: out_proj + LN1 + folded
  cross-attention constant + LN2 -> FFN -> LN3 -> next layer's in_proj] -> fused catalog scorer (K5: arg-max / top-k /
  rank / log-sum-exp); other shapes: tcgen05 linears with fused epilogues (csrc/gemm_tc.cu);
  training: fp32 PIM attention fwd/bwd (K3/K4), torch linears + LayerNorm, tcgen05 softmax-CE fwd/bwd (K5a/K5b), K2.

The parameter containers are the same torch.nn modules the reference instantiates, created in the
same order, so ``torch.manual_seed(s); InfluentialNet(cfg)`` yields bit-identical initial weights.
Deviations from the shipped text are the ones SURVEY.md section 0.1 pins: D1 (PIM through the
``pi_factor`` keyword branch), D6 (gap_len == 0 only), D7 (best item not in the window instead of
"first of top-100"), ties broken by lower item id.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
import torch.optim as optim
from torch.optim import lr_scheduler

from . import ops

W_H = 0.05     # model/influentialRS.py:122 (the --w_h flag never reaches the model, D11)
W_OBJ = 1.0    # model/influentialRS.py:123


class PositionalEncoding(nn.Module):
    """Sinusoidal table as buffer ``pe`` [1,max_len,d] (model/layers.py:17-32)."""

    def __init__(self, d_model, max_len):
        super().__init__()
        pe = torch.zeros((max_len, d_model))
        position = torch.arange(0, max_len, dtype=torch.float).unsqueeze(1)
        div_term = torch.exp(torch.arange(0, d_model, 2).float() * (-math.log(10000.0) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer("pe", pe.unsqueeze(0))

    def forward(self, x):
        return self.pe[:, : x.size(1)]


def _tc_ok(d, ffn):
    """The tcgen05 linear kernel covers K, Nout <= 256 with K % 4 == 0 (every BASELINE config)."""
    return d % 4 == 0 and ffn % 4 == 0 and d <= 256 and ffn <= 256


def _cached(owner, key, ws, make):
    """``make()``, derived from the weights ``ws``, cached on the module ``owner`` per weight version (ops.cached_image)."""
    return ops.cached_image(owner.__dict__.setdefault("_tc_cache", {}), key, ws, make)


def _prepared(owner, key, W):
    """Weight matrix re-tiled for the tensor-core kernels."""
    return _cached(owner, key, (W,), lambda: ops.linear_prepare(W.detach().contiguous()))


def _tc_in_proj(owner, li, sa, x):
    """Packed q,k,v projection [.., 3d] (in_proj of nn.MultiheadAttention) in <= 256-column launches."""
    d = x.shape[-1]
    x2 = x.reshape(-1, d)
    qkv = torch.empty((x2.shape[0], 3 * d), dtype=torch.float32, device=x.device)
    W, b = sa.in_proj_weight, sa.in_proj_bias
    step = 3 * d if 3 * d <= 256 else (2 * d if 2 * d <= 256 else d)      # <= 256 output columns per launch
    for c0 in range(0, 3 * d, step):
        n = min(step, 3 * d - c0)
        ops.linear_tc(x2, _prepared(owner, ("in", li, c0), W[c0:c0 + n]), n, b[c0:c0 + n], ops.EPI_BIAS,
                      out=qkv[:, c0:c0 + n])
    return qkv.view(*x.shape[:-1], 3 * d)


def _tc_layer_tail(owner, li, layer, x, a, c):
    """out_proj + norm1 (+ cross-attention constant + norm2) -> linear1+relu -> linear2 + norm3."""
    sa = layer.self_attn
    d = x.shape[-1]
    shape = x.shape
    x2 = x.reshape(-1, d)
    a2 = a.reshape(-1, d)
    x2 = ops.linear_tc(a2, _prepared(owner, ("out", li), sa.out_proj.weight), d, sa.out_proj.bias, ops.EPI_RESID_LN,
                       resid=x2, g1=layer.norm1.weight, b1=layer.norm1.bias, c2=c.contiguous(), g2=layer.norm2.weight,
                       b2=layer.norm2.bias, eps=layer.norm1.eps)
    ffn = layer.linear1.out_features
    f = ops.linear_tc(x2, _prepared(owner, ("l1", li), layer.linear1.weight), ffn, layer.linear1.bias, ops.EPI_BIAS_RELU)
    x2 = ops.linear_tc(f, _prepared(owner, ("l2", li), layer.linear2.weight), d, layer.linear2.bias, ops.EPI_RESID_LN,
                       resid=x2, g1=layer.norm3.weight, b1=layer.norm3.bias, eps=layer.norm3.eps)
    return x2.view(shape)


def _chain_prepared(owner, key, layer, nxt):
    """Weight stream of the fused decoder-chain kernel for ``layer`` (+ in_proj of the layer ``nxt``)."""
    ws = [layer.self_attn.out_proj.weight, layer.linear1.weight, layer.linear2.weight]
    if nxt is not None:
        ws.append(nxt.self_attn.in_proj_weight)
    return _cached(owner, key, ws, lambda: ops.decoder_chain_prepare(*[w.detach() for w in ws]))


def _cross_const(owner, li, layer):
    """The cross-attention block over the all-zero memory: every key is the bias b_k, so the softmax is uniform and the
    block returns the constant c = W_o b_v + b_o [d] for every row (model/influentialRS.py:172-173,189-193).  Inference
    caches it per weight version (it was six cuBLAS gemv launches per decode); under autograd it is recomputed so that
    gradients reach the cross-attention parameters."""
    ca = layer.multihead_attn
    d = ca.embed_dim
    ws = (ca.in_proj_bias, ca.out_proj.weight, ca.out_proj.bias)
    if torch.is_grad_enabled() and any(w.requires_grad for w in ws):
        return F.linear(ca.in_proj_bias[2 * d:], ca.out_proj.weight, ca.out_proj.bias)
    with torch.no_grad():
        return _cached(owner, ("cross", li), ws,
                       lambda: F.linear(ca.in_proj_bias[2 * d:], ca.out_proj.weight, ca.out_proj.bias).contiguous())


def _cross_rows_dropout(owner, layer, B, L, p_drop, device):
    """Cross-attention block over the all-zero memory WITH attention-probability dropout (train mode): the softmax is
    uniform over the S = max_len memory slots and every value is the bias b_v, so head h returns
    (kept_h / (S (1-p))) b_v[h] with kept_h ~ Binomial(S, 1-p) per (row, head) -- no longer a constant.  Returns [B,L,d],
    differentiable w.r.t. the cross-attention parameters."""
    ca = layer.multihead_attn
    d, H = ca.embed_dim, ca.num_heads
    dh = d // H
    S = float(owner.max_len)
    kept = torch.binomial(torch.full((B, L, H), S, device=device), torch.full((B, L, H), 1.0 - p_drop, device=device))
    mult = kept / (S * (1.0 - p_drop))                                                   # [B,L,H]
    bv = ca.in_proj_bias[2 * d:]
    cv = (ca.out_proj.weight.view(d, H, dh) * bv.view(1, H, dh)).sum(-1)                 # [d,H]: W_o[:, head h] b_v[head h]
    return mult @ cv.t() + ca.out_proj.bias


def _decoder_stack_fused(owner, x, ids, r_u, mask_mode, last_row=None):
    """Inference decoder stack for d=128 / ffn=256: per layer ONE attention kernel and ONE fused
    row-local chain kernel (out_proj+norm1+norm2 -> FFN+norm3 -> in_proj of the next layer).  Same
    arithmetic as ``_decoder_stack``; x and the q/k/v buffer are updated in place.  For windows of
    129..223 positions with 4 heads of 32 the q/k/v projection never exists as fp32 rows: the chain kernel
    writes it as the attention kernel's operand images (csrc/qkv_image.cuh)."""
    H = owner.n_heads
    d = owner.embed_dim
    B, L = x.shape[0], x.shape[1]
    layers = owner.decoder.layers
    n_layers = len(layers)
    use_img = ops.USE_IMG_ATTENTION and ops.USE_TC_ATTENTION and H * 32 == d and ops.attn_img_supported(L, 32)
    if use_img:
        images = ops.qkv_images_buffer(B, L, H, x.device, slot=1)
        l0 = layers[0]
        ops.in_proj_images_tc(x, _chain_prepared(owner, "chain_in0", l0, l0), l0.self_attn.in_proj_bias, images, L, mask_mode)
        qkv = None
    else:
        qkv = _tc_in_proj(owner, 0, layers[0].self_attn, x)
    for li, layer in enumerate(layers):
        sa, ca = layer.self_attn, layer.multihead_attn
        c = _cross_const(owner, li, layer)                                                          # [d]
        last = li == n_layers - 1
        if last and last_row is not None:
            if use_img:
                a = ops.pim_attention_img(images, ids, r_u, B, L, H, mask_mode, W_H, W_OBJ, q_row0=last_row, n_q=1)[:, 0]
            else:
                a = ops.pim_attention(qkv, ids, r_u, H, mask_mode, W_H, W_OBJ, q_row0=last_row, n_q=1)[:, 0]
            return _tc_layer_tail(owner, li, layer, x[:, last_row], a, c)
        if use_img:
            a = ops.pim_attention_img(images, ids, r_u, B, L, H, mask_mode, W_H, W_OBJ)
        else:
            a = ops.pim_attention(qkv, ids, r_u, H, mask_mode, W_H, W_OBJ)
        nxt = None if last else layers[li + 1]
        x, q2 = ops.decoder_chain_tc(a, x, _chain_prepared(owner, ("chain", li), layer, nxt), sa.out_proj.bias,
                                     layer.norm1.weight, layer.norm1.bias, c, layer.norm2.weight, layer.norm2.bias,
                                     layer.linear1.bias, layer.linear2.bias, layer.norm3.weight, layer.norm3.bias,
                                     None if last else nxt.self_attn.in_proj_bias,
                                     eps=(layer.norm1.eps, layer.norm2.eps, layer.norm3.eps),
                                     ffn=layer.linear1.out_features, x_out=x,
                                     qkv_out=None if (last or use_img) else qkv,
                                     qkv_images=images if (use_img and not last) else None, L=L, mask_mode=mask_mode)
        if not last and not use_img:
            qkv = q2
    return x


USE_FUSED_CHAIN = True      # tests flip it to compare against the layer-by-layer kernels


def _draw_seed() -> int:
    """Seed of one sampled generation, from torch's (CPU) generator: reproducible under torch.manual_seed, no device sync."""
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def _decoder_stack(owner, x, ids, r_u, mask_mode, last_row=None):
    """Post-norm decoder over an all-zero memory (model/influentialRS.py:67-74,172-173,189-193).

    x [B,L,d].  If ``last_row`` is given (inference) the last layer computes only that query row and
    the function returns [B,d]; otherwise [B,L,d].  The cross-attention block is the constant
    c = W_o b_v + b_o (softmax over identical keys is uniform), folded into the LN1->LN2 kernel."""
    H = owner.n_heads
    d = owner.embed_dim
    train = torch.is_grad_enabled() and any(p.requires_grad for p in owner.decoder.parameters())
    p_drop = owner.dropout if owner.training else 0.0
    n_layers = len(owner.decoder.layers)
    if (USE_FUSED_CHAIN and not (train or p_drop > 0) and x.dim() == 3
            and ops.decoder_chain_supported(d, owner.decoder.layers[0].linear1.out_features)):
        return _decoder_stack_fused(owner, x.contiguous(), ids, r_u, mask_mode, last_row)
    for li, layer in enumerate(owner.decoder.layers):
        sa, ca = layer.self_attn, layer.multihead_attn
        c = _cross_const(owner, li, layer)                                              # [d]
        only_row = (last_row is not None) and (li == n_layers - 1)
        if not (train or p_drop > 0) and _tc_ok(d, layer.linear1.out_features):
            qkv = _tc_in_proj(owner, li, sa, x)                                          # tcgen05
        else:
            qkv = F.linear(x, sa.in_proj_weight, sa.in_proj_bias)                       # cuBLAS (training / odd dims)
        if only_row:
            a = ops.pim_attention(qkv, ids, r_u, H, mask_mode, W_H, W_OBJ, q_row0=last_row, n_q=1, p_drop=p_drop)[:, 0]
            x = x[:, last_row]
        else:
            # train mode: attention-probability dropout inside the kernel (same p as every dropout of the layer)
            a = ops.pim_attention(qkv, ids, r_u, H, mask_mode, W_H, W_OBJ, p_drop=p_drop)
        if train or p_drop > 0:
            y = F.dropout(F.linear(a, sa.out_proj.weight, sa.out_proj.bias), p_drop, owner.training)
            x = F.layer_norm(x + y, (d,), layer.norm1.weight, layer.norm1.bias, layer.norm1.eps)
            cr = _cross_rows_dropout(owner, layer, x.shape[0], x.shape[1], p_drop, x.device) \
                if (p_drop > 0 and x.dim() == 3) else c.expand_as(x)
            x = F.layer_norm(x + F.dropout(cr, p_drop, owner.training), (d,),
                             layer.norm2.weight, layer.norm2.bias, layer.norm2.eps)
            y = F.linear(F.dropout(F.relu(F.linear(x, layer.linear1.weight, layer.linear1.bias)), p_drop, owner.training),
                         layer.linear2.weight, layer.linear2.bias)
            x = F.layer_norm(x + F.dropout(y, p_drop, owner.training), (d,), layer.norm3.weight, layer.norm3.bias,
                             layer.norm3.eps)
        elif _tc_ok(d, layer.linear1.out_features):
            x = _tc_layer_tail(owner, li, layer, x, a, c)
        else:
            y = F.linear(a, sa.out_proj.weight)
            x = ops.residual_layernorm(x, y, sa.out_proj.bias, layer.norm1.weight, layer.norm1.bias,
                                       c, layer.norm2.weight, layer.norm2.bias, layer.norm1.eps)
            y = F.linear(F.relu(F.linear(x, layer.linear1.weight, layer.linear1.bias)), layer.linear2.weight)
            x = ops.residual_layernorm(x, y, layer.linear2.bias, layer.norm3.weight, layer.norm3.bias,
                                       eps=layer.norm3.eps)
    return x


class InfluentialNet(nn.Module):
    """Influential Recommender Network (model/influentialRS.py:22-216)."""

    def __init__(self, config):
        super().__init__()
        self.PAD_ID = 0
        self.item_embed_path = None
        self.user_embed_path = None
        self.n_item = config.n_item
        self.n_user = config.n_user
        self.use_u = False
        self.max_len = config.max_len
        self.n_layers = config.n_layers
        self.n_heads = config.n_heads
        self.embed_dim = config.emb_dim
        self.u_embed_dim = config.u_emb_dim
        self.ffn_dim = config.ffn_dim
        self.dropout = config.dropout
        # same modules, same order as the reference => same RNG stream => same initial weights
        self.item_embedder = nn.Embedding(self.n_item + 1, self.embed_dim, padding_idx=self.PAD_ID)
        self.user_embedder = nn.Embedding(self.n_user, self.u_embed_dim)
        self.pos_embedder = PositionalEncoding(self.embed_dim, self.max_len)
        self.decoder = nn.TransformerDecoder(
            decoder_layer=nn.TransformerDecoderLayer(d_model=self.embed_dim, nhead=self.n_heads,
                                                     dim_feedforward=self.ffn_dim, dropout=self.dropout,
                                                     activation="relu"),
            num_layers=self.n_layers)
        self.user_mask_layer = nn.Linear(self.u_embed_dim, 1)
        self.project = nn.Linear(self.embed_dim, self.n_item)
        self.optimizer = optim.Adam(filter(lambda x: x.requires_grad, self.parameters()),
                                    betas=(0.9, 0.98), eps=1e-09, lr=config.lr1)
        self.pla_lr_scheduler = lr_scheduler.ReduceLROnPlateau(self.optimizer, factor=0.5, patience=4)

    # -- pieces ------------------------------------------------------------------------------------
    def pi_factor(self, user):
        """r_u = user_mask_layer(user_embedder(user)) [B,1] (model/influentialRS.py:180): one library kernel in
        inference (irs_pif_fwd), torch embedding + linear under autograd."""
        return ops.pif(user, self.user_embedder.weight, self.user_mask_layer.weight, self.user_mask_layer.bias)

    def invalidate_prepared(self):
        """Forget every cached weight image of this module (call after editing weights through ``.data``)."""
        self.__dict__.pop("_tc_cache", None)
        ops.invalidate_prepared()

    def embed(self, dec_input_seq):
        """item_embedder(seq)*sqrt(d) + pe, dropout in training (model/influentialRS.py:174-176)."""
        L = dec_input_seq.size(1)
        x = ops.embed_gather(dec_input_seq, self.item_embedder.weight, self.pos_embedder.pe[0, :L],
                             math.sqrt(self.embed_dim))
        return F.dropout(x, self.dropout, self.training)

    def decoding(self, dec_input_seq, user, return_pi=False, last_row=None):
        """Decoder output [B,L,d] (model/influentialRS.py:157-200).  ``last_row`` (extension) returns
        only that row of the final layer, [B,d] -- what generation and the accuracy metrics read."""
        dec_input_seq = dec_input_seq.contiguous()
        r_u = self.pi_factor(user)
        x = _decoder_stack(self, self.embed(dec_input_seq), dec_input_seq, r_u, ops.MASK_PIM, last_row)
        return (x, r_u) if return_pi else x

    def forward(self, dec_input_seq, user):
        """Logits [B,L,N] (model/influentialRS.py:202-216).  Kept for API parity: it materialises the
        logits on request (cuBLAS); the hot paths below never call it."""
        return self.project(self.decoding(dec_input_seq, user))


class IRSNN(nn.Module):
    """Functionality handler (model/influentialRS.py:219-470)."""

    def __init__(self, config, net, device):
        super().__init__()
        self.PAD_ID = 0
        self.n_item = config.n_item
        self.embed_dim = config.emb_dim
        self.net = net
        self.device = device
        self.loss_function = nn.CrossEntropyLoss()
        self.optimizer = optim.Adam(filter(lambda x: x.requires_grad, self.net.parameters()),
                                    betas=(0.9, 0.98), eps=1e-09, lr=config.lr1)
        self.pla_lr_scheduler = lr_scheduler.ReduceLROnPlateau(self.optimizer, factor=0.5, patience=4)
        self.softmax = nn.Softmax(dim=2)
        self.user_tile = int(getattr(config, "user_tile", 4096))   # users per device pass (activation memory)
        self.grad_sync = None        # set by dist.make_data_parallel(): all-reduce of gradients
        self.scorer = None           # dist.ShardedScorer: catalog-sharded label ranks across GPUs (SURVEY 8e row 3)

    def invalidate_prepared(self):
        """Forget every cached weight image (call after editing weights through ``.data``; see ops.weight_tag)."""
        if hasattr(self.net, "invalidate_prepared"):
            self.net.invalidate_prepared()
        ops.invalidate_prepared()

    # -- loss ---------------------------------------------------------------------------------------
    def _ce(self, seqs, users):
        """mean CE over rows (b, l<L-1) whose next id is non-pad, class = id-1
        (model/influentialRS.py:293-303) -- via the fused scorer, no [M,N] logits."""
        h = self.net.decoding(seqs, users)                                   # [B,L,d]
        B, L, d = h.shape
        tgt = seqs[:, 1:].reshape(-1)
        rows = torch.nonzero(tgt > self.PAD_ID).squeeze(1)                   # the reference's masked_select
        hm = h[:, :-1].reshape(-1, d).index_select(0, rows)
        self.last_ce_rows = int(rows.numel())                                # used by dist.make_data_parallel
        return ops.softmax_ce_mean(hm, self.net.project.weight, self.net.project.bias, tgt.index_select(0, rows) - 1)

    def get_loss_on_eval_data(self, seqs, users):
        self.net.eval()
        with torch.no_grad():
            return self._ce(seqs.clone(), users).item()

    def train_batch(self, seqs, users):
        self.net.train()
        loss = self._ce(seqs.clone(), users)
        self.optimizer.zero_grad()
        loss.backward()
        if self.grad_sync is not None:
            self.grad_sync()
        self.optimizer.step()
        return loss.item()

    def _delete_item_in_history(self, tensor, indices):
        return tensor[~tensor.unsqueeze(1).eq(indices).any(1)]

    def get_pif_in_batch(self, seqs, users):
        """r_u [B,1] as numpy (model/influentialRS.py:325-338) -- without the wasted decode."""
        with torch.no_grad():
            return self.net.pi_factor(users).detach().cpu().numpy()

    # -- accuracy -------------------------------------------------------------------------------------
    @staticmethod
    def _raw_history(raw, device):
        """The ragged raw histories (list of LongTensor, data_provider.py:611) as one zero-padded [B,Lx] id matrix."""
        lens = [int(r.numel()) for r in raw]
        hist = torch.zeros((len(raw), max(lens + [1])), dtype=torch.int64)
        for b, r in enumerate(raw):
            hist[b, : lens[b]] = r.reshape(-1).to("cpu")
        return hist.to(device)

    def _label_rank(self, h, labels, hist_ids):
        """1-based rank of each label among the items not in its raw history (0 = the label is in the history)."""
        if self.scorer is not None:
            return self.scorer.rank(h, labels, hist_ids)
        excl = None if hist_ids is None else ops.sort_exclusions(hist_ids, self.n_item, 1)
        return ops.score_rank(h, self.net.project.weight, self.net.project.bias, labels, excl, 1)

    def get_accuracy_metrics_in_batch(self, raw, seqs, users, targets, labels, top_k=20, gap_len=20, use_h=True):
        """Hit@top_k count and reciprocal ranks (model/influentialRS.py:340-390), by counting the
        items ahead of the label instead of sorting the catalog."""
        B, L = seqs.shape
        pos = L - (gap_len + 1) - 1
        with torch.no_grad():
            h = self.net.decoding(seqs.clone(), users, last_row=pos)         # [B,d]
            hist = self._raw_history(raw, seqs.device) if use_h else None
            rank = self._label_rank(h, labels.to(seqs.device).long(), hist).cpu().numpy()
        found = rank > 0                                   # label filtered out => the reference skips it
        hit_count = int(((rank <= top_k) & found).sum())
        rr = np.reciprocal(rank[found].astype(np.float64))
        return hit_count, rr

    # -- influence-path generation ----------------------------------------------------------------------
    def path_step(self, temp, users, paths, i, excl=None, sample=False, sample_k=3, h=None, seed=None, row_key=None):
        """ONE generation step of a tile of windows ``temp`` [b,L] (updated in place; model/influentialRS.py:412-449):
        decode (row L-2 only in the last layer) -> fused score + window mask + arg-max (or, when ``sample``, top-k and one
        draw from the softmax over the k survivors) -> window shift, pick recorded in ``paths[:, i]``.  ``excl`` is the
        sorted exclusion state of the windows (built on the first call, then updated incrementally: one id slides out,
        the pick comes in) and is returned for the next step.  The draw is a pure function of (``seed``, step ``i``,
        ``row_key``[r]) -- ``row_key`` [b] int64 on the device names each row (default: its index in the tile).  ``seed`` is
        required with ``sample``: one seed held for every step of a path (generate_on_device draws it once per call from
        torch's CPU generator).  No host synchronisation."""
        L = temp.shape[1]
        p = L - 2
        if h is None:
            h = self.net.decoding(temp, users, last_row=p)                              # [b,d]
        if excl is None:
            excl = ops.sort_exclusions(temp[:, : p + 1], self.n_item, 1)
        W, beta = self.net.project.weight, self.net.project.bias
        if not sample:
            nxt = ops.score_argmax(h, W, beta, excl, 1)[1][:, 0].contiguous()          # greedy: the best item not in the window
        else:
            vals, items = ops.score_topk_any(h, W, beta, sample_k, excl, 1)              # tcgen05 top-k: one pass over W
            if seed is None:
                raise ValueError("path_step(sample=True) needs the seed of the whole path (see generate_on_device)")
            if row_key is None:
                row_key = torch.arange(temp.shape[0], dtype=torch.int64, device=temp.device)
            nxt = ops.topk_sample(vals, items, seed, i, row_key)   # softmax over the k survivors, one counter-based draw
        ops.exclusions_update(excl, temp[:, 0], nxt, self.n_item, 1)                     # before the shift: temp[:,0] slides out
        ops.window_shift(temp, nxt, paths, i)
        return excl

    def generate_on_device(self, seqs, users, max_path_len=20, sample=False, sample_k=3, first_h=None):
        """Device loop of get_seq_in_batch: returns paths f32 [B,P] on the device, untrimmed.  ``first_h`` [B,d]
        (optional) is the decoder row L-2 of the unmodified windows, if the caller already has it.  With ``sample`` one
        seed is drawn per call from torch's CPU generator (``torch.manual_seed`` makes runs reproducible) and row b of
        ``seqs`` draws with the key b at every step, so the paths do not depend on ``user_tile`` or on the device."""
        B, L = seqs.shape
        paths = torch.zeros((B, max_path_len), dtype=torch.float32, device=seqs.device)
        seed = _draw_seed() if sample else None
        for b0 in range(0, B, self.user_tile):
            temp = seqs[b0:b0 + self.user_tile].clone()
            us = users[b0:b0 + self.user_tile]
            pt = paths[b0:b0 + self.user_tile]
            keys = torch.arange(b0, b0 + temp.shape[0], dtype=torch.int64, device=seqs.device) if sample else None
            excl = None
            for i in range(max_path_len):
                h = first_h[b0:b0 + self.user_tile] if (i == 0 and first_h is not None) else None
                excl = self.path_step(temp, us, pt, i, excl, sample, sample_k, h, seed, keys)
        return paths

    def test_batch(self, raw, seqs, users, targets, labels, top_k=20, max_path_len=20, use_h=True, sample=False, sample_k=3):
        """One evaluation batch of pipeline.test_model (pipeline.py:187-228) with gap_len = 0: the reference calls
        get_pif_in_batch, get_accuracy_metrics_in_batch and get_seq_in_batch one after the other -- three decodes of the
        same windows, two of them only to read decoder row L-2.  Here that row is decoded once and feeds both the label
        rank and the first generation step.  Returns (r_u [B,1] np, hit_count, rr np, paths np [B,P], targets np,
        histories list, n_early_success): exactly what the three calls return."""
        B, L = seqs.shape
        with torch.no_grad():
            seqs = seqs.contiguous()
            h0, r_u = self.net.decoding(seqs.clone(), users, return_pi=True, last_row=L - 2)
            hist = self._raw_history(raw, seqs.device) if use_h else None
            rank = self._label_rank(h0, labels.to(seqs.device).long(), hist)
            paths = self.generate_on_device(seqs, users, max_path_len, sample, sample_k, first_h=h0)
            rank = rank.cpu().numpy()
        found = rank > 0
        hit_count = int(((rank <= top_k) & found).sum())
        rr = np.reciprocal(rank[found].astype(np.float64))
        from .dist import trim_paths
        p, t, hst, n_early = trim_paths(paths.cpu().numpy(), targets.detach().cpu().numpy(), seqs[:, :-1].detach().cpu().numpy())
        return r_u.detach().cpu().numpy(), hit_count, rr, p, t, hst, n_early

    def get_seq_in_batch(self, seqs, users, targets, max_path_len=20, gap_len=20, sample=False, sample_k=3):
        """Influence paths (model/influentialRS.py:392-470).  Returns (paths f32 np [B,P] zeroed after
        the first occurrence of the target, targets np, list of actual histories, n_early_success)."""
        if gap_len != 0:
            raise NotImplementedError("gap_len > 0 is ill-defined in the reference (SURVEY D6); only gap_len=0 is built")
        with torch.no_grad():
            paths = self.generate_on_device(seqs.contiguous(), users, max_path_len, sample, sample_k)
        from .dist import trim_paths
        return trim_paths(paths.cpu().numpy(), targets.detach().cpu().numpy(), seqs[:, :-1].detach().cpu().numpy())
