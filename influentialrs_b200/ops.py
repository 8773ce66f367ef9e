"""Tensor-level wrappers over the C ABI (include/irs_b200.h).  PyTorch is plumbing here: it owns the
device buffers and the stream; every operator below runs a hand-written sm_100a kernel from
libirs_b200.so and raises if the library is missing or the tensors are not on a CUDA device."""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

from ._lib import lib, check

MASK_PIM, MASK_CAUSAL_PAD, MASK_CAUSAL = 0, 1, 2


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"influentialrs_b200: '{name}' must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"influentialrs_b200: '{name}' must be {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


_error_flags = {}


def _error_flag(device):
    """Device int the tensor-core kernels' pipeline watchdogs write to (0 = healthy)."""
    f = _error_flags.get(device)
    if f is None:
        f = torch.zeros((1,), dtype=torch.int32, device=device)
        _error_flags[device] = f
    return f


# ---- prepared-weight caches ---------------------------------------------------------------------------------------
# Every tensor-core kernel streams a re-tiled bf16 hi/lo IMAGE of its weight matrix, cached per weight version.  The
# version tag is (data_ptr, Tensor._version, shape, epoch): optimizer steps, load_state_dict and every in-place op on
# the parameter bump _version, but edits through ``p.data`` (p.data.copy_ / mul_ / EMA swaps / clipping) do NOT.  After
# such an edit call ``invalidate_prepared()`` (also a method of InfluentialNet / SampleNet / IRSNN / the sharded classes);
# IRS_VERIFY_PREPARED=1 adds a checksum of the weights to the tag (one host sync per lookup: a debug mode).
_prepared_epoch = 0
_VERIFY_PREPARED = __import__("os").environ.get("IRS_VERIFY_PREPARED", "0") == "1"


def invalidate_prepared() -> None:
    """Drop every cached weight image (all modules, this process): the next call re-tiles from the live weights."""
    global _prepared_epoch
    _prepared_epoch += 1
    _prepared_scorer_cache.clear()


def weight_tag(*ws):
    """Cache tag of one or more weight tensors (see the note above)."""
    tag = tuple((w.data_ptr(), w._version, tuple(w.shape)) for w in ws) + (_prepared_epoch,)
    if _VERIFY_PREPARED:
        tag += tuple(float(w.detach().double().sum()) for w in ws)
    return tag


def cached_image(cache: dict, key, ws, make):
    """``make()``, a value derived from the weights ``ws`` (a re-tiled image, a folded constant), cached in ``cache`` under
    ``key`` and rebuilt when weight_tag(*ws) changes.  An entry is (tag, value, weights): it keeps the weights referenced,
    so while it is cached their storage cannot be freed and the address cannot come back as a different tensor with the
    same shape and a fresh version counter (which would silently hit a stale value)."""
    tag = weight_tag(*ws)
    hit = cache.get(key)
    if hit is None or hit[0] != tag:
        hit = (tag, make(), tuple(w.detach() for w in ws))
        cache[key] = hit
    return hit[1]


# bench.py sets this to a dict: kernel class -> list of (start, stop) CUDA events on the launching stream
_timer = None


def _timed(name):
    def deco(fn):
        import functools

        @functools.wraps(fn)
        def wrap(*a, **k):
            t = _timer
            if t is None:
                return fn(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            t.setdefault(name, []).append((e0, e1))
            return r
        return wrap
    return deco


def launch_count() -> int:
    return int(lib().irs_launch_count())


def launch_count_reset() -> None:
    lib().irs_launch_count_reset()


# ------------------------------------------------------------------------------------------------
# K1 / K2
# ------------------------------------------------------------------------------------------------
@_timed("gather")
def embed_gather_raw(ids, table, pe, scale: float) -> torch.Tensor:
    ids = _need(ids, torch.int64, "ids")
    table = _need(table, torch.float32, "table")
    if pe is not None:
        pe = _need(pe, torch.float32, "pe")
    B, L = ids.shape
    d = table.shape[1]
    out = torch.empty((B, L, d), dtype=torch.float32, device=ids.device)
    check(lib().irs_embed_gather_fwd(_ptr(ids), _ptr(table), _ptr(pe), float(scale), _ptr(out),
                                     B * L, L, d, table.shape[0], _stream()), "embed_gather_fwd")
    return out


@_timed("scatter_add")
def embed_scatter_add_raw(ids, d_out, scale: float, d_table, pad_id: int = 0) -> None:
    ids = _need(ids, torch.int64, "ids")
    d_out = _need(d_out, torch.float32, "d_out")
    d = d_table.shape[1]
    check(lib().irs_embed_scatter_add_bwd(_ptr(ids), _ptr(d_out), float(scale), _ptr(d_table),
                                          ids.numel(), d, d_table.shape[0], pad_id, _stream()), "embed_scatter_add_bwd")


class _EmbedGather(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ids, table, pe, scale):
        ctx.save_for_backward(ids)
        ctx.scale = scale
        ctx.table_shape = table.shape
        return embed_gather_raw(ids, table, pe, scale)

    @staticmethod
    def backward(ctx, d_out):
        (ids,) = ctx.saved_tensors
        d_table = torch.zeros(ctx.table_shape, dtype=torch.float32, device=d_out.device)
        embed_scatter_add_raw(ids, d_out, ctx.scale, d_table, 0)      # padding_idx=0 row stays zero
        return None, d_table, None, None


def embed_gather(ids, table, pe, scale: float) -> torch.Tensor:
    """x = table[ids]*scale + pe[:L]  (bit-exact with torch; backward = warp-aggregated scatter-add)."""
    if torch.is_grad_enabled() and table.requires_grad:
        return _EmbedGather.apply(ids, table, pe, scale)
    return embed_gather_raw(ids, table, pe, scale)


def pif(users, user_table, w, c) -> torch.Tensor:
    """r_u [B,1] = user_table[users] @ w^T + c (a2; model/influentialRS.py:180).  Training (autograd needed) goes
    through torch's embedding + linear; inference runs the library kernel."""
    if torch.is_grad_enabled() and (user_table.requires_grad or w.requires_grad):
        return torch.nn.functional.linear(torch.nn.functional.embedding(users, user_table), w, c)
    users = _need(users.reshape(-1), torch.int64, "users")
    user_table = _need(user_table, torch.float32, "user_table")
    out = torch.empty((users.shape[0], 1), dtype=torch.float32, device=users.device)
    check(lib().irs_pif_fwd(_ptr(users), _ptr(user_table), _ptr(_need(w.reshape(-1), torch.float32, "w")), _ptr(c), _ptr(out),
                            users.shape[0], user_table.shape[1], user_table.shape[0], _stream()), "pif_fwd")
    return out


# ------------------------------------------------------------------------------------------------
# K3 / K4
# ------------------------------------------------------------------------------------------------
USE_TC_ATTENTION = True     # tensor-core forward where the shape allows (inference); tests flip it to compare


_image_buffers = {}


def qkv_images_buffer(B: int, L: int, H: int, device, slot: int = 0) -> torch.Tensor:
    """Zero-initialised operand-image buffer for (B, L, H); cached -- the padding rows/columns the
    producers never write must stay zero, and every producer writes the same positions for a given L."""
    key = (B, L, H, str(device), slot)
    buf = _image_buffers.get(key)
    if buf is None:
        nbytes = lib().irs_qkv_images_bytes(B, L, H, 32)
        if nbytes == 0:
            raise RuntimeError(f"operand images need 128 < L <= 223 and dh == 32 (got L={L})")
        for k_old in [k_ for k_ in _image_buffers if k_[3] == key[3] and k_[4] == slot]:
            del _image_buffers[k_old]                     # one live buffer per device and slot
        buf = torch.zeros((nbytes,), dtype=torch.uint8, device=device)
        _image_buffers[key] = buf
    return buf


def attn_img_supported(L: int, dh: int) -> bool:
    return bool(lib().irs_pim_attn_img_supported(int(L), int(dh)))


def qkv_to_images(q, k, v, ld, B, L, H, mode, images=None) -> torch.Tensor:
    if images is None:
        images = qkv_images_buffer(B, L, H, q.device)
    check(lib().irs_qkv_to_images(_ptr(q), _ptr(k), _ptr(v), ld[0], ld[1], ld[2], _ptr(images), B, L, H, 32, int(mode),
                                  _stream()), "qkv_to_images")
    return images


@_timed("attention")
def pim_attention_img(images, ids, r_u, B: int, L: int, H: int, mode: int = MASK_PIM, w_h: float = 0.05, w_obj: float = 1.0,
                      q_row0: int = 0, n_q: Optional[int] = None) -> torch.Tensor:
    """Self-attention from operand images (persistent tcgen05 kernel).  Returns [B, n_q, H*32]."""
    n_q = L if n_q is None else n_q
    if ids is not None:
        ids = _need(ids, torch.int64, "ids")
    if r_u is not None:
        r_u = _need(r_u.reshape(-1), torch.float32, "r_u")
    out = torch.empty((B, n_q, H * 32), dtype=torch.float32, device=images.device)
    check(lib().irs_pim_attn_fwd_img(_ptr(images), _ptr(ids), _ptr(r_u), float(w_h), float(w_obj), int(mode), _ptr(out),
                                     B, L, H, 32, q_row0, n_q, _ptr(_error_flag(images.device)), _stream()), "pim_attn_fwd_img")
    return out


USE_TC_TRAIN_ATTENTION = True   # training forward (lse needed, no attention dropout) on the per-head tcgen05 kernel
USE_IMG_ATTENTION = True    # full windows of 129..223 with dh = 32 go through operand images + the persistent kernel


def _attn_fwd_raw(q, k, v, ld, ids, r_u, w_h, w_obj, mode, B, L, H, dh, q_row0, n_q, need_lse, p_drop=0.0, seed=0):
    # attention-probability dropout lives in the fp32 forward / backward pair only
    if (p_drop == 0 and USE_TC_ATTENTION and USE_IMG_ATTENTION and not need_lse and attn_img_supported(L, dh) and (n_q == L or n_q == 1)
            and ld[0] % 4 == 0 and ld[1] % 4 == 0 and ld[2] % 4 == 0
            and q.data_ptr() % 16 == 0 and k.data_ptr() % 16 == 0 and v.data_ptr() % 16 == 0):
        images = qkv_to_images(q, k, v, ld, B, L, H, mode)
        return pim_attention_img(images, ids, r_u, B, L, H, mode, w_h, w_obj, q_row0, n_q), None
    out = torch.empty((B, n_q, H * dh), dtype=torch.float32, device=q.device)
    lse = torch.empty((B, H, n_q), dtype=torch.float32, device=q.device) if need_lse else None
    # per-(batch, head) tcgen05 kernel: inference at L <= 128 / other head sizes, and the TRAINING forward (it returns the
    # log-sum-exp the backward kernel needs) whenever no attention-probability dropout is asked for
    if (p_drop == 0 and USE_TC_ATTENTION and (USE_TC_TRAIN_ATTENTION or not need_lse) and lib().irs_pim_attn_tc_supported(L, dh)
            and ld[0] % 4 == 0 and ld[1] % 4 == 0 and ld[2] % 4 == 0
            and q.data_ptr() % 16 == 0 and k.data_ptr() % 16 == 0 and v.data_ptr() % 16 == 0):
        check(lib().irs_pim_attn_fwd_tc(_ptr(q), _ptr(k), _ptr(v), ld[0], ld[1], ld[2], _ptr(ids), _ptr(r_u),
                                        float(w_h), float(w_obj), int(mode), _ptr(out), _ptr(lse), B, L, H, dh, q_row0, n_q,
                                        _ptr(_error_flag(q.device)), _stream()), "pim_attn_fwd_tc")
        return out, lse
    check(lib().irs_pim_attn_fwd(_ptr(q), _ptr(k), _ptr(v), ld[0], ld[1], ld[2], _ptr(ids), _ptr(r_u),
                                 float(w_h), float(w_obj), int(mode), _ptr(out), _ptr(lse),
                                 B, L, H, dh, q_row0, n_q, float(p_drop), int(seed), _stream()), "pim_attn_fwd")
    return out, lse


class _PimAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkv, ids, r_u, w_h, w_obj, mode, H, p_drop=0.0):
        B, L, d3 = qkv.shape
        d = d3 // 3
        dh = d // H
        q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
        # dropout seed from torch's (CPU) generator: reproducible under torch.manual_seed, no device sync
        seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if p_drop > 0 else 0
        out, lse = _attn_fwd_raw(q, k, v, (d3, d3, d3), ids, r_u, w_h, w_obj, mode, B, L, H, dh, 0, L, True, p_drop, seed)
        ctx.save_for_backward(qkv, ids, r_u, out, lse)
        ctx.cfg = (w_h, w_obj, mode, H, p_drop, seed)
        return out

    @staticmethod
    def backward(ctx, d_out):
        qkv, ids, r_u, out, lse = ctx.saved_tensors
        w_h, w_obj, mode, H, p_drop, seed = ctx.cfg
        B, L, d3 = qkv.shape
        d = d3 // 3
        dh = d // H
        d_out = d_out.contiguous()
        d_qkv = torch.empty_like(qkv)
        d_ru = torch.zeros(B, dtype=torch.float32, device=qkv.device) if mode == MASK_PIM else None
        q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
        dq, dk, dv = d_qkv[..., :d], d_qkv[..., d:2 * d], d_qkv[..., 2 * d:]
        check(lib().irs_pim_attn_bwd(_ptr(q), _ptr(k), _ptr(v), d3, d3, d3, _ptr(ids), _ptr(r_u),
                                     float(w_h), float(w_obj), int(mode), _ptr(out), _ptr(lse), _ptr(d_out),
                                     _ptr(dq), _ptr(dk), _ptr(dv), _ptr(d_ru), B, L, H, dh, float(p_drop), int(seed),
                                     _stream()), "pim_attn_bwd")
        return d_qkv, None, d_ru, None, None, None, None, None


def pim_attention(qkv, ids, r_u, H: int, mode: int = MASK_PIM, w_h: float = 0.05, w_obj: float = 1.0,
                  q_row0: int = 0, n_q: Optional[int] = None, p_drop: float = 0.0) -> torch.Tensor:
    """Self-attention on the packed in_proj output qkv [B,L,3d] with the mask built in-kernel.
    Returns [B, n_q, d] (heads concatenated, before out_proj).  ``p_drop`` > 0: attention-probability dropout (training
    path only: the fp32 forward / backward kernels regenerate the same counter-based mask)."""
    qkv = _need(qkv, torch.float32, "qkv")
    B, L, d3 = qkv.shape
    d = d3 // 3
    if d % H:
        raise ValueError("embed dim not divisible by heads")
    if ids is not None:
        ids = _need(ids, torch.int64, "ids")
    if r_u is not None:
        r_u = _need(r_u.reshape(-1), torch.float32, "r_u")
    full = (q_row0 == 0 and (n_q is None or n_q == L))
    if torch.is_grad_enabled() and (qkv.requires_grad or (r_u is not None and r_u.requires_grad)):
        if not full:
            raise RuntimeError("row-subset attention is inference-only")
        return _PimAttention.apply(qkv, ids, r_u, w_h, w_obj, mode, H, float(p_drop))
    n_q = L if n_q is None else n_q
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if p_drop > 0 else 0      # train mode under no_grad
    return _attn_fwd_raw(q, k, v, (d3, d3, d3), ids, r_u, w_h, w_obj, mode, B, L, H, d // H, q_row0, n_q, False,
                         float(p_drop), seed)[0]


def attention_qkv(q, k, v, H: int, mode: int = MASK_CAUSAL, ids=None) -> torch.Tensor:
    """Attention with separately laid out q, k, v [B,L,d] (SASRec: queries from LN(x), keys/values from x)."""
    q, k, v = _need(q, torch.float32, "q"), _need(k, torch.float32, "k"), _need(v, torch.float32, "v")
    B, L, d = q.shape
    return _attn_fwd_raw(q, k, v, (d, d, d), ids, None, 0.0, 0.0, mode, B, L, H, d // H, 0, L, False)[0]


# ------------------------------------------------------------------------------------------------
# fused residual + LayerNorm (+ const + LayerNorm)
# ------------------------------------------------------------------------------------------------
def residual_layernorm(x, y, y_bias, g1, b1, c2=None, g2=None, b2=None, eps: float = 1e-5) -> torch.Tensor:
    x = _need(x, torch.float32, "x")
    if y is not None:
        y = _need(y, torch.float32, "y")
    d = x.shape[-1]
    out = torch.empty_like(x)
    check(lib().irs_residual_layernorm(_ptr(x), _ptr(y), _ptr(y_bias), _ptr(g1), _ptr(b1), _ptr(c2), _ptr(g2), _ptr(b2),
                                       float(eps), _ptr(out), x.numel() // d, d, _stream()), "residual_layernorm")
    return out


# ------------------------------------------------------------------------------------------------
# fused scorer family
# ------------------------------------------------------------------------------------------------
def sort_exclusions(excl_ids, n_cols: int, item_base: int = 1) -> Tuple[torch.Tensor, torch.Tensor]:
    excl_ids = _need(excl_ids, torch.int64, "excl_ids")
    M, Lx = excl_ids.shape
    srt = torch.empty((M, Lx), dtype=torch.int32, device=excl_ids.device)
    cnt = torch.empty((M,), dtype=torch.int32, device=excl_ids.device)
    check(lib().irs_sort_exclusions(_ptr(excl_ids), M, Lx, item_base, n_cols, _ptr(srt), _ptr(cnt), _stream()), "sort_exclusions")
    return srt, cnt


def exclusions_update(excl: Tuple[torch.Tensor, torch.Tensor], removed, inserted, n_cols: int, item_base: int = 1) -> None:
    """In place: one window step of the sorted exclusion lists -- ``removed`` [M] (may be a strided column view, e.g.
    windows[:, 0]) slides out, ``inserted`` [M] (the picks) comes in."""
    srt, cnt = excl
    M, Lx = srt.shape
    if removed.dtype != torch.int64 or inserted.dtype != torch.int64 or not removed.is_cuda:
        raise TypeError("exclusions_update: removed / inserted must be CUDA int64 tensors")
    inserted = inserted.contiguous()
    check(lib().irs_exclusions_update(_ptr(srt), _ptr(cnt), _ptr(removed), removed.stride(0), _ptr(inserted), M, Lx, item_base,
                                      n_cols, _stream()), "exclusions_update")


def _rows(h):
    if not h.is_cuda or h.dtype != torch.float32:
        raise RuntimeError("influentialrs_b200: h must be a CUDA float32 tensor")
    if h.dim() != 2 or h.stride(1) != 1:
        h = h.reshape(-1, h.shape[-1]).contiguous()
    return h, h.stride(0)


def _excl(excl):
    """C arguments (sorted ids, counts, Lx) of an exclusion state from sort_exclusions; None = no exclusions."""
    return (None, None, 0) if excl is None else (_ptr(excl[0]), _ptr(excl[1]), excl[0].shape[1])


def _workspace(nbytes: int, like: torch.Tensor) -> torch.Tensor:
    return torch.empty((nbytes,), dtype=torch.uint8, device=like.device)


def _no_rows(h, k: int):
    """(vals [0,k], items [0,k]) of a scorer call without rows: nothing to launch, whichever engine it would pick."""
    return (torch.empty((0, k), dtype=torch.float32, device=h.device),
            torch.empty((0, k), dtype=torch.int64, device=h.device))


# ---- which engine scores a call ------------------------------------------------------------------------------------
# The dispatching ops (score_argmax, score_topk_any, score_rank, score_count_ahead, score_lse_gather and the softmax-CE
# backward) choose between the tcgen05 kernels and the fp32 CUDA-core engine with these rules and nothing else, and take
# the tcgen05 weight image from prepared_scorer_weights.  The arg-max rule is scorer_tc_supported(d).
# Below TC_TOPK_MIN_ITEMS the two-kernel tcgen05 top-k loses to the fp32 engine (measured r2: N=3,706 x 1,024 users, k=50:
# 0.55 ms vs 0.14 ms -- the catalog is 15 tiles, the launch is latency; N=1M x 8,192 users, d=256: 19.6 ms vs 214 ms).
TC_TOPK_MIN_ITEMS = 32768
TC_THREE_MMA_MAX_D = 128    # the three-MMA (hi/lo split) kernels hold hi and lo images of h only for d <= 128
USE_TC_TOPK = True          # top-k (k > 1) on the tensor cores where the shape allows (tests flip each flag to compare)
USE_TC_LSE = True           # log-sum-exp over the catalog on the tensor cores when d <= TC_THREE_MMA_MAX_D
USE_TC_RANK = True          # rank / count-ahead by counting on the tensor cores when d <= TC_THREE_MMA_MAX_D
USE_TC_CE_BWD = True        # softmax-CE backward on the tensor cores when d <= TC_THREE_MMA_MAX_D


def _tc_topk(d: int, k: int, N: int) -> bool:
    # May differ between the catalog shards of one call (their sizes differ by a row): harmless, there is no collective
    # inside the top-k and both engines return the same values, ids and tie order.
    return USE_TC_TOPK and score_topk_tc_supported(d, k) and N >= TC_TOPK_MIN_ITEMS


def _tc_three_mma(flag: bool, d: int) -> bool:
    return flag and d <= TC_THREE_MMA_MAX_D


@_timed("topk")
def score_topk(h, W, bias, k: int = 1, excl: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, item_base: int = 1):
    """Top-k (score desc, item id asc) of h W^T + bias per row among non-excluded items.
    Returns (vals [M,k] f32, items [M,k] i64).  Logits never reach HBM."""
    h, ld = _rows(h)
    W = _need(W, torch.float32, "W")
    M, d = h.shape
    N = W.shape[0]
    vals = torch.empty((M, k), dtype=torch.float32, device=h.device)
    items = torch.empty((M, k), dtype=torch.int64, device=h.device)
    ws = _workspace(lib().irs_score_topk_workspace_bytes(M, N, d, k), h)
    check(lib().irs_score_topk(_ptr(h), ld, _ptr(W), _ptr(bias), item_base, *_excl(excl), k,
                               _ptr(vals), _ptr(items), M, N, d, _ptr(ws), ws.numel(), _stream()), "score_topk")
    return vals, items


def score_topk_any(h, W, bias, k: int = 1, excl=None, item_base: int = 1):
    """Top-k through the fastest engine that covers the shape: the tcgen05 scorer (same values, ids and tie order as the
    fp32 engine) when available, else ``score_topk`` (fp32 CUDA cores)."""
    if h.numel() == 0:
        return _no_rows(h, k)
    if _tc_topk(h.shape[-1], k, W.shape[0]):
        return score_topk_tc(h, W, prepared_scorer_weights(W), bias, k, excl, item_base)
    return score_topk(h, W, bias, k, excl, item_base)


def score_topk_tc_supported(d: int, k: int) -> bool:
    return 1 <= k <= 1024 and scorer_tc_supported(d)


@_timed("topk")
def score_topk_tc(h, W, prepared, bias, k: int, excl=None, item_base: int = 1):
    """Top-k on the tensor cores (d <= 256): chunk maxima from one bf16 tcgen05 MMA per K step, radix-select of the k-th
    largest, exact fp32 re-score of the chunks inside the rounding bound.  Same (vals, items) as score_topk."""
    h, ld = _rows(h)
    W = _need(W, torch.float32, "W")
    M, d = h.shape
    N = W.shape[0]
    vals = torch.empty((M, k), dtype=torch.float32, device=h.device)
    items = torch.empty((M, k), dtype=torch.int64, device=h.device)
    if M == 0:
        return vals, items
    ws = _workspace(lib().irs_score_topk_tc_workspace_bytes(M, N, d, k), h)
    check(lib().irs_score_topk_tc(_ptr(h), ld, _ptr(W), _ptr(prepared), _ptr(bias), item_base, *_excl(excl), k,
                                  _ptr(vals), _ptr(items), M, N, d, _ptr(ws), ws.numel(), _stream()), "score_topk_tc")
    return vals, items


_prepared_scorer_cache = {}


def prepared_scorer_weights(W) -> torch.Tensor:
    """W [N,d] re-tiled for the tcgen05 scorer family, cached per (address, shape) and weight version (cached_image):
    training changes the weights every step (one extra pass over W), inference prepares once.  A catalog shard W[lo:hi]
    gets its own entry next to W's, and shares W's version counter, so an optimizer step on W reaches it too."""
    key = (W.data_ptr(), tuple(W.shape))
    if key not in _prepared_scorer_cache and len(_prepared_scorer_cache) >= 4:
        _prepared_scorer_cache.clear()
    return cached_image(_prepared_scorer_cache, key, (W,), lambda: scorer_prepare_weights(W.detach()))


@_timed("lse")
def score_lse_gather(h, W, bias, sel, item_base: int = 1):
    """(lse [M], logit [M,s]) with logit[m,t] = score of item sel[m,t] (0.0 for an id outside [item_base, item_base + N),
    PAD = 0 included)."""
    h, ld = _rows(h)
    W = _need(W, torch.float32, "W")
    M, d = h.shape
    N = W.shape[0]
    sel = _need(sel.reshape(M, -1 if M else sel.shape[-1]), torch.int64, "sel")      # -1 is ambiguous without rows
    s = sel.shape[1]
    lse = torch.empty((M,), dtype=torch.float32, device=h.device)
    logit = torch.empty((M, s), dtype=torch.float32, device=h.device)
    if M == 0:
        return lse, logit
    if _tc_three_mma(USE_TC_LSE, d):
        ws = _workspace(lib().irs_score_lse_gather_tc_workspace_bytes(M, N, d), h)
        check(lib().irs_score_lse_gather_tc(_ptr(h), ld, _ptr(W), _ptr(prepared_scorer_weights(W)), _ptr(bias), item_base,
                                            _ptr(sel), s, _ptr(lse), _ptr(logit), M, N, d, _ptr(ws), ws.numel(), _stream()),
              "score_lse_gather_tc")
        return lse, logit
    ws = _workspace(lib().irs_score_lse_gather_workspace_bytes(M, N, d, s), h)
    check(lib().irs_score_lse_gather(_ptr(h), ld, _ptr(W), _ptr(bias), item_base, _ptr(sel), s, _ptr(lse), _ptr(logit),
                                     M, N, d, _ptr(ws), ws.numel(), _stream()), "score_lse_gather")
    return lse, logit


@_timed("rank")
def score_rank(h, W, bias, label, excl=None, item_base: int = 1) -> torch.Tensor:
    """1-based rank of ``label`` among non-excluded items (0 if the label is excluded)."""
    h, ld = _rows(h)
    W = _need(W, torch.float32, "W")
    M, d = h.shape
    N = W.shape[0]
    label = _need(label.reshape(-1), torch.int64, "label")
    rank = torch.empty((M,), dtype=torch.int64, device=h.device)
    if M == 0:
        return rank
    if _tc_three_mma(USE_TC_RANK, d):
        ws = _workspace(lib().irs_score_rank_tc_workspace_bytes(M, N, d), h)
        check(lib().irs_score_rank_tc(_ptr(h), ld, _ptr(W), _ptr(prepared_scorer_weights(W)), _ptr(bias), item_base,
                                      _ptr(label), *_excl(excl), _ptr(rank), M, N, d, _ptr(ws), ws.numel(), _stream()),
              "score_rank_tc")
        return rank
    ws = _workspace(lib().irs_score_rank_workspace_bytes(M, N, d), h)
    check(lib().irs_score_rank(_ptr(h), ld, _ptr(W), _ptr(bias), item_base, _ptr(label), *_excl(excl),
                               _ptr(rank), M, N, d, _ptr(ws), ws.numel(), _stream()), "score_rank")
    return rank


class _SoftmaxCE(torch.autograd.Function):
    """mean_m [ lse(h_m W^T + b) - (h_m W^T + b)[target_m] ] with logits recomputed in backward."""

    @staticmethod
    def forward(ctx, h, W, bias, target):
        lse, logit = score_lse_gather(h, W, bias, (target + 1).reshape(-1, 1), item_base=1)
        ctx.save_for_backward(h, W, bias, target, lse)
        return (lse - logit[:, 0]).mean()

    @staticmethod
    def backward(ctx, g):
        h, W, bias, target, lse = ctx.saved_tensors
        M, d = h.shape
        N = W.shape[0]
        d_h = torch.empty_like(h)
        d_W = torch.zeros_like(W)
        d_b = torch.zeros_like(bias) if bias is not None else None
        if M == 0:                                   # no non-pad target row in the batch: zero gradients
            return d_h, d_W, d_b, None
        gscale = float(g) / M                        # upstream gradient of the mean (a host read: the C ABI takes a float)
        ev = None
        if _timer is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
            _timer.setdefault("ce_bwd", []).append(ev)
        try:
            return _SoftmaxCE._backward(h, W, bias, target, lse, gscale, d_h, d_W, d_b, M, N, d)
        finally:
            if ev is not None:
                ev[1].record()

    @staticmethod
    def _backward(h, W, bias, target, lse, gscale, d_h, d_W, d_b, M, N, d):
        if _tc_three_mma(USE_TC_CE_BWD, d):
            ws = _workspace(lib().irs_score_ce_bwd_tc_workspace_bytes(M, N, d), h)
            check(lib().irs_score_ce_bwd_tc(_ptr(h), h.stride(0), _ptr(W), _ptr(bias), _ptr(target), _ptr(lse), gscale,
                                            _ptr(d_h), _ptr(d_W), _ptr(d_b), M, N, d, _ptr(ws), ws.numel(), _stream()),
                  "score_ce_bwd_tc")
            return d_h, d_W, d_b, None
        check(lib().irs_score_ce_bwd(_ptr(h), h.stride(0), _ptr(W), _ptr(bias), _ptr(target), _ptr(lse), gscale,
                                     _ptr(d_h), _ptr(d_W), _ptr(d_b), M, N, d, _stream()), "score_ce_bwd")
        return d_h, d_W, d_b, None


def softmax_ce_mean(h, W, bias, target) -> torch.Tensor:
    """Mean cross-entropy of rows h [M,d] against 0-based classes ``target`` [M] over the catalog
    W [N,d] (+bias), without materialising [M,N] logits in either direction."""
    h = _need(h, torch.float32, "h")
    target = _need(target, torch.int64, "target")
    if h.shape[0] == 0:
        # a batch without a single non-pad target row: the reference's CrossEntropyLoss over zero rows is NaN; return a
        # NaN loss that still backpropagates zeros, so that a data-parallel rank in this state does not dead-lock the
        # others' all-reduce by raising
        return (h.sum() + W.sum() * 0 + (bias.sum() * 0 if bias is not None else 0)) * 0 + float("nan")
    return _SoftmaxCE.apply(h, W, bias, target)


def score_select(h, W, bias, sel, item_base: int = 1) -> torch.Tensor:
    """Exact fp32 scores [M,s] of the items ``sel`` [M,s]; -inf for PAD (0) and for items outside this catalog shard
    [item_base, item_base + N) -- a MAX all-reduce over the shards yields every score."""
    h, ld = _rows(h)
    W = _need(W, torch.float32, "W")
    M, d = h.shape
    sel = _need(sel.reshape(M, -1), torch.int64, "sel")
    out = torch.empty(sel.shape, dtype=torch.float32, device=h.device)
    check(lib().irs_score_select(_ptr(h), ld, _ptr(W), _ptr(bias), item_base, _ptr(sel), sel.shape[1], _ptr(out), M, W.shape[0], d,
                                 _stream()), "score_select")
    return out


@_timed("rank")
def score_count_ahead(h, W, bias, label, label_score, excl=None, item_base: int = 1):
    """(count [M] int64, label_excluded [M] int32): items of THIS catalog shard ahead of (label_score, label id); the label
    may belong to another shard.  rank = 0 if any shard flags the label, else 1 + sum of the counts.  The engine is chosen
    as in score_rank -- the same integers either way."""
    h, ld = _rows(h)
    W = _need(W, torch.float32, "W")
    M, d = h.shape
    N = W.shape[0]
    label = _need(label.reshape(-1), torch.int64, "label")
    label_score = _need(label_score.reshape(-1), torch.float32, "label_score")
    count = torch.empty((M,), dtype=torch.int64, device=h.device)
    flag = torch.empty((M,), dtype=torch.int32, device=h.device)
    if M == 0:
        return count, flag
    if _tc_three_mma(USE_TC_RANK, d):
        ws = _workspace(lib().irs_score_rank_tc_workspace_bytes(M, N, d), h)
        check(lib().irs_score_count_ahead_tc(_ptr(h), ld, _ptr(W), _ptr(prepared_scorer_weights(W)), _ptr(bias), item_base,
                                             _ptr(label), _ptr(label_score), *_excl(excl), _ptr(count), _ptr(flag), M, N, d,
                                             _ptr(ws), ws.numel(), _stream()), "score_count_ahead_tc")
        return count, flag
    ws = _workspace(lib().irs_score_count_ahead_workspace_bytes(M, N, d), h)
    check(lib().irs_score_count_ahead(_ptr(h), ld, _ptr(W), _ptr(bias), item_base, _ptr(label), _ptr(label_score),
                                      *_excl(excl), _ptr(count), _ptr(flag), M, N, d, _ptr(ws), ws.numel(), _stream()),
          "score_count_ahead")
    return count, flag


def topk_merge(vals, items):
    """[G,M,k] per-shard candidates -> best k per row (score desc, item id asc)."""
    vals = _need(vals, torch.float32, "vals")
    items = _need(items, torch.int64, "items")
    G, M, k = vals.shape
    ov = torch.empty((M, k), dtype=torch.float32, device=vals.device)
    oi = torch.empty((M, k), dtype=torch.int64, device=vals.device)
    check(lib().irs_topk_merge(_ptr(vals), _ptr(items), G, M, k, _ptr(ov), _ptr(oi), _stream()), "topk_merge")
    return ov, oi


@_timed("sample")
def topk_sample(vals, items, seed: int, step: int, row_key):
    """One draw per row from the softmax over the k best candidates (score desc, item id asc) of ``vals`` / ``items``
    [G,M,k] (per-shard lists as all-gathered) or [M,k] (G = 1).  The draw is a pure function of (seed, step, row_key[m])
    and of the merged list, so it does not depend on G, on the device or on how rows are tiled (include/irs_b200.h states
    the exact definition).  Returns items [M] int64: -1 for a row with no live candidate, -2 for a row that carries the
    overflow marker of score_topk."""
    vals = _need(vals, torch.float32, "vals")
    items = _need(items, torch.int64, "items")
    row_key = _need(row_key, torch.int64, "row_key")
    if vals.dim() == 2:
        vals, items = vals.unsqueeze(0), items.unsqueeze(0)
    G, M, k = vals.shape
    if tuple(items.shape) != (G, M, k) or row_key.shape != (M,):
        raise ValueError(f"topk_sample: items {tuple(items.shape)} and row_key {tuple(row_key.shape)} must be "
                         f"[{G},{M},{k}] and [{M}]")
    out = torch.empty((M,), dtype=torch.int64, device=vals.device)
    if M == 0:
        return out
    check(lib().irs_topk_sample(_ptr(vals), _ptr(items), G, M, k, int(seed) & (2 ** 64 - 1), int(step), _ptr(row_key),
                                _ptr(out), _stream()), "topk_sample")
    return out


def window_shift(seq, nxt, paths=None, step: int = 0) -> None:
    """In place: seq[b] <- [seq[b,1:L-1], nxt[b], seq[b,L-1]]; paths[b,step] = nxt[b]."""
    B, L = seq.shape
    P = 0 if paths is None else paths.shape[1]
    check(lib().irs_window_shift(_ptr(seq), _ptr(nxt), _ptr(paths), B, L, P, step, _stream()), "window_shift")


# ------------------------------------------------------------------------------------------------
# tensor-core (tcgen05) arg-max scorer
# ------------------------------------------------------------------------------------------------
def scorer_prepare_weights(W) -> torch.Tensor:
    """Re-tile the catalog matrix W [N,d] (d <= 256) into the bf16 hi/lo shared-memory image the
    tcgen05 scorer streams (one 32 KB bulk copy per stage).  Do this once per weight version."""
    W = _need(W, torch.float32, "W")
    N, d = W.shape
    nbytes = lib().irs_scorer_prepared_bytes(N, d)
    if nbytes == 0:
        raise RuntimeError(f"tcgen05 scorer supports d <= 256 (got d={d})")
    out = torch.empty((nbytes,), dtype=torch.uint8, device=W.device)
    check(lib().irs_scorer_prepare_weights(_ptr(W), N, d, _ptr(out), _stream()), "scorer_prepare_weights")
    return out


def scorer_tc_supported(d: int) -> bool:
    """Embedding sizes the tcgen05 scorer family covers (asked of the library, not hard-coded here)."""
    return lib().irs_scorer_prepared_bytes(256, int(d)) > 0


ARGMAX_VARIANT = 2          # 2: single bf16 MMA + rigorous error band (production); 0: three MMAs (hi/lo split)


@_timed("scorer")
def score_argmax_tc(h, W, prepared, bias, excl=None, item_base: int = 1, variant: Optional[int] = None):
    """Arg-max (k = 1) of h W^T + bias among non-excluded items on the tensor cores.
    Returns (vals [M,1], items [M,1]) -- same contract and same winners as score_topk(k=1)."""
    h, ld = _rows(h)
    M, d = h.shape
    N = W.shape[0]
    vals = torch.empty((M, 1), dtype=torch.float32, device=h.device)
    items = torch.empty((M, 1), dtype=torch.int64, device=h.device)
    ws = _workspace(lib().irs_score_argmax_tc_workspace_bytes(M, N, d), h)
    check(lib().irs_score_argmax_tc(_ptr(h), ld, _ptr(W), _ptr(prepared), _ptr(bias), item_base, *_excl(excl),
                                    _ptr(vals), _ptr(items), M, N, d, ARGMAX_VARIANT if variant is None else variant, _ptr(ws),
                                    ws.numel(), _stream()), "score_argmax_tc")
    return vals, items


_pending_phase1 = None      # (start, stop) events of the last timed phase-1 call: merged into the phase-2 record


def score_argmax_tc_phase1(h, W, prepared, bias, excl=None, item_base: int = 1, variant: Optional[int] = None):
    """Phase 1 of the catalog-sharded arg-max: returns (lead [M+1] float32, workspace).  lead[:M] = this shard's best
    tensor-core score per row, lead[M] = its rounding-error scale; max-reduce ``lead`` over the shards, then call
    ``score_argmax_tc_phase2`` with the reduced vector and the same workspace."""
    h, ld = _rows(h)
    M, d = h.shape
    N = W.shape[0]
    lead = torch.empty((M + 1,), dtype=torch.float32, device=h.device)
    ws = _workspace(lib().irs_score_argmax_tc_workspace_bytes(M, N, d), h)
    global _pending_phase1
    ev = None
    if _timer is not None:
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        ev[0].record()
    check(lib().irs_score_argmax_tc_phase1(_ptr(h), ld, _ptr(W), _ptr(prepared), _ptr(bias), item_base, *_excl(excl),
                                           _ptr(lead), M, N, d, ARGMAX_VARIANT if variant is None else variant, _ptr(ws),
                                           ws.numel(), _stream()), "score_argmax_tc_phase1")
    if ev is not None:
        ev[1].record()
    _pending_phase1 = ev
    return lead, ws


def score_argmax_tc_phase2(h, W, prepared, bias, excl, item_base, lead_global, ws, variant: Optional[int] = None):
    """Phase 2: exact re-scoring against the global leaders.  Returns (vals [M,1], items [M,1]); rows whose winner cannot
    be in this shard come back as (-inf, -1)."""
    h, ld = _rows(h)
    M, d = h.shape
    N = W.shape[0]
    lead_global = _need(lead_global, torch.float32, "lead_global")
    vals = torch.empty((M, 1), dtype=torch.float32, device=h.device)
    items = torch.empty((M, 1), dtype=torch.int64, device=h.device)
    global _pending_phase1
    ev = None
    if _timer is not None:
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        ev[0].record()
    check(lib().irs_score_argmax_tc_phase2(_ptr(h), ld, _ptr(W), _ptr(prepared), _ptr(bias), item_base, *_excl(excl),
                                           _ptr(lead_global), _ptr(vals), _ptr(items), M, N, d,
                                           ARGMAX_VARIANT if variant is None else variant, _ptr(ws), ws.numel(), _stream()),
          "score_argmax_tc_phase2")
    if ev is not None:
        ev[1].record()
        # one "scorer" record per step: the two kernels' intervals, without the max-reduction between them
        _timer.setdefault("scorer", []).append(((_pending_phase1 or ()) + ev))
        _pending_phase1 = None
    return vals, items


def score_argmax(h, W, bias, excl=None, item_base: int = 1, reduce_lead=None):
    """Arg-max (k = 1) of h W^T + bias among non-excluded items: (vals [M,1], items [M,1]), the same as score_topk(k=1).
    On the tensor cores when scorer_tc_supported(d), else on the fp32 engine.

    ``reduce_lead``: W is this rank's shard of a catalog split over ranks that all score the same rows h.  The tcgen05
    engine then runs in two phases around ``reduce_lead(lead)``, which must MAX-reduce ``lead`` over the ranks in place,
    so that only the shard that can hold a row's winner re-scores it exactly; rows won in another shard come back as
    (-inf, -1).  So the engine must depend on d alone, never on N: the tcgen05 branch holds that collective, and the
    shards of one catalog differ in size by a row, so a rule on N could leave one rank out of it."""
    if h.numel() == 0:
        return _no_rows(h, 1)
    if not scorer_tc_supported(h.shape[-1]):
        return score_topk(h, W, bias, 1, excl, item_base)
    prep = prepared_scorer_weights(W)
    if reduce_lead is None:
        return score_argmax_tc(h, W, prep, bias, excl, item_base)
    lead, ws = score_argmax_tc_phase1(h, W, prep, bias, excl, item_base)
    reduce_lead(lead)
    return score_argmax_tc_phase2(h, W, prep, bias, excl, item_base, lead, ws)


# ------------------------------------------------------------------------------------------------
# tensor-core (tcgen05) linear layers with fused epilogues
# ------------------------------------------------------------------------------------------------
EPI_BIAS, EPI_BIAS_RELU, EPI_RESID_LN = 0, 1, 2
def linear_supported(Nout: int, K: int) -> bool:
    return 0 < Nout <= 256 and 0 < K <= 256 and K % 4 == 0


def linear_prepare(W) -> torch.Tensor:
    """Re-tile a weight matrix W [Nout,K] (Nout, K <= 256) for linear_tc.  Once per weight version."""
    W = _need(W, torch.float32, "W")
    Nout, K = W.shape
    nbytes = lib().irs_linear_prepared_bytes(Nout, K)
    if nbytes == 0:
        raise RuntimeError(f"linear_tc supports Nout,K <= 256 (got {Nout}x{K})")
    out = torch.empty((nbytes,), dtype=torch.uint8, device=W.device)
    check(lib().irs_linear_prepare_weights(_ptr(W), Nout, K, _ptr(out), _stream()), "linear_prepare_weights")
    return out


def linear_tc(A, prepared, Nout: int, bias=None, epilogue: int = EPI_BIAS, resid=None, g1=None, b1=None, c2=None,
              g2=None, b2=None, eps: float = 1e-5, out=None) -> torch.Tensor:
    """out[R,Nout] = epilogue(A[R,K] W^T) on the tensor cores.  ``A``/``out`` may be column slices of
    wider row-major buffers (stride(0) is the leading dimension)."""
    if not A.is_cuda or A.dtype != torch.float32 or A.dim() != 2 or A.stride(1) != 1:
        raise RuntimeError("linear_tc: A must be a 2-D CUDA float32 tensor with unit inner stride")
    R, K = A.shape
    if out is None:
        out = torch.empty((R, Nout), dtype=torch.float32, device=A.device)
    if resid is not None and (resid.dim() != 2 or resid.stride(1) != 1 or resid.stride(0) % 4 != 0
                              or resid.data_ptr() % 16 != 0):
        # the kernel reads resid rows with 16-byte vector loads: a fresh copy is aligned (contiguous() would return a
        # misaligned contiguous view unchanged)
        resid = resid.clone(memory_format=torch.contiguous_format)
    check(lib().irs_linear_tc(_ptr(A), A.stride(0), _ptr(prepared), _ptr(bias), int(epilogue),
                              _ptr(resid), 0 if resid is None else resid.stride(0), _ptr(g1), _ptr(b1), _ptr(c2), _ptr(g2),
                              _ptr(b2), float(eps), _ptr(out), out.stride(0), R, K, Nout, _ptr(_error_flag(A.device)),
                              _stream()), "linear_tc")
    return out


# ------------------------------------------------------------------------------------------------
# fused decoder-layer chain (out_proj+LN1+LN2 -> FFN+LN3 -> next in_proj) in one tcgen05 kernel
# ------------------------------------------------------------------------------------------------
def decoder_chain_supported(d: int, ffn: int) -> bool:
    return bool(lib().irs_decoder_chain_supported(int(d), int(ffn)))


def decoder_chain_prepare(Wo, W1, W2, Win=None) -> torch.Tensor:
    """Re-tile out_proj / linear1 / linear2 (/ next in_proj) weights into the stream the fused
    decoder-chain kernel consumes.  Once per weight version."""
    Wo, W1, W2 = _need(Wo, torch.float32, "Wo"), _need(W1, torch.float32, "W1"), _need(W2, torch.float32, "W2")
    if Win is not None:
        Win = _need(Win, torch.float32, "Win")
    d, ffn = Wo.shape[0], W1.shape[0]
    nbytes = lib().irs_decoder_chain_prepared_bytes(d, ffn, 0 if Win is None else 1)
    if nbytes == 0:
        raise RuntimeError(f"decoder_chain supports d=128, ffn=256 (got d={d}, ffn={ffn})")
    out = torch.empty((nbytes,), dtype=torch.uint8, device=Wo.device)
    check(lib().irs_decoder_chain_prepare_weights(_ptr(Wo), _ptr(W1), _ptr(W2), _ptr(Win), d, ffn, _ptr(out), _stream()),
          "decoder_chain_prepare_weights")
    return out


@_timed("decoder_chain")
def decoder_chain_tc(attn, x, prepared, bo, g1, b1, c2, g2, b2, bf1, bf2, g3, b3, bin=None, eps=(1e-5, 1e-5, 1e-5),
                     ffn: int = 256, x_out=None, qkv_out=None, qkv_images=None, L: int = 0, mask_mode: int = MASK_PIM):
    """(x', qkv') of one decoder layer's row-local chain; qkv' is None unless ``bin`` is given (the
    prepared stream must then contain the next layer's in_proj).  With ``qkv_images`` (a zero-initialised
    operand-image buffer for windows of L positions) qkv' is written in the attention kernel's operand
    layout instead of fp32 rows and the images tensor is returned in its place."""
    attn = _need(attn, torch.float32, "attn")
    x = _need(x, torch.float32, "x")
    d = x.shape[-1]
    R = x.numel() // d
    if x_out is None:
        x_out = torch.empty_like(x)
    if bin is not None and qkv_out is None and qkv_images is None:
        qkv_out = torch.empty((*x.shape[:-1], 3 * d), dtype=torch.float32, device=x.device)
    if bin is None:
        qkv_out = qkv_images = None
    check(lib().irs_decoder_chain_tc(_ptr(attn), _ptr(x), _ptr(prepared), _ptr(bo), _ptr(g1), _ptr(b1), _ptr(c2), _ptr(g2),
                                     _ptr(b2), _ptr(bf1), _ptr(bf2), _ptr(g3), _ptr(b3), _ptr(bin),
                                     float(eps[0]), float(eps[1]), float(eps[2]), _ptr(x_out),
                                     _ptr(qkv_out) if qkv_images is None else None, _ptr(qkv_images), int(L), int(mask_mode),
                                     R, d, int(ffn), _ptr(_error_flag(x.device)), _stream()), "decoder_chain_tc")
    return x_out, (qkv_images if qkv_images is not None else qkv_out)


@_timed("decoder_chain")
def in_proj_images_tc(x, prepared_with_in_proj, bin, qkv_images, L: int, mask_mode: int = MASK_PIM):
    """First layer's in_proj written straight into operand images: qkv = x Win^T + bin."""
    x = _need(x, torch.float32, "x")
    d = x.shape[-1]
    check(lib().irs_in_proj_images_tc(_ptr(x), _ptr(prepared_with_in_proj), _ptr(bin), _ptr(qkv_images), int(L), int(mask_mode),
                                      x.numel() // d, d, _ptr(_error_flag(x.device)), _stream()), "in_proj_images_tc")
    return qkv_images
