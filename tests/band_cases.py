"""Worst-case inputs for the error bands of the tensor-core scorers, and a float64 emulator of what those kernels compute.

Every tensor-core decision in the library (K5c arg-max ``irs_score_argmax_tc`` and its catalog-sharded phases, K5e top-k
``irs_score_topk_tc``, K5d rank ``irs_score_rank_tc`` / ``irs_score_count_ahead_tc``) is one tensor-core pass followed by
an exact fp32 re-score of the items whose tensor-core score lies inside an error band.  An item outside the band is never
re-scored, so the answer is only right if the band bounds the gap between tensor-core and fp32 scores.  Gaussian data uses a
few percent of a worst-case band; the constructions below use all of it:

* bf16 keeps 8 significant bits, unit roundoff u = 2^-8.  ``C_DN`` rounds down and ``C_UP`` rounds up by almost u, so a
  hi*hi product of two of them is off by almost 2u, all terms of a score the same way.
* ``X3`` is the fp32 value whose three-MMA product X3*X3 (hi*hi + hi*lo + lo*hi) loses the most (``worst_three_mma_value``
  finds it): 2u^2 relative, ~3.0e-5.

A case holds (h, W, bias, excl, expected); ``analyse_*`` computes, on the case's distinct rows, the fp64 and fp32-engine
answers and how far the emulated tensor-core scores sit outside the old band and inside the corrected one.
"""
from __future__ import annotations

import functools
import math
from dataclasses import dataclass, field
from typing import List, Optional

import torch

U = 2.0 ** -8                     # bf16 unit roundoff (8 significant bits, round to nearest even)
BAND_REL = 1e-4                   # floor of every arg-max / top-k band: band_rel * max(1, |s|)
# single_mma_band(): bound on how far two hi*hi scores may swap, times |h_m| max_j |W_j|
OLD_SINGLE = 0.00837              # before: derived from a per-operand error of 2^-9
NEW_SINGLE = 0.016                # 2 (2u + u^2) = 2^-5.99 plus accumulation margin (scorer_tc.cu)
# three_mma_band(): bound on |s_three_mma - s_fp32_engine|, times |h_m| max_j |W_j| (d <= 128)
OLD_THREE = 5e-5
OLD_THREE_LOST = 3 * 2.0 ** -18   # what the old derivation budgeted for the dropped low-order terms
NEW_THREE = 5.7e-5                # 3u^2(1 + 2u) + 3*128/16*2^-23 (accumulation) + 128*2^-24 (engine)
RANK_REL = 1e-6                   # rank band: three_mma_band + 1e-6 |label score|

NUM_SMS, BM, BN, SEG_TILES, CHUNK = 148, 128, 256, 16, 32

C_DN = 1 + 2.0 ** -8 - 2.0 ** -20   # bf16: rounds down to 1
C_UP = 1 + 2.0 ** -8 + 2.0 ** -20   # bf16: rounds up to 1 + 2^-7
X3 = 1 + 2.0 ** -8 + 2.0 ** -17     # hi = 1 + 2^-7, lo = -2^-8 (a tie, to even), 2^-17 dropped
MARGIN = 1e-3                       # fp64 lead of the true winner in the single-MMA pairs (>> fp32 noise)
DELTA3 = 1e-2                       # fp64 lead in the three-MMA cases, whose scores pass through |s| ~ 1e3


# ---------------------------------------------------------------------------------------------- emulator
def bf16_rn(x: torch.Tensor) -> torch.Tensor:
    """Round to bf16, nearest even (as cvt.rn.bf16x2.f32 in split8), returned as float64."""
    return x.float().to(torch.bfloat16).double()


def split_hi_lo(x: torch.Tensor):
    """x = hi + lo + r with hi = bf16_rn(x), lo = bf16_rn(x - hi) (x - hi is exact in fp32)."""
    hi = bf16_rn(x)
    return hi, bf16_rn(x.double() - hi)


def _add_bias(acc: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    acc = acc.float()
    return acc if bias is None else (acc.double() + bias.double()).float()


def score_fp64(h, W, bias=None) -> torch.Tensor:
    s = h.double() @ W.double().t()
    return s if bias is None else s + bias.double()


def score_hihi(h, W, bias=None) -> torch.Tensor:
    """Single-MMA score: bf16 products summed exactly (fp64 stands in for the fp32 accumulator), + bias in fp32."""
    return _add_bias(bf16_rn(h) @ bf16_rn(W).t(), bias)


def score_three(h, W, bias=None) -> torch.Tensor:
    """Three-MMA score hi*hi + hi*lo + lo*hi, summed exactly, + bias in fp32."""
    hh, hl = split_hi_lo(h)
    wh, wl = split_hi_lo(W)
    return _add_bias(hh @ wh.t() + hh @ wl.t() + hl @ wh.t(), bias)


def score_fp32_engine(h, W, bias=None) -> torch.Tensor:
    """The CUDA-core engine and every exact re-score: one sequential fp32 FMA chain over k, then + bias.  Each FMA is
    emulated as fp64 (exact product) rounded to fp32, which is exact up to a rare double rounding."""
    hd, Wd = h.double(), W.double()
    acc = torch.zeros((h.shape[0], W.shape[0]), dtype=torch.float32)
    for k in range(h.shape[1]):
        acc = (acc.double() + hd[:, k:k + 1] * Wd[:, k].unsqueeze(0)).float()
    return _add_bias(acc, bias)


def old_single_band(hn2, wmax2):
    return OLD_SINGLE * math.sqrt(hn2 * wmax2)


def new_single_band(hn2, wmax2):
    return NEW_SINGLE * math.sqrt(hn2 * wmax2)


def old_three_band(hn2, wmax2):
    return OLD_THREE * math.sqrt(hn2 * wmax2)


def new_three_band(hn2, wmax2):
    return NEW_THREE * math.sqrt(hn2 * wmax2)


def plan(M: int, N: int):
    """(m_tiles, n_tiles, tiles_per_split, n_splits) exactly as plan() in scorer_tc.cu."""
    m_tiles = -(-M // BM)
    n_tiles = -(-N // BN)
    ctas = -(-(-(-(m_tiles * n_tiles) // 96)) // NUM_SMS) * NUM_SMS
    splits = min(max(ctas // m_tiles, 1), n_tiles)
    tps = -(-n_tiles // splits)
    return m_tiles, n_tiles, tps, -(-n_tiles // tps)


def locate(col: int, M: int, N: int):
    """(split, segment, 32-column chunk, column half) of a catalog column in the scorer's launch for M rows."""
    _, _, tps, _ = plan(M, N)
    tile = col // BN
    split = tile // tps
    return split, (tile - split * tps) // SEG_TILES, col // CHUNK, (col % BN) // (BN // 2)


def worst_three_mma_value(n: int = 3000):
    """Search fp32 values in [1, 2) (two bf16 hi values, every residual on the 2^-23 grid) for the pair whose three-MMA
    product loses the most.  Returns (x, y, relative error)."""
    base = torch.arange(0, 2 ** 16, dtype=torch.float64) * 2.0 ** -23
    x = torch.cat([1 + base, 1 + 2.0 ** -7 + base]).float()
    hi, lo = split_hi_lo(x)
    r = x.double() - hi - lo
    top = torch.topk((lo / x.double()).abs() * 2 ** 8 + (r / x.double()).abs() * 2 ** 16, n).indices
    xs, H, L = x[top].double(), hi[top], lo[top]
    ex = xs[:, None] * xs[None, :]
    rel = (H[:, None] * H[None, :] + H[:, None] * L[None, :] + L[:, None] * H[None, :] - ex) / ex
    i = int(rel.abs().argmax())
    a, b = divmod(i, rel.shape[1])
    return float(xs[a]), float(xs[b]), float(rel[a, b])


# ---------------------------------------------------------------------------------------------- cases
@dataclass
class Case:
    name: str
    kind: str                          # "argmax1" single-MMA pair, "argmax3" three-MMA pair, "topk", "rank"
    h: torch.Tensor                    # [M, d] float32
    W: torch.Tensor                    # [N, d] float32
    bias: Optional[torch.Tensor]       # [N] float32
    excl: Optional[torch.Tensor]       # [M, Lx] int64 item ids (1-based, 0 = padding)
    k: int
    expected: torch.Tensor             # arg-max / top-k: [M, k] item ids in fp64 order; rank: [M] ranks
    win: int = -1                      # 0-based columns of the true winner and the decoy
    decoy: int = -1
    rows: List[int] = field(default_factory=lambda: [0])     # distinct rows (every other row copies one of them)
    label: Optional[torch.Tensor] = None                     # rank: [M] item ids
    ahead: List[int] = field(default_factory=list)           # rank: columns truly ahead of the label / behind it
    behind: List[int] = field(default_factory=list)
    shard_at: int = 0                  # first column of the second catalog shard (sharded cases)

    @property
    def M(self):
        return self.h.shape[0]

    @property
    def N(self):
        return self.W.shape[0]

    @property
    def d(self):
        return self.h.shape[1]


def _signs(d, g):
    return torch.where(torch.rand(d, generator=g) < 0.5, -1.0, 1.0).double()


def _f32(x) -> float:
    return float(torch.tensor(float(x), dtype=torch.float32))


def _dot(a, b) -> float:
    return float((a.double() * b.double()).sum())


def _background(N, d, g, scale):
    return torch.randn((N, d), generator=g) * scale


def _leader(h, norm, i):
    """Aligned with h over its full support, |w| = norm * (1 - 1e-3 i): scores above a half-support or bias-lifted pair
    without raising max_j |W_j| (the band's scale)."""
    return (h.double() / h.double().norm() * norm * (1 - 1e-3 * i)).float()


def _single_pair(d, use_bias, g):
    """One row h and the pair (w, b) of the true winner and the decoy for the single-MMA (hi*hi) scorer."""
    sg = _signs(d, g)
    if use_bias:
        # h and w_win parallel, every element rounding down by ~u: hi*hi(h, w_win) = (1 - ~2u) h.w_win.  w_dec = -w_win
        # rounds the other way and is lifted by the bias to 2 h.w_win - MARGIN: the decoy leads by ~4u h.w_win on the
        # tensor core, and that is 2u |h| |W| by Cauchy-Schwarz equality
        h = (sg * C_DN).float()
        w = (sg * C_DN / 16).float()
        wd = -w
        P = _dot(h, w)
        return h, w, wd, 0.0, _f32(2 * P - MARGIN)
    # no bias: h rounds down on the even elements and up on the odd ones; the winner lives on the even elements (hi*hi
    # underestimates it by ~2u), the decoy on the odd ones (overestimated by ~2u).  The decoy's last element is lowered so
    # that the winner leads by MARGIN in fp64
    even = (torch.arange(d) % 2 == 0)
    h = (sg * torch.where(even, C_DN, C_UP)).float()
    w = torch.where(even, sg * C_DN / 16, torch.zeros(d, dtype=torch.float64)).float()
    wd = torch.where(~even, sg * C_UP / 16, torch.zeros(d, dtype=torch.float64))
    q = d - 1 if (d - 1) % 2 == 1 else d - 2
    wd[q] -= float(sg[q]) * (_dot(h, wd) - _dot(h, w) + MARGIN) / abs(float(h[q]))
    return h, w, wd.float(), None, None


def _rows(h, M, scales):
    s = torch.tensor([scales[m % len(scales)] for m in range(M)], dtype=torch.float32)
    return (h.unsqueeze(0) * s.unsqueeze(1)).contiguous(), list(range(min(M, len(scales))))


def _expected_topk(case_h, W, bias, excl, k):
    s = score_fp64(case_h, W, bias)
    if excl is not None:
        for m in range(s.shape[0]):
            ids = excl[m][excl[m] > 0] - 1
            s[m, ids] = -math.inf
    return torch.topk(s, k, dim=1).indices + 1


PLACEMENTS = ("segment", "segments", "splits", "tail", "excluded")


@functools.lru_cache(maxsize=None)
def argmax_pair(d: int, placement: str, use_bias: bool) -> Case:
    """Single-MMA arg-max: true winner j and decoy j' in different 32-column chunks, placed
    segment   -- the same 16-tile segment and column half (M = 6, N = 5000);
    segments  -- the same catalog split, segments >= 4096 columns apart (M = 2100, N = 70000: 8 splits of 35 tiles);
    splits    -- different catalog splits, rows in two user tiles (M = 130, N = 70000);
    tail      -- j in the ragged last chunk of a catalog of 5013 items;
    excluded  -- an item above both, in j's chunk, hidden by the row's exclusion list (plus random exclusions)."""
    g = torch.Generator().manual_seed(1000 + d * 10 + PLACEMENTS.index(placement) * 2 + int(use_bias))
    M, N, win, decoy = {"segment": (6, 5000, 37, 101), "segments": (2100, 70000, 1000, 5608),
                        "splits": (130, 70000, 500, 60000), "tail": (6, 5013, 5010, 2000),
                        "excluded": (6, 5000, 37, 101)}[placement]
    h0, w, wd, bw, bd = _single_pair(d, use_bias, g)
    W = _background(N, d, g, 2.0 ** -8)
    W[win], W[decoy] = w, wd
    bias = None
    if use_bias:
        bias = -0.1 * torch.rand(N, generator=g)
        bias[win], bias[decoy] = bw, bd
    # rows: without a bias, power-of-two scalings of the adversarial row (rounding is scale invariant); with one, copies
    h, rows = _rows(h0, M, [1.0] if use_bias else [1.0, 2.0, 0.5])
    excl = None
    if placement == "excluded":
        x = 40                                                       # j's chunk
        W[x] = _leader(h0, min(w.norm(), wd.norm()), 0)
        if use_bias:
            bias[x] = 1.0
        excl = torch.randint(1, N + 1, (M, 8), generator=g)
        excl[excl == win + 1] = 0
        excl[excl == decoy + 1] = 0
        excl[:, 0] = x + 1
        excl[:, 3] = 0
    expected = _expected_topk(h, W, bias, excl, 1)
    return Case(f"argmax1-{placement}-d{d}-{'bias' if use_bias else 'nobias'}", "argmax1", h, W, bias, excl, 1, expected,
                win, decoy, rows)


@functools.lru_cache(maxsize=None)
def sharded_pair(d: int, use_bias: bool) -> Case:
    """Single-MMA arg-max with j in the first of two catalog shards and j' in the second (phase 1 -> MAX -> phase 2 ->
    topk_merge): the first shard must re-score j against the global leader j'."""
    g = torch.Generator().manual_seed(2000 + d * 10 + int(use_bias))
    M, N, win, decoy = 6, 9000, 37, 4500 + 101
    h0, w, wd, bw, bd = _single_pair(d, use_bias, g)
    W = _background(N, d, g, 2.0 ** -8)
    W[win], W[decoy] = w, wd
    bias = None
    if use_bias:
        bias = -0.1 * torch.rand(N, generator=g)
        bias[win], bias[decoy] = bw, bd
    h, rows = _rows(h0, M, [1.0] if use_bias else [1.0, 2.0, 0.5])
    return Case(f"sharded-d{d}-{'bias' if use_bias else 'nobias'}", "argmax1", h, W, bias, None, 1,
                _expected_topk(h, W, bias, None, 1), win, decoy, rows, shard_at=4500)


@functools.lru_cache(maxsize=None)
def topk_boundary(d: int, k: int, use_bias: bool, N: int = 5000) -> Case:
    """Top-k: k-1 clear leaders in chunks of their own, then the pair at ranks k (j) and k+1 (j'), hi*hi order reversed.
    N >= 32768 puts the call through score_topk_any's own dispatch."""
    g = torch.Generator().manual_seed(3000 + d * 100 + k * 2 + int(use_bias) + N)
    M = 5
    win, decoy = (37, 101) if N < 32768 else (1000, N - 7000)
    h0, w, wd, bw, bd = _single_pair(d, use_bias, g)
    W = _background(N, d, g, 2.0 ** -8)
    W[win], W[decoy] = w, wd
    bias = None
    if use_bias:
        bias = -0.1 * torch.rand(N, generator=g)
        bias[win], bias[decoy] = bw, bd
    used = {win // CHUNK, decoy // CHUNK}
    chunks = [c for c in range(8, N // CHUNK) if c not in used][: k - 1]
    r = float(min(w.norm(), wd.norm()))
    for i, c in enumerate(chunks):
        W[c * CHUNK + 5] = _leader(h0, r, i)
        if use_bias:
            bias[c * CHUNK + 5] = 1.0
    h, rows = _rows(h0, M, [1.0] if use_bias else [1.0, 2.0, 0.5])
    return Case(f"topk-k{k}-d{d}-N{N}-{'bias' if use_bias else 'nobias'}", "topk", h, W, bias, None, k,
                _expected_topk(h, W, bias, None, k), win, decoy, rows)


def _three_row(d, g):
    """h = +-4 X3 and the scale of the aligned item w = +-X3 2^e chosen so that |h| |W| = d X3^2 2^(2+e) is in [1e3, 1e4]."""
    sg = _signs(d, g)
    e = next(e for e in range(-4, 12) if d * X3 * X3 * 2.0 ** (2 + e) >= 1e3)
    return sg, (sg * X3 * 4).float(), (sg * X3 * 2.0 ** e).float()


@functools.lru_cache(maxsize=None)
def argmax_three(d: int) -> Case:
    """Three-MMA arg-max (variants 0, 4, ...) with |h| |W| ~ 2e3 and |s| ~ 1: w_win = X3-aligned (three-MMA loses
    ~2u^2 of every product, all the same way), biased down to s = 1; w_dec = -w_win, biased up to s = 1 - DELTA3.  The
    decoy leads by ~4u^2 |h| |W| ~ 0.06 on the tensor cores, far outside the old band 1e-4 max(1, |s|)."""
    g = torch.Generator().manual_seed(4000 + d)
    M, N, win, decoy = 6, 5000, 37, 101
    _, h0, w = _three_row(d, g)
    P = _dot(h0, w)
    W = _background(N, d, g, 2.0 ** -8)
    W[win], W[decoy] = w, -w
    bias = -2.0 - 0.1 * torch.rand(N, generator=g)
    bias[win], bias[decoy] = _f32(1.0 - P), _f32(1.0 + P - DELTA3)
    h, rows = _rows(h0, M, [1.0])
    return Case(f"argmax3-d{d}", "argmax3", h, W, bias, None, 1, _expected_topk(h, W, bias, None, 1), win, decoy, rows)


@functools.lru_cache(maxsize=None)
def rank_three(d: int, crowded: bool) -> Case:
    """Rank: items truly ahead of the label whose three-MMA score errs low, items truly behind it whose score errs high,
    each by ~2u^2 |h| |W| (X3-aligned weights, |h| |W| ~ 2e3) against a true distance to the label of DELTA3 .. 4 DELTA3.
    The three-MMA error alone cannot leave the old rank band (it reaches ~0.6 of 5e-5 |h| |W|; it is ~2.6x the old budget
    of 3 2^-18 for the dropped terms) -- only the tensor core's accumulation can push it out, which this case detects.
    crowded: all 40 of them in one (split, column half) slice, beyond its 30-entry list (the slice is counted exactly)."""
    g = torch.Generator().manual_seed(5000 + d * 2 + int(crowded))
    M, N, label = 4, 20000, 7000
    _, h0, w = _three_row(d, g)
    W = _background(N, d, g, 2.0 ** -8)
    bias = -5.0 - 0.1 * torch.rand(N, generator=g)
    bias[label] = 1.0
    lab = float(score_fp64(h0.unsqueeze(0), W[label:label + 1], bias[label:label + 1])[0, 0])
    cols = [3 * BN + i for i in range(40)] if crowded else [211 + 487 * i for i in range(40)]
    ahead, behind = [], []
    for i, c in enumerate(cols):
        wi = (w * 2.0 ** -(i % 3)).float()
        P = _dot(h0, wi)
        delta = DELTA3 * (1 + (i // 2) % 4)
        if i % 2 == 0:
            W[c], bias[c] = wi, _f32(lab - P + delta)
            ahead.append(c)
        else:
            W[c], bias[c] = -wi, _f32(lab + P - delta)
            behind.append(c)
    h, rows = _rows(h0, M, [1.0])
    labels = torch.full((M,), label + 1, dtype=torch.int64)
    s = score_fp64(h[:1], W, bias)[0]
    expected = torch.full((M,), 1 + int((s > s[label]).sum()), dtype=torch.int64)
    return Case(f"rank-d{d}-{'crowded' if crowded else 'spread'}", "rank", h, W, bias, None, 0, expected, rows=rows,
                label=labels, ahead=ahead, behind=behind, shard_at=N // 2)


# ---------------------------------------------------------------------------------------------- analysis
def _dead(case: Case, rows):
    dead = torch.zeros((len(rows), case.N), dtype=torch.bool)
    if case.excl is not None:
        for i, m in enumerate(rows):
            ids = case.excl[m][case.excl[m] > 0] - 1
            dead[i, ids] = True
    return dead


def _chunk_max(s, dead):
    s = s.double().masked_fill(dead, -math.inf)
    pad = (-s.shape[1]) % CHUNK
    s = torch.nn.functional.pad(s, (0, pad), value=-math.inf)
    return s.view(s.shape[0], -1, CHUNK).max(-1).values


@dataclass
class Analysis:
    fp64_top: torch.Tensor       # [R, k] item ids of the distinct rows, fp64
    engine_top: torch.Tensor     # [R, k] the same from the emulated fp32 engine
    old_ratio: float             # min over rows: (leader - the winner's chunk max) / old band, tensor-core scores
    new_ratio: float             # max over rows: the same / corrected band (must be < 1)
    fp64_margin: float           # min over rows: true lead of j over j' (fp64)


def analyse_pair(case: Case) -> Analysis:
    """Arg-max / top-k: does the winner's chunk fall below (leader - band), i.e. is it never re-scored?"""
    rows = case.rows
    h = case.h[rows]
    three = case.kind == "argmax3"
    tc = (score_three if three else score_hihi)(h, case.W, case.bias)
    dead = _dead(case, rows)
    cm = _chunk_max(tc, dead)
    lead = cm.topk(case.k, dim=1).values[:, -1]                 # arg-max: the leader; top-k: tau, the k-th chunk max
    gap = lead - cm[:, case.win // CHUNK]
    hn2 = (h.double() ** 2).sum(1)
    wmax2 = float((case.W.double() ** 2).sum(1).max())
    floor = BAND_REL * lead.abs().clamp(min=1.0)
    scale = (hn2 * wmax2).sqrt()
    old = floor + (0.0 if three else OLD_SINGLE * scale)
    new = floor + (2 * NEW_THREE * scale if three else NEW_SINGLE * scale)
    s64 = score_fp64(h, case.W, case.bias).masked_fill(dead, -math.inf)
    eng = score_fp32_engine(h, case.W, case.bias).double().masked_fill(dead, -math.inf)
    return Analysis(s64.topk(case.k, dim=1).indices + 1, eng.topk(case.k, dim=1).indices + 1,
                    float((gap / old).min()), float((gap / new).max()),
                    float((s64[:, case.win] - s64[:, case.decoy]).min()))


@dataclass
class RankAnalysis:
    fp64_rank: torch.Tensor      # [R]
    engine_rank: torch.Tensor    # [R] ranks the fp32 engine computes
    wrong_side: float            # max over the constructed items of how far the three-MMA score is on the wrong side of
                                 # the label's exact score
    old_ratio: float             # wrong_side / old rank band
    new_ratio: float             # max |s_three - s_engine| / corrected rank band
    lost_ratio: float            # max |s_three - s_fp64| / (3 2^-18 |h| |W|), the old budget for the dropped terms


def analyse_rank(case: Case) -> RankAnalysis:
    rows = case.rows
    h = case.h[rows]
    l = int(case.label[0]) - 1
    s64 = score_fp64(h, case.W, case.bias)
    eng = score_fp32_engine(h, case.W, case.bias)
    tc = score_three(h, case.W, case.bias)
    lab64, lab = s64[:, l:l + 1], eng[:, l:l + 1].double()
    a, b = case.ahead, case.behind
    wrong = torch.cat([lab - tc[:, a].double(), tc[:, b].double() - lab], 1).max(1).values
    hn2 = (h.double() ** 2).sum(1)
    scale = (hn2 * float((case.W.double() ** 2).sum(1).max())).sqrt()
    cols = a + b
    err = (tc[:, cols].double() - eng[:, cols].double()).abs().max(1).values
    lost = (tc[:, cols].double() - s64[:, cols]).abs().max(1).values
    e_old = OLD_THREE * scale + RANK_REL * lab.abs()[:, 0]
    e_new = NEW_THREE * scale + RANK_REL * lab.abs()[:, 0]
    ids = torch.arange(case.N)
    eng_ahead = (eng.double() > lab) | ((eng.double() == lab) & (ids < l))
    return RankAnalysis(1 + (s64 > lab64).sum(1), 1 + eng_ahead.sum(1), float(wrong.max()),
                        float((wrong / e_old).max()), float((err / e_new).max()),
                        float((lost / (OLD_THREE_LOST * scale)).min()))


def argmax_cases():
    return [argmax_pair(d, p, b) for d in (30, 64, 128) for p in PLACEMENTS for b in (True, False)]


def sharded_cases():
    return [sharded_pair(d, b) for d in (64, 128) for b in (True, False)]


def topk_cases():
    return [topk_boundary(d, k, b) for d in (30, 64, 128, 256) for k in (5, 50) for b in (True, False)]


def topk_any_case():
    return topk_boundary(128, 20, True, N=40000)


def three_cases():
    return [argmax_three(d) for d in (30, 64, 128)]


def rank_cases():
    return [rank_three(d, c) for d in (64, 128) for c in (False, True)]
