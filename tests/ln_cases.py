"""Rows that are hard for a LayerNorm, fp32 emulators of how the kernels compute its statistics, and the error band.

Every LayerNorm of the inference decoder runs in an epilogue: ``irs_linear_tc`` epilogue 2 (one thread owns a row of
Nout <= 256 columns, read in 32-column chunks), the decoder-chain kernel (two threads own 64 columns each of a 128-wide
row and exchange their statistics) and the fp32 ``irs_residual_layernorm`` (a warp per row).  The one-pass variance
E[t^2] - mean^2 loses about u (mean/std)^2 of the variance (u = 2^-24): a row whose mean is large next to its spread gets
the wrong scale, and once the difference goes negative the row is scaled by eps^-1/2.  Zero-mean Gaussian rows never show
it; the rows below do:

* mean/std in RATIOS, both signs, interleaved with well-conditioned rows (a statistic read from the wrong row shows up);
* constant rows (exact output: b);
* a row with one outlier feature;
* a row whose two 64-column halves have different means (the merge of the halves' statistics matters).

The offset sits where an implementation adds it: in the row input (``x`` / ``resid``, placement "row") or in a per-column
bias shared by every row (``y_bias`` / ``bias`` / ``bo`` / ``c2`` / ``bf2``, placement "bias").

The band (``ln_band``) bounds |out - LN(t)| per row, LN in fp64 of the exact t:
  KAPPA u (max_j |t_j| rstd max|g| + max|b|)   -- what holding t (and the output) in fp32 costs any implementation;
  + MARGIN G(K) P rstd max|g|                 -- tensor-core paths: the bf16x3 product error of a K-deep GEMM,
                                                 P = max_j sum_k |a_k w_jk| (G and MARGIN: tests/gemm_cases.py);
  + e rstd max|g| (2 + max_j |z_j|)           -- an error e of t from upstream (LN2 after LN1, LN3 after the FFN).
KAPPA comes from the two-pass and Chan emulators below (KAPPA_MARGIN times the largest ratio they reach on these
cases, tests/test_layernorm_cond_cpu.py), not from GPU output.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np

from tests.gemm_cases import band_rel

U = 2.0 ** -24                  # fp32 unit roundoff
KAPPA = 24.0                    # >= KAPPA_MARGIN x the largest error of the emulators in units of the band: 11.1
KAPPA_MARGIN = 2.0
RATIOS = (1.0, 10.0, 30.0, 100.0, 1e3, 1e4)
DISCRIMINATING = 30.0           # the one-pass statistics leave the band at every |mean|/std >= this


# ---------------------------------------------------------------------------------------------- cases
@dataclass
class Rows:
    name: str
    x: np.ndarray               # [R, n] float32: the row input (x of residual_layernorm / resid of linear_tc / x of the chain)
    bias: np.ndarray            # [n] float32: the per-column offset (zero for placement "row")
    scale: np.ndarray           # [R] float64: the spread (std) of each row, for sizing a product term small next to it
    ratio: np.ndarray           # [R] float64: |mean| / std of t (inf: constant row)

    @property
    def t64(self) -> np.ndarray:
        return self.x.astype(np.float64) + self.bias.astype(np.float64)


def ln_rows(n: int, placement: str, sign: float = 1.0, R: int = 200, seed: int = 0, common: float = 200.0) -> Rows:
    """R rows of width n.  Even rows cycle through the ill-conditioned kinds, odd rows are well conditioned
    (|mean|/std <= 0.1).  placement "row": the offset of each row is in ``x``; "bias": one offset ``sign * common`` for all
    rows sits in ``bias``, and each row's spread sets its ratio."""
    rng = np.random.default_rng(seed + 1000 * n + (0 if placement == "row" else 7) + (0 if sign > 0 else 3))
    kinds = [(r, s) for r in RATIOS for s in (1.0, -1.0)] + ["const", "outlier", "split"]
    x = np.zeros((R, n))
    scale = np.zeros(R)
    ratio = np.zeros(R)
    col = sign * common if placement == "bias" else 0.0
    for i in range(R):
        kind = kinds[(i // 2) % len(kinds)] if i % 2 == 0 else "well"
        if placement == "row":
            sigma = float(np.exp(rng.uniform(-2.0, 2.0)))
        else:
            r = {"well": 10.0 * rng.uniform(1.0, 3.0), "const": np.inf, "outlier": 100.0, "split": 300.0}.get(kind) \
                if not isinstance(kind, tuple) else kind[0]
            sigma = common / r
        z = rng.standard_normal(n)
        z = (z - z.mean()) / z.std()
        if kind == "well":
            off = 0.1 * rng.uniform(-1, 1) * sigma
        elif kind == "const":
            z[:] = 0.0
            off = 37.3 if placement == "row" else 0.0
        elif kind == "outlier":
            z[n // 3] += 0.4 * np.sqrt(n)
            off = 100.0 * sigma
        elif kind == "split":
            z[: n // 2] -= 3.0
            z[n // 2:] += 3.0
            off = 300.0 * sigma
        else:
            off = kind[0] * kind[1] * sigma
        if placement == "bias":
            off = 0.0
        x[i] = z * sigma + off
        scale[i] = sigma
    x32 = x.astype(np.float32)
    bias = np.full(n, col, dtype=np.float32)
    t = x32.astype(np.float64) + bias.astype(np.float64)
    sd = t.std(1)
    with np.errstate(divide="ignore"):
        ratio = np.where(sd > 0, np.abs(t.mean(1)) / np.where(sd > 0, sd, 1.0), np.inf)
    return Rows(f"{placement}{'+' if sign > 0 else '-'}n{n}", x32, bias, np.where(scale > 0, scale, 1.0), ratio)


def ln_params(n: int, seed: int = 0):
    """(g, b) of a LayerNorm: g ~ 1 +- 0.1, b ~ 0.1 N(0, 1), float32."""
    rng = np.random.default_rng(seed + 77 * n)
    return ((1 + 0.1 * rng.standard_normal(n)).astype(np.float32), (0.1 * rng.standard_normal(n)).astype(np.float32))


# ---------------------------------------------------------------------------------------------- reference and band
def ln64(t64: np.ndarray, g, b, eps: float) -> np.ndarray:
    m = t64.mean(1, keepdims=True)
    v = ((t64 - m) ** 2).mean(1, keepdims=True)
    return (t64 - m) / np.sqrt(v + eps) * np.asarray(g, np.float64) + np.asarray(b, np.float64)


def ln_band(t64: np.ndarray, g, b, eps: float, prod: Optional[np.ndarray] = None, k: Optional[int] = None,
            upstream: Optional[np.ndarray] = None) -> np.ndarray:
    """Per-row bound on |out - ln64(t64)| (module docstring).  ``prod`` [R]: product scale of a tensor-core GEMM of depth
    ``k`` inside t; ``upstream`` [R]: a bound on the error of t itself."""
    m = t64.mean(1, keepdims=True)
    rstd = 1.0 / np.sqrt(((t64 - m) ** 2).mean(1) + eps)
    gmax = float(np.abs(np.asarray(g, np.float64)).max())
    bmax = float(np.abs(np.asarray(b, np.float64)).max())
    band = KAPPA * U * (np.abs(t64).max(1) * rstd * gmax + bmax)
    if prod is not None:
        band = band + band_rel(k) * prod * rstd * gmax
    if upstream is not None:
        zmax = (np.abs(t64 - m).max(1)) * rstd
        band = band + upstream * rstd * gmax * (2.0 + zmax)
    return band


def abs_prod(a, w) -> np.ndarray:
    """P = max_j sum_k |a_k w_jk| per row."""
    return (np.abs(np.asarray(a, np.float64)) @ np.abs(np.asarray(w, np.float64)).T).max(1)


def inf_norm(w) -> float:
    return float(np.abs(np.asarray(w, np.float64)).sum(1).max())


def chain_bands(attn, x, P, eps=1e-5):
    """fp64 decoder chain (out_proj + LN1 + LN2, linear1 + relu + linear2 + LN3, next in_proj) and the per-row bands of
    x' and qkv', each GEMM's error propagated with the band of its own depth (128, or 256 for linear2).  P holds the
    float32 parameters by name."""
    D = lambda k: np.asarray(P[k], np.float64)
    t1 = x.astype(np.float64) + attn.astype(np.float64) @ D("Wo").T + D("bo")
    band1 = ln_band(t1, P["g1"], P["b1"], eps, prod=abs_prod(attn, P["Wo"]), k=128)
    t2 = ln64(t1, P["g1"], P["b1"], eps) + D("c2")
    band2 = ln_band(t2, P["g2"], P["b2"], eps, upstream=band1)
    y = ln64(t2, P["g2"], P["b2"], eps)
    f = np.maximum(y @ D("W1").T + D("bf1"), 0.0)
    e_f = inf_norm(P["W1"]) * band2 + band_rel(128) * abs_prod(y, P["W1"]) + 2 * U * np.abs(f).max(1)  # relu: 1-Lipschitz
    t3 = y + f @ D("W2").T + D("bf2")
    band3 = ln_band(t3, P["g3"], P["b3"], eps, prod=abs_prod(f, P["W2"]), k=256, upstream=band2 + inf_norm(P["W2"]) * e_f)
    xo = ln64(t3, P["g3"], P["b3"], eps)
    qkv = xo @ D("Win").T + D("bin")
    band_q = inf_norm(P["Win"]) * band3 + band_rel(128) * abs_prod(xo, P["Win"]) + 2 * U * np.abs(qkv).max(1)
    return xo, band3, qkv, band_q


def row_err(out, want) -> np.ndarray:
    return np.abs(np.asarray(out, np.float64) - np.asarray(want, np.float64)).max(1)


# ---------------------------------------------------------------------------------------------- fp32 emulators
def _fma(a, b, c):
    """fp32 fused multiply-add: the product is exact in fp64, one rounding of the sum (double rounding is rare)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(np.float32)


def _combine(p):
    return p[0] if len(p) == 1 else (p[0] + p[1]) + (p[2] + p[3])


def _seq_sum(t, ways=1):
    """Sum of each row, column j into partial sum j % ways (ways 1 or 4, combined as the kernels do)."""
    p = [np.zeros(t.shape[0], np.float32) for _ in range(ways)]
    for j in range(t.shape[1]):
        p[j % ways] = p[j % ways] + t[:, j]
    return _combine(p)


def _seq_sq(t, c, ways=1):
    p = [np.zeros(t.shape[0], np.float32) for _ in range(ways)]
    for j in range(t.shape[1]):
        e = t[:, j] - c
        p[j % ways] = _fma(e, e, p[j % ways])
    return _combine(p)


def _f(x):
    return np.float32(x)


def stats(t: np.ndarray, method: str, layout: str, eps: float):
    """(mean, rstd, centre) in fp32 of rows t [R, n] float32 as a kernel computes them; ``centre`` [R, n] is the value the
    kernel normalises (t - mean, or t - the half mean for the pair layout).
    method: "one-pass" (E[t^2] - mean^2, clamped at 0, sequential sums), "two-pass" (sequential sums), "chan" (per-chunk
    two-pass in four partial sums + Chan's merge, as the tensor-core kernels);
    layout: "row" (one thread, 32-column chunks: linear_tc), "pair" (two threads of 64 columns: the decoder chain),
    "warp" (two-pass only: lane-strided sums and a butterfly, residual_layernorm)."""
    R, n = t.shape
    inv_n = _f(1.0) / _f(n)
    if method == "one-pass":
        parts = [t] if layout == "row" else [t[:, : n // 2], t[:, n // 2:]]
        s1 = np.zeros(R, np.float32)
        s2 = np.zeros(R, np.float32)
        for p in parts:
            a, b = np.zeros(R, np.float32), np.zeros(R, np.float32)
            for j in range(p.shape[1]):
                a = a + p[:, j]
                b = _fma(p[:, j], p[:, j], b)
            s1, s2 = s1 + a, s2 + b
        mean = s1 * inv_n
        rstd = (_f(1.0) / np.sqrt(np.maximum(s2 * inv_n - mean * mean, _f(0.0)) + _f(eps))).astype(np.float32)
        return mean, rstd, (t - mean[:, None]).astype(np.float32)
    if method == "two-pass" and layout == "warp":     # layernorm.cu: lane-strided sums, then a butterfly over the warp
        def warp_sum(v):
            p = np.zeros((R, 32), np.float32)
            for c in range(n):
                p[:, c % 32] = p[:, c % 32] + v[:, c]
            for s in (16, 8, 4, 2, 1):
                p = p + p[:, np.arange(32) ^ s]
            return p[:, 0]
        mean = warp_sum(t) / _f(n)
        e = t - mean[:, None]
        q = warp_sum(e * e)
        rstd = (_f(1.0) / np.sqrt(q / _f(n) + _f(eps))).astype(np.float32)
        return mean, rstd, e.astype(np.float32)
    if method == "two-pass":
        mean = _seq_sum(t) * inv_n
        q = _seq_sq(t, mean)
        rstd = (_f(1.0) / np.sqrt(q * inv_n + _f(eps))).astype(np.float32)
        return mean, rstd, (t - mean[:, None]).astype(np.float32)
    if layout == "pair":                      # decoder_chain_tc.cu ln_pair_stats
        h = n // 2
        ma, mb = _seq_sum(t[:, :h], 4) * _f(1.0 / h), _seq_sum(t[:, h:], 4) * _f(1.0 / h)
        qa, qb = _seq_sq(t[:, :h], ma, 4), _seq_sq(t[:, h:], mb, 4)
        delta = mb - ma
        mean = _f(0.5) * (ma + mb)
        m2 = _fma(_f(h * h / n) * delta, delta, qa + qb)
        rstd = (_f(1.0) / np.sqrt(m2 * inv_n + _f(eps))).astype(np.float32)
        centre = np.concatenate([t[:, :h] - ma[:, None], t[:, h:] - mb[:, None]], 1).astype(np.float32)
        return mean, rstd, (centre, np.concatenate([np.repeat((ma - mean)[:, None], h, 1),
                                                    np.repeat((mb - mean)[:, None], n - h, 1)], 1).astype(np.float32))
    cnt, mean, m2 = np.zeros(R, np.float32), np.zeros(R, np.float32), np.zeros(R, np.float32)
    for c0 in range(0, n, 32):                 # gemm_tc.cu chan_merge
        c = t[:, c0:c0 + 32]
        nb = _f(c.shape[1])
        cm = _seq_sum(c, 4) / nb
        cq = _seq_sq(c, cm, 4)
        nn = cnt + nb
        delta = cm - mean
        w = nb / nn
        mean = _fma(delta, w, mean)
        m2 = m2 + (cq + delta * delta * (cnt * w))
        cnt = nn
    rstd = (_f(1.0) / np.sqrt(m2 * inv_n + _f(eps))).astype(np.float32)
    return mean, rstd, (t - mean[:, None]).astype(np.float32)


def emulate_ln(t: np.ndarray, g, b, eps: float, method: str, layout: str) -> np.ndarray:
    """fp32 LayerNorm of rows t [R, n] float32 with the statistics of ``stats``, normalised as the kernel does: the
    chain as fma(fma(c, rstd, shift), g, b), linear_tc as (t - mean) rstd g + b."""
    g, b = np.asarray(g, np.float32), np.asarray(b, np.float32)
    mean, rstd, centre = stats(t, method, layout, eps)
    if layout == "pair":
        if method == "chan":
            c, shift = centre
            return _fma(_fma(c, rstd[:, None], shift * rstd[:, None]), g, b)
        return _fma(_fma(t, rstd[:, None], -mean[:, None] * rstd[:, None]), g, b)
    return _fma(centre * rstd[:, None], g, b)


def emulate_input(rows: Rows, prod64: np.ndarray) -> np.ndarray:
    """t as the kernels form it in fp32: (acc + bias) + x, acc the fp32 product."""
    return (prod64.astype(np.float32) + rows.bias) + rows.x
