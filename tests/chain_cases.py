"""Inputs that pin one GEMM stage of the fused decoder chain, and a float64 emulator of the chain's x'.

A LayerNorm with g = 0 outputs exactly its b, so g2 = 0 pins the FFN's input y = b2, and a zero weight matrix with a zero
bias takes a GEMM out.  The stages below are seen only through LN3 (x'), and a LayerNorm removes any error that is
parallel to its input's mean or to the input's own deviation from it.  An error that the three MMAs make coherently
(every product of a worst-rounding row rounded the same way) is close to proportional to the GEMM's output, so each stage
adds a large spread across the columns (+-SPREAD alternating, in y, bf2 or x) that is not parallel to it: the error then
reaches x' and the LN3 band (``ln_cases.chain_bands``) can tell the kernel's arithmetic from one that drops a term
(tests/test_chain_cases_cpu.py).

  linear2     W1 = 0 and bf1 = X3 2^e: the relu output f is exactly a worst-rounding row, read by linear2 (K = 256)
              against worst-rounding columns; y = b2 = +-SPREAD.
  linear1+    y = b2 = X3 rows (all products of the worst+ columns round the same way) through linear1 (K = 128), and a
  linear1+-   0/1 selection W2 (each x' column reads one hidden unit, so ||W2||_inf = 1); bf2 = +-SPREAD.
  out_proj    hard attn rows (gemm_cases.ROW_KINDS) through Wo (K = 128) and LN1, Wo's worst+ columns mirrored by
              negated ones; the FFN off, LN2 and LN3 with g = 1, b = 0; x = +-SPREAD.
"""
from __future__ import annotations

import numpy as np
import torch

from tests import gemm_cases as GC
from tests import ln_cases as C

D, F = 128, 256
SPREAD = 3e3
STAGES = ("linear2", "linear1+", "linear1+-", "out_proj")


def gauss_params(seed: int) -> dict:
    """N(0,1)-scaled parameters of one chain call (float32, by name)."""
    rng = np.random.default_rng(seed)
    f32 = lambda a: np.asarray(a, np.float32)
    rn = lambda *s: rng.standard_normal(s)
    return {"Wo": f32(rn(D, D) / np.sqrt(D)), "bo": f32(0.1 * rn(D)), "g1": f32(1 + 0.1 * rn(D)), "b1": f32(0.1 * rn(D)),
            "c2": f32(0.3 * rn(D)), "g2": f32(1 + 0.1 * rn(D)), "b2": f32(0.1 * rn(D)), "W1": f32(rn(F, D) / np.sqrt(D)),
            "bf1": f32(0.1 * rn(F)), "W2": f32(rn(D, F) / np.sqrt(F)), "bf2": f32(0.1 * rn(D)),
            "g3": f32(1 + 0.1 * rn(D)), "b3": f32(0.1 * rn(D)), "Win": f32(rn(3 * D, D) / np.sqrt(D)),
            "bin": f32(0.1 * rn(3 * D))}


def weights(N: int, K: int, scaled: bool = True):
    W, b, _ = GC.gemm_weights(N, K, scaled=scaled)
    return W.numpy(), b.numpy()


def row_of(kind: str, K: int) -> np.ndarray:
    A, rk = GC.gemm_rows(len(GC.ROW_KINDS), K)
    return A[GC.ROW_KINDS.index(kind)].numpy()


def _alternating(n: int) -> np.ndarray:
    return np.where(np.arange(n) % 2 == 0, SPREAD, -SPREAD).astype(np.float32)


def stage_case(stage: str, R: int = 333):
    """(attn, x, P, row kinds) of one chain call in which ``stage`` carries the error (module docstring)."""
    rng = np.random.default_rng(STAGES.index(stage))
    P = gauss_params(20 + STAGES.index(stage))
    attn = rng.standard_normal((R, D)).astype(np.float32)
    x = rng.standard_normal((R, D)).astype(np.float32)
    kinds = [stage] * R
    zD, zF = np.zeros(D, np.float32), np.zeros(F, np.float32)
    if stage == "linear2":
        P.update(g2=zD, b2=_alternating(D), W1=np.zeros((F, D), np.float32),
                 bf1=(GC.worst_pair()[0] * 2.0 ** (np.arange(F) % 9 - 4)).astype(np.float32))
        P["W2"], P["bf2"] = weights(D, F, scaled=False)
    elif stage.startswith("linear1"):
        P.update(g2=zD, b2=row_of("worst+" if stage == "linear1+" else "worst+-", D), bf2=_alternating(D))
        P["W1"], P["bf1"] = weights(F, D, scaled=False)
        W2 = np.zeros((D, F), np.float32)
        W2[np.arange(D), np.arange(D) * 2 + (np.arange(D) // 64)] = 1.0          # hidden units of every column kind
        P["W2"] = W2
    else:
        P["Wo"], P["bo"] = weights(D, D, scaled=False)
        # columns 2 mod 4 mirror the worst+ columns 0 mod 4: on a worst+ row the coherent error is then +e, -e on the
        # even columns, orthogonal to the mean and to x's alternating spread, so LN1 passes all of it on
        P["Wo"][2::4], P["bo"][2::4] = -P["Wo"][0::4], 0.0
        P.update(c2=zD, g2=np.ones(D, np.float32), b2=zD, W1=np.zeros((F, D), np.float32), bf1=zF,
                 W2=np.zeros((D, F), np.float32), bf2=zD, g3=np.ones(D, np.float32), b3=zD)
        A, rk = GC.gemm_rows(R, D)
        attn = A.numpy()
        x = (_alternating(D)[None, :] + rng.standard_normal((R, D))).astype(np.float32)
        kinds = [GC.ROW_KINDS[k] for k in rk]
    return attn, x, P, kinds


def emulate_chain_x(attn, x, P, mode: str = "rn", terms=("lohi", "hilo", "hihi"), eps: float = 1e-5) -> np.ndarray:
    """x' of the chain with its GEMMs and their fp32 epilogue additions as the kernel does them (``gemm_cases.emulate``;
    ``terms`` drops products), the LayerNorms in float64 on the fp32 inputs (their own fp32 error is the KAPPA term of
    the band, checked in tests/test_layernorm_cond_cpu.py)."""
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    f32 = lambda a: np.asarray(a, np.float32)
    acc1 = GC.emulate(t(attn), t(P["Wo"]), t(P["bo"]), mode, terms).numpy()
    t1 = f32(acc1 + x)
    y1 = f32(C.ln64(t1.astype(np.float64), P["g1"], f32(P["b1"] + P["c2"]), eps))
    y = f32(C.ln64(y1.astype(np.float64), P["g2"], P["b2"], eps))
    f = np.maximum(GC.emulate(t(y), t(P["W1"]), t(P["bf1"]), mode, terms).numpy(), 0)
    t3 = f32(GC.emulate(t(f), t(P["W2"]), t(P["bf2"]), mode, terms).numpy() + y)
    return C.ln64(t3.astype(np.float64), P["g3"], P["b3"], eps)
