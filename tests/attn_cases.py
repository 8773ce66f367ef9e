"""Hard inputs for the PIM attention kernels, their float64 reference, per-row error bounds derived from each kernel's
arithmetic, and a float64 emulator of the persistent tensor-core kernel.

The attention of one (batch, head) item, in natural-log units (mask M of oracle/irn_oracle.py::pim_mask for mode 0, the
causal mask for modes 1 and 2, key padding -inf in modes 0 and 1):

    s_ij = q_i . k_j / sqrt(dh) + M_ij,   w_ij = softmax_j(s_ij),   o_i = sum_j w_ij v_j,   lse_i = log sum_j exp(s_ij)

The tensor-core kernels work in log2 units: q~ = fp32(q * qscale) with qscale = log2(e) / sqrt(dh), so sigma_ij =
s_ij log2(e) and b_ij = M_ij log2(e) is the additive bias.  A_ij = sum_t |q~_t k_jt| (log2 units) is the scale of the
score's rounding.  Symbols below: J = visible keys of row i, u = 2^-8 (bf16 unit roundoff), rho = RHO.

Cases (``hard_case``; regimes mixed inside every 128-row tile, a window regime per batch row):

* control   -- q, k, v ~ N(0,1): the old tests' data, so the bound can be compared with their tolerances;
* trained   -- keys around a shared direction (|k| ~ sqrt(dh)), rows whose component along it gives scores of tens of
               nats, an "attention sink" key that most rows favour (in PIM mode the objective column L-1), and rows of
               the regimes saturated (a leader ahead by 10, 30 and 60 log2 units, lifted as ce_cases does) and
               tie (two near-equal keys far above the rest);
* worst     -- q~ and k made of band_cases.X3 values with one sign pattern, so every q~_t k_jt of a key has one sign and
               the three-MMA error reaches 2u^2 A_ij coherently; in PIM mode the objective key is anti-aligned and its
               bias lifts it level with the aligned keys, so the two leaders err in opposite directions;
* v offset  -- trained q, k and v = c + w, |c| / |w| = 1e3 (c made of X3 values), one outlier key: the P.V rounding is
               then measured against sum_j w_j |v_j| ~ |c|, not against the spread of v;
* masks     -- pre-padded windows with 1 and L-2 PADs, only the objective visible (L-1 PADs), post-padded windows, an
               all-PAD window (NaN rows and NaN lse), the objective key PAD; objective weights r_u include +-40 and -80.

``threshold_case`` is the persistent kernel's shift-free shortcut (attention_tc2.cu): an item skips the row-max pass when
``1.02 sqrt(max|q~_hi|^2 max|k_hi|^2) + max|bias| <= 80``.  Its items land at 79..79.9 (shift-free, p up to 2^+-78) and
80.1..81 (exact pass) by the producer warp's own fp32 arithmetic (``producer_bound``), alternate between the two kinds
from one item to the next, and are more than 4 x 148 so that each CTA's two staging buffers carry both kinds.

Error model, per query row i (float64, from the reference; every term carries the factor MARGIN = 2 at the end):

1. score error E_ij (log2 units):
   * tensor cores (tcgen05 kernels, the persistent kernel, its one-row kernel): NEW_THREE A_ij -- the three-MMA
     product (band_cases.NEW_THREE: 3u^2(1+2u) dropped terms + TMEM accumulation) -- plus 4 2^-24 A_ij for the fp32
     rounding of q * qscale and of qscale itself (log2(e), sqrtf, the division); the one-row kernel rebuilds q~ and k
     as hi + lo (2u^2 A_ij, inside NEW_THREE);
   * fp32 kernels: (dh + 4) 2^-24 A_ij (the FMA chain over dh, the product with 1/sqrt(dh));
   * both: 2^-23 (2|sigma_ij| + |b_ij| + |sigma_ij - m_i|) for the bias addition, the subtraction of the row maximum
     m_i (0 on the shift-free path: |sigma - m| covers both) and the exponent's argument.
   E_i = max_{j in J} E_ij.
2. exponent: rho = 2^-22 relative, i.e. 2 ulp.  The CUDA C++ Programming Guide (appendix "Mathematical Functions",
   single-precision table) gives 2 ulp as the maximum error of expf and exp2f over the full range; for the intrinsic
   __expf it gives 2 + floor(|1.173 x|) ulp, of which 2 ulp are ex2.approx.ftz.f32 (the persistent kernel's
   exponent) and the rest the rounding of x log2(e), which item 1 already counts.
3. weights: with p^_j = p_j 2^{d_j} (1 + r_j), |d_j| <= E_i, |r_j| <= rho, the computed output is
       o^_i - o_i = (1/Z) sum_j w_j (2^{d_j}(1 + r_j) - 1)(v_j - o_i),   Z = sum_j w_j 2^{d_j}(1 + r_j) >= 2^-E_i (1 - rho)
   (sum_j w_j (v_j - o_i) = 0), so |o^_i - o_i| <= F_i sum_j w_j |v_j - o_i|,
       F_i = 2^E_i (2^E_i (1 + rho) - 1) / (1 - rho):
   the spread of v under the row's own softmax, not max|v|.  (This is the exact form of the first-order
   2^{2 E_i} (1 + rho)^2 - 1: the normalisation Z shares the error of the numerator.)
4. P.V and normalisation, times sum_j w_j |v_j| (n = key columns of the window):
   * tensor cores: P_hi.[V_hi | V_lo] + P_lo.V_hi drops P_lo V_lo and the residuals of both splits, 3u^2(1 + 2u) (the
     same product term as NEW_THREE); TMEM accumulation, one fp32 truncation of the running partial per K = 16 MMA
     (test_three_mma_accumulation_probe in tests/test_gpu_scorer_bands.py): 6 MMAs per 32 keys, 2^-23 each;
   * fp32 kernels: an FMA chain over the n keys, (n + 8) 2^-24; the key-blocked kernel also rescales its running
     output and sum once per 64-key block by expf (rho + 2 2^-24 each);
   * the one-row kernel: v rebuilt as hi + lo (u^2) and lane-parallel FMAs ((n/32 + 6) 2^-24, inside (n + 8) 2^-24);
   * all: the fp32 sum of the unrounded p over a chain of depth n + 8, (n + 8) 2^-24, and the final 1/sum and
     product, 2 2^-23; plus, absolutely, (n + 8) 2^-126 max_j |v_j| for weights below the smallest normal fp32 (the
     row maximum's weight is 1, and ex2.approx.ftz flushes smaller results to zero).
5. lse (natural log; kernels that return it): ln2 E_i + 2 rho + (n + 8) 2^-22 + 2^-22 (|lse| + ln2 |m_i| + 1), as
   ce_cases.forward_bound (log of a sum whose terms each move by at most E_i + rho, the fp32 sum, max + log).
6. backward (fp32 kernels; P recomputed from the lse the kernel received, D_i = dO_i . O_i from the out it received),
   element-wise from absolute-value sums as ce_cases.backward_bound:
       dP_ij <= P_ij (exp(ln2 E_ij(fp32) + rho + 2^-23 (|s_ij| + |lse_i|) + dlse_i) - 1),  dlse_i = the lse bound of
       the forward that produced lse (tcgen05 or fp32, items 1-5 without the margin);
       d(dp_ij) <= (dh + 1) 2^-24 sum_t |dO_it V_jt|;  dD_i <= sum_t |dO_it| dO_i + (dh + 1) 2^-24 sum_t |dO_it O_it|
       with dO_i the forward's out bound of row i;
       d(dS_ij) <= dP_ij (|dp_ij - D_i| + d(dp) + dD) + P_ij (d(dp) + dD) + 2^-23 |dS_ij|;
       dQ, dK = scale (d(dS) |K|, d(dS)^T |Q|) + L 2^-24 scale (|dS| |K|, |dS|^T |Q|) + 2^-23 |result|;
       dV = dP^T |dO| + L 2^-24 P^T |dO|;   d r_u[b] = |w_obj| sum_{h,i} (d(dS_{i,L-1}) + L 2^-24 |dS_{i,L-1}|);
       and the gradients' subnormal range: expf below 2^-149 is 0 and a subnormal result rounds to a multiple of
       2^-149, so dP, d(dS) and each of the L steps of every sum gain 2^-149 absolutely.

Every constant above comes from this derivation; none from a GPU measurement except the accumulation-probe figure (one
truncation per MMA) that NEW_THREE and item 4 reuse.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional

import torch

from tests.band_cases import C_DN, NEW_THREE, U, X3, bf16_rn, split_hi_lo
from tests.ce_cases import _bisect, f32, trunc32

W_H, W_OBJ = 0.05, 1.0
PIM, CAUSAL_PAD, CAUSAL = 0, 1, 2
U24, U23, U22 = 2.0 ** -24, 2.0 ** -23, 2.0 ** -22
FTZ, TINY = 2.0 ** -126, 2.0 ** -149   # smallest normal / subnormal fp32 (items 4 and 6 of the module docstring)
RHO = 2.0 ** -22                      # 2 ulp: expf, exp2f, ex2.approx.ftz.f32 (item 2 of the module docstring)
MARGIN = 2.0
LN2 = math.log(2.0)
L2E = float(torch.tensor(1.4426950408889634, dtype=torch.float32))       # log2(e) as the kernels hold it
NO_SHIFT_SAFE = 80.0                  # attention_tc2.cu: shift-free when the item's score bound is <= this
NUM_SMS = 148
C_PV_TC = 3 * U * U * (1 + 2 * U)     # item 4: the dropped u^2 terms of the two- / three-MMA P.V
ENGINES = ("fp32", "fp32_blocked", "tc", "tc_blocked", "img", "row")

# window regimes
CONTROL, TRAINED, WORST, VOFF = range(4)
_WINDOW_CYCLE = (TRAINED, WORST, VOFF, CONTROL)
# row regimes (inside trained / v-offset windows)
R_CONTROL, R_TRAINED, R_SAT10, R_SAT30, R_SAT60, R_TIE, R_WORST = range(7)
_ROW_CYCLE = (R_TRAINED, R_SAT10, R_SAT30, R_SAT60, R_TIE, R_CONTROL)
SAT_LEAD = {R_SAT10: 10.0, R_SAT30: 30.0, R_SAT60: 60.0}
# window masks (ids), cycled over the batch with a period prime to the regimes' so that they combine
MASKS = {PIM: ("none", "pre1", "pre_L-2", "post", "obj_only", "all_pad", "obj_pad"),
         CAUSAL_PAD: ("none", "pre1", "pre_L-2", "post", "all_pad"),
         CAUSAL: ("none",)}
TRAIN_MASKS = {PIM: ("none", "pre1", "pre_L-2", "obj_only", "obj_pad"), CAUSAL_PAD: ("none", "post"), CAUSAL: ("none",)}
_RU_CYCLE = (None, 40.0, -80.0, 2.0, -40.0)


@dataclass
class Case:
    name: str
    qkv: torch.Tensor                  # [B, L, 3 H dh] float32 (q | k | v, heads contiguous dh-slices)
    ids: torch.Tensor                  # [B, L] int64, 0 = PAD
    r_u: torch.Tensor                  # [B] float32 objective weight of each window
    H: int
    mode: int
    regime: torch.Tensor               # [B, H, L] int64 row regime
    window: torch.Tensor               # [B] int64 window regime
    shift_free: Optional[torch.Tensor] = None    # threshold case: [B*H] intended side of NO_SHIFT_SAFE

    @property
    def B(self):
        return self.qkv.shape[0]

    @property
    def L(self):
        return self.qkv.shape[1]

    @property
    def dh(self):
        return self.qkv.shape[2] // (3 * self.H)


# ---------------------------------------------------------------------------------------------- helpers
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _unit(v):
    return v / v.norm()


def qscale(dh: int) -> float:
    """log2(e) / sqrtf(dh) in fp32, as the tensor-core kernels and qkv_to_images compute it."""
    return float(torch.tensor(L2E, dtype=torch.float32) / torch.tensor(float(dh), dtype=torch.float32).sqrt())


def q_from_scaled(qt: torch.Tensor, dh: int) -> torch.Tensor:
    """fp32 q with fp32(q * qscale) == qt wherever an fp32 q reaches it (the nearest otherwise)."""
    qs = torch.tensor(qscale(dh), dtype=torch.float32)
    want = qt.float()
    q0 = (qt.double() / float(qs)).float()
    best = q0.clone()
    for cand in (torch.nextafter(q0, torch.full_like(q0, math.inf)), torch.nextafter(q0, torch.full_like(q0, -math.inf)), q0):
        best = torch.where((cand * qs) == want, cand, best)
    return best


def x_of(H: float) -> float:
    """H - 2^-8 + 2^-17 for an 8-bit mantissa H in (1, 2): bf16 hi = H, lo = -2^-8 (a tie, to even), 2^-17 dropped --
    the X3 construction (band_cases) with another hi.  x_of(1 + 2^-7) == X3."""
    return H - 2.0 ** -8 + 2.0 ** -17


def mask_bias(ids, r_u, L, mode, dtype=torch.float64):
    """[B, L, L] additive mask in natural-log units: oracle/irn_oracle.py::pim_mask (mode 0) or causal_mask, plus the
    key padding of modes 0 and 1."""
    from oracle import irn_oracle as O
    B = ids.shape[0]
    if mode == PIM:
        m = O.pim_mask(L, r_u.reshape(B, 1).to(dtype), W_H, W_OBJ).to(dtype)
    else:
        m = O.causal_mask(L, dtype).unsqueeze(0).expand(B, L, L)
    if mode != CAUSAL:
        m = m.masked_fill(ids.eq(0)[:, None, :], float("-inf"))
    return m


def _apply_mask(ids_row, kind, L):
    if kind == "pre1":
        ids_row[:1] = 0
    elif kind == "pre_L-2":
        ids_row[: max(L - 2, 0)] = 0
    elif kind == "obj_only":
        ids_row[: L - 1] = 0
    elif kind == "post":
        ids_row[L - L // 4:] = 0
    elif kind == "all_pad":
        ids_row.zero_()
    elif kind == "obj_pad":
        ids_row[L - 1] = 0


# ---------------------------------------------------------------------------------------------- cases
def _lift(q0, k, bias_row, vis, t, lead, dh, excl=()):
    """q0 + lam (k_t - mean_J k) with the key t ahead of every other visible key (outside excl) by ``lead`` log2
    units (None when out of reach)."""
    J = vis.nonzero().flatten()
    if J.numel() < 2 or not bool(vis[t]):
        return None
    d = _unit(k[t] - k[J].mean(0))
    others = vis.clone()
    others[t] = False
    for e in excl:
        others[e] = False
    if not bool(others.any()):
        return None
    rate = (k @ d) / math.sqrt(dh) * L2E
    s0 = ((k @ q0) / math.sqrt(dh) + bias_row) * L2E

    def f(lam):
        s = s0 + lam * rate
        return float(s[t] - s[others].max())
    lam = _bisect(f, lead, 1.0 if lead > f(0.0) else -1.0)
    return None if lam is None else q0 + lam * d


def _worst_window(g, L, dh, mode, obj_visible):
    """X3 rows and keys (module docstring, "worst"); returns (q~ target, k, v, r_u or None)."""
    sg = torch.where(torch.rand(dh, generator=g) < 0.5, -1.0, 1.0).double()
    n = round(math.log2(32.0 / (dh * X3 * X3)))                 # aligned top scores ~ 32 log2 units
    j = torch.arange(L)
    eps = torch.where(j % 2 == 0, 1.0, -1.0).double()
    m = (j // 2) % 3
    k = eps[:, None] * sg[None, :] * X3 * (2.0 ** -m.double())[:, None]
    i = torch.arange(L)
    eta = torch.where((i // 2) % 2 == 0, 1.0, -1.0).double()
    qt = eta[:, None] * sg[None, :] * X3 * (2.0 ** (n - (i % 2)).double())[:, None]
    r_u = None
    if mode == PIM and obj_visible:
        # the objective key anti-aligned; its bias lifts it level with the aligned keys (+s_a): -s_a + b = s_a
        k[L - 1] = -sg * X3
        s_a = dh * X3 * X3 * 2.0 ** n
        r_u = 2 * s_a / (L2E * W_OBJ)
    # a C_DN-made key (bf16 rounds it down by ~u): its hi x hi product errs the same way in every term
    if L > 4:
        k[3] = sg * C_DN
    v = torch.randn((L, dh), generator=g, dtype=torch.float64)
    return qt, k, v, r_u


def hard_case(B: int, L: int, H: int, dh: int, mode: int, seed: int, train: bool = False, windows=_WINDOW_CYCLE) -> Case:
    """All regimes and masks of the module docstring: window regime b % len(windows), mask b % len(masks), row regimes
    cycled inside trained and v-offset windows.  train: only masks under which every row sees a key."""
    g = _gen(seed)
    masks = (TRAIN_MASKS if train else MASKS)[mode]
    d = H * dh
    qkv = torch.zeros((B, L, 3 * d), dtype=torch.float64)
    ids = torch.randint(1, 1000, (B, L), generator=g)
    r_u = torch.randn(B, generator=g, dtype=torch.float64) * 0.7
    regime = torch.zeros((B, H, L), dtype=torch.int64)
    window = torch.zeros(B, dtype=torch.int64)
    qs = qscale(dh)
    for b in range(B):
        _apply_mask(ids[b], masks[b % len(masks)], L)
        ru = _RU_CYCLE[b % len(_RU_CYCLE)]
        if ru is not None:
            r_u[b] = ru
        wr = windows[b % len(windows)]
        window[b] = wr
        obj_visible = bool(ids[b, L - 1] != 0)
        for h in range(H):
            sl = slice(h * dh, (h + 1) * dh)
            if wr == WORST:
                qt, k, v, ru_w = _worst_window(g, L, dh, mode, obj_visible)
                if ru_w is not None:
                    r_u[b] = ru_w
                q = q_from_scaled(qt, dh).double()
                regime[b, h] = R_WORST
            elif wr == CONTROL:
                q = torch.randn((L, dh), generator=g, dtype=torch.float64)
                k = torch.randn((L, dh), generator=g, dtype=torch.float64)
                v = torch.randn((L, dh), generator=g, dtype=torch.float64)
                regime[b, h] = R_CONTROL
            else:
                u = _unit(torch.randn(dh, generator=g, dtype=torch.float64))
                beta = 0.3 * torch.randn(dh, generator=g, dtype=torch.float64)          # per-feature offset
                z = torch.randn((L, dh), generator=g, dtype=torch.float64)
                k = 0.5 * math.sqrt(dh) * u + 0.9 * z + beta
                sink = L - 1 if mode == PIM else 0
                k[sink] = 2.0 * math.sqrt(dh) * u + 0.3 * z[sink]
                if L > 3:
                    k[2] = k[1] + 1e-3 * torch.randn(dh, generator=g, dtype=torch.float64)   # near-tied pair
                c = torch.tensor([0.3, 0.6, 1.0], dtype=torch.float64)[torch.arange(L) % 3]
                q = c[:, None] * math.sqrt(dh) * u + torch.randn((L, dh), generator=g, dtype=torch.float64) + beta
                if wr == VOFF:
                    cv = 1e3 * X3 * torch.where(torch.rand(dh, generator=g) < 0.5, -1.0, 1.0).double()
                    w = torch.randn((L, dh), generator=g, dtype=torch.float64)
                    w[L // 2] *= 30.0                                                    # the outlier key
                    v = cv + w
                else:
                    v = torch.randn((L, dh), generator=g, dtype=torch.float64)
                rg = torch.tensor([_ROW_CYCLE[i % len(_ROW_CYCLE)] for i in range(L)])
                # lift the saturated and tie rows against the window's mask (float64, before the fp32 cast)
                mb = mask_bias(ids[b:b + 1], r_u[b:b + 1], L, mode)[0]
                kf = k.float().double()
                for i in range(L):
                    r = int(rg[i])
                    if r not in SAT_LEAD and r != R_TIE:
                        continue
                    vis = torch.isfinite(mb[i])
                    J = vis.nonzero().flatten().tolist()
                    if r == R_TIE:
                        new = _lift(q[i], kf, mb[i], vis, 1, 20.0, dh, excl=(2,)) if (1 in J and 2 in J) else None
                    else:
                        t = J[(i * 7) % len(J)] if J else 0
                        new = _lift(q[i], kf, mb[i], vis, t, SAT_LEAD[r], dh)
                    if new is None:
                        rg[i] = R_TRAINED
                    else:
                        q[i] = new
                regime[b, h] = rg
            qkv[b, :, sl] = q
            qkv[b, :, d + h * dh: d + (h + 1) * dh] = k
            qkv[b, :, 2 * d + h * dh: 2 * d + (h + 1) * dh] = v
    return Case(f"hard-B{B}-L{L}-H{H}-dh{dh}-m{mode}{'-train' if train else ''}", qkv.float().contiguous(), ids,
                r_u.float(), H, mode, regime, window)


def control_case(B: int, L: int, H: int, dh: int, mode: int, seed: int) -> Case:
    return hard_case(B, L, H, dh, mode, seed, windows=(CONTROL,))


# ---------------------------------------------------------------------------------------------- the persistent kernel's bound
def _fma_norm2(x, rows=False):
    """max over rows (rows=True: each row) of the producer warp's sum of squares: per 8-wide slab acc = fmaf(a0, a0, acc); fmaf(a1, a1, acc)
    over the 4 packed pairs, then (a[0] + a[1]) + (a[2] + a[3]) (x: bf16 hi values as float64, [R, 32])."""
    a = []
    for sl in range(4):
        acc = torch.zeros(x.shape[0], dtype=torch.float64)
        for e in range(8):
            acc = f32(acc + x[:, sl * 8 + e] * x[:, sl * 8 + e])        # bf16^2 is exact in float64: one rounding = fmaf
        a.append(acc)
    n2 = f32(f32(a[0] + a[1]) + f32(a[2] + a[3]))
    return n2 if rows else float(n2.max())


def _bound_of(q2, k2, babs):
    c = float(torch.tensor(1.02, dtype=torch.float32))
    return f32(f32(c * f32(torch.sqrt(f32(q2 * k2)))) + babs)


def producer_bound(qt_hi, k_hi, babs: float) -> float:
    """ks[0] of pim_attn_persistent_kernel: 1.02f * sqrtf(q2 * k2) + babs in fp32 (babs < 0: +inf)."""
    if babs < 0:
        return math.inf
    return float(_bound_of(torch.tensor(_fma_norm2(qt_hi), dtype=torch.float64), _fma_norm2(k_hi), babs))


def item_operands(case: Case, b: int, h: int):
    """(q~ [L, dh], k, v, column order, column bias kb [L] in log2 units) of one item as the tensor-core kernels see
    them: q~ = fp32(q * qscale); columns in kernel order (PIM: column 0 = the objective key L-1)."""
    L, dh, d = case.L, case.dh, case.H * case.dh
    q = case.qkv[b, :, h * dh:(h + 1) * dh]
    k = case.qkv[b, :, d + h * dh:d + (h + 1) * dh].double()
    v = case.qkv[b, :, 2 * d + h * dh:2 * d + (h + 1) * dh].double()
    qt = (q * torch.tensor(qscale(dh), dtype=torch.float32)).double()
    pim = case.mode == PIM
    cols = torch.tensor(([L - 1] + list(range(L - 1))) if pim else list(range(L)))
    obj = float(torch.tensor(W_OBJ, dtype=torch.float32) * case.r_u[b])
    kb = torch.empty(L, dtype=torch.float64)
    for c in range(L):
        key = int(cols[c])
        if case.mode != CAUSAL and int(case.ids[b, key]) == 0:
            kb[c] = -math.inf
        else:
            w = obj if (pim and c == 0) else (W_H if pim else 0.0)
            kb[c] = float(torch.tensor(L2E, dtype=torch.float32) * torch.tensor(w, dtype=torch.float32))
    return qt, k[cols], v[cols], cols, kb


def item_bound(case: Case, b: int, h: int) -> float:
    qt, k, _, _, kb = item_operands(case, b, h)
    fin = torch.isfinite(kb)
    babs = float(kb[fin].abs().max()) if bool(fin.any()) else -1.0
    return producer_bound(bf16_rn(qt), bf16_rn(k), babs)


def threshold_case(seed: int = 11, n_items: int = 4 * NUM_SMS, H: int = 4, L: int = 201) -> Case:
    """Items at 79..79.9 (shift-free) and 80.1..81 (exact) by the producer's arithmetic, PIM mode, dh = 32; the kind of
    item k alternates with k and, per CTA (k mod 148), as A B B A over its consecutive items, so both staging buffers
    carry both kinds.  Windows beyond n_items / H carry r_u = +-80 (|bias| 115: exact pass).  Rows and keys are
    X3-type (``x_of``): q~ = eta sg x_of(Hq) 2^n (half of the rows at half scale), k = eps sg X3 2^-m, and in most
    windows the objective bias is 2 s_a, so that rows see the objective key level with their top keys with opposite
    product signs (the "worst" construction) and rows aligned with the objective reach 2^+-78."""
    dh = 32
    B = n_items // H + 2
    g = _gen(seed)
    d = H * dh
    qkv = torch.zeros((B, L, 3 * d), dtype=torch.float64)
    ids = torch.randint(1, 1000, (B, L), generator=g)
    r_u = torch.zeros(B, dtype=torch.float64)
    shift = torch.zeros(B * H, dtype=torch.bool)
    khi = 1 + 2.0 ** -7
    s_ref = 26.3                                       # top score: 1.02 s + 2 s ~ 79.5
    cand = [(1 + mm / 128, n) for n in (-3, -2, -1, 0, 1) for mm in range(1, 128)]
    cand_q = torch.tensor([[Hq * 2.0 ** n] * dh for Hq, n in cand], dtype=torch.float64)
    k2 = _fma_norm2(torch.full((1, dh), khi))
    for b in range(B):
        sgn = 1.0 if b % 2 == 0 else -1.0
        if b * H >= n_items:
            r_u[b] = 80.0 * sgn
        elif b % 5 == 4:
            r_u[b] = 40.0 * sgn
        else:
            r_u[b] = 2 * s_ref / (L2E * W_OBJ) * sgn
        r_u[b] = float(torch.tensor(float(r_u[b]), dtype=torch.float32))
        babs = abs(float(torch.tensor(L2E, dtype=torch.float32) * torch.tensor(float(r_u[b]), dtype=torch.float32)))
        for h in range(H):
            it = b * H + h
            want_free = it < n_items and (((it // NUM_SMS) % 4 in (0, 3)) != (it % 2 == 1))
            shift[it] = want_free
            lo, hi = (79.0, 79.9) if want_free else (80.1, 81.0)
            # choose (Hq, n): the producer bound of the row image with the largest norm, closest to the window centre
            bd = _bound_of(_fma_norm2(cand_q, rows=True), k2, babs)
            ok = (bd >= lo) & (bd <= hi)
            if bool(ok.any()):
                pick = int(torch.where(ok, (bd - 0.5 * (lo + hi)).abs(), torch.full_like(bd, math.inf)).argmin())
                best = (0.0, cand[pick][0], cand[pick][1])
            else:                                      # r_u = +-80: every scale is an exact item
                best = (0.0, 1 + 2.0 ** -7, -1)
            _, Hq, n = best
            sg = torch.where(torch.rand(dh, generator=g) < 0.5, -1.0, 1.0).double()
            j = torch.arange(L)
            eps = torch.where((j + h) % 2 == 0, 1.0, -1.0).double()
            m = (j // 2) % 3
            k = eps[:, None] * sg[None, :] * X3 * (2.0 ** -m.double())[:, None]
            k[L - 1] = sg * X3 * (1.0 if r_u[b] < 0 else -1.0)     # the objective key: m = 0
            i = torch.arange(L)
            eta = torch.where((i // 2) % 2 == 0, 1.0, -1.0).double()
            qt = eta[:, None] * sg[None, :] * x_of(Hq) * (2.0 ** (n - (i % 2)).double())[:, None]
            q = q_from_scaled(qt, dh).double()
            v = torch.randn((L, dh), generator=g, dtype=torch.float64)
            qkv[b, :, h * dh:(h + 1) * dh] = q
            qkv[b, :, d + h * dh:d + (h + 1) * dh] = k
            qkv[b, :, 2 * d + h * dh:2 * d + (h + 1) * dh] = v
    regime = torch.full((B, H, L), R_WORST, dtype=torch.int64)
    return Case(f"threshold-B{B}-L{L}-H{H}", qkv.float().contiguous(), ids, r_u.float(), H, PIM, regime,
                torch.full((B,), WORST, dtype=torch.int64), shift)


# ---------------------------------------------------------------------------------------------- reference
def split_heads(qkv, H):
    B, L, d3 = qkv.shape
    d = d3 // 3
    dh = d // H
    return [qkv[..., i * d:(i + 1) * d].reshape(B, L, H, dh).transpose(1, 2) for i in range(3)]


def reference(case: Case, go: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """float64: out [B, L, d], lse [B, H, L] (NaN where a row sees no key, as the kernels; torch's softmax gives NaN rows
    there), and with ``go`` the gradients d_qkv [B, L, 3d] and d_r_u [B] by autograd."""
    qkv = case.qkv.double().requires_grad_(go is not None)
    r_u = case.r_u.double().requires_grad_(go is not None)
    q, k, v = split_heads(qkv, case.H)
    s = q @ k.transpose(-1, -2) / math.sqrt(case.dh) + mask_bias(case.ids, r_u, case.L, case.mode).unsqueeze(1)
    lse = torch.logsumexp(s, -1)
    dead = torch.isinf(s).all(-1) & (s < 0).all(-1)
    a = torch.softmax(s, -1)
    out = (a @ v).transpose(1, 2).reshape(case.B, case.L, -1)
    res = {"out": out.detach(), "lse": torch.where(dead, torch.full_like(lse, math.nan), lse).detach()}
    if go is not None:
        out.backward(go.double())
        res["d_qkv"] = qkv.grad
        res["d_r_u"] = r_u.grad
    return res


def _stats(case: Case):
    """Float64 quantities of the error model, [B, H, L(, L)]."""
    q, k, v = (x.double() for x in split_heads(case.qkv, case.H))
    dh, L = case.dh, case.L
    mb = mask_bias(case.ids, case.r_u.double(), L, case.mode).unsqueeze(1)           # [B, 1, L, L]
    s = q @ k.transpose(-1, -2) / math.sqrt(dh) + mb
    vis = torch.isfinite(s)
    dead = ~vis.any(-1)
    sig = s * (1 / LN2)                                # log2 units
    bias = torch.where(vis, mb.expand_as(s) * (1 / LN2), torch.zeros((), dtype=s.dtype))
    A = (q.abs() @ k.abs().transpose(-1, -2)) * (1 / (LN2 * math.sqrt(dh)))
    m = torch.where(vis, sig, torch.full_like(sig, -math.inf)).max(-1).values
    m = torch.where(dead, torch.zeros_like(m), m)
    w = torch.softmax(torch.where(dead[..., None], torch.zeros_like(s), s), -1) * vis
    o = w @ v
    spread = (w[..., None] * (v[:, :, None, :, :] - o[..., None, :]).abs()).sum(-2).amax(-1) if L * L * dh <= 2 ** 26 \
        else _spread_chunked(w, v, o)
    absv = (w @ v.abs()).amax(-1)
    lse = torch.logsumexp(torch.where(vis, s, torch.full_like(s, -math.inf)), -1)
    return dict(q=q, k=k, v=v, s=s, vis=vis, dead=dead, sig=sig, bias=bias, A=A, m=m, w=w, o=o, spread=spread,
                absv=absv, lse=lse)


def _spread_chunked(w, v, o):
    """max over head dims of sum_j w_ij |v_jt - o_it|, in row chunks (long windows)."""
    out = torch.empty(w.shape[:-1], dtype=w.dtype)
    for i0 in range(0, w.shape[2], 64):
        sl = slice(i0, i0 + 64)
        out[:, :, sl] = (w[:, :, sl, :, None] * (v[:, :, None, :, :] - o[:, :, sl, None, :]).abs()).sum(-2).amax(-1)
    return out


def _score_coef(engine: str, dh: int) -> float:
    return (dh + 4) * U24 if engine in ("fp32", "fp32_blocked") else NEW_THREE + 4 * U24


def _pv_coef(engine: str, n: int) -> float:
    acc = (n + 8) * U24 + 2 * U23                                  # fp32 sum of p, 1 / sum and the product
    if engine in ("tc", "tc_blocked", "img"):
        return C_PV_TC + 6 * math.ceil(n / 32) * U23 + acc
    if engine == "row":
        return U * U + (n + 8) * U24 + acc
    c = (n + 8) * U24 + acc
    if engine == "fp32_blocked":
        c += math.ceil(n / 64) * (RHO + 2 * U24) * 2
    return c


def forward_bound_raw(case: Case, engine: str, st=None):
    """Per-row bounds (items 1-5 of the module docstring, without MARGIN): out [B, H, L] (on every head dim of the row),
    lse [B, H, L], and E_i [B, H, L] (log2 units)."""
    st = st or _stats(case)
    L = case.L
    E = _score_coef(engine, case.dh) * st["A"] + U23 * (2 * st["sig"].abs() + st["bias"].abs()
                                                         + (st["sig"] - st["m"][..., None]).abs())
    E = torch.where(st["vis"], E, torch.zeros_like(E)).amax(-1)
    two_e = torch.pow(2.0, E)
    F = two_e * (two_e * (1 + RHO) - 1) / (1 - RHO)
    vmax = st["v"].abs().amax((-1, -2))[..., None]
    out_b = F * st["spread"] + _pv_coef(engine, L) * st["absv"] + (L + 8) * FTZ * vmax
    lse_b = LN2 * E + 2 * RHO + (L + 8) * U22 + U22 * (st["lse"].abs() + LN2 * st["m"].abs() + 1)
    zero = torch.zeros_like(out_b)
    return torch.where(st["dead"], zero, out_b), torch.where(st["dead"], zero, lse_b), E


def forward_bound(case: Case, engine: str, st=None):
    out_b, lse_b, _ = forward_bound_raw(case, engine, st)
    return MARGIN * out_b, MARGIN * lse_b


def row_ratios(case: Case, got_out, got_lse, engine: str, rows=None, st=None):
    """(max out ratio [B, H, n], max lse ratio [B, H, n]) of |got - ref| over the row's bound; ``rows``: the window rows
    got_out / got_lse hold (default all).  NaN rows must be NaN in both (checked by the caller with ``dead``)."""
    st = st or _stats(case)
    ref = reference(case)
    ob, lb = forward_bound(case, engine, st)
    rows = torch.arange(case.L) if rows is None else torch.as_tensor(rows)
    B, H, dh = case.B, case.H, case.dh
    go = got_out.double().reshape(B, len(rows), H, dh).transpose(1, 2)
    ro = ref["out"].reshape(B, case.L, H, dh).transpose(1, 2)[:, :, rows]
    err = (go - ro).abs().amax(-1)
    dead = st["dead"][:, :, rows]
    err = torch.where(dead, torch.zeros_like(err), err)
    r_out = _ratio(err, ob[:, :, rows])
    r_lse = None
    if got_lse is not None:
        el = (got_lse.double() - ref["lse"][:, :, rows]).abs()
        el = torch.where(dead, torch.zeros_like(el), el)
        r_lse = _ratio(el, lb[:, :, rows])
    return r_out, r_lse, dead


def _ratio(err, bound):
    return torch.where(bound > 0, err / bound, torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))


def backward_bound(case: Case, go: torch.Tensor, fwd_engine: str):
    """Element-wise bounds (item 6) of d_qkv [B, L, 3d] and d_r_u [B] for the fp32 backward fed by ``fwd_engine``'s
    out and lse (their raw bounds enter as dO and dlse)."""
    st = _stats(case)
    q, k, v, vis = st["q"], st["k"], st["v"], st["vis"]
    B, H, L, dh = case.B, case.H, case.L, case.dh
    scale = 1 / math.sqrt(dh)
    ob, lb, _ = forward_bound_raw(case, fwd_engine, st)
    gO = go.double().reshape(B, L, H, dh).transpose(1, 2)
    P = st["w"]
    s = st["s"]
    Es = _score_coef("fp32", dh) * st["A"] * LN2 + RHO + U23 * (s.abs() + st["lse"].abs()[..., None]).nan_to_num(0.0) \
        + lb[..., None]
    dP = torch.where(vis, P * torch.expm1(Es) + TINY, torch.zeros_like(P))
    dp = gO @ v.transpose(-1, -2)
    ddp = (dh + 1) * U24 * (gO.abs() @ v.abs().transpose(-1, -2))
    O = st["o"]
    D = (gO * O).sum(-1)
    dD = gO.abs().sum(-1) * ob + (dh + 1) * U24 * (gO.abs() * O.abs()).sum(-1)
    dS = P * (dp - D[..., None])
    ddS = dP * ((dp - D[..., None]).abs() + ddp + dD[..., None]) + P * (ddp + dD[..., None]) + U23 * dS.abs() + TINY
    ddS = torch.where(vis, ddS, torch.zeros_like(ddS))
    dQ = scale * (dS @ k)
    bq = scale * (ddS @ k.abs() + L * U24 * (dS.abs() @ k.abs())) + U23 * dQ.abs() + L * TINY
    dK = scale * (dS.transpose(-1, -2) @ q)
    bk = scale * (ddS.transpose(-1, -2) @ q.abs() + L * U24 * (dS.abs().transpose(-1, -2) @ q.abs())) + U23 * dK.abs() + L * TINY
    bv = dP.transpose(-1, -2) @ gO.abs() + L * U24 * (P.transpose(-1, -2) @ gO.abs()) + L * TINY
    cat = lambda x: x.transpose(1, 2).reshape(B, L, H * dh)
    b_qkv = MARGIN * torch.cat([cat(bq), cat(bk), cat(bv)], -1)
    b_ru = MARGIN * abs(W_OBJ) * (ddS[..., L - 1] + L * U24 * dS[..., L - 1].abs() + TINY).sum((1, 2)) if case.mode == PIM else None
    return b_qkv, b_ru


# ---------------------------------------------------------------------------------------------- emulator
def emulate_persistent(case: Case, b: int, h: int, force_exact: bool = False, fault: Optional[str] = None):
    """float64 model of pim_attn_persistent_kernel on one item: S = three bf16 MMAs (lo*hi, hi*lo, hi*hi) per K = 16
    step, each truncated to fp32; x = fp32(fp32(S + kb) - mx) with mx = 0 when the producer bound is <= 80 (unless
    force_exact), the visible row maximum otherwise; p = fp32(2^x) (the exponent without its approximation error);
    sum = the sequential fp32 sum of the unrounded p in column order; P split into bf16 hi / lo; per 16 keys
    ACC1 += P_hi V_hi, ACC2 += P_hi V_lo, ACC1 += P_lo V_hi, each MMA truncated to fp32; o = fp32(ACC1 + ACC2) / sum.
    fault = "pv_hi_only": P.V as the single product P_hi V_hi.  Returns (out [L, dh] in window row order, shift_free)."""
    qt, k, v, cols, kb = item_operands(case, b, h)
    L, dh = case.L, case.dh
    pim = case.mode == PIM
    koff = 1 if pim else 0
    fin = torch.isfinite(kb)
    babs = float(kb[fin].abs().max()) if bool(fin.any()) else -1.0
    qh, ql = split_hi_lo(qt)
    kh, kl = split_hi_lo(k)
    free = (not force_exact) and producer_bound(qh, kh, babs) <= NO_SHIFT_SAFE
    kp = -(-dh // 16) * 16
    S = torch.zeros((L, L), dtype=torch.float64)
    for k0 in range(0, kp, 16):
        S = trunc32(S + ql[:, k0:k0 + 16] @ kh[:, k0:k0 + 16].t())
        S = trunc32(S + qh[:, k0:k0 + 16] @ kl[:, k0:k0 + 16].t())
        S = trunc32(S + qh[:, k0:k0 + 16] @ kh[:, k0:k0 + 16].t())
    i = torch.arange(L)[:, None]
    c = torch.arange(L)[None, :]
    vis = ((c <= i + koff) | ((c == 0) & pim)) & fin[None, :]
    sb = f32(S + kb[None, :])
    if free:
        mx = torch.zeros(L, dtype=torch.float64)
    else:
        mx = torch.where(vis, sb, torch.full_like(sb, -math.inf)).max(1).values
    x = f32(sb - mx[:, None])
    p = torch.where(vis, f32(torch.exp2(x)), torch.zeros_like(x))
    ssum = torch.zeros(L, dtype=torch.float64)
    for cc in range(L):
        ssum = f32(ssum + p[:, cc])
    ph, pl = split_hi_lo(p)
    vh, vl = split_hi_lo(v)
    acc1 = torch.zeros((L, dh), dtype=torch.float64)
    acc2 = torch.zeros((L, dh), dtype=torch.float64)
    for k0 in range(0, L, 16):
        ks = slice(k0, k0 + 16)
        acc1 = trunc32(acc1 + ph[:, ks] @ vh[ks])
        if fault != "pv_hi_only":
            acc2 = trunc32(acc2 + ph[:, ks] @ vl[ks])
            acc1 = trunc32(acc1 + pl[:, ks] @ vh[ks])
    o = f32(f32(acc1 + acc2) * f32(1.0 / ssum)[:, None])
    dead = ~vis.any(1)
    o[dead] = math.nan
    return o, free
