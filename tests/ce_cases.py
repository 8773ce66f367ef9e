"""Hard inputs for the softmax cross-entropy kernels, their float64 reference, per-element error bounds for both engines,
and a float64 emulator of the tensor-core backward.

The CE path is the log-sum-exp forward ``irs_score_lse_gather[_tc]`` (lse and selected logits per row) and the backward
``irs_score_ce_bwd[_tc]``:

    g[m,j] = (exp(s[m,j] - lse[m]) - [j == target[m]]) * gscale,   s = h W^T + bias
    d_h = g W,    d_W += g^T h,    d_bias += colsum(g)

Logits of an untrained model (h ~ N(0,1), W ~ N(0,1/d)) have |s| ~ 1 and a nearly uniform softmax.  The cases here look
like a model after training, mixed inside every 128-row tile:

* anisotropic -- W_j = mu + sigma z_j with the shared direction mu carrying half of E|W_j|^2, and LayerNorm-like rows h
  (|h| ~ sqrt(d), a per-feature offset), so the catalog sums of d_h and the user sums of d_W are coherent;
* confident   -- the target leads the runner-up by DELTAS nats (p_t from ~0.7 to 1 - 1e-17);
* large       -- rows whose best score is +LARGE and rows whose scores are all <= -LARGE (beyond fp32 exp's +-88.7);
* popularity  -- bias = -alpha log(1 + popularity rank), POP_SPAN nats wide; rows whose target is a tail item;
* ties        -- three identical W rows (and biases) at the top, the target among them;
* worst       -- rows and items made of band_cases.X3 (the fp32 value the three-MMA product rounds worst) and of C_DN, so
                 the three-MMA score error reaches NEW_THREE sum_k |h_k W_jk|.

Targets include column 0, column N-1 (last partial tile) and -1 (a skipped row).

Error model (per element, computed in float64 from the reference, for the engine that ran):

* score error E[m,j]: three-MMA (tensor cores) NEW_THREE sum_k |h_k W_jk|; fp32 FMA chain d 2^-24 sum_k |h_k W_jk|; both
  plus 2^-24 |s| for the fp32 bias addition.
* exponent argument eps[m,j]: 2^-23 (|lse| + |b_j| + |s - lse|) + 2^-21 (rounding of the shifted argument, log2(e) in
  fp32, and ex2.approx / expf at <= 2 ulp).
* forward lse: log(sum_j p_j exp(E + eps)) (the largest shift of a log-sum-exp whose terms each move by at most E + eps)
  + D 2^-22 for the fp32 sum of positive terms over a dependency chain of depth D taken from the kernel's plan (2^-22,
  not 2^-24: each step may also rescale the running sum by an approximate exp) + 2^-23 (|lse| + ln N + 1) for max + log.
* backward, out = G Y with X rows resident and Y rows streamed in 128-row tiles (d_h: X = users, Y = items; d_W: the
  two swap):  sum_y |p~ - p| |Y_yk|  with |p~ - p| <= p (exp(E + eps) - 1),  plus C sum_y |g_y Y_yk| for the product
  (C = NEW_THREE + 2^-23 on the tensor cores, whose G and Y are bf16 hi/lo pairs; 2^-23 on the fp32 engine), plus the
  accumulation: every accumulation step loses at most one fp32 ulp of the running partial, i.e. 2^-23 |partial| on the
  tensor cores (one truncation per K = 16 tcgen05.mma, as measured by test_three_mma_accumulation_probe in
  tests/test_gpu_scorer_bands.py: ~one ulp per MMA when the partial sums have one sign) and 2^-24 |partial| per fp32
  FMA.  The partials are the reference's, in the kernel's own Y-tile order, restarted at every catalog split:
  sum over tiles of steps_per_tile * unit * (max(|P_before|, |P_after|) + sum_{y in tile} |g_y Y_yk|).  Finally
  2^-23 (|out| + |prefill|) (n_splits + 1) for the gscale product and the additions into the output.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import torch

from tests.band_cases import C_DN, NEW_THREE, X3, bf16_rn

NUM_SMS, BM = 148, 128
MAX_RUN_TILES = 256                  # scorer_ce_tc.cu: Y tiles one tensor-memory accumulation may span
U24, U23, U22, U21 = 2.0 ** -24, 2.0 ** -23, 2.0 ** -22, 2.0 ** -21
L2E = float(torch.tensor(1.4426950408889634, dtype=torch.float32))       # log2(e) as the kernels hold it
EXP_LIMIT = 88.72                    # fp32 exp overflows above this argument
LARGE = 120.0
DELTAS = (1.0, 5.0, 15.0, 40.0)
POP_SPAN = 35.0                      # width of the popularity bias in nats
NORTH_STAR = 1e-3                    # gradients within 1e-3 of the compared tensor's max (README, tests/helpers.py)

# regime of a row
CONTROL, ANISO, CONF, LARGE_POS, LARGE_NEG, POP_TAIL, TIES, WORST_X3, WORST_DN = range(9)
REGIME_NAMES = ("control", "anisotropic", "confident", "large+", "large-", "popularity-tail", "ties", "worst-x3",
                "worst-cdn")
DISTINCT_ROWS = 1536
_ROW_CYCLE = (ANISO, CONF, LARGE_POS, POP_TAIL, CONF, TIES, LARGE_NEG, CONF, WORST_X3, ANISO, CONF, WORST_DN)


# ---------------------------------------------------------------------------------------------- plans
def _cdiv(a, b):
    return -(-a // b)


def plan_ce_tc(RX: int, RY: int):
    """(n_x, n_y, n_splits, tiles_per_split) exactly as plan() in scorer_ce_tc.cu (one pass: X resident, Y streamed)."""
    n_x, n_y = _cdiv(RX, BM), _cdiv(RY, BM)
    splits = 1
    if n_x < 2 * NUM_SMS:
        splits = _cdiv(2 * NUM_SMS, n_x)
    max_splits = max(_cdiv(n_y, 16), 1)
    splits = min(splits, max_splits)
    tps = min(_cdiv(n_y, splits), MAX_RUN_TILES)
    return n_x, n_y, _cdiv(n_y, tps), tps


def plan_lse_simt(M: int, N: int):
    """(n_splits, tiles_per_split) of the fp32 engine's MODE_LSE launch (launch_score_simt, BN = 128)."""
    m_tiles, n_tiles = _cdiv(M, 128), _cdiv(N, 128)
    splits = min(max((NUM_SMS * 4) // m_tiles, 1), n_tiles)
    tps = _cdiv(n_tiles, splits)
    return _cdiv(n_tiles, tps), tps


def plan_lse_tc(M: int, N: int):
    """(n_splits, tiles_per_split) of the tensor-core scorer (band_cases.plan = plan() in scorer_tc.cu, BN = 256)."""
    from tests.band_cases import plan
    _, _, tps, n_splits = plan(M, N)
    return n_splits, tps


def lse_sum_depth(M: int, N: int, engine: str) -> int:
    """Depth of the fp32 dependency chain that sums the exponentials of one row (see the module docstring)."""
    if engine == "tc":
        n_splits, tps = plan_lse_tc(M, N)
        # per (split, column half) thread: 4 chunks per tile, each (8-term lanes, 2 combines, 1 add + 1 rescale);
        # finalise: n_part / 32 terms per lane, a 5-level warp sum, the exp of the merge
        return tps * 4 * 2 + 11 + _cdiv(2 * n_splits, 32) + 7
    n_splits, tps = plan_lse_simt(M, N)
    # per thread: 8 expf terms per tile + (rescale, add) per tile; 4-level shuffle merge; n_splits sequential adds
    return tps * (8 + 2) + 8 + n_splits + 2


# ---------------------------------------------------------------------------------------------- cases
@dataclass
class Case:
    name: str
    h: torch.Tensor                    # [M, d] float32
    W: torch.Tensor                    # [N, d] float32
    bias: torch.Tensor                 # [N] float32
    target: torch.Tensor               # [M] int64, 0-based, -1 = skipped row
    sel: torch.Tensor                  # [M, 2] int64 1-based ids: target + 1, then another id (0, > N, < 0 included)
    regime: torch.Tensor               # [M] int64 regime of each row
    lead: Dict[int, float] = field(default_factory=dict)     # confident rows: intended lead of the target (nats)

    @property
    def M(self):
        return self.h.shape[0]

    @property
    def N(self):
        return self.W.shape[0]

    @property
    def d(self):
        return self.h.shape[1]

    def rows(self, regime: int) -> List[int]:
        return (self.regime == regime).nonzero().flatten().tolist()


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _unit(v):
    return v / v.norm()


def _bisect(f, goal, step, iters=80):
    """lam with f(lam) = goal for f monotone in the direction of ``step`` (bracketed by doubling ``step``), or the last
    bracket end when the goal is out of reach."""
    lo, hi = 0.0, step
    up = goal > f(0.0)
    for _ in range(24):
        if (f(hi) >= goal) == up:
            break
        lo, hi = hi, hi * 2
    else:
        return None
    for _ in range(iters):
        mid = 0.5 * (lo + hi)
        if (f(mid) >= goal) == up:
            hi = mid
        else:
            lo = mid
    return 0.5 * (lo + hi)


def _solve_lift(h0, v, W, b, target_max):
    """lam such that max_j (h0 + lam v) . W_j + b_j = target_max (all in float64)."""
    rate, s0 = W @ v, W @ h0 + b
    f = lambda lam: float((s0 + lam * rate).max())
    lam = _bisect(f, target_max, 1.0 if target_max > f(0.0) else -1.0)
    return None if lam is None else h0 + lam * v


def _ortho(v, rows):
    for w in rows:
        v = v - (v @ w) * w / (w @ w)
    return _unit(v)


def _confident_row(h0, W, b, Wmean, t, delta, excl=(), avoid=()):
    """h0 + lam v with v = W_t - mean(W) (orthogonal to the rows ``avoid``): the target's score leads every other item
    (outside excl) by ``delta``.  None when no lam reaches it."""
    v = _ortho(W[t] - Wmean, [W[j] for j in avoid])
    rate, s0 = W @ v, W @ h0 + b
    mask = torch.zeros(W.shape[0], dtype=torch.bool)
    mask[[t] + list(excl)] = True

    def lead(lam):
        s = s0 + lam * rate
        return float(s[t] - s.masked_fill(mask, -math.inf).max())
    lam = _bisect(lead, delta, 1.0 if delta > lead(0.0) else -1.0)
    return None if lam is None else h0 + lam * v


def control_case(M: int, N: int, d: int, seed: int, h_scale: float = 1.0) -> Case:
    """Today's Gaussian data: h ~ N(0,1), W ~ N(0,1/d), bias ~ 0.1 N(0,1).  ``h_scale`` < 1 gives the small scores of
    a model at initialisation, where the score error of either engine is far below 1e-4 nats."""
    g = _gen(seed)
    h = torch.randn((M, d), generator=g) * h_scale
    W = torch.randn((N, d), generator=g) / math.sqrt(d)
    bias = torch.randn(N, generator=g) * 0.1
    target = torch.randint(0, N, (M,), generator=g)
    _edges(target, N, g)
    return Case(f"control-M{M}-N{N}-d{d}" + ("" if h_scale == 1.0 else f"-x{h_scale:g}"), h, W, bias, target, _sel(target, N, g),
                torch.full((M,), CONTROL, dtype=torch.int64))


def _edges(target, N, g):
    M = target.shape[0]
    for m, t in ((0, 0), (1, N - 1), (2, -1)):
        if m < M:
            target[m] = t
    if M > 40:
        target[torch.randperm(M, generator=g)[: max(1, M // 50)]] = -1


def _sel(target, N, g):
    M = target.shape[0]
    sel = torch.zeros((M, 2), dtype=torch.int64)
    sel[:, 0] = (target + 1).clamp(min=0)
    sel[:, 1] = torch.randint(1, N + 1, (M,), generator=g)
    m = torch.arange(M)
    sel[m % 7 == 0, 1] = 0
    sel[m % 7 == 1, 1] = N + 1                 # just past the catalog: inside the last partial tile unless N % 128 == 0
    sel[m % 7 == 2, 1] = -3
    sel[m % 7 == 3, 1] = N                     # the last item
    sel[m % 7 == 4, 1] = 1                     # the first
    return sel


def mixed_case(M: int, N: int, d: int, seed: int) -> Case:
    """All regimes of the module docstring, cycled row by row so that every 128-row tile mixes them.  At most
    DISTINCT_ROWS rows are constructed; longer cases repeat them (same regimes, same position in the tile)."""
    g = _gen(seed)
    sigma = 1.0 / math.sqrt(d)
    mu = _unit(torch.randn(d, generator=g, dtype=torch.float64)) * sigma * math.sqrt(d)     # |mu|^2 = sigma^2 d
    W = mu + sigma * torch.randn((N, d), generator=g, dtype=torch.float64)
    alpha = POP_SPAN / math.log(N) if N > 1 else 0.0
    bias = -alpha * torch.log1p(torch.randperm(N, generator=g).double())
    R = min(M, DISTINCT_ROWS)
    # LayerNorm-like rows: unit-variance features around zero mean, then a per-feature offset beta
    beta = 0.6 * torch.randn(d, generator=g, dtype=torch.float64)
    z = torch.randn((R, d), generator=g, dtype=torch.float64)
    h = (z - z.mean(1, keepdim=True)) / z.std(1, keepdim=True) + beta
    target = torch.randint(0, N, (R,), generator=g)
    regime = torch.tensor([_ROW_CYCLE[m % len(_ROW_CYCLE)] for m in range(R)], dtype=torch.int64)
    specials = N >= 16
    if not specials:
        keep = (ANISO, CONF, POP_TAIL) if N > 1 else (ANISO,)
        regime[~torch.isin(regime, torch.tensor(keep))] = ANISO
    tie, avoid = [], []
    u = _unit(mu)
    if specials:
        order = torch.argsort(bias, descending=True)
        tie = [int(order[0]), int(order[1]), int(order[2])]               # the three most popular items
        for j in tie[1:]:
            W[j] = W[tie[0]]
            bias[j] = bias[tie[0]]
        x3_item, dn_item = int(order[N // 2]), int(order[N // 2 + 1])
        sg = torch.where(torch.rand(d, generator=g) < 0.5, -1.0, 1.0).double()
        sg2 = torch.where(torch.rand(d, generator=g) < 0.5, -1.0, 1.0).double()
        # |h| |W| ~ 1e3 on the worst-rounding pairs (as band_cases.argmax_three): the three-MMA error of the pair's score
        # is ~ NEW_THREE |h| |W| ~ 0.05 nats
        e1 = next(e for e in range(-8, 16) if d * 4 * X3 * X3 * 2.0 ** e >= 1e3)
        e2 = next(e for e in range(-8, 16) if d * 4 * C_DN * C_DN * 2.0 ** e >= 1e3)
        W[x3_item] = sg * X3 * 2.0 ** e1
        W[dn_item] = sg2 * C_DN * 2.0 ** e2
        h_x3, h_dn = sg * X3 * 4, sg2 * C_DN * 4
        avoid = [x3_item, dn_item]                  # the confident and large rows leave these two alone
        u = _ortho(u, [W[j] for j in avoid])
    Wf = W.float().double()
    Wmean = Wf.mean(0)
    if specials:
        # lift each worst-rounding item 3 nats above everything else on its rows (p ~ 0.95 on the item whose three-MMA
        # score carries the largest error); with |h| |W| ~ 1e3 its bias sinks it far below every other row's scores (set
        # before the rows are built: the large rows must see it)
        for item, hv in ((x3_item, h_x3), (dn_item, h_dn)):
            hv = hv.float().double()
            s = Wf @ hv + bias.float().double()
            s[item] = -math.inf
            bias[item] = float(s.max()) + 3.0 - float(Wf[item] @ hv)
    tail = [j for j in torch.argsort(bias).tolist() if j not in avoid][: max(1, N // 100)]
    for m in range(R):
        r = int(regime[m])
        if r == POP_TAIL:
            target[m] = tail[m % len(tail)]
        elif r == CONF and int(target[m]) in avoid:
            target[m] = (int(target[m]) + 2) % N
        elif r == TIES:
            target[m] = tie[1 + m % 2]
        elif r in (WORST_X3, WORST_DN):
            target[m] = x3_item if r == WORST_X3 else dn_item
    _edges(target, N, g)
    biasf = bias.float().double()
    lead = {}
    for m in range(R):
        r = int(regime[m])
        t = int(target[m])
        new = None
        if r == CONF and t >= 0:
            delta = DELTAS[(m // len(_ROW_CYCLE)) % len(DELTAS)]
            new = _confident_row(h[m], Wf, biasf, Wmean, t, delta, tie if t in tie else (), avoid)
            if new is not None:
                lead[m] = delta
        elif r == TIES:
            new = _confident_row(h[m], Wf, biasf, Wmean, tie[0], 3.0, tie, avoid)
        elif r in (LARGE_POS, LARGE_NEG):
            new = _solve_lift(h[m], u, Wf, biasf, LARGE if r == LARGE_POS else -LARGE)
        if r in (CONF, TIES, LARGE_POS, LARGE_NEG):
            if new is None:                        # out of reach on this catalog: an ordinary anisotropic row
                regime[m] = ANISO
            else:
                h[m] = new
        elif r in (WORST_X3, WORST_DN):
            h[m] = h_x3 if r == WORST_X3 else h_dn
    reps = _cdiv(M, R)
    h = h.repeat(reps, 1)[:M]
    target = target.repeat(reps)[:M]
    regime = regime.repeat(reps)[:M]
    if M > R:
        target[M - 1] = N - 1 if target[M - 1] >= 0 else target[M - 1]
        lead = {m: lead[m % R] for m in range(M) if (m % R) in lead and int(target[m]) >= 0}
    return Case(f"mixed-M{M}-N{N}-d{d}", h.float().contiguous(), W.float(), bias.float(), target, _sel(target, N, g),
                regime, lead)


def training_case(M: int, N: int, d: int, seed: int, device="cpu") -> Case:
    """The training shape: anisotropic items, LayerNorm-like rows, half of them confident (the target lifted along
    W_t - mu by 0, 4, 10 or 25 |W_t - mu|-units: leads of a few to tens of nats), a popularity bias 20 nats wide.  Built
    without scoring the rows (a full [M, N] pass per Newton step would cost minutes at M = 200k, N = 500k)."""
    g = torch.Generator(device=device).manual_seed(seed)
    sigma = 1.0 / math.sqrt(d)
    mu = _unit(torch.randn(d, generator=g, device=device)) * sigma * math.sqrt(d)
    W = mu + sigma * torch.randn((N, d), generator=g, device=device)
    bias = -(20.0 / math.log(N)) * torch.log1p(torch.randperm(N, generator=g, device=device).float())
    beta = 0.6 * torch.randn(d, generator=g, device=device)
    z = torch.randn((M, d), generator=g, device=device)
    h = (z - z.mean(1, keepdim=True)) / z.std(1, keepdim=True) + beta
    target = torch.randint(0, N, (M,), generator=g, device=device)
    target[0], target[M - 1] = N - 1, 0
    m = torch.arange(M, device=device)
    lift = torch.tensor([0.0, 4.0, 10.0, 25.0], device=device)[(m // 2) % 4] * (m % 2 == 1)
    v = W[target] - mu
    h = h + lift[:, None] * v / v.norm(dim=1, keepdim=True) * math.sqrt(d) / 4
    regime = torch.where(lift > 0, CONF, ANISO)
    sel = torch.stack([target + 1, torch.randint(1, N + 1, (M,), generator=g, device=device)], 1)
    return Case(f"training-M{M}-N{N}-d{d}", h.contiguous(), W.contiguous(), bias.contiguous(), target, sel, regime)


# ---------------------------------------------------------------------------------------------- reference
def scores64(h, W, bias):
    s = h.double() @ W.double().t()
    return s if bias is None else s + bias.double()


def abs_dot(h, W):
    """sum_k |h_k W_jk| [M, N]."""
    return h.double().abs() @ W.double().abs().t()


def forward_ref(h, W, bias, sel, item_base: int = 1):
    """(lse [M], logit [M, s]) in float64; ids outside [item_base, item_base + N) give 0.0."""
    s = scores64(h, W, bias)
    lse = torch.logsumexp(s, 1)
    col = sel.to(s.device) - item_base
    ok = (col >= 0) & (col < W.shape[0])
    logit = torch.where(ok, torch.gather(s, 1, col.clamp(0, W.shape[0] - 1)), torch.zeros((), dtype=s.dtype, device=s.device))
    return lse, logit


def forward_bound(h, W, bias, sel, engine: str, item_base: int = 1, plan_M: Optional[int] = None):
    """Per-row bound of |lse_kernel - lse| and per-element bound of |logit_kernel - logit| (module docstring); plan_M:
    the row count of the launch when h holds some of its rows."""
    M, d = h.shape
    N = W.shape[0]
    s = scores64(h, W, bias)
    lse = torch.logsumexp(s, 1)
    mx = s.max(1).values
    a = abs_dot(h, W)
    E = (NEW_THREE if engine == "tc" else d * U24) * a + U24 * s.abs()
    eps = U23 * (mx.abs()[:, None] + s.abs() + (s - mx[:, None]).abs()) + U21
    shift = torch.logsumexp(s - lse[:, None] + E + eps, 1)
    D = lse_sum_depth(plan_M or M, N, engine)
    lse_b = shift + D * U22 + U23 * (lse.abs() + math.log(N) + 1)
    col = sel.to(s.device) - item_base
    ok = (col >= 0) & (col < N)
    cc = col.clamp(0, N - 1)
    chain = max(d, d // 32 + 6)
    logit_b = torch.where(ok, chain * U24 * torch.gather(a, 1, cc) + U24 * torch.gather(s, 1, cc).abs(),
                          torch.zeros((), dtype=s.dtype, device=s.device))
    return lse_b, logit_b


def grad_matrix(h, W, bias, target, lse_in, gscale):
    """(G, P, s) in float64 given the lse the kernel received: G = (p - onehot) gscale; rows with target -1 are zero,
    target -2 marks a live row whose target is not among W's rows."""
    s = scores64(h, W, bias)
    P = torch.exp(s - lse_in.double().to(s.device)[:, None])
    target = target.to(s.device)
    P = torch.where(((target >= 0) | (target == -2))[:, None], P, torch.zeros((), dtype=s.dtype, device=s.device))
    live = target >= 0
    G = P.clone()
    rows = live.nonzero().flatten()
    G[rows, target.to(s.device)[rows]] -= 1.0
    return G * gscale, P, s


def backward_ref(h, W, bias, target, lse_in, gscale):
    """(d_h, d_W, d_bias) in float64 given lse_in (no prefill)."""
    G, _, _ = grad_matrix(h, W, bias, target, lse_in, gscale)
    return G @ W.double(), G.t() @ h.double(), G.sum(0)


def _side_bound(G, Y, dP, c_prod, steps_per_tile, unit, tps, ref, prefill, n_splits):
    """Bound of out = G Y (+ prefill) for an X-resident kernel streaming the rows of Y in 128-row tiles."""
    absY = Y.abs()
    absG = G.abs()
    b = dP @ absY + c_prod * (absG @ absY)
    acc = torch.zeros_like(b)
    P = torch.zeros_like(b)
    n_tiles = _cdiv(Y.shape[0], BM)
    for t in range(n_tiles):
        if t % tps == 0:
            P = torch.zeros_like(b)
        sl = slice(t * BM, min((t + 1) * BM, Y.shape[0]))
        Pn = P + G[:, sl] @ Y[sl]
        acc += torch.maximum(P.abs(), Pn.abs()) + absG[:, sl] @ absY[sl]
        P = Pn
    pre = 0.0 if prefill is None else prefill.double().abs()
    return b + steps_per_tile * unit * acc + U23 * (ref.abs() + pre) * (n_splits + 1)


def backward_bound(h, W, bias, target, lse_in, gscale, engine: str, prefill_W=None, prefill_b=None, rows=None, cols=None,
                   plan_M: Optional[int] = None):
    """Per-element bounds (d_h [M|rows, d], d_W [N|cols, d], d_bias [N|cols]) and the float64 results they bound, given
    the lse the kernel received.  ``rows`` / ``cols`` restrict d_h to some users and d_W / d_bias to some items (the
    sums still run over the whole catalog / all users).  plan_M: the row count of the launch when h holds some of its
    rows (d_h only)."""
    M, d = h.shape
    N = W.shape[0]
    hd, Wd = h.double(), W.double()
    out = {}
    tc = engine == "tc"
    c_prod = (NEW_THREE + U23) if tc else U23
    steps, unit = (24, U23) if tc else (BM, U24)

    def pieces(hr, Wc, br, tr, lr):
        G, P, s = grad_matrix(hr, Wc, br, tr, lr, gscale)
        E = (NEW_THREE if tc else d * U24) * abs_dot(hr, Wc) + U24 * s.abs()
        lsd = lr.double()[:, None]
        bb = 0.0 if br is None else br.double().abs()[None, :]
        eps = U23 * (lsd.abs() + bb + (s - lsd).abs()) + U21
        return G, P * torch.expm1(E + eps) * abs(gscale)

    # d_h: X = users, Y = items
    r = torch.arange(M, device=h.device) if rows is None else rows.to(h.device)
    G, dP = pieces(hd[r], Wd, bias, target[r], lse_in[r])
    ref = G @ Wd
    _, _, n_splits, tps = plan_ce_tc(plan_M or M, N) if tc else (0, 0, 1, _cdiv(N, BM))
    out["d_h"] = (ref, _side_bound(G, Wd, dP, c_prod, steps, unit, tps, ref, None, n_splits))
    # d_W, d_bias: X = items, Y = users
    c = torch.arange(N, device=h.device) if cols is None else cols.to(h.device)
    G, dP = pieces(hd, Wd[c], None if bias is None else bias[c], _local_target(target, c), lse_in)
    Gt, dPt = G.t(), dP.t()
    refW = Gt @ hd
    refb = Gt.sum(1)
    _, _, n_splits, tps = plan_ce_tc(N, M) if tc else (0, 0, 1, _cdiv(M, BM))
    if prefill_W is not None:
        refW = refW + prefill_W.double()[c]
    if prefill_b is not None:
        refb = refb + prefill_b.double()[c]
    out["d_W"] = (refW, _side_bound(Gt, hd, dPt, c_prod, steps, unit, tps, refW, None if prefill_W is None else prefill_W[c], n_splits))
    n_add = _cdiv(M, BM) * 24 + 32
    preb = 0.0 if prefill_b is None else prefill_b.double()[c].abs()
    out["d_bias"] = (refb, dPt.sum(1) + (n_add * U24 + U23) * Gt.abs().sum(1) + U23 * (refb.abs() + preb) * (n_splits + 1))
    return out


def _local_target(target, cols):
    """Targets re-indexed into the item subset ``cols`` (-2: the target is another item; -1 stays skipped)."""
    pos = torch.full((int(cols.max()) + 1 if cols.numel() else 1,), -2, dtype=torch.int64, device=cols.device)
    pos[cols] = torch.arange(cols.numel(), device=cols.device)
    t = target.to(cols.device)
    inside = (t >= 0) & (t < pos.shape[0])
    loc = torch.where(inside, pos[t.clamp(0, pos.shape[0] - 1)], torch.full_like(t, -2))
    return torch.where(t < 0, t, loc)


def ratio(got, ref, bound):
    """max |got - ref| / bound (0/0 = 0)."""
    err = (got.double().to(ref.device) - ref).abs()
    r = torch.where(bound > 0, err / bound, torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    return float(r.max()) if r.numel() else 0.0


# ---------------------------------------------------------------------------------------------- emulator
FAULTS = ("no_bias", "target_off_by_one", "skip_tile", "pad_as_zero", "g_hi_only", "lse_shift")


def trunc32(x: torch.Tensor) -> torch.Tensor:
    """float64 -> the fp32 value nearest to x in the direction of zero (truncation), as float64."""
    f = x.float()
    over = f.double().abs() > x.abs()
    return torch.where(over, torch.nextafter(f, torch.zeros_like(f)), f).double()


def f32(x: torch.Tensor) -> torch.Tensor:
    return x.float().double()


def _pad_rows(x, n):
    return torch.cat([x, x.new_zeros((n - x.shape[0],) + tuple(x.shape[1:]))]) if n > x.shape[0] else x


def _split(x):
    hi = bf16_rn(x)
    return hi, bf16_rn(f32(x.double() - hi))


def _mma_acc(acc, Ahi, Alo, Bhi, Blo, k0, k1):
    """One K = 16 step of the three-MMA product (lo*hi, hi*lo, hi*hi), each MMA truncated to fp32."""
    acc = trunc32(acc + Alo[:, k0:k1] @ Bhi[k0:k1])
    acc = trunc32(acc + Ahi[:, k0:k1] @ Blo[k0:k1])
    return trunc32(acc + Ahi[:, k0:k1] @ Bhi[k0:k1])


def emulate_tc_backward(h, W, bias, target, lse_in, gscale, fault: Optional[str] = None, rows=None,
                        prefill_W=None, prefill_b=None, passes=("d_h", "d_W"), plan_M: Optional[int] = None):
    """float64 model of irs_score_ce_bwd_tc: S = three bf16 MMAs per K = 16 step, G = exp2(S log2e + (bias - lse) log2e)
    in fp32 (minus 1 at the target) split into bf16 hi/lo, ACC += G Y with the same three MMAs over Y tiles in the
    kernel's order, every MMA truncated to fp32, a fresh ACC per catalog split, results scaled by gscale and added.
    ``fault`` seeds one of FAULTS.  Returns {"d_h": [M|rows, d], "d_W": [N, d], "d_bias": [N]} (fp32 values)."""
    M, d = h.shape
    N = W.shape[0]
    Mp, Np = _cdiv(M, BM) * BM, _cdiv(N, BM) * BM
    hp = _pad_rows(h.double(), Mp)
    Wp = _pad_rows(W.double(), Np)
    kp = _cdiv(d, 16) * 16
    hp = torch.nn.functional.pad(hp, (0, kp - d))
    Wp = torch.nn.functional.pad(Wp, (0, kp - d))
    hh, hl = _split(hp)
    wh, wl = _split(Wp)
    # S [Mp, Np]: 16-wide K steps (zero K padding adds nothing)
    S = torch.zeros((Mp, Np), dtype=torch.float64)
    for k0 in range(0, kp, 16):
        S = _mma_acc(S, hh, hl, wh.t(), wl.t(), k0, k0 + 16)
    lse = lse_in.double() + (1e-4 if fault == "lse_shift" else 0.0)
    b = torch.zeros(N, dtype=torch.float64) if (bias is None or fault == "no_bias") else bias.double()
    rowterm = f32(-f32(lse) * L2E)
    colterm = f32(b.float().double() * L2E)
    tgt = target.clone()
    if fault == "target_off_by_one":
        tgt = torch.where(tgt >= 0, (tgt + 1) % N, tgt)
    live = tgt >= 0
    rt = torch.full((Mp,), -math.inf, dtype=torch.float64)
    rt[:M] = torch.where(live, rowterm, torch.full_like(rowterm, -math.inf))
    ct = torch.full((Np,), 0.0 if fault == "pad_as_zero" else -math.inf, dtype=torch.float64)
    ct[:N] = colterm
    if fault == "pad_as_zero":
        rt[M:] = 0.0                               # padded users: their -lse term counted as 0
    arg = f32(S * L2E + f32(rt[:, None] + ct[None, :]))
    Gm = f32(torch.exp2(arg))
    rr = live.nonzero().flatten()
    Gm[rr, tgt[rr]] = f32(Gm[rr, tgt[rr]] - 1.0)
    Gm = torch.nan_to_num(Gm, nan=0.0)
    if fault == "pad_as_zero":
        Gm[:M, N:] = 0.0                           # the item side of the padding is W = 0 anyway
    gh, gl = _split(Gm)
    if fault == "g_hi_only":
        gl = torch.zeros_like(gl)
    out = {}
    skip = None

    def run(Ghi, Glo, Yhi, Ylo, RX, RY):
        _, n_y, n_splits, tps = plan_ce_tc(RX, RY)
        n_y = _cdiv(Yhi.shape[0], BM)
        sk = n_y // 2 if fault == "skip_tile" else None
        res = torch.zeros((Ghi.shape[0], kp), dtype=torch.float64)
        for sp in range(n_splits):
            acc = torch.zeros_like(res)
            for t in range(sp * tps, min((sp + 1) * tps, n_y)):
                if t == sk:
                    continue
                for k0 in range(t * BM, (t + 1) * BM, 16):
                    acc = _mma_acc(acc, Ghi, Glo, Yhi, Ylo, k0, k0 + 16)
            res = f32(res + f32(f32(acc) * gscale))
        return res[:, :d]

    if "d_h" in passes:
        r = torch.arange(M) if rows is None else rows
        out["d_h"] = run(gh[r], gl[r], wh, wl, plan_M or M, N)
    if "d_W" in passes:
        dW = run(gh.t()[:N], gl.t()[:N], hh, hl, N, M)
        G_sum = Gm.sum(0)[:N]
        if fault == "skip_tile":
            sk = _cdiv(M, BM) // 2
            G_sum = G_sum - Gm[sk * BM:(sk + 1) * BM, :N].sum(0)
        db = f32(G_sum * gscale)
        out["d_W"] = dW if prefill_W is None else f32(dW + prefill_W.double())
        out["d_bias"] = db if prefill_b is None else f32(db + prefill_b.double())
    return out
