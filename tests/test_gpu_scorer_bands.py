"""The tensor-core scorers on the worst-case inputs of tests/band_cases.py: every decision must be the fp32 engine's,
bit for bit (winners, values and tie order), and the fp64 oracle's wherever its margin exceeds fp32 noise (all cases
here lead by >= 5e-4).  A band that is too narrow drops the true winner before the exact re-score and returns the decoy."""
import math

import pytest
import torch

from tests import band_cases as B

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


def _dev(case, ops):
    h, W = case.h.to(DEV), case.W.to(DEV)
    b = None if case.bias is None else case.bias.to(DEV)
    e = None if case.excl is None else ops.sort_exclusions(case.excl.to(DEV), case.N, 1)
    return h, W, b, e


def _healthy(ops):
    torch.cuda.synchronize()
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def _same(got, want, expected, name):
    gv, gi = got
    wv, wi = want
    assert torch.equal(wi.cpu(), expected), f"{name}: fp32 engine disagrees with the fp64 oracle"
    assert torch.equal(gi, wi), f"{name}: tensor-core items {gi[:, -1].tolist()[:4]} != fp32 engine {wi[:, -1].tolist()[:4]}"
    assert torch.equal(gv, wv), f"{name}: tensor-core values differ from the fp32 engine's"


@pytest.mark.parametrize("variant", [2, 10, 0, 4])
@pytest.mark.parametrize("d", [30, 64, 128])
@pytest.mark.parametrize("placement", B.PLACEMENTS)
@pytest.mark.parametrize("use_bias", [True, False])
def test_argmax_single_mma_pair(ops, d, placement, use_bias, variant):
    """Variants 2 / 10: one bf16 MMA, the single-MMA band; 0 / 4: three MMAs (the same cases are easy for them)."""
    case = B.argmax_pair(d, placement, use_bias)
    h, W, b, e = _dev(case, ops)
    want = ops.score_topk(h, W, b, 1, e, 1)
    got = ops.score_argmax_tc(h, W, ops.scorer_prepare_weights(W), b, e, 1, variant=variant)
    _same(got, want, case.expected, case.name)
    _healthy(ops)


@pytest.mark.parametrize("variant", [0, 4, 2, 10])
@pytest.mark.parametrize("d", [30, 64, 128])
def test_argmax_three_mma_pair(ops, d, variant):
    """|h| |W| ~ 2e3 with |s| ~ 1: the three-MMA band must scale with |h| |W|, not with |s|."""
    case = B.argmax_three(d)
    h, W, b, e = _dev(case, ops)
    want = ops.score_topk(h, W, b, 1, e, 1)
    got = ops.score_argmax_tc(h, W, ops.scorer_prepare_weights(W), b, e, 1, variant=variant)
    _same(got, want, case.expected, case.name)
    _healthy(ops)


@pytest.mark.parametrize("variant", [2, 0])
@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("use_bias", [True, False])
def test_argmax_sharded_pair(ops, d, use_bias, variant):
    """Phase 1 per shard -> MAX of the leaders -> phase 2 per shard -> topk_merge, with j and j' in different shards."""
    case = B.sharded_pair(d, use_bias)
    h, W, b, _ = _dev(case, ops)
    want = ops.score_topk(h, W, b, 1, None, 1)
    bounds = [(0, case.shard_at), (case.shard_at, case.N)]
    leads, state = [], []
    for lo, hi in bounds:
        Wg = W[lo:hi].contiguous()
        bg = None if b is None else b[lo:hi].contiguous()
        prep = ops.scorer_prepare_weights(Wg)
        lead, ws = ops.score_argmax_tc_phase1(h, Wg, prep, bg, None, lo + 1, variant=variant)
        leads.append(lead)
        state.append((Wg, bg, prep, ws, lo))
    lead_g = torch.stack(leads).max(0).values
    vals, items = [], []
    for Wg, bg, prep, ws, lo in state:
        v, i = ops.score_argmax_tc_phase2(h, Wg, prep, bg, None, lo + 1, lead_g, ws, variant=variant)
        vals.append(v)
        items.append(i)
    got = ops.topk_merge(torch.stack(vals), torch.stack(items))
    _same(got, want, case.expected, case.name)
    _healthy(ops)


@pytest.mark.parametrize("d", [30, 64, 128, 256])
@pytest.mark.parametrize("k", [5, 50])
@pytest.mark.parametrize("use_bias", [True, False])
def test_topk_boundary_pair(ops, d, k, use_bias):
    case = B.topk_boundary(d, k, use_bias)
    h, W, b, e = _dev(case, ops)
    want = ops.score_topk(h, W, b, k, e, 1)
    got = ops.score_topk_tc(h, W, ops.scorer_prepare_weights(W), b, k, e, 1)
    _same(got, want, case.expected, case.name)
    _healthy(ops)


def test_topk_any_pair(ops, monkeypatch):
    """A catalog of 40,000 items: score_topk_any picks the tensor-core top-k by itself."""
    case = B.topk_any_case()
    assert case.N >= ops.TC_TOPK_MIN_ITEMS and ops.score_topk_tc_supported(case.d, case.k)
    h, W, b, e = _dev(case, ops)
    monkeypatch.setattr(ops, "USE_TC_TOPK", False)
    want = ops.score_topk_any(h, W, b, case.k, e, 1)
    monkeypatch.setattr(ops, "USE_TC_TOPK", True)
    got = ops.score_topk_any(h, W, b, case.k, e, 1)
    _same(got, want, case.expected, case.name)
    _healthy(ops)


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("crowded", [False, True])
def test_rank_three_mma(ops, d, crowded, monkeypatch):
    case = B.rank_three(d, crowded)
    h, W, b, _ = _dev(case, ops)
    lab = case.label.to(DEV)
    monkeypatch.setattr(ops, "USE_TC_RANK", False)
    want = ops.score_rank(h, W, b, lab, None, 1)
    monkeypatch.setattr(ops, "USE_TC_RANK", True)
    got = ops.score_rank(h, W, b, lab, None, 1)
    assert torch.equal(want.cpu(), case.expected)
    assert torch.equal(got, want), (got.tolist(), want.tolist())
    _healthy(ops)


@pytest.mark.parametrize("tc", [True, False])
@pytest.mark.parametrize("d", [64, 128])
def test_count_ahead_three_mma_across_shards(ops, d, tc, monkeypatch):
    """rank = 1 + sum over two catalog shards of score_count_ahead, label score = MAX of score_select, on the tensor-core
    count-ahead (tc) and on the fp32 engine."""
    monkeypatch.setattr(ops, "USE_TC_RANK", tc)
    case = B.rank_three(d, False)
    h, W, b, _ = _dev(case, ops)
    lab = case.label.to(DEV)
    bounds = [(0, case.shard_at), (case.shard_at, case.N)]
    assert any(c >= case.shard_at for c in case.ahead) and any(c < case.shard_at for c in case.ahead)
    score = torch.full((case.M,), -math.inf, device=DEV)
    for lo, hi in bounds:
        score = torch.maximum(score, ops.score_select(h, W[lo:hi], b[lo:hi], lab.view(-1, 1), lo + 1)[:, 0])
    total = torch.zeros((case.M,), dtype=torch.int64, device=DEV)
    for lo, hi in bounds:
        Ws, bs = W[lo:hi].contiguous(), b[lo:hi].contiguous()
        c, f = ops.score_count_ahead(h, Ws, bs, lab, score, None, lo + 1)
        assert int(f.sum()) == 0
        total += c
    assert torch.equal((total + 1).cpu(), case.expected)
    _healthy(ops)


def _probe_inputs(K):
    """Rows of A and W whose partial sums all have one sign: the worst coherent three-MMA value X3 at one scale, X3 at
    scales spread over 2^0 .. 2^-12 (the accumulator aligns ever smaller terms), and random fp32 values in [1, 2)."""
    g = torch.Generator().manual_seed(7)
    A = [torch.full((K,), B.X3), B.X3 * 2.0 ** -(torch.arange(K) % 13).double(), 1 + torch.rand(K, generator=g, dtype=torch.float64),
         B.X3 * 2.0 ** -(torch.arange(K) * 12 // K).double()]
    Wr = [torch.full((K,), B.X3), torch.full((K,), B.X3), 1 + torch.rand(K, generator=g, dtype=torch.float64),
          B.X3 * 2.0 ** -(torch.arange(K) % 7).double()]
    A = torch.stack([a.float() for a in A] * 64)                                   # 256 rows
    Wm = torch.stack([w.float() for w in Wr] * 32 + [(1 + torch.rand(K, generator=g)) for _ in range(128)])   # 256 outputs
    return A, Wm


def test_three_mma_accumulation_probe(ops):
    """linear_tc (epilogue 0, no bias) runs the same split8 and the same bf16 x3 tcgen05.mma kind as the scorer.  With
    every partial sum of one sign, |out - exact three-MMA sum| / sum_k |a_k w_k| is the tensor core's own fp32
    accumulation error; three_mma_band() budgets 3 K / 16 2^-23 for it (one truncation per K = 16 MMA)."""
    K = 128
    A, Wm = _probe_inputs(K)
    out = ops.linear_tc(A.to(DEV), ops.linear_prepare(Wm.to(DEV)), Wm.shape[0], None, 0).cpu().double()
    _healthy(ops)
    exact = A.double() @ Wm.double().t()
    three = B.score_three(A, Wm).double()              # exact sum of the three products, rounded once to fp32
    ah, al = B.split_hi_lo(A)
    wh, wl = B.split_hi_lo(Wm)
    three_exact = ah @ wh.t() + ah @ wl.t() + al @ wh.t()
    mag = A.double().abs() @ Wm.double().abs().t()
    acc = float(((out - three_exact).abs() / mag).max())
    total = float(((out - exact).abs() / mag).max())
    budget = 3 * K // 16 * 2.0 ** -23
    assert float(((three - three_exact).abs() / mag).max()) <= 2.0 ** -24
    assert acc <= budget, f"tensor-core accumulation error {acc:.3e} of sum|a w| exceeds the budget {budget:.3e}"
    assert total <= B.NEW_THREE, f"three-MMA error {total:.3e} of sum|a w| exceeds three_mma_band's {B.NEW_THREE:.1e}"
    print(f"\naccumulation probe K={K}: accumulation error {acc:.3e}, total three-MMA error {total:.3e} "
          f"(of sum|a w|; budget {budget:.3e} / {B.NEW_THREE:.1e})")
