"""The worst-case constructions of tests/band_cases.py mean what they claim, checked without a GPU: the fp64 order (and the
emulated fp32 engine's, which the GPU tests compare bit for bit) puts the true winner first, the emulated tensor-core
scores put it outside the OLD error band of the leader by the stated ratio, and inside the corrected band."""
import math

import pytest
import torch

from tests import band_cases as B


def test_bf16_unit_roundoff_is_2_to_the_minus_8():
    for c, direction in ((B.C_DN, -1), (B.C_UP, 1)):
        x = torch.tensor([c], dtype=torch.float32)
        rel = float((B.bf16_rn(x) - x.double()) / x.double())
        assert direction * rel > 0.99 * B.U                    # not 2^-9, as the old single-MMA band assumed
    hi, lo = B.split_hi_lo(torch.tensor([B.X3], dtype=torch.float32))
    assert float(hi) == 1 + 2 ** -7 and float(lo) == -2 ** -8


def test_worst_three_mma_value_is_the_search_optimum():
    """X3 * X3 loses 2u^2 of the product in the three-MMA scheme, 2.65x the old budget of 3 * 2^-18."""
    x, y, rel = B.worst_three_mma_value()
    assert x == y == B.X3
    assert abs(rel) > 1.98 * B.U ** 2 and abs(rel) / B.OLD_THREE_LOST > 2.6
    assert abs(rel) <= 3 * B.U ** 2 * (1 + 2 * B.U)            # the lost-terms part of the corrected band


def test_plan_and_placements():
    assert B.plan(2100, 70000) == (17, 274, 35, 8)
    assert B.plan(130, 70000)[2:] == (4, 69)
    for d in (30, 64, 128):
        seg = B.argmax_pair(d, "segment", True)
        a, b = B.locate(seg.win, seg.M, seg.N), B.locate(seg.decoy, seg.M, seg.N)
        assert a[:2] == b[:2] and a[3] == b[3] and a[2] != b[2]        # same split, segment and half; other chunk
        segs = B.argmax_pair(d, "segments", False)
        a, b = B.locate(segs.win, segs.M, segs.N), B.locate(segs.decoy, segs.M, segs.N)
        assert a[0] == b[0] and a[1] != b[1] and abs(segs.win - segs.decoy) >= 4096
        spl = B.argmax_pair(d, "splits", True)
        assert spl.M >= 130 and B.plan(spl.M, spl.N)[0] == 2
        assert B.locate(spl.win, spl.M, spl.N)[0] != B.locate(spl.decoy, spl.M, spl.N)[0]
        tail = B.argmax_pair(d, "tail", False)
        assert tail.N % 32 and tail.win // 32 == (tail.N - 1) // 32
        ex = B.argmax_pair(d, "excluded", True)
        hidden = int(ex.excl[0, 0]) - 1
        assert hidden // 32 == ex.win // 32
        s = B.score_fp64(ex.h[:1], ex.W, ex.bias)[0]
        t = B.score_hihi(ex.h[:1], ex.W, ex.bias)[0]
        assert s[hidden] > s[ex.win] and t[hidden] > t[ex.decoy]      # above both, exactly and on the tensor core
        sh = B.sharded_pair(d, False) if d != 30 else None
        if sh is not None:
            assert sh.win < sh.shard_at <= sh.decoy


def _check_pair(case, min_old_ratio):
    a = B.analyse_pair(case)
    rows = case.rows
    assert torch.equal(a.fp64_top, case.expected[rows]), "fp64 order"
    assert torch.equal(a.engine_top, a.fp64_top), "fp32 engine order"
    assert int(case.expected[rows[0], -1]) == case.win + 1 and case.decoy + 1 not in case.expected[rows[0]].tolist()
    assert a.fp64_margin > 4e-4
    assert case.win // B.CHUNK != case.decoy // B.CHUNK
    assert a.old_ratio >= min_old_ratio, f"{case.name}: tensor-core gap is only {a.old_ratio:.3f}x the old band"
    assert a.new_ratio < 1.0, f"{case.name}: tensor-core gap is {a.new_ratio:.3f}x the corrected band"
    return a


@pytest.mark.parametrize("d", [30, 64, 128])
@pytest.mark.parametrize("placement", B.PLACEMENTS)
@pytest.mark.parametrize("use_bias", [True, False])
def test_single_mma_argmax_pair(d, placement, use_bias):
    """With a bias the decoy leads the winner by 1.77..1.83x the old single-MMA band (0.93..0.96 of the corrected one).
    Without a bias the two items need disjoint supports, so Cauchy-Schwarz loses sqrt(2): the lead reaches 1.18x (d = 30)
    .. 1.28x (d = 128) of the old band -- still outside it, but not 1.5x."""
    _check_pair(B.argmax_pair(d, placement, use_bias), 1.5 if use_bias else 1.15)


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("use_bias", [True, False])
def test_sharded_pair(d, use_bias):
    """Same ratios as the unsharded pair: phase 2 bands around the global leader with the largest weight norm of any shard."""
    _check_pair(B.sharded_pair(d, use_bias), 1.5 if use_bias else 1.15)


@pytest.mark.parametrize("d", [30, 64, 128, 256])
@pytest.mark.parametrize("k", [5, 50])
@pytest.mark.parametrize("use_bias", [True, False])
def test_topk_boundary_pair(d, k, use_bias):
    """tau (the k-th largest chunk maximum) is the decoy's; the winner's chunk lies 1.77..1.83x (bias) / 1.18..1.29x (no
    bias) the old band below it."""
    _check_pair(B.topk_boundary(d, k, use_bias), 1.5 if use_bias else 1.15)


def test_topk_any_pair_goes_through_the_tensor_cores():
    case = B.topk_any_case()
    assert case.N >= 32768 and case.k > 1
    _check_pair(case, 1.5)


@pytest.mark.parametrize("d", [30, 64, 128])
def test_three_mma_argmax_pair(d):
    """|h| |W| ~ 2e3 with |s| ~ 1: the decoy leads by ~500x the old band 1e-4 max(1, |s|), and by ~0.45 of the corrected
    band 2 three_mma_band(|h|^2, max |W|^2)."""
    case = B.argmax_three(d)
    hn = float(case.h[0].double().norm())
    wm = float(case.W.double().norm(dim=1).max())
    assert 1e3 <= hn * wm <= 1e4
    assert abs(float(B.score_fp64(case.h[:1], case.W, case.bias)[0, case.win])) < 2
    _check_pair(case, 100.0)


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("crowded", [False, True])
def test_rank_three_mma_pairs(d, crowded):
    """Items truly ahead of the label score below it on the three-MMA tensor-core path, items behind score above it.
    Without accumulation error this cannot leave the old band: it reaches 0.41x of it (the dropped terms alone are 2.65x
    the old budget 3 2^-18 for them); the corrected band holds it at 0.53x."""
    case = B.rank_three(d, crowded)
    a = B.analyse_rank(case)
    assert torch.equal(a.fp64_rank, case.expected[case.rows])
    assert torch.equal(a.engine_rank, a.fp64_rank)
    assert a.wrong_side > 0                                    # the tensor-core order is wrong for some of them
    assert a.lost_ratio > 2.6
    assert 0.35 < a.old_ratio < 1.0
    assert a.new_ratio < 0.6
    if crowded:
        slices = {B.locate(c, case.M, case.N)[0::3] for c in case.ahead + case.behind}
        assert len(slices) == 1 and len(case.ahead) + len(case.behind) > 30


def test_corrected_band_constants():
    """The constants of scorer_tc.cu, re-derived from u = 2^-8."""
    single = 2 * (2 * B.U + B.U ** 2)                          # two scores, each off by (2u + u^2) |h| |W_j|
    acc = 2 * (256 * 2.0 ** -23 + 256 * 2.0 ** -24)            # tensor-core accumulation + engine FMA chain, d <= 256
    assert single + acc < B.NEW_SINGLE < 1.03 * (single + acc)
    assert math.log2(B.NEW_SINGLE) == pytest.approx(-5.97, abs=0.01)
    three = 3 * B.U ** 2 * (1 + 2 * B.U) + 3 * 128 // 16 * 2.0 ** -23 + 128 * 2.0 ** -24
    assert three < B.NEW_THREE < 1.01 * three
    assert B.OLD_SINGLE < single and B.OLD_THREE < three
