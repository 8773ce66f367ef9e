"""tests/ce_cases.py without a GPU: every case has the property its regime advertises, the float64 emulator of the
tensor-core backward stays inside the bound, and each seeded fault of that emulator leaves the bound on some case -- which
is what makes the bound worth asserting on the GPU (tests/test_gpu_ce_bounds.py)."""
import math

import pytest
import torch

from tests import ce_cases as C

SHAPES = [(129, 300, 64), (300, 1000, 30), (260, 640, 128), (40, 127, 16), (1, 300, 64), (200, 1, 16), (128, 129, 100)]


def _lse_scores(c):
    s = C.scores64(c.h, c.W, c.bias)
    return s, torch.logsumexp(s, 1)


def test_plan_branches():
    """The ported plan() of scorer_ce_tc.cu at the shapes the GPU tests rely on."""
    assert C.plan_ce_tc(37760, 5000) == (295, 40, 2, 20)           # d_h: two splits
    assert C.plan_ce_tc(37888, 5000) == (296, 40, 1, 40)           # d_h: owner path
    assert C.plan_ce_tc(5000, 37760) == (40, 295, 8, 37)           # d_W: 8 splits, the last one 36 tiles
    assert C.plan_ce_tc(700, 40000) == (6, 313, 20, 16)            # d_h split 20 ways, the last split 9 tiles
    assert C.plan_ce_tc(40000, 700) == (313, 6, 1, 6)
    assert C.plan_ce_tc(200704, 500000) == (1568, 3907, 16, 256)   # cfg4 d_h: runs of <= 256 tiles, not one of 3,907
    assert C.plan_ce_tc(500000, 200704) == (3907, 1568, 7, 256)    # cfg4 d_W
    assert C.plan_ce_tc(37888, 40000) == (296, 313, 2, 256)        # owner-sized X, split only by the run cap


def test_cases_have_their_regimes():
    c = C.mixed_case(300, 1000, 64, 11)
    s, lse = _lse_scores(c)
    mx = s.max(1).values
    live = c.target >= 0
    loss = torch.where(live, lse - s[torch.arange(c.M), c.target.clamp(min=0)], torch.zeros_like(lse))
    assert (c.target == 0).any() and (c.target == c.N - 1).any() and (c.target == -1).any()
    big, small = c.rows(C.LARGE_POS), c.rows(C.LARGE_NEG)
    assert big and small
    assert float(mx[big].min()) >= C.LARGE - 1e-3 > C.EXP_LIMIT
    assert float(mx[small].max()) <= -C.LARGE + 1e-3
    for m, delta in c.lead.items():
        t = int(c.target[m])
        other = s[m].clone()
        other[t] = -math.inf
        assert abs(float(s[m, t] - other.max()) - delta) < 1e-4
    p40 = [m for m, dl in c.lead.items() if dl == 40.0]
    p1 = [m for m, dl in c.lead.items() if dl == 1.0]
    assert p40 and p1
    assert float(loss[p40].max()) < 1e-15                           # p_t = 1 - O(1e-17)
    assert 0.05 < float(loss[p1].min()) and float(loss[p1].max()) < 1.0
    tail = [m for m in c.rows(C.POP_TAIL) if c.target[m] >= 0]
    assert tail and 30 <= float(loss[tail].min()) and float(loss[tail].max()) <= 50
    assert float(c.bias.max() - c.bias.min()) >= 30                   # popularity: tens of nats
    ties = c.rows(C.TIES)
    assert ties
    for m in ties:
        p = torch.exp(s[m] - lse[m])
        assert float(p[c.target[m]]) > 0.25                          # shared with its two copies
    # anisotropic: half of E|W_j|^2 in the shared direction; rows |h| ~ sqrt(d) with an offset
    W = c.W.double()
    W = W[W.norm(dim=1) < 3]                                         # without the two worst-rounding items
    mu = W.mean(0)
    assert 0.35 < float(mu @ mu) / float((W * W).sum(1).mean()) < 0.65
    hn = c.h.double()[c.rows(C.ANISO)]
    assert 0.8 * math.sqrt(c.d) < float(hn.norm(dim=1).mean()) < 1.6 * math.sqrt(c.d)
    assert float(hn.mean(0).norm()) > 0.3 * math.sqrt(c.d)
    # worst rounding: the three-MMA score error on the X3 / C_DN pairs is a good part of NEW_THREE sum_k |h_k W_jk|
    from tests.band_cases import score_three
    for r in (C.WORST_X3, C.WORST_DN):
        m = c.rows(r)[0]
        j = int(c.target[m])
        err = abs(float(score_three(c.h[m:m + 1], c.W[j:j + 1]).double()) - float(c.h[m].double() @ c.W[j].double()))
        assert err > 0.2 * C.NEW_THREE * float(C.abs_dot(c.h[m:m + 1], c.W[j:j + 1]))
    # selected ids: 0, past the catalog, negative, first, last
    assert {0, c.N + 1, -3, c.N, 1} <= set(c.sel[:, 1].tolist())


def test_every_tile_mixes_the_regimes():
    c = C.mixed_case(1000, 640, 64, 11)
    for t0 in range(0, c.M - 127, 128):
        assert len(set(c.regime[t0:t0 + 128].tolist())) >= 7


@pytest.mark.parametrize("M,N,d", SHAPES)
def test_emulator_inside_bound(M, N, d):
    c = C.mixed_case(M, N, d, 11)
    lse = C.forward_ref(c.h, c.W, c.bias, c.sel)[0].float()
    gscale = 1.0 / M
    out = C.backward_bound(c.h, c.W, c.bias, c.target, lse, gscale, "tc")
    emu = C.emulate_tc_backward(c.h, c.W, c.bias, c.target, lse, gscale)
    for k in out:
        assert C.ratio(emu[k], *out[k]) <= 1.0, k


def test_emulator_inside_bound_with_prefill_and_splits():
    """700 users x 5,000 items: the d_h pass splits 3 ways (red.global), d_W and d_bias are accumulated into."""
    c = C.mixed_case(700, 5000, 64, 13)
    assert C.plan_ce_tc(700, 5000)[2] == 3
    lse = C.forward_ref(c.h, c.W, c.bias, c.sel)[0].float()
    g = torch.Generator().manual_seed(1)
    pW, pb = torch.randn((c.N, c.d), generator=g) * 1e-3, torch.randn(c.N, generator=g) * 1e-3
    out = C.backward_bound(c.h, c.W, c.bias, c.target, lse, 1 / 700, "tc", prefill_W=pW, prefill_b=pb)
    emu = C.emulate_tc_backward(c.h, c.W, c.bias, c.target, lse, 1 / 700, prefill_W=pW, prefill_b=pb)
    for k in out:
        assert C.ratio(emu[k], *out[k]) <= 1.0, k


def _fault_cases():
    return [C.mixed_case(129, 300, 64, 11), C.mixed_case(300, 1000, 30, 11), C.control_case(129, 300, 64, 3),
            C.control_case(129, 300, 64, 3, h_scale=1 / 16)]


@pytest.mark.parametrize("fault", C.FAULTS)
def test_seeded_fault_leaves_the_bound(fault):
    worst = 0.0
    for c in _fault_cases():
        lse = C.forward_ref(c.h, c.W, c.bias, c.sel)[0].float()
        out = C.backward_bound(c.h, c.W, c.bias, c.target, lse, 1.0 / c.M, "tc")
        emu = C.emulate_tc_backward(c.h, c.W, c.bias, c.target, lse, 1.0 / c.M, fault=fault)
        worst = max(worst, max(C.ratio(emu[k], *out[k]) for k in out))
    assert worst > 2.0, f"fault {fault}: at most {worst:.3g} x the bound"


def test_forward_bound_separates_a_dropped_tile():
    """The forward bound is tight enough that losing one 128-item tile of a 1,000-item catalog (or counting the padded
    columns of the last tile as score 0) leaves it, on the fp32 engine and on the tensor cores."""
    c = C.mixed_case(129, 1000, 64, 11)
    s = C.scores64(c.h, c.W, c.bias)
    lse = torch.logsumexp(s, 1)
    dropped = torch.logsumexp(s[:, 128:], 1)
    padded = torch.logsumexp(torch.cat([s, torch.zeros((c.M, 1024 - 1000), dtype=s.dtype)], 1), 1)
    for engine in ("simt", "tc"):
        b, _ = C.forward_bound(c.h, c.W, c.bias, c.sel, engine)
        assert C.ratio(dropped, lse, b) > 2 and C.ratio(padded, lse, b) > 2, engine


def test_training_shape_prediction():
    """The emulator at the training shape's d_h sweep (N = 500,000: 3,907 item tiles, 93,768 truncating MMAs into one
    accumulator) on four rows: anisotropic and confident.  Predicts the tensor-core d_h error before a GPU runs it: inside
    the bound and the north star."""
    N, d, M = 500000, 128, 200704
    c = C.training_case(8, N, d, 21)
    rows = torch.tensor([0, 2, 3, 7])                                  # lift 0, 4, 10, 25 (x sqrt(d) / 4)
    h, tgt = c.h, c.target
    lse = torch.logsumexp(C.scores64(h, c.W, c.bias), 1).float()
    gscale = 1.0 / M
    # the emulator's d_h pass for these rows (a shortened copy of emulate_tc_backward without the d_W pass)
    emu = C.emulate_tc_backward(h[rows], c.W, c.bias, tgt[rows], lse[rows], gscale, passes=("d_h",), plan_M=M)["d_h"]
    ref, bound = C.backward_bound(h[rows], c.W, c.bias, tgt[rows], lse[rows], gscale, "tc", plan_M=M)["d_h"]
    err = (emu - ref).abs()
    print(f"\npredicted cfg4 d_h (tensor cores): max|err| / max|ref| = {float(err.max() / ref.abs().max()):.3e}, "
          f"err / bound {C.ratio(emu, ref, bound):.3f}")
    assert C.ratio(emu, ref, bound) <= 1.0
    assert float(err.max()) <= C.NORTH_STAR * float(ref.abs().max())
