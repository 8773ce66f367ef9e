"""The GEMM bound of tests/gemm_cases.py, checked on the float64 emulator (no device): the kernel's arithmetic stays inside
the derived bound (half the band) on every case and shape with the accumulator rounded either way, the worst-rounding elements use a large part of
the bound and exceed the suite's earlier 3e-5, and emulations that drop a product term leave the band.  So the GPU tests
(tests/test_gpu_gemm_bounds.py) can tell a correct kernel from one that loses a term."""
import numpy as np
import pytest
import torch

from tests import gemm_cases as GC

R_CPU = (1, 128, 129)


def _ratios(case, K, mode="rn", terms=("lohi", "hilo", "hihi")):
    C, P = GC.reference(case.A, case.W, case.bias)
    err = (GC.emulate(case.A, case.W, case.bias, mode, terms).double() - C).abs()
    return (err / GC.bound(C, P, K)).numpy(), (err / P).numpy()


def test_bound_constants():
    assert GC.G(16) == GC.G(4) < GC.G(36) < GC.G(128) < GC.G(256)
    assert abs(GC.G(256) - (3 * 2.0 ** -16 * (1 + 2.0 ** -7) + 48 * 2.0 ** -23)) < 1e-15
    x, y, rel = GC.worst_pair()
    assert 3.0e-5 < abs(rel) < 3 * GC.U ** 2                       # the worst product, inside the product part of G


def test_cases_cover_every_kind_in_one_tile():
    case = GC.gemm_case(128, 36, 24)
    assert set(case.row_kind.tolist()) == set(range(len(GC.ROW_KINDS)))
    assert set(case.col_kind.tolist()) == set(range(len(GC.COL_KINDS)))
    C, P = GC.reference(case.A, case.W, case.bias)
    cancel = GC.cancel_mask(case)
    assert cancel.any() and ((C.abs() / P).numpy()[cancel] < 2e-4).all()
    assert GC.hard_mask(case).any() and GC.control_mask(case).any()
    scales = case.A.abs().amax(1)
    assert scales.max() / scales.min() > 1e5                         # rows from ~1e-3 to ~1e3
    cs = case.W.abs().amax(1)
    assert cs.max() / cs.min() > 1e5


@pytest.mark.parametrize("K", GC.KS)
@pytest.mark.parametrize("N", GC.NOUTS)
def test_emulator_inside_the_bound(K, N):
    for R in R_CPU:
        case = GC.gemm_case(R, K, N)
        for mode in ("rn", "rz"):
            r, _ = _ratios(case, K, mode)
            assert r.max() <= 1.0, (R, mode, float(r.max()))              # the band on the GPU is MARGIN x this


@pytest.mark.parametrize("K", GC.KS)
def test_worst_rounding_is_hard_and_controls_are_not(K):
    """Hard elements reach at least half of the derived bound (a quarter of the band with its margin); the N(0,1)
    controls stay below that.  Every hard element loses more than 3e-5 sum |a||w|: the old constant is not a bound."""
    case = GC.gemm_case(128, K, 256)
    hard, ctrl = GC.hard_mask(case), GC.control_mask(case)
    for mode in ("rn", "rz"):
        r, rel = _ratios(case, K, mode)
        assert r[hard].min() >= 0.5, (mode, float(r[hard].min()))
        assert r[ctrl].max() < 0.4, (mode, float(r[ctrl].max()))
        assert rel[hard].min() > GC.OLD_REL, (mode, float(rel[hard].min()))


@pytest.mark.parametrize("K", GC.KS)
@pytest.mark.parametrize("terms", [("hihi",), ("hilo", "hihi")])
def test_dropped_terms_leave_the_band(K, terms):
    """hi*hi alone, or hi*hi + hi*lo without lo*hi, leaves the band on every hard element and on controls."""
    case = GC.gemm_case(128, K, 256)
    r, _ = _ratios(case, K, "rn", terms)
    band = r / GC.MARGIN
    assert band[GC.hard_mask(case)].min() > 10.0
    assert band[GC.control_mask(case)].max() > 2.0


def test_image_addressing_is_a_bijection():
    """The port of qkv_image.cuh maps every (token, piece) to its own 16 bytes, inside its item."""
    for L in (129, 160, 161, 192, 193, 223):
        for mode in (0, 1, 2):
            off = GC.image_offsets(2, L, 4, mode)
            flat = np.concatenate([off.ravel(), off[..., :16].ravel() + GC.Q_PART, off[..., 16:].ravel() + GC.K_PART])
            assert len(np.unique(flat)) == flat.size
            assert (flat % 16 == 0).all() and flat.max() < 2 * 4 * GC.ITEM_BYTES


def test_split8_bits_reassemble():
    x = torch.randn(1000) * 10.0 ** torch.randint(-3, 4, (1000,)).float()
    hi, lo = GC.split8_bits(x)
    h = hi.view(torch.bfloat16).double()
    l_ = lo.view(torch.bfloat16).double()
    assert ((h + l_ - x.double()).abs() <= 2.0 ** -16 * x.double().abs()).all()
