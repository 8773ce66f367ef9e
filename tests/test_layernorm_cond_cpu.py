"""The LayerNorm error band of tests/ln_cases.py, checked on the fp32 emulators (no device): two-pass and Chan-merged
statistics stay inside it on every case, and the one-pass E[t^2] - mean^2 leaves it at every |mean|/std the GPU tests
(tests/test_gpu_layernorm_cond.py) rely on, in both the linear_tc and the decoder-chain layouts.  So the GPU tests can
tell the two apart."""
import math

import numpy as np
import pytest

from tests import ln_cases as C

WIDTHS = (30, 64, 120, 128, 256, 1000)
CASES = [(n, pl, sg) for n in WIDTHS for pl in ("row", "bias") for sg in (1.0, -1.0)]


def _layouts(n):
    """(method, layout) pairs of a width: residual_layernorm takes any width, linear_tc Nout <= 256, the chain 128.  The
    plain two-pass over a whole row, one sequential sum (no kernel here does it), is checked up to n = 128: the rounding
    error of its mean grows with n, which the per-chunk and per-lane sums of the kernels avoid."""
    out = [("two-pass", "warp")]
    if n <= 128:
        out += [("two-pass", "row")]
    if n <= 256:
        out += [("chan", "row")]
    if n == 128:
        out += [("two-pass", "pair"), ("chan", "pair")]
    return out


def _ln1(n, pl, sg, eps):
    rows = C.ln_rows(n, pl, sg)
    g, b = C.ln_params(n)
    prod = np.random.default_rng(5).standard_normal(rows.x.shape) * rows.scale[:, None] * 0.01
    prod[np.isinf(rows.ratio)] = 0.0                                    # constant rows stay constant
    t64 = rows.t64 + prod
    return rows, g, b, t64, C.emulate_input(rows, prod), C.ln64(t64, g, b, eps), C.ln_band(t64, g, b, eps)


def _ratio_groups(rows):
    return [q for q in C.RATIOS if q >= C.DISCRIMINATING and np.isclose(rows.ratio, q, rtol=0.05).any()]


def test_cases_cover_the_hard_rows():
    rows = C.ln_rows(128, "row", 1.0)
    assert np.isinf(rows.ratio).any()                                    # constant rows
    for q in C.RATIOS:
        assert np.isclose(rows.ratio, q, rtol=0.05).sum() >= 6          # each ratio, both signs, several rows
    ill = rows.ratio[:128] >= 30
    assert ill[0::2].sum() > 20 and not ill[1::2].any()                 # interleaved inside one 128-row tile
    mean = rows.t64.mean(1)
    assert (mean[0::2] > 0).any() and (mean[0::2] < 0).any()
    b = C.ln_rows(128, "bias", -1.0)
    assert (b.bias == -200.0).all() and np.isclose(b.ratio, 1e4, rtol=0.05).any()


@pytest.mark.parametrize("eps", [1e-5, 1e-8])
@pytest.mark.parametrize("n,pl,sg", CASES)
def test_two_pass_and_chan_stay_inside_the_band(n, pl, sg, eps):
    rows, g, b, t64, t, want, band = _ln1(n, pl, sg, eps)
    for meth, lay in _layouts(n):
        err = C.row_err(C.emulate_ln(t, g, b, eps, meth, lay), want)
        worst = int(np.argmax(err / band))
        assert (err <= band / C.KAPPA_MARGIN).all(), \
            f"{meth}/{lay}: row {worst} (|mean|/std {rows.ratio[worst]:.3g}) err {err[worst]:.3e} band {band[worst]:.3e}"
    const = np.isinf(rows.ratio)
    if pl == "row" and const.any():                                     # a constant row comes out as b
        for meth, lay in _layouts(n):
            out = C.emulate_ln(t, g, b, eps, meth, lay)[const]
            assert np.abs(out.astype(np.float64) - b).max() <= C.ln_band(t64, g, b, eps)[const].max()


@pytest.mark.parametrize("eps", [1e-5, 1e-8])
@pytest.mark.parametrize("n,pl,sg", [c for c in CASES if c[0] <= 256])
def test_one_pass_leaves_the_band(n, pl, sg, eps):
    rows, g, b, t64, t, want, band = _ln1(n, pl, sg, eps)
    groups = _ratio_groups(rows)
    assert groups
    for lay in ("row", "pair") if n == 128 else ("row",):
        r = C.row_err(C.emulate_ln(t, g, b, eps, "one-pass", lay), want) / band
        for q in groups:
            m = np.isclose(rows.ratio, q, rtol=0.05)
            assert r[m].max() > 3.0, f"one-pass/{lay} stays inside the band at |mean|/std = {q:g}"


def _ln2(n, c2, lay, method):
    """LN2(LN1(t) + c2): LN1 of mixed rows, then the common offset c2 (folded into b1 in the chain, as V_B1 does)."""
    eps = 1e-5
    rows, g1, b1, t64, t, want1, band1 = _ln1(n, "row", 1.0, eps)
    g2, b2 = C.ln_params(n, seed=1)
    c2v = np.full(n, c2, np.float32)
    if lay == "pair":
        y1 = C.emulate_ln(t, g1, (b1 + c2v).astype(np.float32), eps, method, lay)
    else:
        y1 = (C.emulate_ln(t, g1, b1, eps, method, lay) + c2v).astype(np.float32)
    t2 = want1 + c2v.astype(np.float64)
    want = C.ln64(t2, g2, b2, eps)
    band = C.ln_band(t2, g2, b2, eps, upstream=band1)
    return C.row_err(C.emulate_ln(y1, g2, b2, eps, method, lay), want), band


@pytest.mark.parametrize("c2", [30.0, -1e3, 1e4])
@pytest.mark.parametrize("n,lay", [(128, "pair"), (128, "row"), (256, "row"), (120, "row")])
def test_second_layernorm_offset_by_c2(n, lay, c2):
    err, band = _ln2(n, c2, lay, "chan")
    assert (err <= band / C.KAPPA_MARGIN).all()
    err, band = _ln2(n, c2, lay, "one-pass")
    assert (err / band).max() > 3.0


def test_kappa_has_its_margin():
    """KAPPA is KAPPA_MARGIN times (at least) the largest error of the two-pass and Chan emulators on these cases."""
    worst = 0.0
    for n, pl, sg in CASES:
        rows, g, b, t64, t, want, band = _ln1(n, pl, sg, 1e-5)
        unit = band / C.KAPPA
        for meth, lay in _layouts(n):
            worst = max(worst, float((C.row_err(C.emulate_ln(t, g, b, 1e-5, meth, lay), want) / unit).max()))
    assert 4.0 < worst <= C.KAPPA / C.KAPPA_MARGIN, worst


@pytest.mark.parametrize("placement", ["row", "bias"])
@pytest.mark.parametrize("K,Nout", [(32, 16), (120, 120), (128, 128), (256, 256)])
def test_one_pass_leaves_the_band_with_the_product_term(K, Nout, placement):
    """The linear_tc cases of tests/test_gpu_layernorm_cond.py, band and all: the tensor-core product term (2 G(K) P,
    up to about a fifth of the band at |mean|/std = 30) does not hide the one-pass statistics."""
    import math
    eps = 1e-5
    for sign in (1.0, -1.0):
        rows = C.ln_rows(Nout, placement, sign)
        rng = np.random.default_rng(K + Nout)
        A = (rng.standard_normal((rows.x.shape[0], K)) * rows.scale[:, None] * 0.01).astype(np.float32)
        W = (rng.standard_normal((Nout, K)) / math.sqrt(K)).astype(np.float32)
        g, b = C.ln_params(Nout)
        prod64 = A.astype(np.float64) @ W.astype(np.float64).T
        t64 = rows.t64 + prod64
        band = C.ln_band(t64, g, b, eps, prod=C.abs_prod(A, W), k=K)
        r = C.row_err(C.emulate_ln(C.emulate_input(rows, prod64), g, b, eps, "one-pass", "row"), C.ln64(t64, g, b, eps)) / band
        for q in _ratio_groups(rows):
            assert r[np.isclose(rows.ratio, q, rtol=0.05)].max() > 3.0, f"one-pass inside the band at |mean|/std = {q:g}"
