"""The decoder-body tensor-core GEMMs against the per-element bound of tests/gemm_cases.py, on worst-case bf16 rounding:
``linear_tc`` (epilogues 0 and 1 element by element, epilogue 2 through the LayerNorm band of tests/ln_cases.py), the
four GEMMs of the fused decoder chain one stage at a time and as a whole, and the chain's operand-image writers, which
must put exactly split8 of the chain's own fp32 q, k and v where the attention kernel reads them and nothing anywhere
else.  Also the ``resid`` alignment rule of ``irs_linear_tc``.  The largest err/band per kernel and case kind is printed
at the end (pytest -s)."""
import functools

import numpy as np
import pytest
import torch

from tests import gemm_cases as GC
from tests import chain_cases as CC
from tests import ln_cases as C

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WORST = {}                     # (kernel, case kind) -> largest err / band
OLD = {}                       # kernel -> largest err / (3e-5 sum |a||w|) on the hard elements


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


def _flag_ok(ops):
    torch.cuda.synchronize()
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def _note(kernel, kind, ratio):
    WORST[(kernel, kind)] = max(WORST.get((kernel, kind), 0.0), float(ratio))


def _note_old(kernel, rel):
    OLD[kernel] = max(OLD.get(kernel, 0.0), float(rel) / GC.OLD_REL)


@functools.lru_cache(maxsize=None)
def _rows(R, K):
    return GC.gemm_rows(R, K)


def _case(R, K, N):
    A, rk = _rows(R, K)
    W, bias, ck = GC.gemm_weights(N, K)
    return GC.GemmCase(A, W, bias, rk, ck)


def _check_elements(kernel, case, got, K, relu, what):
    """got [R, N] on the device against fp64, element by element; records the ratios per case kind."""
    A, W, b = case.A.to(DEV), case.W.to(DEV), case.bias.to(DEV)
    Cref, P = GC.reference(A, W, b)
    band = GC.MARGIN * GC.bound(Cref, P, K)
    want = Cref.clamp_min(0) if relu else Cref
    err = (got.double() - want).abs()
    ratio = err / band
    worst = float(ratio.max())
    if worst > 1.0:
        i = int(ratio.argmax())
        r, j = divmod(i, ratio.shape[1])
        raise AssertionError(f"{what}: element ({r}, {j}) rows {GC.ROW_KINDS[case.row_kind[r]]} col "
                             f"{GC.COL_KINDS[case.col_kind[j]]}: err {float(err.flatten()[i]):.3e} band "
                             f"{float(band.flatten()[i]):.3e} (ratio {worst:.3f})")
    masks = {"hard": GC.hard_mask(case), "cancel": GC.cancel_mask(case), "control": GC.control_mask(case)}
    masks["other"] = ~(masks["hard"] | masks["cancel"] | masks["control"])
    for kind, m in masks.items():
        if m.any():
            _note(kernel, kind, ratio[torch.from_numpy(m).to(DEV)].max())
    if masks["hard"].any() and not relu:
        _note_old(kernel, (err / P)[torch.from_numpy(masks["hard"]).to(DEV)].max())


# ---------------------------------------------------------------------------------------------- linear_tc
def _slice(t, pad=4):
    """t as a column slice of a wider row-major buffer (leading dimension + 2 pad, 16-byte aligned start)."""
    R, n = t.shape
    wide = torch.full((R, n + 2 * pad), float("nan"), device=DEV)
    wide[:, pad:pad + n] = t
    return wide, wide[:, pad:pad + n]


@pytest.mark.parametrize("N", GC.NOUTS)
@pytest.mark.parametrize("K", GC.KS)
def test_linear_tc_bias_and_relu(ops, K, N):
    """Epilogues 0 and 1, every R of gemm_cases.RS; A and C are contiguous for R = 1 and 129, column slices of wider
    buffers for R = 127 and the multi-pass R."""
    for i, R in enumerate(GC.RS):
        case = _case(R, K, N)
        prep = ops.linear_prepare(case.W.to(DEV))
        sliced = i % 2 == 1
        A = case.A.to(DEV)
        if sliced:
            _, A = _slice(A)
        for epi in (ops.EPI_BIAS, ops.EPI_BIAS_RELU):
            wide, out = _slice(torch.empty((R, N), device=DEV)) if sliced else (None, None)
            got = ops.linear_tc(A, prep, N, case.bias.to(DEV), epi, out=out)
            _flag_ok(ops)
            if sliced:
                assert torch.isnan(wide[:, :4]).all() and torch.isnan(wide[:, 4 + N:]).all()   # nothing outside C
            _check_elements(f"linear_tc epi{epi}", case, got, K, epi == ops.EPI_BIAS_RELU, f"epi {epi} R {R} K {K} N {N}")


@pytest.mark.parametrize("N", GC.NOUTS)
@pytest.mark.parametrize("K", GC.KS)
def test_linear_tc_layernorm(ops, K, N):
    """Epilogue 2, LN(resid + A W^T + bias) [-> LN(. + c2)], per row within ln_band with prod = sum |a||w| and G(K)."""
    eps = 1e-5
    g1, b1 = C.ln_params(N)
    g2, b2 = C.ln_params(N, seed=1)
    c2 = np.full(N, 3.0, np.float32)
    d = lambda a: torch.as_tensor(a, dtype=torch.float32, device=DEV)
    for R in (1, 129, GC.RS[-1]):
        case = _case(R, K, N)
        prep = ops.linear_prepare(case.W.to(DEV))
        resid = torch.randn((R, N), generator=torch.Generator().manual_seed(R + N))
        _, rs = _slice(resid.to(DEV))
        Cref, P = GC.reference(case.A.to(DEV), case.W.to(DEV), case.bias.to(DEV))
        t = (Cref + resid.double().to(DEV)).cpu().numpy()
        prod = P.max(1).values.cpu().numpy()
        band1 = C.ln_band(t, g1, b1, eps, prod=prod, k=K)
        want1 = C.ln64(t, g1, b1, eps)
        got1 = ops.linear_tc(case.A.to(DEV), prep, N, case.bias.to(DEV), ops.EPI_RESID_LN, resid=rs, g1=d(g1), b1=d(b1),
                             eps=eps)
        got2 = ops.linear_tc(case.A.to(DEV), prep, N, case.bias.to(DEV), ops.EPI_RESID_LN, resid=rs, g1=d(g1), b1=d(b1),
                             c2=d(c2), g2=d(g2), b2=d(b2), eps=eps)
        _flag_ok(ops)
        t2 = want1 + c2
        band2 = C.ln_band(t2, g2, b2, eps, upstream=band1)
        for name, got, want, band in (("LN1", got1, want1, band1), ("LN2", got2, C.ln64(t2, g2, b2, eps), band2)):
            r = C.row_err(got.cpu().numpy(), want) / band
            assert r.max() <= 1.0, f"{name} R {R} K {K} N {N}: row {int(r.argmax())} " \
                                   f"({GC.ROW_KINDS[case.row_kind[int(r.argmax())]]}) err/band {r.max():.3f}"
            for i, kind in enumerate(GC.ROW_KINDS):
                if (case.row_kind == i).any():
                    _note(f"linear_tc epi2 {name}", kind, r[case.row_kind == i].max())


def test_linear_tc_rejects_misaligned_resid(ops):
    """Epilogue 2 reads resid with 16-byte vector loads: a resid pointer off 16 bytes, or a leading dimension that is not
    a multiple of 4, is refused with IRS_E_SHAPE (-2) before anything is launched."""
    R, K, N = 64, 32, 128
    A = torch.randn((R, K), device=DEV)
    prep = ops.linear_prepare(torch.randn((N, K), device=DEV))
    wide = torch.randn((R, N + 8), device=DEV)
    g1, b1 = torch.ones(N, device=DEV), torch.zeros(N, device=DEV)
    out = torch.empty((R, N), device=DEV)
    lib = ops.lib()
    flag = ops._ptr(ops._error_flag(A.device))

    def call(resid_ptr, ldr):
        return lib.irs_linear_tc(A.data_ptr(), K, prep.data_ptr(), None, 2, resid_ptr, ldr, g1.data_ptr(), b1.data_ptr(),
                                 None, None, None, 1e-5, out.data_ptr(), N, R, K, N, flag, ops._stream())
    assert call(wide.data_ptr() + 4, N + 8) == -2
    assert call(wide.data_ptr() + 8, N + 8) == -2
    assert call(wide.data_ptr(), N + 2) == -2
    assert call(wide.data_ptr() + 16, N + 8) == 0
    _flag_ok(ops)


@pytest.mark.parametrize("N", [128, 120])
def test_linear_tc_unaligned_resid_view(ops, N):
    """ops.linear_tc copies a resid view that breaks the alignment rule; the result equals the contiguous one."""
    R, K = 300, 128
    g = torch.Generator().manual_seed(N)
    A = torch.randn((R, K), generator=g).to(DEV)
    prep = ops.linear_prepare((torch.randn((N, K), generator=g) / 11).to(DEV))
    wide = torch.randn((R, N + 3), generator=g).to(DEV)            # leading dimension not a multiple of 4
    wide4 = torch.randn((R, N + 4), generator=g).to(DEV)           # leading dimension fine, start off 16 bytes
    g1, b1 = torch.ones(N, device=DEV), torch.zeros(N, device=DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    for view in (wide[:, 1:1 + N], wide[:, 3:3 + N], wide4[:, 1:1 + N], wide4[:, 2:2 + N]):
        got = ops.linear_tc(A, prep, N, bias, ops.EPI_RESID_LN, resid=view, g1=g1, b1=b1)
        want = ops.linear_tc(A, prep, N, bias, ops.EPI_RESID_LN, resid=view.contiguous(), g1=g1, b1=b1)
        _flag_ok(ops)
        assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------- decoder chain
D_, F_ = CC.D, CC.F


def _run_chain(ops, attn, x, P, with_qkv=True, inplace=False, **kw):
    Pd = {k: torch.as_tensor(v, device=DEV) for k, v in P.items()}
    xd = torch.as_tensor(x, device=DEV).clone()
    prep = ops.decoder_chain_prepare(Pd["Wo"], Pd["W1"], Pd["W2"], Pd["Win"] if with_qkv else None)
    got_x, got_q = ops.decoder_chain_tc(torch.as_tensor(attn, device=DEV), xd, prep, Pd["bo"], Pd["g1"], Pd["b1"],
                                        Pd["c2"], Pd["g2"], Pd["b2"], Pd["bf1"], Pd["bf2"], Pd["g3"], Pd["b3"],
                                        Pd["bin"] if with_qkv else None, x_out=xd if inplace else None, **kw)
    _flag_ok(ops)
    if inplace:
        assert got_x.data_ptr() == xd.data_ptr()
    return got_x, got_q, prep


def _check_rows(kernel, kinds, got, want, band, what):
    r = C.row_err(got.cpu().numpy() if torch.is_tensor(got) else got, want) / band
    w = int(r.argmax())
    assert r.max() <= 1.0, f"{what}: row {w} ({kinds[w] if kinds is not None else ''}) err/band {r.max():.3f}"
    if kinds is None:
        _note(kernel, "hard", r.max())
        return
    for kind in set(kinds):
        _note(kernel, kind, r[np.asarray(kinds) == kind].max())


B3_KINDS = ("worst+", "worst+-", "gauss", "scaled", "dominant", "cancel+")


def _row_of(kind, K, seed=0):
    A, rk = _rows(len(GC.ROW_KINDS) * 2, K)
    return A[int(np.nonzero(rk == GC.ROW_KINDS.index(kind))[0][seed])].numpy()


@pytest.mark.parametrize("kind", B3_KINDS)
def test_chain_in_proj_stage(ops, kind):
    """g3 = 0 makes x' = b3 exactly: the next layer's in_proj (K = 128) is observed raw in qkv_out, element by element,
    with b3 a hard row and Win of worst-rounding and scaled columns (the q, k and v blocks of different scales)."""
    R = 300
    P = CC.gauss_params(11)
    P["g3"] = np.zeros(D_, np.float32)
    P["b3"] = _row_of(kind, D_)
    P["Win"], P["bin"] = CC.weights(3 * D_, D_)
    attn = np.random.default_rng(1).standard_normal((R, D_)).astype(np.float32)
    x = np.random.default_rng(2).standard_normal((R, D_)).astype(np.float32)
    got_x, got_q, _ = _run_chain(ops, attn, x, P)
    assert torch.equal(got_x.cpu(), torch.from_numpy(P["b3"]).expand(R, D_))
    A = torch.from_numpy(P["b3"]).expand(R, D_).contiguous()
    case = GC.GemmCase(A, torch.from_numpy(P["Win"]), torch.from_numpy(P["bin"]),
                       np.full(R, GC.ROW_KINDS.index(kind)), np.arange(3 * D_) % len(GC.COL_KINDS))
    _check_elements("chain in_proj", case, got_q, D_, False, f"in_proj, b3 {kind}")


@pytest.mark.parametrize("stage", CC.STAGES)
def test_chain_stage(ops, stage):
    """One GEMM stage carries the error, seen through LN3 (tests/chain_cases.py): linear2 (K = 256) on an exact
    worst-rounding relu output, linear1 (K = 128) on X3 rows read back through a 0/1 selection W2, out_proj (K = 128)
    on hard attn rows.  tests/test_chain_cases_cpu.py shows that an FFN or out_proj dropping lo*hi leaves this band."""
    attn, x, P, kinds = CC.stage_case(stage)
    want_x, band_x, _, _ = C.chain_bands(attn, x, P)
    got_x, _, _ = _run_chain(ops, attn, x, P, with_qkv=False)
    _check_rows(f"chain stage {stage} (LN3 band)", kinds, got_x, want_x, band_x, f"{stage} stage")


@pytest.mark.parametrize("R,inplace", [(333, False), (333, True), (148 * 128 * 2 + 77, True), (128 * 5, False)])
def test_chain_whole_on_hard_inputs(ops, R, inplace):
    """All four GEMMs with worst-rounding and scaled weights and hard attn rows, x' and qkv' against the propagated
    bands of ln_cases.chain_bands, with and without x' aliasing x."""
    P = CC.gauss_params(14)
    P["Wo"], P["bo"] = CC.weights(D_, D_)
    P["W1"], P["bf1"] = CC.weights(F_, D_)
    P["W2"], P["bf2"] = CC.weights(D_, F_)
    P["Win"], P["bin"] = CC.weights(3 * D_, D_)
    A, rk = _rows(R, D_)
    attn = A.numpy()
    x = np.random.default_rng(R).standard_normal((R, D_)).astype(np.float32)
    want_x, band_x, want_q, band_q = C.chain_bands(attn, x, P)
    got_x, got_q, _ = _run_chain(ops, attn, x, P, inplace=inplace)
    kinds = [GC.ROW_KINDS[k] for k in rk]
    _check_rows("chain whole x'", kinds, got_x, want_x, band_x, f"R {R} x'")
    _check_rows("chain whole qkv'", kinds, got_q, want_q, band_q, f"R {R} qkv'")


# ---------------------------------------------------------------------------------------------- operand images
SENTINEL = 0xA5
H = 4


def _decode(images, B, L, mode):
    """(hi, lo) int16 bit patterns [B*L, 384] of every token's q | k | v, and a mask of the bytes that hold them."""
    img = images.cpu().numpy()
    off = GC.image_offsets(B, L, H, mode)
    lo_off = off + np.where(np.arange(off.shape[-1]) < 4 * H, GC.Q_PART, GC.K_PART)
    words = img.view(np.int16)
    e = np.arange(8)
    hi = words[(off[..., None] // 2) + e].reshape(B * L, -1)
    lo = words[(lo_off[..., None] // 2) + e].reshape(B * L, -1)
    used = np.zeros(img.size, bool)
    for o in (off, lo_off):
        used[(o.reshape(-1)[:, None] + np.arange(16)).reshape(-1)] = True
    return torch.from_numpy(hi.copy()), torch.from_numpy(lo.copy()), used, img


def _bits_to_f64(b):
    return b.view(torch.bfloat16).double()


def _interval_distance(hi, lo, target):
    """Distance from target to the fp32 values whose split8 is (hi, lo): hi + lo +- half a bf16 spacing of lo."""
    h, l_ = _bits_to_f64(hi), _bits_to_f64(lo)
    sp = torch.where(l_ != 0, torch.exp2(torch.floor(torch.log2(l_.abs().clamp_min(1e-300))) - 7), torch.zeros_like(l_))
    return ((h + l_ - target).abs() - sp / 2).clamp_min(0)


def _sentinel_images(ops, B, L):
    n = ops.lib().irs_qkv_images_bytes(B, L, H, 32)
    assert n > 0
    return torch.full((n,), SENTINEL, dtype=torch.uint8, device=DEV)


def _image_inputs(L, mode):
    B = 2
    R = B * L
    rng = np.random.default_rng(L * 3 + mode)
    attn = rng.standard_normal((R, D_)).astype(np.float32)
    x = rng.standard_normal((R, D_)).astype(np.float32)
    return B, attn, x, CC.gauss_params(100 + L + mode)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("L", [129, 160, 161, 192, 193, 223])
def test_chain_images_are_split8_of_qkv(ops, L, mode):
    """k and v halves bit-equal to split8 of the same kernel's fp32 qkv_out; q (bin_q = 0) bit-equal to split8 of
    fl32(qkv_out log2(e)/sqrt(32)), and with bin_q != 0 within the two roundings of the folded FFMA; every byte no
    token maps to still holds the sentinel."""
    B, attn, x, P = _image_inputs(L, mode)
    for q_bias in (False, True):
        if not q_bias:
            P["bin"][:D_] = 0.0
        else:
            P["bin"][:D_] = np.random.default_rng(L).standard_normal(D_).astype(np.float32)
        x1, qkv, _ = _run_chain(ops, attn, x, P)
        images = _sentinel_images(ops, B, L)
        x2, im, _ = _run_chain(ops, attn, x, P, qkv_images=images, L=L, mask_mode=mode)
        assert torch.equal(x1, x2)
        hi, lo, used, raw = _decode(im, B, L, mode)
        assert (raw[~used] == SENTINEL).all(), f"{int((raw[~used] != SENTINEL).sum())} bytes outside the map written"
        q = qkv.cpu()
        kh, kl = GC.split8_bits(q[:, D_:])
        assert torch.equal(hi[:, D_:], kh) and torch.equal(lo[:, D_:], kl), "k / v halves differ from split8(qkv_out)"
        s = float(GC.QSCALE)
        if not q_bias:
            qh, ql = GC.split8_bits(q[:, :D_] * torch.tensor(GC.QSCALE))
            assert torch.equal(hi[:, :D_], qh) and torch.equal(lo[:, :D_], ql), "q halves differ from split8(fl(qkv s))"
        else:
            target = q[:, :D_].double() * s
            sb = (torch.from_numpy(P["bin"][:D_]).double() * s).abs()
            tol = GC.MARGIN * GC.U32 * (2 * target.abs() + sb)
            dist = _interval_distance(hi[:, :D_], lo[:, :D_], target)
            assert (dist <= tol).all(), f"q off by {float((dist / tol).max()):.2f} of two fp32 roundings"
            _note("chain q image (folded scale)", "ulp", float((dist / tol).max()))


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("L", [129, 161, 223])
def test_in_proj_images(ops, L, mode):
    """irs_in_proj_images_tc: q, k and v halves decode to within the G(128) band of fp64 x Win^T + bin (q scaled), the
    sentinel survives everywhere else."""
    B, _, x, P = _image_inputs(L, mode)
    P["Win"], P["bin"] = CC.weights(3 * D_, D_)
    Pd = {k: torch.as_tensor(v, device=DEV) for k, v in P.items()}
    prep = ops.decoder_chain_prepare(Pd["Wo"], Pd["W1"], Pd["W2"], Pd["Win"])
    images = _sentinel_images(ops, B, L)
    ops.in_proj_images_tc(torch.as_tensor(x, device=DEV), prep, Pd["bin"], images, L, mode)
    _flag_ok(ops)
    hi, lo, used, raw = _decode(images, B, L, mode)
    assert (raw[~used] == SENTINEL).all()
    Cref, Pp = GC.reference(torch.from_numpy(x), torch.from_numpy(P["Win"]), torch.from_numpy(P["bin"]))
    band = GC.MARGIN * GC.bound(Cref, Pp, D_)
    scale = torch.ones(3 * D_, dtype=torch.float64)
    scale[:D_] = float(GC.QSCALE)
    target = Cref * scale
    tol = band * scale + GC.MARGIN * 2 * GC.U32 * target.abs() * (scale != 1)
    ratio = _interval_distance(hi, lo, target) / tol
    assert float(ratio.max()) <= 1.0, float(ratio.max())
    _note("in_proj images", "q", ratio[:, :D_].max())
    _note("in_proj images", "k,v", ratio[:, D_:].max())


def test_zz_report():
    """Largest err/band per kernel and case kind of the tests above (run with -s to see it)."""
    print("\nlargest err/band per kernel and case kind:")
    for (kernel, kind), r in sorted(WORST.items()):
        print(f"  {kernel:36s} {kind:10s} {r:.3f}")
    for kernel, r in sorted(OLD.items()):
        print(f"  {kernel:36s} hard elements: err / (3e-5 sum|a||w|) up to {r:.3f}")
