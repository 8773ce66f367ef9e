"""LayerNorms of the inference decoder on rows whose mean is large next to their spread, against fp64 within the per-row
band of tests/ln_cases.py: the fp32 ``residual_layernorm``, ``linear_tc`` epilogue 2 (LN1, optional LN2), each of the
three LayerNorms of the fused decoder chain, and a whole IRN whose biases carry a common offset on every route."""
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import irn_oracle as O
from tests import ln_cases as C
from tests.helpers import assert_close_rel, RTOL

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PROD = 0.01                    # the matrix-product term of t, next to the row's spread


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


def _d(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(DEV)


def _check(got, want, band, what, ratio=None):
    err = C.row_err(got.detach().cpu().numpy() if torch.is_tensor(got) else got, want)
    bad = np.nonzero(err > band)[0]
    if len(bad):
        w = bad[np.argmax((err / band)[bad])]
        where = "" if ratio is None else f", |mean|/std {ratio[w]:.3g}"
        raise AssertionError(f"{what}: {len(bad)} of {len(err)} rows outside the band; worst row {w}{where}: "
                             f"err {err[w]:.3e} band {band[w]:.3e}")


# ---------------------------------------------------------------------------------------------- residual_layernorm
@pytest.mark.parametrize("two", [False, True])
@pytest.mark.parametrize("eps", [1e-5, 1e-8])
@pytest.mark.parametrize("placement", ["row", "bias"])
@pytest.mark.parametrize("d", [30, 64, 128, 256, 1000])
def test_residual_layernorm_large_mean(ops, d, placement, eps, two):
    """The fp32 kernel already takes two passes: the control of this file."""
    for sign in (1.0, -1.0):
        rows = C.ln_rows(d, placement, sign)
        rng = np.random.default_rng(d)
        y = (rng.standard_normal(rows.x.shape) * rows.scale[:, None] * PROD).astype(np.float32)
        g1, b1 = C.ln_params(d)
        g2, b2 = C.ln_params(d, seed=1)
        c2 = np.full(d, -sign * 1e3, np.float32)
        t = rows.x.astype(np.float64) + y + rows.bias
        band1 = C.ln_band(t, g1, b1, eps)
        if not two:
            got = ops.residual_layernorm(_d(rows.x), _d(y), _d(rows.bias), _d(g1), _d(b1), eps=eps)
            _check(got, C.ln64(t, g1, b1, eps), band1, f"{rows.name} LN1", rows.ratio)
            continue
        got = ops.residual_layernorm(_d(rows.x), _d(y), _d(rows.bias), _d(g1), _d(b1), _d(c2), _d(g2), _d(b2), eps=eps)
        t2 = C.ln64(t, g1, b1, eps) + c2
        _check(got, C.ln64(t2, g2, b2, eps), C.ln_band(t2, g2, b2, eps, upstream=band1), f"{rows.name} LN2", rows.ratio)


# ---------------------------------------------------------------------------------------------- linear_tc epilogue 2
@pytest.mark.parametrize("two", [False, True])
@pytest.mark.parametrize("placement", ["row", "bias"])
@pytest.mark.parametrize("K,Nout", [(32, 16), (120, 120), (128, 128), (256, 256)])
def test_linear_tc_layernorm_large_mean(ops, K, Nout, placement, two):
    """LN(resid + A W^T + bias) [-> LN(. + c2)], the offset in ``resid`` or ``bias``; Nout 120 ends in a partial chunk."""
    eps = 1e-5
    for sign in (1.0, -1.0):
        rows = C.ln_rows(Nout, placement, sign)
        rng = np.random.default_rng(K + Nout)
        A = (rng.standard_normal((rows.x.shape[0], K)) * rows.scale[:, None] * PROD).astype(np.float32)
        W = (rng.standard_normal((Nout, K)) / math.sqrt(K)).astype(np.float32)
        g1, b1 = C.ln_params(Nout)
        g2, b2 = C.ln_params(Nout, seed=1)
        c2 = np.full(Nout, sign * 1e3, np.float32)
        t = rows.x.astype(np.float64) + A.astype(np.float64) @ W.astype(np.float64).T + rows.bias
        band1 = C.ln_band(t, g1, b1, eps, prod=C.abs_prod(A, W), k=K)
        prep = ops.linear_prepare(_d(W))
        if not two:
            got = ops.linear_tc(_d(A), prep, Nout, _d(rows.bias), ops.EPI_RESID_LN, resid=_d(rows.x), g1=_d(g1), b1=_d(b1),
                                eps=eps)
            _check(got, C.ln64(t, g1, b1, eps), band1, f"{rows.name} K{K} LN1", rows.ratio)
        else:
            got = ops.linear_tc(_d(A), prep, Nout, _d(rows.bias), ops.EPI_RESID_LN, resid=_d(rows.x), g1=_d(g1), b1=_d(b1),
                                c2=_d(c2), g2=_d(g2), b2=_d(b2), eps=eps)
            t2 = C.ln64(t, g1, b1, eps) + c2
            _check(got, C.ln64(t2, g2, b2, eps), C.ln_band(t2, g2, b2, eps, upstream=band1), f"{rows.name} K{K} LN2",
                   rows.ratio)
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


# ---------------------------------------------------------------------------------------------- decoder chain
CHAIN = [("ln1", "row", 1.0), ("ln1", "bias", 1.0), ("ln1", "bias", -1.0), ("ln2", None, 300.0), ("ln2", None, -1e3),
         ("ln2", None, 1e4), ("ln3", None, -100.0), ("ln3", None, 1e3), ("ln3", None, 1e4)]


def _chain_case(stage, placement, v, R=333, d=128, ffn=256):
    """Inputs of one chain call with exactly one LayerNorm conditioned: LN1 through x (placement "row") or bo ("bias",
    v = sign), LN2 through c2 = v, LN3 through bf2 = v.  The GEMM terms are small next to the spread of each row."""
    rng = np.random.default_rng(CHAIN.index((stage, placement, v)))
    f32 = lambda a: np.asarray(a, np.float32)
    rn = lambda *s: rng.standard_normal(s)
    if stage == "ln1":
        rows = C.ln_rows(d, placement, v, R=R)
        x, bo, scale, ratio = rows.x, rows.bias, rows.scale, rows.ratio
    else:
        x, bo, scale, ratio = f32(rn(R, d)), f32(0.1 * rn(d)), np.ones(R), None
    P = {"Wo": f32(rn(d, d) / math.sqrt(d)), "bo": bo, "g1": f32(1 + 0.1 * rn(d)), "b1": f32(0.1 * rn(d)),
         "c2": f32(np.full(d, v) if stage == "ln2" else 0.3 * rn(d)), "g2": f32(1 + 0.1 * rn(d)), "b2": f32(0.1 * rn(d)),
         "W1": f32(rn(ffn, d) / d), "bf1": f32(0.1 * rn(ffn)), "W2": f32(rn(d, ffn) / (2 * ffn)),
         "bf2": f32(np.full(d, v) if stage == "ln3" else 0.1 * rn(d)), "g3": f32(1 + 0.1 * rn(d)), "b3": f32(0.1 * rn(d)),
         "Win": f32(rn(3 * d, d) / math.sqrt(d)), "bin": f32(0.1 * rn(3 * d))}
    attn = f32(rn(R, d) * scale[:, None] * PROD)
    return attn, x, P, ratio


@pytest.mark.parametrize("with_qkv,inplace", [(True, False), (False, True), (True, True)])
@pytest.mark.parametrize("stage,placement,v", CHAIN)
def test_decoder_chain_layernorms_large_mean(ops, stage, placement, v, with_qkv, inplace):
    """One of LN1 / LN2 / LN3 conditioned at a time, R = 333 (a partial tile), in place or not, with and without the
    next layer's in_proj; x' and qkv' against the same fp64 chain."""
    attn, x, P, ratio = _chain_case(stage, placement, v)
    want_x, band_x, want_q, band_q = C.chain_bands(attn, x, P)
    Pd = {k: _d(a) for k, a in P.items()}
    xd = _d(x)
    prep = ops.decoder_chain_prepare(Pd["Wo"], Pd["W1"], Pd["W2"], Pd["Win"] if with_qkv else None)
    got_x, got_q = ops.decoder_chain_tc(_d(attn), xd, prep, Pd["bo"], Pd["g1"], Pd["b1"], Pd["c2"], Pd["g2"], Pd["b2"],
                                        Pd["bf1"], Pd["bf2"], Pd["g3"], Pd["b3"], Pd["bin"] if with_qkv else None,
                                        x_out=xd if inplace else None)
    torch.cuda.synchronize()
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0
    _check(got_x, want_x, band_x, f"chain {stage} {placement} {v:g}: x'", ratio)
    if with_qkv:
        _check(got_q, want_q, band_q, f"chain {stage} {placement} {v:g}: qkv'", ratio)
    else:
        assert got_q is None
    if inplace:
        assert got_x.data_ptr() == xd.data_ptr()


# ---------------------------------------------------------------------------------------------- model level
OFFSET = 200.0


def _offset_irn(pkg, L, seed):
    """IRN d = 128, ffn = 256, 2 layers, 4 heads; +OFFSET on self_attn.out_proj.bias, multihead_attn.out_proj.bias (so on
    the folded cross-attention constant c2) and linear2.bias of every layer.  The offsets live only inside LayerNorm
    inputs: the normalised outputs, and the attention scores, keep their usual scale."""
    N, U_ = 3000, 30
    cfg = SimpleNamespace(n_item=N, n_user=U_, max_len=L, n_layers=2, n_heads=4, emb_dim=128, u_emb_dim=10, ffn_dim=256,
                          dropout=0.0, lr1=1e-3)
    sd = O.synth_irn_state(N, U_, L, 128, 2, 256, seed=seed)
    for i in range(2):
        for k in ("self_attn.out_proj.bias", "multihead_attn.out_proj.bias", "linear2.bias"):
            sd[f"decoder.layers.{i}.{k}"] += OFFSET
    net = pkg.InfluentialNet(cfg)
    net.load_state_dict(sd)
    net.to(DEV).eval()
    g = torch.Generator().manual_seed(seed + 1)
    B = 6
    seqs = torch.zeros((B, L), dtype=torch.long)
    for b in range(B):
        n = L if b < 2 else int(torch.randint(L // 4, L + 1, (1,), generator=g))
        seqs[b, L - n:] = torch.randperm(N, generator=g)[:n] + 1
    users = torch.randint(0, U_, (B,), generator=g)
    return cfg, sd, net, seqs, users


@pytest.fixture(scope="module")
def pkg(ops):
    import influentialrs_b200 as p
    return p


@pytest.mark.parametrize("route", ["fused", "linear_tc", "residual_layernorm"])
@pytest.mark.parametrize("L", [201, 60])
def test_irn_decoding_with_offset_biases(pkg, monkeypatch, L, route):
    """net.decoding against the fp64 oracle at RTOL: the fused chain (image attention at L = 201), the linear_tc tail
    (USE_FUSED_CHAIN off) and residual_layernorm (no tensor-core linears)."""
    from influentialrs_b200 import irn
    if route != "fused":
        monkeypatch.setattr(irn, "USE_FUSED_CHAIN", False)
    if route == "residual_layernorm":
        monkeypatch.setattr(irn, "_tc_ok", lambda d, ffn: False)
    cfg, sd, net, seqs, users = _offset_irn(pkg, L, 21 + L)
    with torch.no_grad():
        h = net.decoding(seqs.to(DEV), users.to(DEV)).cpu()
    want, _ = O.irn_decoding(O.to_dtype(sd, torch.float64), seqs, users, 4, fold_cross=True)
    ok = seqs.ne(0)
    assert_close_rel(h[ok], want[ok], RTOL, f"decoder with +{OFFSET:g} biases, {route}, L={L}")


@pytest.mark.parametrize("L", [201, 60])
def test_irn_generation_with_offset_biases(pkg, L):
    """Greedy generation on the fused route against the fp64 oracle wherever the decision margins exceed fp32 noise."""
    cfg, sd, net, seqs, users = _offset_irn(pkg, L, 41 + L)
    irn_ = pkg.IRSNN(cfg, net, DEV)
    P = 4
    want, _, _, _, margins = O.generate_paths(O.to_dtype(sd, torch.float64), seqs, users, seqs[:, -1], 4, P,
                                              return_margins=True, fold_cross=True)
    got, _, _, _ = irn_.get_seq_in_batch(seqs.to(DEV), users.to(DEV), seqs[:, -1].to(DEV), max_path_len=P, gap_len=0)
    safe = margins.min(1) > 1e-4
    assert safe.mean() > 0.5
    for b in np.nonzero(safe)[0]:
        np.testing.assert_array_equal(got[b], want[b])
