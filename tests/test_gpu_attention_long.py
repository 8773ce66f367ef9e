"""Long windows (up to 2048 positions): the key-blocked attention kernels against an fp64 oracle, the routing of the
attention entry points, and the models at windows whose attention no longer fits on chip."""
import math

import numpy as np
import pytest
import torch

from oracle import irn_oracle as O
from oracle.ref_shim import irn_config
from tests.helpers import assert_close_rel, RTOL

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
W_H, W_OBJ = 0.05, 1.0


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


def _oracle(qkv, ids, r_u, H, mode, keep=None, p=0.0):
    """fp64 attention with the mask of include/irs_b200.h; keep (bool [B,H,L,L]) applies dropout after the softmax.
    Returns (out [B,L,d], lse [B,H,L])."""
    B, L, d3 = qkv.shape
    d = d3 // 3
    dh = d // H
    q, k, v = (qkv[..., i * d:(i + 1) * d].reshape(B, L, H, dh).transpose(1, 2) for i in range(3))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
    s = s + (O.pim_mask(L, r_u.reshape(B, 1), W_H, W_OBJ).to(s.dtype).unsqueeze(1) if mode == 0
             else O.causal_mask(L, s.dtype))
    if mode != 2:
        s = s.masked_fill(ids.eq(0)[:, None, None, :], float("-inf"))
    lse = torch.logsumexp(s, -1)
    a = torch.softmax(s, -1)
    if keep is not None:
        a = a * keep.to(a.dtype) / (1 - p)
    return (a @ v).transpose(1, 2).reshape(B, L, d), lse


def _drop_mask(seed, B, H, L, p):
    """The counter-based keep mask of the attention kernels (drop_scale in csrc/attention.cu), restated in numpy."""
    bh = np.arange(B * H, dtype=np.uint64).reshape(B * H, 1, 1)
    i = np.arange(L, dtype=np.uint64).reshape(1, L, 1)
    j = np.arange(L, dtype=np.uint64).reshape(1, 1, L)
    with np.errstate(over="ignore"):
        x = np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * ((bh * np.uint64(L) + i) * np.uint64(L) + j + np.uint64(1))
        x ^= x >> np.uint64(33); x *= np.uint64(0xff51afd7ed558ccd)
        x ^= x >> np.uint64(33); x *= np.uint64(0xc4ceb9fe1a85ec53)
        x ^= x >> np.uint64(33)
    return torch.from_numpy(((x >> np.uint64(32)) >= np.uint64(int(p * 4294967296.0))).reshape(B, H, L, L))


def _case(B, L, H, dh, mode, seed):
    """Random q/k/v over B windows plus the edge windows: pre- and post-padded; in PIM mode one where only the
    objective is visible; with key padding an all-PAD one (NaN rows).  Objective weights r_u include 40 and -80."""
    edits = [lambda i: i[: L // 3].zero_(), lambda i: i[L - L // 4:].zero_()]
    if mode == 0:
        edits.append(lambda i: i[: L - 1].zero_())
    if mode != 2:
        edits.append(lambda i: i.zero_())
    Bt = B + len(edits)
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn((Bt, L, 3 * H * dh), generator=g)
    ids = torch.randint(1, 100, (Bt, L), generator=g)
    r_u = torch.randn(Bt, generator=g)
    r_u[0], r_u[1] = 40.0, -80.0
    for b, f in enumerate(edits):
        f(ids[B + b])
    return qkv, ids, r_u


def _call(ops, fn, qkv, ids, r_u, H, mode, q_row0, n_q, lse=True):
    from influentialrs_b200._lib import lib, check
    B, L, d3 = qkv.shape
    d = d3 // 3
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    out = torch.full((B, n_q, d), 7.0, device=DEV)
    l = torch.full((B, H, n_q), 7.0, device=DEV) if lse else None
    args = (ops._ptr(q), ops._ptr(k), ops._ptr(v), d3, d3, d3, ops._ptr(ids), ops._ptr(r_u) if mode == 0 else None,
            W_H, W_OBJ, mode, ops._ptr(out), ops._ptr(l), B, L, H, d // H, q_row0, n_q)
    if fn.endswith("_tc") or fn.endswith("_tc_blocked"):
        check(getattr(lib(), fn)(*args, ops._ptr(ops._error_flag(qkv.device)), ops._stream()), fn)
    else:
        check(getattr(lib(), fn)(*args, 0.0, 0, ops._stream()), fn)
    torch.cuda.synchronize()
    return out.cpu(), (l.cpu() if lse else None)


def _check(got, want, tol, what):
    o, l = got
    wo, wl = want
    assert torch.equal(torch.isnan(o), torch.isnan(wo)), f"{what}: NaN rows differ"
    ok = ~torch.isnan(wo)
    assert_close_rel(o[ok], wo[ok], tol, what)
    if l is not None:
        fin = torch.isfinite(wl)
        assert torch.equal(torch.isnan(l), ~fin), f"{what}: lse of fully masked rows"
        assert_close_rel(l[fin], wl[fin], tol, what + " lse")


TC_SHAPES = [(2, 224, 2, 32, 0), (2, 257, 4, 32, 0), (2, 300, 2, 16, 1), (2, 512, 4, 32, 0),
             (1, 777, 2, 48, 2), (2, 1024, 2, 64, 0), (1, 2048, 1, 32, 0), (1, 2048, 2, 16, 1)]


@pytest.mark.parametrize("B,L,H,dh,mode", TC_SHAPES)
def test_tc_blocked_forward_against_fp64(ops, B, L, H, dh, mode):
    qkv, ids, r_u = _case(B, L, H, dh, mode, seed=L + dh)
    want_o, want_l = _oracle(qkv.double(), ids, r_u.double(), H, mode)
    dq, di, dr = qkv.to(DEV), ids.to(DEV), r_u.to(DEV)
    for fn in ("irs_pim_attn_fwd_tc", "irs_pim_attn_fwd_tc_blocked"):
        _check(_call(ops, fn, dq, di, dr, H, mode, 0, L), (want_o, want_l), 3e-5, f"{fn} L={L}")
        # one row (generation reads row L-2) and a 5-row subset straddling a 128-row tile boundary
        r = L - 2
        _check(_call(ops, fn, dq, di, dr, H, mode, r, 1), (want_o[:, r:r + 1], want_l[:, :, r:r + 1]), 3e-5, f"{fn} row")
        r = 126
        _check(_call(ops, fn, dq, di, dr, H, mode, r, 5), (want_o[:, r:r + 5], want_l[:, :, r:r + 5]), 3e-5, f"{fn} subset")
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


@pytest.mark.parametrize("L", [1, 2, 12, 127, 128, 129, 201, 223])
@pytest.mark.parametrize("dh,mode", [(32, 0), (16, 1), (64, 2)])
def test_blocked_entry_points_at_short_windows(ops, L, dh, mode):
    """The blocked kernels cover every window length, short ones included: against the oracle and the resident kernels."""
    B, H = 3, 2
    qkv, ids, r_u = _case(B, L, H, dh, mode, seed=100 + L)
    want = _oracle(qkv.double(), ids, r_u.double(), H, mode)
    dq, di, dr = qkv.to(DEV), ids.to(DEV), r_u.to(DEV)
    tc_b = _call(ops, "irs_pim_attn_fwd_tc_blocked", dq, di, dr, H, mode, 0, L)
    tc_r = _call(ops, "irs_pim_attn_fwd_tc", dq, di, dr, H, mode, 0, L)
    f_b = _call(ops, "irs_pim_attn_fwd_blocked", dq, di, dr, H, mode, 0, L)
    f_r = _call(ops, "irs_pim_attn_fwd", dq, di, dr, H, mode, 0, L)
    _check(tc_b, want, 3e-5, "tcgen05 blocked")
    _check(f_b, want, 2e-5, "fp32 blocked")
    _check(tc_b, tc_r, 3e-5, "tcgen05 blocked vs resident")
    _check(f_b, f_r, 2e-5, "fp32 blocked vs resident")
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def _fp32_fwd_bwd(ops, qkv, ids, r_u, H, mode, p, seed, blocked):
    """Forward + backward through the fp32 entry points (blocked or routed), all rows; returns out, d_qkv, d_r_u."""
    from influentialrs_b200._lib import lib, check
    B, L, d3 = qkv.shape
    d = d3 // 3
    dh = d // H
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    out = torch.empty((B, L, d), device=DEV)
    lse = torch.empty((B, H, L), device=DEV)
    rp = ops._ptr(r_u) if mode == 0 else None
    fwd = "irs_pim_attn_fwd_blocked" if blocked else "irs_pim_attn_fwd"
    bwd = "irs_pim_attn_bwd_blocked" if blocked else "irs_pim_attn_bwd"
    check(getattr(lib(), fwd)(ops._ptr(q), ops._ptr(k), ops._ptr(v), d3, d3, d3, ops._ptr(ids), rp, W_H, W_OBJ, mode,
                              ops._ptr(out), ops._ptr(lse), B, L, H, dh, 0, L, float(p), int(seed), ops._stream()), fwd)
    g = torch.Generator().manual_seed(L)
    go = torch.randn((B, L, d), generator=g).to(DEV)
    d_qkv = torch.full_like(qkv, 7.0)                      # written, not accumulated
    d_ru = torch.zeros(B, device=DEV)
    dq, dk, dv = d_qkv[..., :d], d_qkv[..., d:2 * d], d_qkv[..., 2 * d:]
    check(getattr(lib(), bwd)(ops._ptr(q), ops._ptr(k), ops._ptr(v), d3, d3, d3, ops._ptr(ids), rp, W_H, W_OBJ, mode,
                              ops._ptr(out), ops._ptr(lse), ops._ptr(go), ops._ptr(dq), ops._ptr(dk), ops._ptr(dv),
                              ops._ptr(d_ru) if mode == 0 else None, B, L, H, dh, float(p), int(seed), ops._stream()), bwd)
    torch.cuda.synchronize()
    return out.cpu(), d_qkv.cpu(), d_ru.cpu(), go.cpu()


def _ref_fwd_bwd(qkv, ids, r_u, H, mode, go, keep=None, p=0.0):
    a = qkv.double().requires_grad_(True)
    r = r_u.double().requires_grad_(True)
    out, _ = _oracle(a, ids, r, H, mode, keep, p)
    out.backward(go.double())
    return out.detach(), a.grad, r.grad


def _train_case(B, L, H, dh, mode, seed):
    """Windows every row of which sees a key (training never meets a fully masked row): PIM pre-padded, CAUSAL_PAD
    post-padded."""
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn((B, L, 3 * H * dh), generator=g)
    ids = torch.randint(1, 100, (B, L), generator=g)
    for b in range(B):
        if mode == 0:
            ids[b, : (b * 37) % (L - 1)] = 0
        elif mode == 1 and b:
            ids[b, L - (b * 29) % (L - 1):] = 0
    return qkv, ids, torch.randn(B, generator=g)


@pytest.mark.parametrize("B,L,H,dh,mode", [(2, 287, 4, 32, 0), (2, 201, 2, 64, 0), (1, 93, 1, 128, 1),
                                           (2, 700, 6, 5, 0), (1, 1500, 2, 32, 1), (1, 2048, 4, 8, 2)])
def test_fp32_blocked_forward_backward_against_fp64_autograd(ops, B, L, H, dh, mode):
    qkv, ids, r_u = _train_case(B, L, H, dh, mode, seed=L)
    out, d_qkv, d_ru, go = _fp32_fwd_bwd(ops, qkv.to(DEV), ids.to(DEV), r_u.to(DEV), H, mode, 0.0, 0, True)
    want, wa, wr = _ref_fwd_bwd(qkv, ids, r_u, H, mode, go)
    assert_close_rel(out, want, 2e-5, "out")
    assert_close_rel(d_qkv, wa, 5e-5, "d_qkv")
    if mode == 0:
        assert_close_rel(d_ru, wr, 5e-5, "d_r_u")
    # the routed entry points give the same (blocked where the resident layout does not fit)
    out2, d_qkv2, d_ru2, _ = _fp32_fwd_bwd(ops, qkv.to(DEV), ids.to(DEV), r_u.to(DEV), H, mode, 0.0, 0, False)
    assert_close_rel(out2, want, 2e-5, "routed out")
    assert_close_rel(d_qkv2, wa, 5e-5, "routed d_qkv")


@pytest.mark.parametrize("L", [300, 1024])
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_fp32_blocked_dropout_mask_rebuilt_from_seed(ops, L, p):
    B, H, dh, mode = 2, 2, 32, 0
    qkv, ids, r_u = _train_case(B, L, H, dh, mode, seed=L + 1)
    seed = 0x1234567890ABCD + L
    keep = _drop_mask(seed, B, H, L, p)
    out, d_qkv, d_ru, go = _fp32_fwd_bwd(ops, qkv.to(DEV), ids.to(DEV), r_u.to(DEV), H, mode, p, seed, True)
    want, wa, wr = _ref_fwd_bwd(qkv, ids, r_u, H, mode, go, keep, p)
    assert_close_rel(out, want, 2e-5, "dropout out")
    assert_close_rel(d_qkv, wa, 5e-5, "dropout d_qkv")
    assert_close_rel(d_ru, wr, 5e-5, "dropout d_r_u")
    if L <= 300:        # the resident kernels draw the same mask
        out_r, d_qkv_r, _, _ = _fp32_fwd_bwd(ops, qkv.to(DEV), ids.to(DEV), r_u.to(DEV), H, mode, p, seed, False)
        assert_close_rel(out_r, out, 2e-5, "resident vs blocked under dropout")


def test_every_attention_entry_point_rejects_windows_longer_than_2048(ops):
    from influentialrs_b200._lib import lib
    x = torch.zeros((1, 2049, 96), device=DEV)
    ids = torch.ones((1, 2049), dtype=torch.long, device=DEV)
    r = torch.zeros(1, device=DEV)
    o = torch.zeros((1, 2049, 32), device=DEV)
    args = (ops._ptr(x), ops._ptr(x[..., 32:]), ops._ptr(x[..., 64:]), 96, 96, 96, ops._ptr(ids), ops._ptr(r), W_H, W_OBJ, 0,
            ops._ptr(o), ops._ptr(o), 1, 2049, 1, 32, 0, 2049)
    for fn in ("irs_pim_attn_fwd", "irs_pim_attn_fwd_blocked"):
        assert getattr(lib(), fn)(*args, 0.0, 0, None) == -2
    for fn in ("irs_pim_attn_fwd_tc", "irs_pim_attn_fwd_tc_blocked"):
        assert getattr(lib(), fn)(*args, None, None) == -2
    for fn in ("irs_pim_attn_bwd", "irs_pim_attn_bwd_blocked"):
        assert getattr(lib(), fn)(*args[:11], ops._ptr(o), ops._ptr(o), ops._ptr(o), ops._ptr(o), ops._ptr(o), ops._ptr(o),
                                  ops._ptr(r), 1, 2049, 1, 32, 0.0, 0, None) == -2
    assert lib().irs_pim_attn_tc_supported(2048, 32) == 1 and lib().irs_pim_attn_tc_supported(2049, 32) == 0


# ---------------------------------------------------------------------------------------------- routing
def _kernels(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


def _attn_names(names):
    return {n.split("(")[0].split("<")[0].replace("void ", "").replace("irs::", "") for n in names if "attn" in n}


@pytest.mark.parametrize("L,dh,fwd_infer,fwd_train,bwd", [
    (201, 32, {"tcp::pim_attn_row_kernel"}, {"pim_attn_tc_kernel"}, {"pim_attn_bwd_kernel"}),
    (201, 64, {"pim_attn_tc_kernel"}, {"pim_attn_tc_kernel"}, {"pim_attn_bwd_dq_blocked_kernel", "pim_attn_bwd_dkv_blocked_kernel"}),
    (512, 32, {"tcb::pim_attn_tc_blocked_kernel"}, {"tcb::pim_attn_tc_blocked_kernel"},
     {"pim_attn_bwd_dq_blocked_kernel", "pim_attn_bwd_dkv_blocked_kernel"}),
])
def test_routing_by_kernel_name(ops, L, dh, fwd_infer, fwd_train, bwd):
    B, H = 2, 2
    qkv, ids, r_u = _train_case(B, L, H, dh, 0, seed=3)
    qkv, ids, r_u = qkv.to(DEV), ids.to(DEV), r_u.to(DEV)
    with torch.no_grad():
        got = _attn_names(_kernels(lambda: ops.pim_attention(qkv, ids, r_u, H, 0, n_q=1, q_row0=L - 2)))
    assert {n.replace("tca::", "") for n in got} == fwd_infer, got
    a = qkv.clone().requires_grad_(True)
    holder = {}
    got = _attn_names(_kernels(lambda: holder.setdefault("o", ops.pim_attention(a, ids, r_u, H, 0))))
    assert {n.replace("tca::", "") for n in got} == fwd_train, got
    got = _attn_names(_kernels(lambda: holder["o"].backward(torch.ones_like(holder["o"]))))
    assert got == bwd, got


# ---------------------------------------------------------------------------------------------- models
@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import influentialrs_b200 as p
    return p


def _irn(pkg, N, L, n_layers, H, d, ffn, seed, dropout=0.0):
    sd = O.synth_irn_state(n_item=N, n_user=40, max_len=L, d=d, n_layers=n_layers, ffn=ffn, seed=seed)
    cfg = irn_config(N, 40, L, n_layers, H, d, ffn, u_emb_dim=10, dropout=dropout)
    net = pkg.InfluentialNet(cfg)
    net.load_state_dict(sd, strict=True)
    net.to(DEV).eval()
    return sd, net, pkg.IRSNN(cfg, net, DEV)


def _seqs(B, L, N, seed, n_min=20):
    g = torch.Generator().manual_seed(seed)
    seqs = torch.zeros((B, L), dtype=torch.long)
    for b in range(B):
        n = L if b < 2 else int(torch.randint(n_min, L + 1, (1,), generator=g))
        seqs[b, L - n:] = torch.randperm(N, generator=g)[:n] + 1
    return seqs, torch.randint(0, 40, (B,), generator=g)


def test_irn_decoding_at_512(pkg):
    N, L, H = 3000, 512, 4
    sd, net, irn = _irn(pkg, N, L, 2, H, 128, 256, seed=21)
    seqs, users = _seqs(4, L, N, 22)
    with torch.no_grad():
        h = net.decoding(seqs.to(DEV), users.to(DEV)).cpu()
        h_row = net.decoding(seqs.to(DEV), users.to(DEV), last_row=L - 2).cpu()
    want, _ = O.irn_decoding(O.to_dtype(sd, torch.float64), seqs, users, H, fold_cross=True)
    ok = seqs.ne(0)
    assert_close_rel(h[ok], want[ok], RTOL, "decoding L=512")
    assert_close_rel(h_row, want[:, L - 2], RTOL, "decoding last_row")


def test_irn_generation_at_600(pkg):
    N, L, P, B = 3000, 600, 4, 8
    sd, net, irn = _irn(pkg, N, L, 2, 4, 128, 256, seed=31)
    seqs, users = _seqs(B, L, N, 32)
    want, _, _, _, margins = O.generate_paths(O.to_dtype(sd, torch.float64), seqs, users, seqs[:, -1], 4, P,
                                              return_margins=True, fold_cross=True)
    got, _, _, _ = irn.get_seq_in_batch(seqs.to(DEV), users.to(DEV), seqs[:, -1].to(DEV), max_path_len=P, gap_len=0)
    for b in range(B):
        if margins[b].min() > 1e-5:
            np.testing.assert_array_equal(got[b], np.asarray(want[b]))
    assert (margins.min(1) > 1e-5).mean() > 0.7


@pytest.mark.parametrize("L,H", [(300, 4), (201, 2)])
def test_irn_train_batch_long_windows(pkg, L, H):
    N = 2000
    sd, net, irn = _irn(pkg, N, L, 2, H, 128, 256, seed=41 + L)
    seqs, users = _seqs(4, L, N, 42)
    want_loss, want_g = O.irn_loss_and_grads(O.to_dtype(sd, torch.float64), seqs, users, H)
    loss = irn.train_batch(seqs.to(DEV), users.to(DEV))
    assert abs(loss - float(want_loss)) < 1e-4 * max(1.0, abs(float(want_loss)))
    for k, p_ in net.named_parameters():
        ref = want_g[k]
        got = torch.zeros_like(p_) if p_.grad is None else p_.grad
        if float(ref.abs().max()) == 0:
            assert float(got.abs().max()) < 1e-7, k
        else:
            assert_close_rel(got.cpu(), ref, RTOL, "grad " + k)


def test_irn_dropout_training_step_at_400(pkg):
    N, L = 2000, 400
    sd, net, irn = _irn(pkg, N, L, 2, 4, 128, 256, seed=51, dropout=0.1)
    seqs, users = _seqs(4, L, N, 52)
    torch.manual_seed(5)
    loss = irn.train_batch(seqs.to(DEV), users.to(DEV))
    assert math.isfinite(loss)
    for k, p_ in net.named_parameters():
        if "multihead_attn.in_proj_weight" in k:
            continue
        assert p_.grad is not None and torch.isfinite(p_.grad).all(), k


def test_evaluator_pp_at_400(pkg):
    from types import SimpleNamespace
    N, L, H = 500, 400, 2
    cfg = SimpleNamespace(n_item=N, max_len=L + 1, n_layers=2, n_heads=H, emb_dim=64, ffn_dim=128, dropout=0.0, lr1=1e-3)
    torch.manual_seed(61)
    net = pkg.SampleNet(cfg)
    sd = {k: v.detach().clone().double() if v.is_floating_point() else v.clone() for k, v in net.state_dict().items()}
    net.to(DEV).eval()
    ev = pkg.Evaluator(cfg, net, torch.device(DEV))
    g = torch.Generator().manual_seed(62)
    B = 4
    new = torch.randint(1, N + 1, (B, L + 1), generator=g)
    new[1, :100] = 0                                            # pre-padded
    start = torch.tensor([300, 150, 1, 390])
    lpath = torch.tensor([20, 40, 10, 10])
    want = O.evaluator_pp(sd, new, start, lpath, H)
    got = ev.get_pp_in_batch(new.to(DEV), start.to(DEV), lpath.to(DEV))
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-4)


def test_sas_predict_at_300(pkg):
    from types import SimpleNamespace
    N, T, H = 800, 300, 2
    cfg = SimpleNamespace(n_user=9, n_item=N, hidden_units=64, max_len=T, dropout_rate=0.2, num_blocks=2, num_heads=H)
    torch.manual_seed(71)
    net = pkg.SAS(cfg, torch.device(DEV))
    sd = {k: v.detach().clone().double() for k, v in net.state_dict().items()}
    net.to(DEV).eval()
    g = torch.Generator().manual_seed(72)
    B = 5
    seqs = torch.randint(1, N + 1, (B, T), generator=g)
    seqs[0, :120] = 0
    rats = torch.randint(1, 6, (B, T), generator=g) * seqs.ne(0)
    with torch.no_grad():
        got = net.predict(np.arange(B), seqs.numpy(), rats.numpy()).cpu()
    want = O.sas_predict(sd, seqs, rats, H)
    assert_close_rel(got, want, RTOL, "SAS.predict at T=300")
