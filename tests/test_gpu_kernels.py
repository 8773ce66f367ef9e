"""GPU parity tests, kernel by kernel, through the C ABI (ctypes) against the CPU oracle on the same
seeded inputs.  Bit-exact for gathered embeddings, indices, ranks; RTOL (1e-3 of the tensor's max
magnitude, tests/helpers.py) for floating point."""
import math

import numpy as np
import pytest
import torch

from oracle import irn_oracle as O
from tests.helpers import assert_close_rel, RTOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


DEV = "cuda:0"


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ---------------------------------------------------------------------------------------------- K1
@pytest.mark.parametrize("B,L,d,N", [(7, 13, 128, 1000), (3, 5, 30, 50), (64, 201, 128, 20000), (2, 60, 64, 3415)])
def test_embed_gather_bit_exact(ops, B, L, d, N):
    g = _gen(1)
    table = torch.randn((N + 1, d), generator=g)
    table[0] = 0
    ids = torch.randint(0, N + 1, (B, L), generator=g)
    ids[0, : L // 2] = 0
    pe = O.positional_table(L + 3, d)
    want = O.embed(ids, table, pe)
    got = ops.embed_gather(ids.to(DEV), table.to(DEV), pe[:L].contiguous().to(DEV), math.sqrt(d)).cpu()
    assert torch.equal(got, want)


def test_embed_gather_empty_and_no_pe(ops):
    table = torch.randn((10, 8))
    ids = torch.zeros((0, 4), dtype=torch.long)
    assert ops.embed_gather(ids.to(DEV), table.to(DEV), None, 2.0).shape == (0, 4, 8)
    ids = torch.tensor([[1, 2, 9]])
    got = ops.embed_gather(ids.to(DEV), table.to(DEV), None, 2.0).cpu()
    assert torch.equal(got, table[ids] * 2.0)


# ---------------------------------------------------------------------------------------------- K2
@pytest.mark.parametrize("rows,d,N,skew", [(1000, 128, 50, True), (4096, 64, 100000, False), (77, 30, 20, True)])
def test_embed_scatter_add(ops, rows, d, N, skew):
    g = _gen(2)
    if skew:   # Zipf-like: many duplicates inside a warp chunk
        ids = (torch.rand(rows, generator=g) ** 3 * (N + 1)).long().clamp(0, N)
    else:
        ids = torch.randint(0, N + 1, (rows,), generator=g)
    ids[::7] = 0
    d_out = torch.randn((rows, d), generator=g)
    scale = math.sqrt(d)
    want = torch.zeros((N + 1, d), dtype=torch.float64)
    keep = ids != 0
    want.index_add_(0, ids[keep], d_out[keep].double() * scale)
    got = torch.zeros((N + 1, d), device=DEV)
    ops.embed_scatter_add_raw(ids.to(DEV).view(1, -1), d_out.to(DEV), scale, got, 0)
    assert float(got[0].abs().max()) == 0.0
    assert_close_rel(got.cpu(), want, 1e-5, "scatter-add")


# ---------------------------------------------------------------------------------------------- LN
@pytest.mark.parametrize("rows,d", [(5, 30), (1000, 128), (33, 64), (9, 256)])
def test_residual_layernorm(ops, rows, d):
    g = _gen(3)
    x, y = torch.randn((rows, d), generator=g), torch.randn((rows, d), generator=g)
    yb, c2 = torch.randn(d, generator=g), torch.randn(d, generator=g)
    g1, b1, g2, b2 = (torch.randn(d, generator=g) for _ in range(4))
    t = torch.nn.functional.layer_norm(x + y + yb, (d,), g1, b1, 1e-5)
    want2 = torch.nn.functional.layer_norm(t + c2, (d,), g2, b2, 1e-5)
    D = lambda a: a.to(DEV)
    got1 = ops.residual_layernorm(D(x), D(y), D(yb), D(g1), D(b1)).cpu()
    got2 = ops.residual_layernorm(D(x), D(y), D(yb), D(g1), D(b1), D(c2), D(g2), D(b2)).cpu()
    assert_close_rel(got1, t, 1e-5, "ln1")
    assert_close_rel(got2, want2, 1e-5, "ln1+ln2")


# ---------------------------------------------------------------------------------------------- K3
def _attn_oracle(qkv, ids, r_u, H, mode):
    B, L, d3 = qkv.shape
    d = d3 // 3
    dh = d // H
    q, k, v = (qkv[..., i * d:(i + 1) * d].reshape(B, L, H, dh).transpose(1, 2) for i in range(3))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
    if mode == 0:
        s = s + O.pim_mask(L, r_u.reshape(B, 1)).unsqueeze(1)
    else:
        s = s + O.causal_mask(L)
    if mode != 2:
        s = s.masked_fill(ids.eq(0)[:, None, None, :], float("-inf"))
    return (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, L, d)


@pytest.mark.parametrize("tc", [True, False])
@pytest.mark.parametrize("B,L,H,dh,mode", [(3, 12, 2, 16, 0), (2, 201, 4, 32, 0), (4, 60, 6, 5, 0),
                                           (3, 14, 2, 16, 1), (2, 20, 3, 40, 2), (5, 33, 1, 64, 0),
                                           (3, 128, 2, 32, 0), (2, 129, 2, 32, 1), (2, 223, 1, 16, 2), (70, 60, 4, 32, 0),
                                           # full windows of 129..223 with dh = 32: the persistent tcgen05 kernel
                                           (5, 201, 4, 32, 1), (3, 201, 4, 32, 2), (3, 150, 4, 32, 0), (2, 223, 2, 32, 0),
                                           (2, 161, 1, 32, 1), (2, 193, 3, 32, 0), (160, 201, 4, 32, 0)])
def test_pim_attention_forward(ops, B, L, H, dh, mode, tc, monkeypatch):
    """tc=True: tcgen05 kernel where the shape allows (dh % 16 == 0, L <= 223), else the fp32 kernel;
    tc=False: always the fp32 CUDA-core kernel."""
    monkeypatch.setattr(ops, "USE_TC_ATTENTION", tc)
    g = _gen(4)
    d = H * dh
    qkv = torch.randn((B, L, 3 * d), generator=g)
    ids = torch.randint(1, 100, (B, L), generator=g)
    if mode == 0:      # pre-padded, objective slot never PAD
        for b in range(B):
            ids[b, : (b * 3) % (L - 1)] = 0
    elif mode == 1:    # post-padded
        for b in range(1, B):
            ids[b, L - (b * 2) % (L - 1):] = 0
    r_u = torch.randn(B, generator=g)
    want = _attn_oracle(qkv.double(), ids, r_u.double(), H, mode)
    got = ops.pim_attention(qkv.to(DEV), ids.to(DEV), r_u.to(DEV) if mode == 0 else None, H, mode).cpu()
    ok = ~torch.isnan(want)          # fully masked rows (post-padded queries never are; keep generic)
    assert torch.equal(torch.isnan(got), torch.isnan(want.float()))
    assert_close_rel(got[ok], want[ok], 3e-5 if tc else 2e-5, "attention")
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0
    # row subset (generation reads one row of the last layer)
    row = L - 2
    sub = ops.pim_attention(qkv.to(DEV), ids.to(DEV), r_u.to(DEV) if mode == 0 else None, H, mode, q_row0=row, n_q=1).cpu()
    if ops.attn_img_supported(L, dh) and tc:       # one-row requests of the image path run on the CUDA cores
        assert_close_rel(sub[:, 0][ok[:, row]], want[:, row][ok[:, row]], 3e-5, "one-row attention")
    else:
        assert torch.equal(sub[:, 0], got[:, row])


@pytest.mark.parametrize("scale", [0.05, 1.0, 2.8, 12.0])
@pytest.mark.parametrize("mode", [0, 1])
def test_pim_attention_image_kernel_softmax_shift(ops, scale, mode):
    """The persistent kernel skips the row-max pass (softmax shift 0) when |q_i| max_j|k_j| + max|bias| proves every score
    of the warp's rows small, and runs the exact row-max pass otherwise: small, typical, borderline (some warps each way)
    and huge activations, large |r_u| (objective bias) and a fully padded history.  The error of a bf16x3 score is
    relative to |q||k|, so the tolerance grows with the square of the activation scale."""
    B, L, H, dh = 6, 201, 4, 32
    g = _gen(77)
    d = H * dh
    qkv = torch.randn((B, L, 3 * d), generator=g) * scale
    qkv[..., 2 * d:] /= scale                                   # keep v O(1): the comparison is relative to max|out|
    ids = torch.randint(1, 100, (B, L), generator=g)
    if mode == 0:
        ids[1, : L - 1] = 0                                     # only the objective is visible
        ids[2, : 100] = 0
    else:
        ids[1, 50:] = 0
    r_u = torch.randn(B, generator=g)
    r_u[3] = 40.0                                               # objective bias 40 * log2(e) = 58: still no shift needed
    r_u[4] = -80.0                                              # |bias| 115: forces the exact pass for that item
    want = _attn_oracle(qkv.double(), ids, r_u.double(), H, mode)
    got = ops.pim_attention(qkv.to(DEV), ids.to(DEV), r_u.to(DEV) if mode == 0 else None, H, mode).cpu()
    ok = ~torch.isnan(want)
    assert torch.equal(torch.isnan(got), torch.isnan(want.float()))
    assert_close_rel(got[ok], want[ok], 3e-5 * max(1.0, scale * scale), f"attention, activations x{scale}")
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


@pytest.mark.parametrize("B,L,H,dh,mode", [(3, 12, 2, 16, 0), (2, 50, 4, 32, 0), (2, 17, 6, 5, 0), (3, 14, 2, 16, 1)])
def test_pim_attention_backward(ops, B, L, H, dh, mode):
    g = _gen(5)
    d = H * dh
    qkv = torch.randn((B, L, 3 * d), generator=g)
    ids = torch.randint(1, 100, (B, L), generator=g)
    for b in range(B):
        if mode == 0:
            ids[b, : (b * 3) % (L - 1)] = 0
        elif b:
            ids[b, L - (b * 2) % (L - 1):] = 0
    r_u = torch.randn(B, generator=g)
    go = torch.randn((B, L, d), generator=g)
    a = qkv.double().requires_grad_(True)
    r = r_u.double().requires_grad_(True)
    _attn_oracle(a, ids, r, H, mode).backward(go.double())
    q_dev = qkv.to(DEV).requires_grad_(True)
    r_dev = r_u.to(DEV).requires_grad_(True)
    out = ops.pim_attention(q_dev, ids.to(DEV), r_dev if mode == 0 else None, H, mode)
    out.backward(go.to(DEV))
    assert_close_rel(q_dev.grad.cpu(), a.grad, 5e-5, "d_qkv")
    if mode == 0:
        assert_close_rel(r_dev.grad.cpu(), r.grad, 5e-5, "d_r_u")


# ---------------------------------------------------------------------------------------------- K5
def _score_case(M, N, d, Lx, seed, zipf=False):
    g = _gen(seed)
    h = torch.randn((M, d), generator=g)
    W = torch.randn((N, d), generator=g) / math.sqrt(d)
    bias = torch.randn(N, generator=g) * 0.1
    if zipf:
        excl = (torch.rand((M, Lx), generator=g) ** 4 * N).long().clamp(0, N - 1) + 1
    else:
        excl = torch.randint(1, N + 1, (M, Lx), generator=g)
    excl[:, ::5] = 0
    return h, W, bias, excl


@pytest.mark.parametrize("M,N,d,Lx,k", [(5, 300, 32, 7, 1), (130, 5000, 128, 200, 1), (48, 3415, 64, 59, 1),
                                        (9, 3415, 64, 50, 50), (33, 20000, 128, 20, 5), (3, 40, 30, 4, 3),
                                        (200, 1000, 16, 3, 20)])
def test_score_topk_matches_oracle(ops, M, N, d, Lx, k):
    h, W, bias, excl = _score_case(M, N, d, Lx, 6 + k, zipf=True)
    s = (h.double() @ W.double().t() + bias.double())
    wv, wi = O.topk_excluding(s, excl, k)
    e = ops.sort_exclusions(excl.to(DEV), N, 1)
    gv, gi = ops.score_topk(h.to(DEV), W.to(DEV), bias.to(DEV), k, e, 1)
    gv, gi = gv.cpu(), gi.cpu()
    # decisions closer than fp32 noise may legitimately swap; everything else must be identical
    assert_close_rel(gv, wv, 1e-5, "top-k values")
    gap = (wv[:, :-1] - wv[:, 1:]).min().item() if k > 1 else 1.0
    if gap > 1e-5:
        assert torch.equal(gi, wi)
    else:
        assert (gi == wi).float().mean() > 0.99
    # excluded items never appear
    for m in range(M):
        assert not set(gi[m].tolist()) & set(excl[m][excl[m] > 0].tolist())


def test_score_topk_no_exclusion_no_bias_and_ties(ops):
    # exact ties: duplicate catalog rows -> the lower item id must win, and order inside top-k is by id
    g = _gen(9)
    h = torch.randn((4, 16), generator=g)
    W = torch.randn((300, 16), generator=g)
    W[250] = W[7]
    W[100] = W[7]
    s = h @ W.t()
    _, wi = O.topk_excluding(s.double(), None, 300 if False else 10)
    gv, gi = ops.score_topk(h.to(DEV), W.to(DEV), None, 10, None, 1)
    assert torch.equal(gi.cpu(), wi)
    _, g1 = ops.score_topk(h.to(DEV), W.to(DEV), None, 1, None, 1)
    assert torch.equal(g1.cpu(), wi[:, :1])


def test_score_topk_everything_excluded_and_small_catalog(ops):
    h = torch.randn((2, 8))
    W = torch.randn((5, 8))
    excl = torch.tensor([[1, 2, 3, 4, 5], [1, 0, 0, 0, 0]])
    e = ops.sort_exclusions(excl.to(DEV), 5, 1)
    gv, gi = ops.score_topk(h.to(DEV), W.to(DEV), None, 1, e, 1)
    assert gi.cpu()[0, 0].item() == -1 and gv.cpu()[0, 0].item() == float("-inf")
    gv, gi = ops.score_topk(h.to(DEV), W.to(DEV), None, 8, e, 1)       # k > live items
    assert gi.cpu()[1].tolist()[4:] == [-1] * 4
    want = O.topk_excluding((h @ W.t()).double()[1:], excl[1:], 4)[1]
    assert gi.cpu()[1, :4].tolist() == want[0].tolist()


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("M,N,d,Lx", [(6, 150, 32, 9), (130, 5000, 128, 60), (64, 3415, 64, 0), (300, 70001, 128, 40)])
def test_score_rank_matches_oracle(ops, M, N, d, Lx, tc, monkeypatch):
    """tc=False: fp32 CUDA-core counter; tc=True: tcgen05 counting + exact re-scoring of the columns inside the error band."""
    monkeypatch.setattr(ops, "USE_TC_RANK", tc)
    h, W, bias, excl = _score_case(M, N, d, max(Lx, 1), 21)
    g = _gen(22)
    label = torch.randint(1, N + 1, (M,), generator=g)
    if Lx:
        label[0] = excl[0][excl[0] > 0][0]      # excluded label -> rank 0
    s = (h @ W.t() + bias)
    e = ops.sort_exclusions(excl.to(DEV), N, 1) if Lx else None
    got = ops.score_rank(h.to(DEV), W.to(DEV), bias.to(DEV), label.to(DEV), e, 1).cpu()
    want = O.rank_excluding(s.double(), label, excl if Lx else None)
    # a rank can move by the number of items within fp32 noise of the label's score
    sl = s.double()[torch.arange(M), label - 1].unsqueeze(1)
    near = ((s.double() - sl).abs() < 1e-5).sum(1) - 1
    assert ((got - want).abs() <= near).all()
    if Lx:
        assert got[0].item() == 0


@pytest.mark.parametrize("M,N,d,Lx", [(130, 5000, 128, 60), (257, 70001, 128, 0), (40, 3415, 64, 20), (9, 700, 30, 5)])
def test_score_rank_tc_equals_fp32_engine_with_ties(ops, M, N, d, Lx, monkeypatch):
    """The tensor-core rank must be the SAME integer as the fp32 engine's, including exact ties (twin catalog rows of
    the label: lower id ahead), near-ties, an overflowing uncertain list (> 30 twins in one slice), labels out of range
    and excluded labels."""
    h, W, bias, excl = _score_case(M, N, d, max(Lx, 1), 51)
    g = _gen(52)
    label = torch.randint(1, N + 1, (M,), generator=g)
    # twins of row 0's label (exact ties), 40 of them contiguous so that one (split, half) slice overflows its list
    l0 = int(label[0]) - 1
    tw = torch.randint(0, N, (12,), generator=g)
    W[tw] = W[l0].clone(); bias[tw] = bias[l0].clone()
    start = min(max(l0 - 20, 0), N - 40)
    W[start:start + 40] = W[l0].clone(); bias[start:start + 40] = bias[l0].clone()
    # near-ties of row 1's label: relative perturbations around fp32 resolution
    l1 = int(label[1]) - 1
    nt = torch.randint(0, N, (16,), generator=g)
    W[nt] = W[l1].clone() * (1 + torch.linspace(-3e-6, 3e-6, 16).unsqueeze(1)); bias[nt] = bias[l1].clone()
    label[2] = N + 5                                  # out of range -> 0
    if Lx:
        label[3] = excl[3][excl[3] > 0][0]            # excluded -> 0
    e = ops.sort_exclusions(excl.to(DEV), N, 1) if Lx else None
    args = (h.to(DEV), W.to(DEV), bias.to(DEV), label.to(DEV), e, 1)
    monkeypatch.setattr(ops, "USE_TC_RANK", False)
    want = ops.score_rank(*args).cpu()
    monkeypatch.setattr(ops, "USE_TC_RANK", True)
    got = ops.score_rank(*args).cpu()
    assert torch.equal(got, want), (got - want).abs().max()
    assert got[2].item() == 0
    if Lx:
        assert got[3].item() == 0


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("M,N,d,s", [(7, 150, 32, 1), (130, 5000, 128, 2), (300, 3415, 64, 1), (1000, 70001, 128, 2), (5, 300, 30, 1)])
def test_score_lse_gather(ops, M, N, d, s, tc, monkeypatch):
    """tc=False: fp32 CUDA-core engine; tc=True: tcgen05 online log-sum-exp (d <= 128) + exact selected logits."""
    monkeypatch.setattr(ops, "USE_TC_LSE", tc)
    h, W, bias, _ = _score_case(M, N, d, 1, 31)
    g = _gen(32)
    sel = torch.randint(1, N + 1, (M, s), generator=g)
    sel[0, 0] = 0
    sc = (h.double() @ W.double().t() + bias.double())
    wl, wg = O.lse_gather(sc, sel)
    wg[0, 0] = 0.0
    gl, gg = ops.score_lse_gather(h.to(DEV), W.to(DEV), bias.to(DEV), sel.to(DEV), 1)
    assert_close_rel(gl.cpu(), wl, 1e-5 if tc else 1e-6, "lse")
    assert_close_rel(gg.cpu(), wg, 1e-5, "gathered logits")


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("M,N,d", [(50, 300, 32), (260, 1000, 128), (17, 3415, 64), (9, 130, 30), (700, 40000, 128), (40000, 700, 128)])
def test_softmax_ce_forward_backward(ops, M, N, d, tc, monkeypatch):
    """tc=False: fp32 CUDA-core kernels; tc=True: tcgen05 log-sum-exp forward and the two-pass tcgen05 backward."""
    monkeypatch.setattr(ops, "USE_TC_LSE", tc)
    monkeypatch.setattr(ops, "USE_TC_CE_BWD", tc)
    g = _gen(41)
    h = torch.randn((M, d), generator=g)
    W = torch.randn((N, d), generator=g) / math.sqrt(d)
    bias = torch.randn(N, generator=g) * 0.1
    tgt = torch.randint(0, N, (M,), generator=g)
    hh, WW, bb = (t.double().requires_grad_(True) for t in (h, W, bias))
    loss = torch.nn.functional.cross_entropy(hh @ WW.t() + bb, tgt)
    loss.backward()
    hd, Wd, bd = (t.to(DEV).requires_grad_(True) for t in (h, W, bias))
    got = ops.softmax_ce_mean(hd, Wd, bd, tgt.to(DEV))
    got.backward()
    assert abs(got.item() - loss.item()) < 1e-5 * max(1.0, abs(loss.item()))
    tol = 1e-4 if tc else 2e-5                     # north-star: gradients within 1e-3; bf16x3 measured ~2e-5
    assert_close_rel(hd.grad.cpu(), hh.grad, tol, "d_h")
    assert_close_rel(Wd.grad.cpu(), WW.grad, tol, "d_W")
    assert_close_rel(bd.grad.cpu(), bb.grad, tol, "d_bias")
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def test_topk_merge_equals_unsharded(ops):
    """Catalog sharding on one GPU: G logical shards scored separately + merge == unsharded top-k."""
    M, N, d, k, G = 40, 4000, 64, 6, 4
    h, W, bias, excl = _score_case(M, N, d, 30, 51)
    e = ops.sort_exclusions(excl.to(DEV), N, 1)
    fv, fi = ops.score_topk(h.to(DEV), W.to(DEV), bias.to(DEV), k, e, 1)
    vs, its = [], []
    for gidx in range(G):
        lo, hi = gidx * N // G, (gidx + 1) * N // G
        es = ops.sort_exclusions(excl.to(DEV), hi - lo, lo + 1)
        v, i = ops.score_topk(h.to(DEV), W[lo:hi].contiguous().to(DEV), bias[lo:hi].contiguous().to(DEV), k, es, lo + 1)
        vs.append(v)
        its.append(i)
    mv, mi = ops.topk_merge(torch.stack(vs), torch.stack(its))
    assert torch.equal(mi, fi)
    assert torch.equal(mv, fv)


def test_window_shift(ops):
    g = _gen(61)
    B, L, P = 37, 201, 4
    seq = torch.randint(1, 1000, (B, L), generator=g)
    nxt = torch.randint(1, 1000, (B,), generator=g)
    want = torch.cat([seq[:, 1:L - 1], nxt[:, None], seq[:, L - 1:]], 1)
    sd, paths = seq.to(DEV), torch.zeros((B, P), device=DEV)
    ops.window_shift(sd, nxt.to(DEV), paths, 2)
    assert torch.equal(sd.cpu(), want)
    assert torch.equal(paths[:, 2].cpu(), nxt.float())


def test_missing_cuda_inputs_fail_loudly(ops):
    with pytest.raises(RuntimeError):
        ops.embed_gather(torch.zeros((1, 2), dtype=torch.long), torch.zeros((3, 4)), None, 1.0)


# ---------------------------------------------------------------------------------------------- K5c (tcgen05)
@pytest.mark.parametrize("M,N,d,Lx", [(5, 300, 32, 7), (130, 5000, 128, 200), (48, 3415, 64, 59), (257, 70000, 128, 31),
                                      (9, 1000, 30, 4), (128, 256, 16, 1),
                                      # 17 user tiles x 8 catalog splits of 35 tiles: three candidate segments per split,
                                      # the last split (29 tiles) has only two
                                      (2100, 70000, 128, 40)])
@pytest.mark.parametrize("variant", [2, 0, 6, 4, 10])
def test_score_argmax_tensor_core_equals_fp32_engine(ops, M, N, d, Lx, variant, monkeypatch):
    """The tcgen05 arg-max (variant 2: one bf16 MMA + rigorous error band; variant 0: bf16x3) + exact re-score returns
    the same winners AND the same fp32 score bits as the CUDA-core engine, and both agree with the oracle outside
    fp32-noise near-ties."""
    monkeypatch.setattr(ops, "ARGMAX_VARIANT", variant)
    h, W, bias, excl = _score_case(M, N, d, Lx, 77, zipf=True)
    e = ops.sort_exclusions(excl.to(DEV), N, 1)
    hd, Wd, bd = h.to(DEV), W.to(DEV), bias.to(DEV)
    prep = ops.scorer_prepare_weights(Wd)
    tv, ti = ops.score_argmax_tc(hd, Wd, prep, bd, e, 1)
    rv, ri = ops.score_topk(hd, Wd, bd, 1, e, 1)
    assert torch.equal(ti, ri)
    assert torch.equal(tv, rv)
    s = (h.double() @ W.double().t() + bias.double())
    wv, wi = O.topk_excluding(s, excl, 2)
    safe = (wv[:, 0] - wv[:, 1]) > 1e-5
    assert torch.equal(ti.cpu()[safe], wi[safe][:, :1])
    # no bias / no exclusions
    tv, ti = ops.score_argmax_tc(hd, Wd, prep, None, None, 1)
    rv, ri = ops.score_topk(hd, Wd, None, 1, None, 1)
    assert torch.equal(ti, ri) and torch.equal(tv, rv)


@pytest.mark.parametrize("variant", [2, 0])
@pytest.mark.parametrize("M,N,d,Lx,shards", [(130, 5000, 128, 60, 2), (300, 70001, 128, 40, 3), (64, 3415, 64, 0, 4)])
def test_score_argmax_two_phase_sharded_equals_unsharded(ops, M, N, d, Lx, shards, variant, monkeypatch):
    """Catalog-sharded arg-max in two phases (phase 1 per shard -> max-reduce of the leaders -> phase 2 per shard -> merge)
    returns exactly the winners and fp32 scores of the unsharded call, and every row is re-scored by at least one shard;
    shards that cannot hold a row's winner return (-inf, -1) for it.  One shard has much larger weight norms (its
    rounding-error scale must widen the band of the others)."""
    monkeypatch.setattr(ops, "ARGMAX_VARIANT", variant)
    h, W, bias, excl = _score_case(M, N, d, max(Lx, 1), 91)
    bounds = [N * g // shards for g in range(shards + 1)]
    W[bounds[1]:bounds[2]] *= 3.0                              # shard 1: larger norms and scores
    hd, Wd, bd = h.to(DEV), W.to(DEV), bias.to(DEV)
    ex_full = ops.sort_exclusions(excl.to(DEV), N, 1) if Lx else None
    want_v, want_i = ops.score_argmax_tc(hd, Wd, ops.scorer_prepare_weights(Wd), bd, ex_full, 1)
    leads, state = [], []
    for g in range(shards):
        lo, hi = bounds[g], bounds[g + 1]
        Wg, bg = Wd[lo:hi].contiguous(), bd[lo:hi].contiguous()
        prep = ops.scorer_prepare_weights(Wg)
        ex = ops.sort_exclusions(excl.to(DEV), hi - lo, lo + 1) if Lx else None
        lead, ws = ops.score_argmax_tc_phase1(hd, Wg, prep, bg, ex, lo + 1)
        leads.append(lead); state.append((Wg, bg, prep, ex, ws, lo))
    lead_g = torch.stack(leads).max(0).values                  # what the all-reduce (MAX) computes
    vals, items = [], []
    for Wg, bg, prep, ex, ws, lo in state:
        v, i = ops.score_argmax_tc_phase2(hd, Wg, prep, bg, ex, lo + 1, lead_g, ws)
        vals.append(v); items.append(i)
    vals, items = torch.stack(vals), torch.stack(items)        # [G, M, 1]
    got_v, got_i = ops.topk_merge(vals, items)
    assert torch.equal(got_i, want_i) and torch.equal(got_v, want_v)
    live = (items[:, :, 0] >= 0).sum(0)
    assert int(live.min()) >= 1                                # somebody re-scored every row
    assert float((live == 1).float().mean()) > 0.5            # and mostly only the shard that holds the winner


@pytest.mark.parametrize("variant", [2, 0])
def test_score_argmax_tensor_core_near_ties(ops, variant, monkeypatch):
    monkeypatch.setattr(ops, "ARGMAX_VARIANT", variant)
    _near_ties(ops)


def test_score_argmax_single_mma_large_dynamic_range(ops):
    """Single-MMA mode with rows / items of very different norms (the band scales with |h_m| max_j |W_j|) and scores that
    differ only in the bits a lone bf16 product loses."""
    g = _gen(89)
    M, N, d = 200, 50000, 128
    h = torch.randn((M, d), generator=g) * torch.logspace(-2, 2, M).unsqueeze(1)
    W = torch.randn((N, d), generator=g) / math.sqrt(d)
    W[::7] *= 8.0
    W[1000:1100] = W[2000:2100] * (1 + 1e-3)          # pairs 0.1 % apart: invisible to hi*hi alone
    hd, Wd = h.to(DEV), W.to(DEV)
    prep = ops.scorer_prepare_weights(Wd)
    tv, ti = ops.score_argmax_tc(hd, Wd, prep, None, None, 1, variant=2)
    rv, ri = ops.score_topk(hd, Wd, None, 1, None, 1)
    assert torch.equal(ti, ri) and torch.equal(tv, rv)


def _near_ties(ops):
    """Adversarial: many catalog rows are tiny perturbations of each other, so dozens of scores sit
    inside the bf16x3 error band.  The exact re-scoring (chunk re-score + ambiguous-slice scan) must
    still return the fp32 engine's winner, ties by lower id."""
    g = _gen(88)
    M, N, d = 64, 6000, 128
    h = torch.randn((M, d), generator=g)
    base = torch.randn((40, d), generator=g) / math.sqrt(d)
    W = base[torch.randint(0, 40, (N,), generator=g)] + torch.randn((N, d), generator=g) * 1e-6
    W[100] = W[4000]                                    # exact duplicates -> exact ties
    W[17] = W[5000]
    hd, Wd = h.to(DEV), W.to(DEV)
    prep = ops.scorer_prepare_weights(Wd)
    tv, ti = ops.score_argmax_tc(hd, Wd, prep, None, None, 1)
    rv, ri = ops.score_topk(hd, Wd, None, 1, None, 1)
    assert torch.equal(ti, ri) and torch.equal(tv, rv)


# ---------------------------------------------------------------------------------------------- tcgen05 linear
@pytest.mark.parametrize("R,K,Nout,epi", [(300, 128, 128, 0), (1000, 128, 256, 1), (129, 256, 128, 2), (5000, 128, 128, 2),
                                          (77, 64, 192, 0), (40, 120, 120, 2), (128, 32, 16, 1), (20000, 128, 256, 0)])
def test_linear_tensor_core(ops, R, K, Nout, epi):
    g = _gen(101)
    A = torch.randn((R, K), generator=g)
    W = torch.randn((Nout, K), generator=g) / math.sqrt(K)
    bias = torch.randn(Nout, generator=g) * 0.1
    resid = torch.randn((R, Nout), generator=g)
    g1, b1, c2, g2, b2 = (torch.randn(Nout, generator=g) for _ in range(5))
    acc = A.double() @ W.double().t() + bias.double()
    D = lambda t: t.to(DEV)
    prep = ops.linear_prepare(D(W))
    if epi == 0:
        want = acc
        got = ops.linear_tc(D(A), prep, Nout, D(bias), 0)
    elif epi == 1:
        want = torch.relu(acc)
        got = ops.linear_tc(D(A), prep, Nout, D(bias), 1)
    else:
        F = torch.nn.functional
        t = F.layer_norm(resid.double() + acc, (Nout,), g1.double(), b1.double(), 1e-5)
        want1 = t
        want = F.layer_norm(t + c2.double(), (Nout,), g2.double(), b2.double(), 1e-5)
        got1 = ops.linear_tc(D(A), prep, Nout, D(bias), 2, resid=D(resid), g1=D(g1), b1=D(b1))
        assert_close_rel(got1.cpu(), want1, 3e-5, "linear+LN")
        got = ops.linear_tc(D(A), prep, Nout, D(bias), 2, resid=D(resid), g1=D(g1), b1=D(b1), c2=D(c2), g2=D(g2), b2=D(b2))
    assert_close_rel(got.cpu(), want, 3e-5, f"linear_tc epi={epi}")   # bf16x3: ~1e-5 of the tensor's scale
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def test_linear_tensor_core_into_column_slice(ops):
    g = _gen(102)
    R, K = 333, 128
    A = torch.randn((R, K), generator=g)
    W = torch.randn((384, K), generator=g) / math.sqrt(K)
    b = torch.randn(384, generator=g)
    out = torch.zeros((R, 384), device=DEV)
    Wd, bd = W.to(DEV), b.to(DEV)
    ops.linear_tc(A.to(DEV), ops.linear_prepare(Wd[:256].contiguous()), 256, bd[:256].contiguous(), 0, out=out[:, :256])
    ops.linear_tc(A.to(DEV), ops.linear_prepare(Wd[256:].contiguous()), 128, bd[256:].contiguous(), 0, out=out[:, 256:])
    assert_close_rel(out.cpu(), A.double() @ W.double().t() + b.double(), 3e-5, "qkv in two launches")


# --------------------------------------------------------------- fused decoder-layer chain (tcgen05)
def _chain_reference(attn, x, P, with_qkv):
    """fp64 restatement: LN2(LN1(x + attn Wo^T + bo) + c2) -> FFN -> LN3 -> next in_proj
    (nn.TransformerDecoderLayer post-norm order, model/influentialRS.py:67-74)."""
    F = torch.nn.functional
    dd = lambda t: t.double()
    d = x.shape[1]
    t = F.layer_norm(dd(x) + dd(attn) @ dd(P["Wo"]).t() + dd(P["bo"]), (d,), dd(P["g1"]), dd(P["b1"]), 1e-5)
    y = F.layer_norm(t + dd(P["c2"]), (d,), dd(P["g2"]), dd(P["b2"]), 1e-5)
    f = torch.relu(y @ dd(P["W1"]).t() + dd(P["bf1"]))
    xo = F.layer_norm(y + f @ dd(P["W2"]).t() + dd(P["bf2"]), (d,), dd(P["g3"]), dd(P["b3"]), 1e-5)
    qkv = xo @ dd(P["Win"]).t() + dd(P["bin"]) if with_qkv else None
    return xo, qkv


@pytest.mark.parametrize("R,with_qkv,inplace", [(128, True, False), (300, True, False), (37, False, False),
                                                (148 * 128 * 2 + 77, True, True), (5000, False, True)])
def test_decoder_chain_tensor_core(ops, R, with_qkv, inplace):
    g = _gen(300 + R % 97)
    d, ffn = 128, 256
    P = {"Wo": torch.randn((d, d), generator=g) / math.sqrt(d), "bo": 0.1 * torch.randn(d, generator=g),
         "g1": 1 + 0.1 * torch.randn(d, generator=g), "b1": 0.1 * torch.randn(d, generator=g),
         "c2": 0.3 * torch.randn(d, generator=g),
         "g2": 1 + 0.1 * torch.randn(d, generator=g), "b2": 0.1 * torch.randn(d, generator=g),
         "W1": torch.randn((ffn, d), generator=g) / math.sqrt(d), "bf1": 0.1 * torch.randn(ffn, generator=g),
         "W2": torch.randn((d, ffn), generator=g) / math.sqrt(ffn), "bf2": 0.1 * torch.randn(d, generator=g),
         "g3": 1 + 0.1 * torch.randn(d, generator=g), "b3": 0.1 * torch.randn(d, generator=g),
         "Win": torch.randn((3 * d, d), generator=g) / math.sqrt(d), "bin": 0.1 * torch.randn(3 * d, generator=g)}
    attn = torch.randn((R, d), generator=g)
    x = torch.randn((R, d), generator=g)
    want_x, want_qkv = _chain_reference(attn, x, P, with_qkv)
    Pd = {k: v.to(DEV) for k, v in P.items()}
    prep = ops.decoder_chain_prepare(Pd["Wo"], Pd["W1"], Pd["W2"], Pd["Win"] if with_qkv else None)
    xd = x.to(DEV)
    got_x, got_qkv = ops.decoder_chain_tc(attn.to(DEV), xd, prep, Pd["bo"], Pd["g1"], Pd["b1"], Pd["c2"], Pd["g2"], Pd["b2"],
                                          Pd["bf1"], Pd["bf2"], Pd["g3"], Pd["b3"], Pd["bin"] if with_qkv else None,
                                          x_out=xd if inplace else None)
    torch.cuda.synchronize()
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0
    assert_close_rel(got_x.cpu(), want_x, 3e-5, "decoder chain x'")
    if with_qkv:
        assert_close_rel(got_qkv.cpu(), want_qkv, 3e-5, "decoder chain qkv'")
    else:
        assert got_qkv is None
    if inplace:
        assert got_x.data_ptr() == xd.data_ptr()


@pytest.mark.parametrize("B,L,mode", [(3, 201, 0), (2, 150, 1), (2, 223, 2)])
def test_decoder_chain_writes_operand_images(ops, B, L, mode):
    """The chain kernel's image output (and the first-layer in_proj-only mode) feed the persistent attention
    kernel exactly like irs_qkv_to_images applied to the fp32 projection."""
    g = _gen(400 + L)
    d, ffn, H = 128, 256, 4
    R = B * L
    rn = lambda *s: torch.randn(*s, generator=g)
    P = {"Wo": rn(d, d) / math.sqrt(d), "bo": 0.1 * rn(d), "g1": 1 + 0.1 * rn(d), "b1": 0.1 * rn(d), "c2": 0.3 * rn(d),
         "g2": 1 + 0.1 * rn(d), "b2": 0.1 * rn(d), "W1": rn(ffn, d) / math.sqrt(d), "bf1": 0.1 * rn(ffn),
         "W2": rn(d, ffn) / math.sqrt(ffn), "bf2": 0.1 * rn(d), "g3": 1 + 0.1 * rn(d), "b3": 0.1 * rn(d),
         "Win": rn(3 * d, d) / math.sqrt(d), "bin": 0.1 * rn(3 * d)}
    attn, x = rn(R, d), rn(R, d)
    ids = torch.randint(1, 50, (B, L), generator=g)
    if mode == 0:
        ids[1, :7] = 0
    elif mode == 1:
        ids[1, L - 9:] = 0
    r_u = rn(B)
    Pd = {k: v.to(DEV) for k, v in P.items()}
    prep = ops.decoder_chain_prepare(Pd["Wo"], Pd["W1"], Pd["W2"], Pd["Win"])
    args = (Pd["bo"], Pd["g1"], Pd["b1"], Pd["c2"], Pd["g2"], Pd["b2"], Pd["bf1"], Pd["bf2"], Pd["g3"], Pd["b3"], Pd["bin"])
    ru_d = r_u.to(DEV) if mode == 0 else None
    # fp32 route: chain -> fp32 qkv -> (converter + persistent kernel inside pim_attention)
    x1, qkv = ops.decoder_chain_tc(attn.to(DEV), x.to(DEV), prep, *args)
    want = ops.pim_attention(qkv.view(B, L, 3 * d), ids.to(DEV), ru_d, H, mode)
    # image route
    images = torch.zeros_like(ops.qkv_images_buffer(B, L, H, torch.device(DEV), slot=7))
    x2, im = ops.decoder_chain_tc(attn.to(DEV), x.to(DEV), prep, *args, qkv_images=images, L=L, mask_mode=mode)
    got = ops.pim_attention_img(im, ids.to(DEV), ru_d, B, L, H, mode)
    torch.cuda.synchronize()
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0
    assert torch.equal(x1, x2)
    # The two routes differ by one ulp in q.  P is carried as two bf16 (16 significant bits): with the row maximum as the
    # shift the largest weight of a row is exactly 1.0, without a shift it is rounded at 2^-17 like every other weight,
    # so a one-ulp change of a score can move the output by ~2^-17 of it (both agree with fp64 to 3e-5, tested above).
    assert_close_rel(got.cpu(), want.cpu(), 1e-5, "image route vs fp32 route (same MMAs; q scale folded into an FFMA)")
    row = ops.pim_attention_img(im, ids.to(DEV), ru_d, B, L, H, mode, q_row0=L - 2, n_q=1)
    assert_close_rel(row[:, 0].cpu(), want[:, L - 2].cpu(), 1e-5, "one-row attention (CUDA-core kernel) vs full kernel")
    # first-layer mode: qkv = x Win^T + bin only
    images2 = torch.zeros_like(images)
    ops.in_proj_images_tc(x.to(DEV), prep, Pd["bin"], images2, L, mode)
    got0 = ops.pim_attention_img(images2, ids.to(DEV), ru_d, B, L, H, mode).cpu()
    qkv0 = (x.double() @ P["Win"].double().t() + P["bin"].double()).view(B, L, 3 * d)
    want0 = _attn_oracle(qkv0, ids, r_u.double(), H, mode)
    assert_close_rel(got0, want0, 3e-5, "in_proj images + attention")


def test_ce_backward_tensor_core_skips_negative_targets(ops):
    """C-ABI contract of irs_score_ce_bwd(_tc): rows whose target is < 0 contribute nothing (d_h row = 0, no d_W / d_bias
    term).  The tcgen05 kernel must agree with the fp32 CUDA-core kernel."""
    from influentialrs_b200._lib import lib, check
    g = _gen(43)
    M, N, d = 300, 2000, 128
    h = torch.randn((M, d), generator=g).to(DEV)
    W = (torch.randn((N, d), generator=g) / math.sqrt(d)).to(DEV)
    bias = (0.1 * torch.randn(N, generator=g)).to(DEV)
    tgt = torch.randint(0, N, (M,), generator=g)
    tgt[::3] = -1
    tgt = tgt.to(DEV)
    lse, _ = ops.score_lse_gather(h, W, bias, torch.ones((M, 1), dtype=torch.long, device=DEV), 1)
    gscale = 1.0 / 200
    s = torch.cuda.current_stream().cuda_stream
    out = {}
    for name in ("simt", "tc"):
        dh = torch.full((M, d), 7.0, device=DEV)                 # d_h is WRITTEN, whatever it held
        dW = torch.zeros((N, d), device=DEV)
        db = torch.zeros((N,), device=DEV)
        if name == "simt":
            check(lib().irs_score_ce_bwd(h.data_ptr(), d, W.data_ptr(), bias.data_ptr(), tgt.data_ptr(), lse.data_ptr(), gscale,
                                         dh.data_ptr(), dW.data_ptr(), db.data_ptr(), M, N, d, s), "ce_bwd")
        else:
            nb = lib().irs_score_ce_bwd_tc_workspace_bytes(M, N, d)
            ws = torch.empty((nb,), dtype=torch.uint8, device=DEV)
            check(lib().irs_score_ce_bwd_tc(h.data_ptr(), d, W.data_ptr(), bias.data_ptr(), tgt.data_ptr(), lse.data_ptr(), gscale,
                                            dh.data_ptr(), dW.data_ptr(), db.data_ptr(), M, N, d, ws.data_ptr(), nb, s), "ce_bwd_tc")
        out[name] = (dh.cpu(), dW.cpu(), db.cpu())
    assert float(out["tc"][0][::3].abs().max()) == 0.0           # skipped rows
    assert float(out["simt"][0][::3].abs().max()) == 0.0
    for a, b, what in zip(out["tc"], out["simt"], ("d_h", "d_W", "d_bias")):
        assert_close_rel(a, b, 1e-4, what + " tcgen05 vs fp32 kernel with skipped rows")


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("M,N,d,Lx,shards", [(130, 5000, 128, 60, 2), (300, 70001, 128, 40, 3), (64, 3415, 64, 0, 4), (9, 700, 30, 5, 2),
                                             (40, 40000, 192, 20, 3), (17, 9001, 256, 9, 2), (128, 5000, 160, 0, 4),
                                             (9, 700, 129, 5, 2)])
def test_sharded_rank_select_and_count_equal_unsharded(ops, M, N, d, Lx, shards, tc, monkeypatch):
    """Catalog-sharded rank (SURVEY 8e row 3), shards emulated on one GPU: label score = MAX over shards of irs_score_select,
    rank = 1 + SUM over shards of irs_score_count_ahead[_tc] -- the same integers as irs_score_rank over the whole catalog,
    with exact ties of the label straddling shard boundaries, excluded labels and uneven shards; irs_score_select is
    bit-identical to the scorer's own label scores.  ``tc`` sets USE_TC_RANK; for d > 128 both count-ahead and rank take
    the fp32 engine whatever the flag."""
    monkeypatch.setattr(ops, "USE_TC_RANK", tc)
    h, W, bias, excl = _score_case(M, N, d, max(Lx, 1), 61)
    g = _gen(62)
    label = torch.randint(1, N + 1, (M,), generator=g)
    l0 = int(label[0]) - 1
    tw = torch.randint(0, N, (16,), generator=g)              # twins of row 0's label all over the catalog (every shard)
    W[tw] = W[l0].clone(); bias[tw] = bias[l0].clone()
    if Lx:
        label[3] = excl[3][excl[3] > 0][0]                    # excluded label -> rank 0
    hd, Wd, bd, ld_, ed = h.to(DEV), W.to(DEV), bias.to(DEV), label.to(DEV), excl.to(DEV)
    want = ops.score_rank(hd, Wd, bd, ld_, ops.sort_exclusions(ed, N, 1) if Lx else None, 1)
    bounds = [(s * N // shards, (s + 1) * N // shards) for s in range(shards)]
    score = torch.full((M,), float("-inf"), device=DEV)
    for lo, hi in bounds:
        score = torch.maximum(score, ops.score_select(hd, Wd[lo:hi], bd[lo:hi], ld_.view(-1, 1), lo + 1)[:, 0])
    exact = ops.score_select(hd, Wd, bd, ld_.view(-1, 1), 1)[:, 0]
    assert torch.equal(score, exact)
    ref = (h.double() * W[label - 1].double()).sum(1) + bias[label - 1].double()
    assert (exact.cpu().double() - ref).abs().max() < 1e-4
    total = torch.zeros((M,), dtype=torch.int64, device=DEV)
    flags = torch.zeros((M,), dtype=torch.int64, device=DEV)
    for lo, hi in bounds:
        Ws, bs = Wd[lo:hi].contiguous(), bd[lo:hi].contiguous()
        e = ops.sort_exclusions(ed, hi - lo, lo + 1) if Lx else None
        c, f = ops.score_count_ahead(hd, Ws, bs, ld_, score, e, lo + 1)
        total += c
        flags += f.long()
    got = torch.where(flags > 0, torch.zeros_like(total), total + 1)
    assert torch.equal(got, want), (got - want).abs().max()
    if Lx:
        assert got[3].item() == 0
    # PAD / foreign items select to -inf
    sel = torch.tensor([[0, N + 7]], device=DEV).expand(M, 2).contiguous()
    assert torch.isinf(ops.score_select(hd, Wd, bd, sel, 1)).all()


def test_score_topk_few_rows_large_catalog(ops):
    """Few rows x large catalog, k > 1: the split count must stay inside what the threshold kernel can sort (regression:
    M <= ~300 rows over 300k items returned IRS_E_SHAPE)."""
    M, N, d, k = 5, 300_007, 128, 20
    h, W, bias, excl = _score_case(M, N, d, 30, 71)
    got_v, got_i = ops.score_topk(h.to(DEV), W.to(DEV), bias.to(DEV), k, ops.sort_exclusions(excl.to(DEV), N, 1), 1)
    want_v, want_i = O.topk_excluding(h.double() @ W.double().t() + bias.double(), excl, k)
    gaps = (want_v[:, :-1] - want_v[:, 1:]).min(1).values
    safe = gaps > 1e-5
    assert torch.equal(got_i.cpu()[safe], want_i[safe])
    assert_close_rel(got_v.cpu(), want_v, 1e-5, "top-k values")


@pytest.mark.parametrize("M,N,d,Lx,k", [(5, 300, 32, 7, 3), (130, 5000, 128, 200, 50), (48, 3415, 64, 59, 20), (257, 70001, 128, 31, 64),
                                        (64, 20000, 256, 40, 50), (9, 700, 30, 5, 20), (33, 4100, 200, 0, 7), (300, 9000, 120, 20, 50)])
def test_score_topk_tensor_core_equals_fp32_engine(ops, M, N, d, Lx, k):
    """irs_score_topk_tc (tcgen05 chunk maxima + radix select + exact re-score; d <= 256) must return the SAME values, item ids
    and tie order as the fp32 CUDA-core engine irs_score_topk, and both must match the fp64 oracle outside fp32 near-ties:
    exclusions, catalog tails, exact ties (twin catalog rows -> lower id first), near-ties, k larger than what one chunk holds."""
    h, W, bias, excl = _score_case(M, N, d, max(Lx, 1), 81)
    g = _gen(82)
    # exact ties and near-ties among the leaders of rows 0 and 1
    s = h @ W.t() + bias
    top = s.topk(3, dim=1).indices
    tw = torch.randint(0, N, (6,), generator=g)
    W[tw] = W[top[0, 0]].clone(); bias[tw] = bias[top[0, 0]].clone()
    nt = torch.randint(0, N, (6,), generator=g)
    W[nt] = W[top[1, 1]].clone() * (1 + torch.linspace(-3e-6, 3e-6, 6).unsqueeze(1)); bias[nt] = bias[top[1, 1]].clone()
    hd, Wd, bd = h.to(DEV), W.to(DEV), bias.to(DEV)
    e = ops.sort_exclusions(excl.to(DEV), N, 1) if Lx else None
    want_v, want_i = ops.score_topk(hd, Wd, bd, k, e, 1)
    prep = ops.scorer_prepare_weights(Wd)
    got_v, got_i = ops.score_topk_tc(hd, Wd, prep, bd, k, e, 1)
    assert torch.equal(got_i, want_i), (got_i != want_i).sum()
    assert torch.equal(got_v, want_v)
    ov, oi = O.topk_excluding(h.double() @ W.double().t() + bias.double(), excl if Lx else None, k)
    kk = min(k, N - Lx)
    gaps = (ov[:, : kk - 1] - ov[:, 1:kk]).abs().min(1).values
    safe = gaps > 1e-5
    assert torch.equal(got_i.cpu()[safe][:, :kk], oi[safe][:, :kk])
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def test_score_topk_tensor_core_everything_excluded_and_item_base(ops):
    """Fewer live items than k -> (-inf, -1) padding like the fp32 engine; a catalog shard (item_base > 1) reports global ids."""
    M, N, d, k = 6, 40, 32, 50
    h, W, bias, _ = _score_case(M, N, d, 1, 91)
    excl = torch.arange(1, N + 1).unsqueeze(0).expand(M, -1).clone()
    excl[1:, 5:] = 0                                           # row 0: everything excluded; others: items 1..5 excluded
    hd, Wd, bd = h.to(DEV), W.to(DEV), bias.to(DEV)
    e = ops.sort_exclusions(excl.to(DEV), N, 1)
    prep = ops.scorer_prepare_weights(Wd)
    want = ops.score_topk(hd, Wd, bd, k, e, 1)
    got = ops.score_topk_tc(hd, Wd, prep, bd, k, e, 1)
    assert torch.equal(got[1], want[1]) and torch.equal(got[0].nan_to_num(neginf=-1e30), want[0].nan_to_num(neginf=-1e30))
    assert (got[1][0] == -1).all() and (got[1][1, : N - 5] > 5).all() and (got[1][1, N - 5:] == -1).all()
    e2 = ops.sort_exclusions(excl.to(DEV) + 1000, N, 1001)
    got2 = ops.score_topk_tc(hd, Wd, prep, bd, 4, e2, 1001)
    want2 = ops.score_topk(hd, Wd, bd, 4, e2, 1001)
    assert torch.equal(got2[1], want2[1]) and int(got2[1][1].min()) > 1005


def test_score_argmax_tensor_core_d256(ops):
    """128 < d <= 256: the single-MMA arg-max (hi image of h spans both operand regions) equals the fp32 engine."""
    M, N, d, Lx = 70, 9000, 256, 30
    h, W, bias, excl = _score_case(M, N, d, Lx, 95)
    hd, Wd, bd = h.to(DEV), W.to(DEV), bias.to(DEV)
    e = ops.sort_exclusions(excl.to(DEV), N, 1)
    want = ops.score_topk(hd, Wd, bd, 1, e, 1)
    got = ops.score_argmax_tc(hd, Wd, ops.scorer_prepare_weights(Wd), bd, e, 1, variant=2)
    assert torch.equal(got[1], want[1]) and torch.equal(got[0], want[0])


def test_score_topk_tensor_core_k_larger_than_chunk_count(ops):
    """k = 100 over a 700-item catalog (22 chunks < k: every live column is a candidate) against the fp64 oracle."""
    M, N, d, Lx, k = 9, 700, 30, 5, 100
    h, W, bias, excl = _score_case(M, N, d, Lx, 97)
    hd, Wd, bd = h.to(DEV), W.to(DEV), bias.to(DEV)
    e = ops.sort_exclusions(excl.to(DEV), N, 1)
    gv, gi = ops.score_topk_tc(hd, Wd, ops.scorer_prepare_weights(Wd), bd, k, e, 1)
    ov, oi = O.topk_excluding(h.double() @ W.double().t() + bias.double(), excl, k)
    safe = (ov[:, :-1] - ov[:, 1:]).min(1).values > 1e-5
    assert safe.any()
    assert torch.equal(gi.cpu()[safe], oi[safe])
    assert_close_rel(gv.cpu(), ov, 1e-5, "top-100 values")


@pytest.mark.parametrize("M,L,N,lo,hi", [(37, 14, 50, 0, 50), (300, 201, 5000, 0, 5000), (64, 60, 900, 300, 650), (5, 3, 10, 0, 10)])
def test_exclusions_update_equals_resort(ops, M, L, N, lo, hi):
    """One window step applied incrementally to the sorted exclusion lists (one id slides out, the pick comes in) equals
    re-sorting the shifted windows: duplicates inside a window, PAD entries, ids outside the catalog shard [lo+1, hi], several
    steps in a row."""
    g = _gen(33)
    win = torch.randint(0, N + 1, (M, L), generator=g)          # 0 = PAD; duplicates are likely for small N
    win[:, : L // 3][torch.rand((M, L // 3), generator=g) < 0.5] = 0
    w = win.to(DEV)
    excl = ops.sort_exclusions(w[:, :-1].contiguous(), hi - lo, lo + 1)
    for step in range(2 * L):
        nxt = torch.randint(1, N + 1, (M,), generator=g).to(DEV)
        ops.exclusions_update(excl, w[:, 0], nxt, hi - lo, lo + 1)
        ops.window_shift(w, nxt, None, 0)
        want = ops.sort_exclusions(w[:, :-1].contiguous(), hi - lo, lo + 1)
        assert torch.equal(excl[1], want[1]), f"counts differ at step {step}"
        assert torch.equal(excl[0], want[0]), f"lists differ at step {step}"


def _drop_mask(seed, B, H, L, p):
    """The kernels' counter-based keep mask (csrc/attention.cu: drop_scale) restated with numpy uint64 arithmetic."""
    import numpy as np
    bh = np.arange(B * H, dtype=np.uint64).reshape(B * H, 1, 1)
    i = np.arange(L, dtype=np.uint64).reshape(1, L, 1)
    j = np.arange(L, dtype=np.uint64).reshape(1, 1, L)
    with np.errstate(over="ignore"):
        idx = (bh * np.uint64(L) + i) * np.uint64(L) + j + np.uint64(1)
        x = np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * idx
        x ^= x >> np.uint64(33); x *= np.uint64(0xff51afd7ed558ccd)
        x ^= x >> np.uint64(33); x *= np.uint64(0xc4ceb9fe1a85ec53)
        x ^= x >> np.uint64(33)
    keep = (x >> np.uint64(32)) >= np.uint64(int(p * 4294967296.0))
    return torch.from_numpy(keep.reshape(B, H, L, L))


@pytest.mark.parametrize("B,L,H,dh,mode,p", [(3, 12, 2, 16, 0, 0.3), (2, 50, 4, 32, 0, 0.05), (3, 14, 2, 16, 1, 0.5)])
def test_pim_attention_probability_dropout(ops, B, L, H, dh, mode, p):
    """Train-mode attention-probability dropout (nn.MultiheadAttention(dropout=p); ADVICE r1): forward and backward of the
    fp32 kernels against autograd of  (softmax(s) o M / (1-p)) V  in fp64, with M regenerated from the same seed."""
    g = _gen(15)
    d = H * dh
    qkv = torch.randn((B, L, 3 * d), generator=g)
    ids = torch.randint(1, 100, (B, L), generator=g)
    r_u = torch.randn(B, generator=g)
    go = torch.randn((B, L, d), generator=g)
    torch.manual_seed(321)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())       # what ops._PimAttention.forward will draw
    keep = _drop_mask(seed, B, H, L, p)
    assert abs(float(keep.float().mean()) - (1 - p)) < 0.05
    a = qkv.double().requires_grad_(True)
    r = r_u.double().requires_grad_(True)
    q, k, v = (a[..., i * d:(i + 1) * d].reshape(B, L, H, dh).transpose(1, 2) for i in range(3))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
    s = s + (O.pim_mask(L, r.reshape(B, 1)).unsqueeze(1) if mode == 0 else O.causal_mask(L))
    s = s.masked_fill(ids.eq(0)[:, None, None, :], float("-inf"))
    want = ((torch.softmax(s, -1) * keep.double() / (1 - p)) @ v).transpose(1, 2).reshape(B, L, d)
    want.backward(go.double())
    q_dev = qkv.to(DEV).requires_grad_(True)
    r_dev = r_u.to(DEV).requires_grad_(True)
    torch.manual_seed(321)
    out = ops.pim_attention(q_dev, ids.to(DEV), r_dev if mode == 0 else None, H, mode, p_drop=p)
    assert_close_rel(out.detach().cpu(), want.detach(), 1e-5, "dropout forward")
    out.backward(go.to(DEV))
    assert_close_rel(q_dev.grad.cpu(), a.grad, 5e-5, "d_qkv with dropout")
    if mode == 0:
        assert_close_rel(r_dev.grad.cpu(), r.grad, 5e-5, "d_r_u with dropout")
    # p = 0 is the undropped kernel bit for bit
    o0 = ops.pim_attention(qkv.to(DEV).requires_grad_(True), ids.to(DEV), r_u.to(DEV) if mode == 0 else None, H, mode, p_drop=0.0)
    o1 = ops.pim_attention(qkv.to(DEV).requires_grad_(True), ids.to(DEV), r_u.to(DEV) if mode == 0 else None, H, mode)
    assert torch.equal(o0, o1)


@pytest.mark.parametrize("B,L,H,dh,mode", [(3, 50, 4, 32, 0), (2, 60, 2, 16, 1), (2, 201, 4, 32, 0)])
def test_training_forward_attention_on_tensor_cores_returns_lse(ops, B, L, H, dh, mode, monkeypatch):
    """The training forward (lse needed) runs on the per-head tcgen05 kernel: its output and log-sum-exp equal the fp32
    kernel's (which the backward kernel was written against) to tensor-core accuracy, fully padded heads included."""
    g = _gen(25)
    d = H * dh
    qkv = torch.randn((B, L, 3 * d), generator=g).to(DEV)
    ids = torch.randint(1, 100, (B, L), generator=g)
    ids[0, : L // 3] = 0
    ids = ids.to(DEV)
    r_u = torch.randn(B, generator=g).to(DEV) if mode == 0 else None
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    monkeypatch.setattr(ops, "USE_TC_TRAIN_ATTENTION", True)
    pkg_launch0 = ops.launch_count()
    o_tc, l_tc = ops._attn_fwd_raw(q, k, v, (3 * d,) * 3, ids, r_u, 0.05, 1.0, mode, B, L, H, dh, 0, L, True)
    monkeypatch.setattr(ops, "USE_TC_TRAIN_ATTENTION", False)
    o_32, l_32 = ops._attn_fwd_raw(q, k, v, (3 * d,) * 3, ids, r_u, 0.05, 1.0, mode, B, L, H, dh, 0, L, True)
    assert ops.launch_count() == pkg_launch0 + 2
    ok = torch.isfinite(l_32)                                   # rows that see no key at all are NaN / -inf in both
    assert ok.float().mean() > 0.5
    assert_close_rel(l_tc[ok].cpu(), l_32[ok].cpu(), 2e-5, "lse")
    okr = torch.isfinite(o_32).all(-1)
    assert_close_rel(o_tc[okr].cpu(), o_32[okr].cpu(), 5e-5, "attention output")
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0
