"""The softmax cross-entropy kernels on the cases of tests/ce_cases.py, each engine against float64 within its own
per-element error bound: the log-sum-exp forward (score_lse_gather), softmax_ce_mean forward and backward, and the raw
C ABI of irs_score_ce_bwd[_tc] (accumulation into d_W / d_bias, NULL outputs, selected ids outside the catalog), at
shapes that take every branch of the tensor-core backward's plan(), at the training shape, and through the catalog-sharded
log-sum-exp merge of ShardedScorer."""
import functools
import math

import pytest
import torch

from tests import ce_cases as C

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ENGINES = ("simt", "tc")

# (M, N, d): M / N in {1, 127, 128, 129}; d in {16, 30, 64, 100, 128}; 295 vs 296 user tiles (2 splits vs owner path of
# the d_h pass at N = 5000); short last splits (40000 x 700: 20 splits of 16 user tiles, the last 9 long; 37760 x 5000:
# 8 splits of 37, the last 36); 700 x 40000 (d_W owner path, d_h split 20 ways)
SHAPES = [(1, 300, 64), (127, 1000, 128), (128, 129, 30), (129, 127, 100), (300, 1, 16), (1000, 128, 64),
          (260, 5000, 16), (37760, 5000, 64), (37888, 5000, 64), (700, 40000, 128), (40000, 700, 128)]


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


@functools.lru_cache(maxsize=4)
def _case(M, N, d, kind="mixed"):
    c = C.mixed_case(M, N, d, 11) if kind == "mixed" else C.control_case(M, N, d, 12)
    return c, tuple(t.to(DEV) for t in (c.h, c.W, c.bias, c.target, c.sel))


def _engine(ops, monkeypatch, engine):
    monkeypatch.setattr(ops, "USE_TC_LSE", engine == "tc")
    monkeypatch.setattr(ops, "USE_TC_CE_BWD", engine == "tc")


def _healthy(ops):
    torch.cuda.synchronize()
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def _inside(got, ref, bound, what):
    r = C.ratio(got, ref, bound)
    assert r <= 1.0, f"{what}: error {r:.3g} x its bound"
    return r


def raw_bwd(engine, h, W, b, tgt, lse, gscale, dh, dW, db):
    """irs_score_ce_bwd (simt) or irs_score_ce_bwd_tc through the C ABI; any of dh, dW, db may be None (NULL)."""
    from influentialrs_b200._lib import lib, check
    p = lambda t: None if t is None else t.data_ptr()
    M, d = h.shape
    N = W.shape[0]
    s = torch.cuda.current_stream().cuda_stream
    if engine == "simt":
        check(lib().irs_score_ce_bwd(p(h), d, p(W), p(b), p(tgt), p(lse), gscale, p(dh), p(dW), p(db), M, N, d, s), "ce_bwd")
        return
    nb = lib().irs_score_ce_bwd_tc_workspace_bytes(M, N, d)
    ws = torch.empty((nb,), dtype=torch.uint8, device=DEV)
    check(lib().irs_score_ce_bwd_tc(p(h), d, p(W), p(b), p(tgt), p(lse), gscale, p(dh), p(dW), p(db), M, N, d,
                                    p(ws), nb, s), "ce_bwd_tc")


# ---------------------------------------------------------------------------------------------- forward
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("M,N,d", SHAPES)
def test_lse_gather_inside_bound(ops, M, N, d, engine, monkeypatch):
    _engine(ops, monkeypatch, engine)
    c, (h, W, b, _, sel) = _case(M, N, d)
    lse, logit = ops.score_lse_gather(h, W, b, sel, 1)
    _healthy(ops)
    want_lse, want_logit = C.forward_ref(h, W, b, sel)
    lse_b, logit_b = C.forward_bound(h, W, b, sel, engine)
    _inside(lse, want_lse, lse_b, f"{c.name} {engine} lse")
    _inside(logit, want_logit, logit_b, f"{c.name} {engine} selected logits")
    off = (sel < 1) | (sel > N)
    assert bool((logit[off] == 0).all()), f"{engine}: ids outside the catalog must give 0.0, got {logit[off].unique()}"


# ---------------------------------------------------------------------------------------------- softmax_ce_mean
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("M,N,d", SHAPES)
def test_softmax_ce_inside_bound(ops, M, N, d, engine, monkeypatch):
    """Loss and gradients of softmax_ce_mean (rows with a target; the backward gets the forward's own lse)."""
    _engine(ops, monkeypatch, engine)
    c, (h, W, b, tgt, _) = _case(M, N, d)
    live = tgt >= 0
    h, tgt = h[live].contiguous(), tgt[live].contiguous()
    Ml = h.shape[0]
    hd, Wd, bd = (t.clone().requires_grad_(True) for t in (h, W, b))
    loss = ops.softmax_ce_mean(hd, Wd, bd, tgt)
    loss.backward()
    _healthy(ops)
    sel = (tgt + 1).view(-1, 1)
    want_lse, want_logit = C.forward_ref(h, W, b, sel)
    lse_b, logit_b = C.forward_bound(h, W, b, sel, engine)
    rows = want_lse - want_logit[:, 0]
    tol = float((lse_b + logit_b[:, 0]).mean()) + (math.log2(Ml) + 2) * C.U24 * float(rows.abs().mean())
    assert abs(float(loss) - float(rows.mean())) <= tol, (float(loss), float(rows.mean()), tol)
    lse_k, _ = ops.score_lse_gather(h, W, b, sel, 1)            # the lse the backward received
    out = C.backward_bound(h, W, b, tgt, lse_k, 1.0 / Ml, engine)
    for name, got in (("d_h", hd.grad), ("d_W", Wd.grad), ("d_bias", bd.grad)):
        _inside(got, *out[name], f"{c.name} {engine} {name}")


# ---------------------------------------------------------------------------------------------- raw C ABI
@pytest.mark.parametrize("lse_from", ["fp64", "kernel"])
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("M,N,d", SHAPES)
def test_ce_bwd_accumulates_inside_bound(ops, M, N, d, engine, lse_from, monkeypatch):
    """irs_score_ce_bwd[_tc] with skipped rows, d_h prefilled with garbage (it is written), d_W and d_bias prefilled with
    nonzero values (they are accumulated into, on the owner path and on the red.global split path)."""
    _engine(ops, monkeypatch, engine)
    c, (h, W, b, tgt, _) = _case(M, N, d)
    if lse_from == "fp64":
        lse = C.forward_ref(h, W, b, tgt.view(-1, 1) + 1)[0].float()
    else:
        lse = ops.score_lse_gather(h, W, b, (tgt.clamp(min=0) + 1).view(-1, 1), 1)[0]
    g = torch.Generator(device=DEV).manual_seed(5)
    gscale = 1.0 / max(1, int((tgt >= 0).sum()))
    pre_W = torch.randn((N, d), generator=g, device=DEV) * 1e-3
    pre_b = torch.randn((N,), generator=g, device=DEV) * 1e-3
    dh = torch.full((M, d), 7.0, device=DEV)
    dW, db = pre_W.clone(), pre_b.clone()
    raw_bwd(engine, h, W, b, tgt, lse, gscale, dh, dW, db)
    _healthy(ops)
    out = C.backward_bound(h, W, b, tgt, lse, gscale, engine, prefill_W=pre_W, prefill_b=pre_b)
    _inside(dh, *out["d_h"], f"{c.name} {engine} d_h")
    _inside(dW, *out["d_W"], f"{c.name} {engine} d_W += ")
    _inside(db, *out["d_bias"], f"{c.name} {engine} d_bias += ")
    assert float(dh[tgt < 0].abs().max()) == 0.0 if bool((tgt < 0).any()) else True


@pytest.mark.parametrize("null", ["d_h", "d_W", "d_bias"])
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("M,N,d", [(700, 40000, 128), (40000, 700, 128), (129, 127, 100)])
def test_ce_bwd_null_output(ops, M, N, d, engine, null):
    """Each of d_h, d_W, d_bias may be NULL; the other outputs are still right."""
    c, (h, W, b, tgt, _) = _case(M, N, d)
    lse = C.forward_ref(h, W, b, tgt.view(-1, 1) + 1)[0].float()
    gscale = 1.0 / M
    bufs = {"d_h": torch.zeros((M, d), device=DEV), "d_W": torch.zeros((N, d), device=DEV), "d_bias": torch.zeros((N,), device=DEV)}
    bufs[null] = None
    raw_bwd(engine, h, W, b, tgt, lse, gscale, bufs["d_h"], bufs["d_W"], bufs["d_bias"])
    torch.cuda.synchronize()
    out = C.backward_bound(h, W, b, tgt, lse, gscale, engine)
    for name, got in bufs.items():
        if got is not None:
            _inside(got, *out[name], f"{c.name} {engine} {name} with {null} NULL")


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("N", [300, 384])
def test_selected_ids_outside_catalog_give_zero(ops, N, engine, monkeypatch):
    """sel = 0, > N (inside the last partial tile and beyond it) or negative: logit 0.0 on both engines."""
    _engine(ops, monkeypatch, engine)
    c, (h, W, b, _, _) = _case(40, N, 64)
    bad = torch.tensor([0, N + 1, N + 2, N + 100, 10 ** 6, -1, -3], dtype=torch.int64)
    sel = torch.stack([bad.roll(i) for i in range(40)]).to(DEV)
    sel[:, 0] = torch.arange(1, 41, device=DEV)
    _, logit = ops.score_lse_gather(h, W, b, sel, 1)
    torch.cuda.synchronize()
    assert torch.equal(logit[:, 1:].cpu(), torch.zeros((40, sel.shape[1] - 1))), logit[:, 1:].unique()
    want = C.forward_ref(h, W, b, sel[:, :1])[1]
    _inside(logit[:, :1], want, C.forward_bound(h, W, b, sel[:, :1], engine)[1], f"{engine} in-catalog logits")


# ---------------------------------------------------------------------------------------------- sharded lse
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("M,N,d", [(300, 1000, 64), (129, 5000, 128), (1000, 129, 30), (127, 40000, 100)])
def test_sharded_lse_gather_matches_unsharded(ops, M, N, d, engine, monkeypatch):
    """ShardedScorer's per-shard _lse_cuda (item_base = lo + 1) and _select_cuda on the real kernels, merged as lse_gather
    merges them (float64 logsumexp over the shards, MAX over the selects, 0.0 outside the catalog): within the bound of
    the float64 result, and of the unsharded score_lse_gather."""
    from influentialrs_b200.dist import ShardedScorer
    _engine(ops, monkeypatch, engine)
    c, (h, W, b, _, sel) = _case(M, N, d)
    lses, logits, bounds = [], [], []
    for g in range(3):
        sc = ShardedScorer(W, b, rank=g, world=3)
        lses.append(sc._lse_cuda(h))
        logits.append(sc._select_cuda(h, sel))
        bounds.append(C.forward_bound(h, sc.W, sc.b, sel, engine, item_base=sc.lo + 1)[0])
    _healthy(ops)
    lse = torch.logsumexp(torch.stack(lses).double(), 0).float()
    logit = torch.stack(logits).max(0).values
    logit = torch.where((sel < 1) | (sel > N), torch.zeros_like(logit), logit)
    # merging is 1-Lipschitz in the per-shard errors; + the fp32 rounding of the merged value
    want_lse, want_logit = C.forward_ref(h, W, b, sel)
    lse_b = torch.stack(bounds).max(0).values + C.U23 * want_lse.abs()
    logit_b = C.forward_bound(h, W, b, sel, engine)[1]
    _inside(lse, want_lse, lse_b, f"{c.name} {engine} sharded lse")
    _inside(logit, want_logit, logit_b, f"{c.name} {engine} sharded logits")
    # and the merge done by ShardedScorer.lse_gather itself (world = 1 path of the same code on the whole catalog)
    full_lse, full_logit = ops.score_lse_gather(h, W, b, sel, 1)
    lse_fb, logit_fb = C.forward_bound(h, W, b, sel, engine)
    _inside(lse, full_lse.double(), lse_b + lse_fb, f"{c.name} {engine} sharded vs unsharded lse")
    _inside(logit, full_logit.double(), 2 * logit_fb, f"{c.name} {engine} sharded vs unsharded logits")
    sc1 = ShardedScorer(W, b, rank=0, world=1)
    l1, g1 = sc1.lse_gather(h, sel)
    _inside(l1, want_lse, lse_fb + C.U23 * want_lse.abs(), f"{engine} ShardedScorer.lse_gather world 1")
    _inside(g1, want_logit, logit_fb, f"{engine} ShardedScorer.lse_gather logits world 1")


# ---------------------------------------------------------------------------------------------- training shape
TRAIN_M, TRAIN_N, TRAIN_D = 200704, 500000, 128          # bench cfg4: 4096 users x 49 targets, 500k items, d = 128


@functools.lru_cache(maxsize=1)
def _training():
    c = C.training_case(TRAIN_M, TRAIN_N, TRAIN_D, 21, device=DEV)
    g = torch.Generator().manual_seed(22)
    rows = torch.cat([torch.tensor([0, 1, 127, 128, TRAIN_M - 129, TRAIN_M - 1]),
                      torch.randperm(TRAIN_M, generator=g)[:506]]).unique()
    cols = torch.cat([torch.tensor([0, 1, 127, 128, TRAIN_N - 33, TRAIN_N - 1]), c.target[rows[:200]].cpu(),
                      torch.randperm(TRAIN_N, generator=g)[:306]]).unique()
    return c, rows.to(DEV), cols.to(DEV)


@pytest.mark.parametrize("engine", ENGINES)
def test_training_shape(ops, engine, monkeypatch):
    """M = 200,704 CE rows, N = 500,000 items, d = 128 (the d_h pass sweeps 3,907 item tiles into one accumulator, the
    d_W pass 1,568 user tiles), anisotropic and confident rows.  lse and loss on 512 sampled rows, d_h on the same rows,
    d_W and d_bias on ~512 sampled items, all against float64 given the lse the backward received: inside the bound, and
    within 1e-3 of each compared tensor's max."""
    _engine(ops, monkeypatch, engine)
    c, rows, cols = _training()
    h, W, b, tgt = c.h, c.W, c.bias, c.target
    M, N, d = TRAIN_M, TRAIN_N, TRAIN_D
    sel = (tgt + 1).view(-1, 1)
    lse, logit = ops.score_lse_gather(h, W, b, sel, 1)
    dh = torch.empty((M, d), device=DEV)
    dW = torch.zeros((N, d), device=DEV)
    db = torch.zeros((N,), device=DEV)
    gscale = 1.0 / M
    raw_bwd(engine, h, W, b, tgt, lse, gscale, dh, dW, db)                 # warm-up (module load, weight images)
    torch.cuda.synchronize()
    dW.zero_()
    db.zero_()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    raw_bwd(engine, h, W, b, tgt, lse, gscale, dh, dW, db)
    t1.record()
    _healthy(ops)
    ms = t0.elapsed_time(t1)
    want_lse, want_logit = C.forward_ref(h[rows], W, b, sel[rows])
    lse_b, logit_b = C.forward_bound(h[rows], W, b, sel[rows], engine, plan_M=M)
    r_lse = _inside(lse[rows], want_lse, lse_b, f"{engine} cfg4 lse")
    loss_ref = want_lse - want_logit[:, 0]
    loss = lse[rows].double() - logit[rows, 0].double()
    r_loss = _inside(loss, loss_ref, lse_b + logit_b[:, 0] + C.U24 * loss_ref.abs(), f"{engine} cfg4 per-row loss")
    out = C.backward_bound(h, W, b, tgt, lse, gscale, engine, rows=rows, cols=cols)
    bad = []
    report = [f"\ncfg4 shape {engine}: backward {ms:.1f} ms (one call, both passes); lse err/bound {r_lse:.3f}, "
              f"loss err/bound {r_loss:.3f}; loss rows: max|err| {float((loss - loss_ref).abs().max()):.3e}"]
    for name, got in (("d_h", dh[rows]), ("d_W", dW[cols]), ("d_bias", db[cols])):
        ref, bound = out[name]
        r = C.ratio(got, ref, bound)
        err = float((got.double() - ref).abs().max())
        scale = float(ref.abs().max())
        report.append(f"  {name}: max|err| / max|ref| = {err / scale:.3e} (north star {C.NORTH_STAR:g}), err/bound {r:.3f}")
        bad += [f"{name}: {r:.3g} x its bound"] if r > 1.0 else []
        bad += [f"{name}: {err / scale:.3e} of max|ref|"] if err > C.NORTH_STAR * scale else []
    print("\n".join(report))
    assert not bad, f"{engine} cfg4: " + "; ".join(bad)
