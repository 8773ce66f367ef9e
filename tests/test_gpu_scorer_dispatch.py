"""GPU: the dispatching scorer ops of ops.py.  Each picks its engine by one rule, returns empty outputs for zero rows
without a launch whichever engine it would pick, and takes its weight image from one cache keyed on (address, shape)
and weight version.  The catalog-sharded classes go through the same ops, so at world size 1 they give what one GPU
gives and share that cache."""
import math
import socket

import numpy as np
import pytest
import torch

from oracle.ref_shim import irn_config
from tests.helpers import load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


def _problem(N, M, d, seed, Lx=8):
    g = torch.Generator(device=DEV).manual_seed(seed)
    W = torch.randn((N, d), generator=g, device=DEV) / math.sqrt(d)
    bias = 0.1 * torch.randn((N,), generator=g, device=DEV)
    h = torch.randn((M, d), generator=g, device=DEV)
    window = torch.randint(1, N + 1, (M, Lx), generator=g, device=DEV)
    label = torch.randint(1, N + 1, (M,), generator=g, device=DEV)
    return W, bias, h, window, label


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("d", [64, 192])
def test_zero_rows_give_empty_outputs_without_a_launch(ops, tc, d, monkeypatch):
    for flag in ("USE_TC_TOPK", "USE_TC_LSE", "USE_TC_RANK", "USE_TC_CE_BWD"):
        monkeypatch.setattr(ops, flag, tc)
    N = 40_000                                                   # >= TC_TOPK_MIN_ITEMS: the top-k flag decides
    W, b, _, _, _ = _problem(N, 1, d, seed=d)
    h = torch.empty((0, d), device=DEV)
    lab = torch.empty((0,), dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    ops.launch_count_reset()
    v, i = ops.score_topk_any(h, W, b, 5, None, 1)
    assert v.shape == i.shape == (0, 5) and v.dtype == torch.float32 and i.dtype == torch.int64
    for reduce_lead in (None, lambda t: pytest.fail("no rows: no collective")):
        v, i = ops.score_argmax(h, W, b, None, 1, reduce_lead)
        assert v.shape == i.shape == (0, 1) and v.dtype == torch.float32 and i.dtype == torch.int64
    r = ops.score_rank(h, W, b, lab, None, 1)
    assert r.shape == (0,) and r.dtype == torch.int64
    c, f = ops.score_count_ahead(h, W, b, lab, torch.empty((0,), device=DEV), None, 1)
    assert c.shape == f.shape == (0,) and c.dtype == torch.int64 and f.dtype == torch.int32
    lse, logit = ops.score_lse_gather(h, W, b, torch.empty((0, 3), dtype=torch.int64, device=DEV), 1)
    assert lse.shape == (0,) and logit.shape == (0, 3)
    hg, Wg = h.clone().requires_grad_(True), W.clone().requires_grad_(True)
    loss = ops._SoftmaxCE.apply(hg, Wg, b, lab)                 # forward (lse) and backward dispatchers
    loss.backward()
    assert math.isnan(float(loss)) and hg.grad.shape == (0, d) and float(Wg.grad.abs().max()) == 0.0
    assert ops.launch_count() == 0


@pytest.mark.parametrize("d", [64, 192])
def test_world1_sharded_rank_equals_score_rank(ops, d):
    """d = 192 is outside the three-MMA kernels: the sharded count-ahead must take the fp32 engine as score_rank does."""
    from influentialrs_b200.dist import ShardedScorer
    N, M = 5_000, 300
    W, b, h, window, label = _problem(N, M, d, seed=7 + d)
    label[:5] = window[:5, 0]                                    # labels inside their own window -> rank 0
    want = ops.score_rank(h, W, b, label, ops.sort_exclusions(window, N, 1), 1)
    got = ShardedScorer(W, b, 0, 1).rank(h, label, window)
    assert torch.equal(got, want)
    assert bool((got[:5] == 0).all())


@pytest.mark.parametrize("N", [3_001, 40_000])
def test_world1_sharded_topk_equals_topk_any(ops, N):
    """The same values, ids and engine (the same launches) as score_topk_any, on both sides of TC_TOPK_MIN_ITEMS."""
    from influentialrs_b200.dist import ShardedScorer
    M, d, k = 256, 128, 20
    W, b, h, window, _ = _problem(N, M, d, seed=N)
    sc = ShardedScorer(W, b, 0, 1)
    runs = []
    for fn in (lambda: ops.score_topk_any(h, W, b, k, ops.sort_exclusions(window, N, 1), 1),
               lambda: sc.topk(h, k, window)):
        fn()                                                     # warm: the weight image, if any, is prepared here
        torch.cuda.synchronize()
        ops.launch_count_reset()
        out = fn()
        runs.append((out, ops.launch_count()))
    (wv, wi), n_want = runs[0]
    (gv, gi), n_got = runs[1]
    assert torch.equal(gi, wi) and torch.equal(gv, wv)
    assert n_got == n_want


def test_a_catalog_and_its_leading_shard_keep_their_images(ops):
    """W and W[:N//2] start at one address: alternating calls re-tile nothing after the first pass."""
    N, M, d = 70_000, 64, 128
    W, b, h, _, _ = _problem(N, M, d, seed=70)
    assert N // 2 >= ops.TC_TOPK_MIN_ITEMS
    torch.cuda.synchronize()
    ops.launch_count_reset()
    ops.scorer_prepare_weights(W)
    n_prep = ops.launch_count()                                  # launches of one re-tiling
    assert n_prep > 0
    ops.invalidate_prepared()
    counts = []
    for _ in range(3):
        for Wx, bx in ((W, b), (W[: N // 2], b[: N // 2])):
            torch.cuda.synchronize()
            ops.launch_count_reset()
            ops.score_topk_any(h, Wx, bx, 5, None, 1)
            counts.append(ops.launch_count())
    assert counts[0] == counts[2] + n_prep and counts[1] == counts[3] + n_prep  # one prepare each, in the first pass
    assert counts[2:] == counts[2:4] * 2


def test_irsnn_and_the_sharded_classes_prepare_project_weight_once(ops):
    import influentialrs_b200 as pkg
    import torch.distributed as dist
    from influentialrs_b200.dist import ShardedGenerator, ShardedScorer
    sd, g = load_golden("irn_ml1m")
    cfgv = g["cfg"]
    cfg = irn_config(*[int(x) for x in cfgv[:7]], u_emb_dim=int(cfgv[7]), dropout=0.0)
    net = pkg.InfluentialNet(cfg)
    net.load_state_dict(sd, strict=True)
    net.to(DEV).eval()
    irn = pkg.IRSNN(cfg, net, DEV)
    assert cfg.emb_dim <= ops.TC_THREE_MMA_MAX_D                  # arg-max and rank both read the tcgen05 image
    seqs, users = torch.from_numpy(g["seqs"]).to(DEV), torch.from_numpy(g["users"]).to(DEV)
    targets = seqs[:, -1]
    with torch.no_grad():
        h = net.decoding(seqs, users, last_row=seqs.shape[1] - 2)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        sg = ShardedGenerator(irn, 0, 1)
        sc = ShardedScorer(net.project.weight, net.project.bias, 0, 1)
        calls = (lambda: irn.get_seq_in_batch(seqs, users, targets, max_path_len=3, gap_len=0)[0],
                 lambda: sg.get_seq_in_batch(seqs, users, targets, max_path_len=3)[0],
                 lambda: sc.rank(h, targets, seqs[:, :-1]))
        passes = []
        for _ in range(2):
            counts, outs = [], []
            for fn in calls:
                torch.cuda.synchronize()
                ops.launch_count_reset()
                outs.append(fn())
                torch.cuda.synchronize()
                counts.append(ops.launch_count())
            passes.append((counts, outs))
        (first, outs), (again, _) = passes
        assert first[0] > again[0]                               # IRSNN's first pass prepares the images
        assert first[1:] == again[1:]                            # the sharded classes find project.weight's in the cache
        np.testing.assert_array_equal(outs[1], outs[0])
        excl = ops.sort_exclusions(seqs[:, :-1], cfg.n_item, 1)
        assert torch.equal(outs[2], ops.score_rank(h, net.project.weight, net.project.bias, targets, excl, 1))
    finally:
        dist.destroy_process_group()
