"""GPU: the on-device top-k sampler irs_topk_sample (ops.topk_sample) and sampled influence-path generation.

The kernel's picks equal the numpy emulator of tests/test_sample_cpu.py bit for bit; its draws follow the softmax over
the survivors and are independent from step to step; they do not depend on how the candidates are split over catalog
shards, on the user tile or on the number of ranks."""
import math
import socket

import numpy as np
import pytest
import torch

from oracle.ref_shim import irn_config
from tests.helpers import load_golden
from tests.test_sample_cpu import emulate_sample, merged_topk

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import influentialrs_b200 as p
    return p


def _candidates(rng, G, M, k, n_items=1_000_000):
    """Per-shard lists [G,M,k] as a scorer leaves them: item ids distinct within a row, exact score ties across shards, a
    few rows with fewer live candidates than k ((-inf, -1) slots); every shard's list shuffled."""
    n = G * k
    vals = (2.0 * rng.standard_normal((M, n))).astype(np.float32)
    if n > 1:
        j = k if G > 1 else 1                                 # the first candidate of shard 1 (or the second of shard 0)
        vals[: M // 4, j] = vals[: M // 4, 0]                 # an exact tie in a quarter of the rows
    span = n_items // n
    items = rng.integers(0, span, (M, n)) + np.arange(n) * span + 1                  # distinct within a row
    items = np.take_along_axis(items, np.argsort(rng.random((M, n)), 1), 1)          # ids in random slot order
    vals = np.ascontiguousarray(vals.reshape(M, G, k).transpose(1, 0, 2))
    items = np.ascontiguousarray(items.reshape(M, G, k).transpose(1, 0, 2))
    short = rng.random((G, M, k)) < 0.02
    vals[short], items[short] = -np.inf, -1
    perm = rng.permutation(k)
    return np.ascontiguousarray(vals[:, :, perm]), np.ascontiguousarray(items[:, :, perm])


@pytest.mark.parametrize("G", [1, 3])
@pytest.mark.parametrize("k", [1, 3, 50])
def test_kernel_draw_equals_the_emulator_bit_for_bit(pkg, G, k):
    ops = pkg.ops
    rng = np.random.default_rng(100 * G + k)
    M = 20_000 if k < 50 else 4_000
    vals, items = _candidates(rng, G, M, k)
    keys = rng.integers(-2 ** 62, 2 ** 62, M)
    for seed, step in ((0, 0), (2 ** 62 - 1, 19), (123456789, -1)):
        got = ops.topk_sample(torch.from_numpy(vals).to(DEV), torch.from_numpy(items).to(DEV), seed, step,
                              torch.from_numpy(keys).to(DEV)).cpu().numpy()
        want, gap = emulate_sample(vals, items, seed, step, keys, return_margin=True)
        close = gap <= 1e-12                     # |u S - C_i| <= 1e-12 S: CUDA's and numpy's exp may differ by an ulp
        assert close.mean() < 1e-6
        np.testing.assert_array_equal(got[~close], want[~close])
        if k > 1:
            sv, si, live, _ = merged_topk(vals, items)
            assert (got != si[:, 0]).mean() > 0.1          # a draw, not the arg-max
    # the [M,k] form is G = 1; G = 3 equals G = 1 on the merged list
    if G == 3:
        v3, i3 = torch.from_numpy(vals).to(DEV), torch.from_numpy(items).to(DEV)
        mv, mi = ops.topk_merge(v3, i3)
        kt = torch.from_numpy(keys).to(DEV)
        assert torch.equal(ops.topk_sample(v3, i3, 5, 2, kt), ops.topk_sample(mv, mi, 5, 2, kt))


def test_draws_follow_the_softmax_and_are_independent_across_steps(pkg):
    from scipy import stats
    ops = pkg.ops
    s = torch.tensor([2.0, 1.0, 0.5, 0.0, -1.0])
    M = 2 ** 20
    vals = s.view(1, 5).expand(M, 5).contiguous().to(DEV)
    items = torch.arange(1, 6).view(1, 5).expand(M, 5).contiguous().to(DEV)
    keys = torch.arange(M, dtype=torch.int64, device=DEV)
    a = ops.topk_sample(vals, items, 20261020, 4, keys).cpu().numpy()
    b = ops.topk_sample(vals, items, 20261020, 5, keys).cpu().numpy()
    p = torch.softmax(s.double(), 0).numpy()
    for x in (a, b):
        obs = np.bincount(x, minlength=6)[1:]
        assert obs.sum() == M
        assert stats.chisquare(obs, p * M).pvalue > 1e-3
    table = np.zeros((5, 5))
    np.add.at(table, (a - 1, b - 1), 1)
    assert stats.chi2_contingency(table).pvalue > 1e-3


def _problem(N, M, d, Lx, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    W = torch.randn((N, d), generator=g, device=DEV) / math.sqrt(d)
    bias = 0.1 * torch.randn((N,), generator=g, device=DEV)
    h = torch.randn((M, d), generator=g, device=DEV)
    window = torch.randint(1, N + 1, (M, Lx), generator=g, device=DEV)
    return W, bias, h, window


@pytest.mark.parametrize("N", [40_000, 3_001])
@pytest.mark.parametrize("k", [3, 50])
def test_shards_emulated_on_one_gpu_draw_what_the_full_catalog_draws(pkg, N, k):
    """Per-shard top-k over row slices of W (item_base) fed to the sampler as G = 3 gives the picks of G = 1 over the full
    catalog's top-k: tensor-core top-k for N = 40,000 (>= TC_TOPK_MIN_ITEMS), the fp32 engine for the small catalog."""
    ops = pkg.ops
    M, d = 512, 128
    W, bias, h, window = _problem(N, M, d, 40, seed=N + k)
    tc = N >= ops.TC_TOPK_MIN_ITEMS
    full_v, full_i = ops.score_topk_any(h, W, bias, k, ops.sort_exclusions(window, N, 1), 1)
    vs, its = [], []
    for g in range(3):
        lo, hi = g * N // 3, (g + 1) * N // 3
        excl = ops.sort_exclusions(window, hi - lo, lo + 1)
        if tc:
            v, i = ops.score_topk_tc(h, W[lo:hi], ops.scorer_prepare_weights(W[lo:hi].contiguous()), bias[lo:hi], k, excl,
                                     lo + 1)
        else:
            v, i = ops.score_topk(h, W[lo:hi], bias[lo:hi], k, excl, lo + 1)
        vs.append(v)
        its.append(i)
    vals, items = torch.stack(vs), torch.stack(its)
    mv, mi = ops.topk_merge(vals, items)
    assert torch.equal(mi, full_i) and torch.equal(mv, full_v)
    keys = torch.arange(M, dtype=torch.int64, device=DEV) + 1000
    for step in range(4):
        one = ops.topk_sample(full_v, full_i, 77, step, keys)
        three = ops.topk_sample(vals, items, 77, step, keys)
        assert torch.equal(one, three)
        assert not (window == one.view(-1, 1)).any()                      # never a window item
        assert bool(((one.view(-1, 1) == full_i).any(1)).all())          # always one of the k best


def test_edge_rows(pkg):
    ops = pkg.ops
    N, d, k = 6, 16, 4
    W, bias, h, _ = _problem(N, 3, d, 1, seed=3)
    window = torch.tensor([[1, 2, 3, 0, 0, 0],                 # three live items for k = 4
                           [1, 2, 3, 4, 5, 6],                 # every item excluded
                           [1, 2, 3, 4, 0, 0]], device=DEV)
    v, i = ops.score_topk(h, W, bias, k, ops.sort_exclusions(window, N, 1), 1)
    keys = torch.arange(3, dtype=torch.int64, device=DEV)
    for step in range(20):
        pick = ops.topk_sample(v, i, 9, step, keys).cpu()
        assert int(pick[0]) in (4, 5, 6)                                   # three live items for k = 4
        assert int(pick[1]) == -1                                           # every item excluded: what the arg-max gives
        assert int(pick[2]) in (5, 6)
    # the overflow marker of score_topk is never sampled around
    v2, i2 = v.clone(), i.clone()
    v2[0, 2], i2[0, 2] = float("nan"), -2
    pick = ops.topk_sample(v2, i2, 9, 0, keys).cpu()
    assert int(pick[0]) == -2 and int(pick[2]) in (5, 6)
    pick3 = ops.topk_sample(torch.stack([v, v2]), torch.stack([i, i2]), 9, 0, keys).cpu()     # in any shard
    assert int(pick3[0]) == -2
    with pytest.raises(RuntimeError):
        ops.topk_sample(v.expand(2000, 3, k).contiguous(), i.expand(2000, 3, k).contiguous(), 0, 0, keys)   # G k > 4096


# ---- end to end ---------------------------------------------------------------------------------------------------
def _build(pkg, name, user_tile=None):
    sd, g = load_golden(name)
    cfgv = g["cfg"]
    cfg = irn_config(*[int(x) for x in cfgv[:7]], u_emb_dim=int(cfgv[7]), dropout=0.0)
    if user_tile is not None:
        cfg.user_tile = user_tile
    net = pkg.InfluentialNet(cfg)
    net.load_state_dict(sd, strict=True)
    net.to(DEV).eval()
    return g, pkg.IRSNN(cfg, net, DEV)


@pytest.mark.parametrize("name", ["irn_small", "irn_d30", "irn_ml1m"])
def test_sample_k1_is_greedy(pkg, name):
    g, irn = _build(pkg, name)
    seqs, users = torch.from_numpy(g["seqs"]).to(DEV), torch.from_numpy(g["users"]).to(DEV)
    targets = torch.from_numpy(g["targets"]).to(DEV)
    P = g["paths"].shape[1]
    paths, _, _, ne = irn.get_seq_in_batch(seqs, users, targets, max_path_len=P, gap_len=0, sample=True, sample_k=1)
    np.testing.assert_array_equal(paths, g["paths"])
    assert ne == int(g["n_early"])


def test_sampled_paths_do_not_depend_on_the_user_tile(pkg):
    runs = []
    for tile in (4096, 7):
        g, irn = _build(pkg, "irn_ml1m", user_tile=tile)
        seqs, users = torch.from_numpy(g["seqs"]).to(DEV), torch.from_numpy(g["users"]).to(DEV)
        torch.manual_seed(31)
        runs.append(irn.get_seq_in_batch(seqs, users, seqs[:, -1], max_path_len=8, gap_len=0, sample=True, sample_k=5)[0])
    np.testing.assert_array_equal(runs[0], runs[1])
    torch.manual_seed(32)
    other = irn.get_seq_in_batch(seqs, users, seqs[:, -1], max_path_len=8, gap_len=0, sample=True, sample_k=5)[0]
    assert not np.array_equal(other, runs[0])                                # another torch seed, other paths


def test_sampled_test_batch_equals_the_separate_calls(pkg):
    g, irn = _build(pkg, "irn_small")
    seqs, users = torch.from_numpy(g["seqs"]).to(DEV), torch.from_numpy(g["users"]).to(DEV)
    targets, labels = torch.from_numpy(g["targets"]).to(DEV), torch.from_numpy(g["labels"]).to(DEV)
    raw = list(torch.split(torch.from_numpy(g["raw_flat"]), g["raw_lens"].tolist()))
    P = g["paths"].shape[1]
    torch.manual_seed(5)
    r_u, hit, rr, paths, tg, hist, ne = irn.test_batch(raw, seqs, users, targets, labels, top_k=20, max_path_len=P,
                                                       sample=True, sample_k=3)
    torch.manual_seed(5)
    hit2, rr2 = irn.get_accuracy_metrics_in_batch(raw, seqs, users, targets, labels, 20, 0, True)
    p2, t2, h2, ne2 = irn.get_seq_in_batch(seqs, users, targets, max_path_len=P, gap_len=0, sample=True, sample_k=3)
    assert hit == hit2 and ne == ne2
    np.testing.assert_array_equal(rr, rr2)
    np.testing.assert_array_equal(paths, p2)


def test_world1_sharded_sampling_equals_single_gpu(pkg):
    import torch.distributed as dist
    from influentialrs_b200.dist import ShardedGenerator
    g, irn = _build(pkg, "irn_ml1m", user_tile=16)
    seqs, users = torch.from_numpy(g["seqs"]).to(DEV), torch.from_numpy(g["users"]).to(DEV)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        sg = ShardedGenerator(irn, 0, 1)
        for k in (3, 20):
            torch.manual_seed(k)
            got = sg.get_seq_in_batch(seqs, users, seqs[:, -1], max_path_len=6, sample=True, sample_k=k)[0]
            torch.manual_seed(k)
            want = irn.get_seq_in_batch(seqs, users, seqs[:, -1], max_path_len=6, gap_len=0, sample=True, sample_k=k)[0]
            np.testing.assert_array_equal(got, want)
    finally:
        dist.destroy_process_group()
