"""CPU: the on-device top-k sampler (irs_topk_sample) without a GPU -- a numpy emulator written from the definition in
include/irs_b200.h, the C entry point's argument checks, and sampled catalog-sharded generation (ShardedGenerator over
gloo, world 2) with the oracle's top-k and the emulator injected, against a single-process replay over the whole batch."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import irn_oracle as O

MASK64 = (1 << 64) - 1
PHI = 0x9E3779B97F4A7C15


def fmix64(x: np.ndarray) -> np.ndarray:
    """murmur3 finaliser on uint64 arrays (wrap-around arithmetic)."""
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xFF51AFD7ED558CCD)
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xC4CEB9FE1A85EC53)
        x = x ^ (x >> np.uint64(33))
    return x


def uniform(seed: int, step: int, row_key) -> np.ndarray:
    """u in [0, 1) of every row: x = fmix64(seed + phi (step + 1)); x = fmix64(x + phi (row_key + 1)); u = (x >> 11) 2^-53."""
    x = fmix64(np.array([(seed + PHI * (step + 1)) & MASK64], dtype=np.uint64))
    keys = np.asarray(row_key, dtype=np.int64).reshape(-1).astype(np.uint64)      # two's complement
    with np.errstate(over="ignore"):
        x = fmix64(x + np.uint64(PHI) * (keys + np.uint64(1)))
    return (x >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def merged_topk(vals, items):
    """[G,M,k] per-shard lists -> (vals [M,k], items [M,k], live [M,k], marker [M]): the best k by (score desc, id asc) of
    the candidates with an item id >= 0 and a non-NaN score; marker = a candidate is (NaN, -2) or has a NaN score."""
    vals, items = np.asarray(vals, dtype=np.float32), np.asarray(items, dtype=np.int64)
    if vals.ndim == 2:
        vals, items = vals[None], items[None]
    G, M, k = vals.shape
    v = vals.transpose(1, 0, 2).reshape(M, G * k)
    it = items.transpose(1, 0, 2).reshape(M, G * k)
    marker = ((it == -2) | np.isnan(v)).any(1)
    ok = (it >= 0) & ~np.isnan(v)
    order = np.lexsort((it, -np.where(ok, v, 0), ~ok), axis=1)[:, :k]
    take = lambda a: np.take_along_axis(a, order, 1)
    return take(v), take(it), take(ok), marker


def emulate_sample(vals, items, seed, step, row_key, return_margin=False):
    """The draw of irs_topk_sample: picks [M] int64 (and, optionally, min_i |u S - C_i| / S of every row: how close the
    draw came to a boundary, where CUDA's and numpy's exp may round differently)."""
    sv, si, live, marker = merged_topk(vals, items)
    M, k = sv.shape
    fin = live & np.isfinite(sv)
    any_fin = fin.any(1)
    first = fin.argmax(1)
    v0 = sv[np.arange(M), first].astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        w = np.where(fin, np.exp(sv.astype(np.float64) - v0[:, None]), 0.0)
    C = np.cumsum(w, axis=1)                       # sequential: adding the 0.0 of a non-finite slot changes nothing
    S = C[:, -1]
    t = uniform(seed, step, row_key) * S
    above = (C > t[:, None]) & fin
    last = k - 1 - np.argmax(fin[:, ::-1], axis=1)
    idx = np.where(above.any(1), above.argmax(1), last)
    pick = si[np.arange(M), idx]
    pick = np.where(any_fin, pick, -1)
    pick = np.where(marker, -2, pick)
    if not return_margin:
        return pick
    with np.errstate(invalid="ignore"):
        gap = np.where(fin, np.abs(t[:, None] - C), np.inf).min(1) / np.where(any_fin, S, 1.0)
    return pick, np.where(any_fin & ~marker, gap, np.inf)


def sample_fn_emulated(vals, items, seed, step, row_key):
    """ShardedGenerator.sample_fn on CPU tensors."""
    return torch.from_numpy(emulate_sample(vals.numpy(), items.numpy(), seed, step, row_key.numpy()))


# ---- the emulator itself --------------------------------------------------------------------------------------------
def test_uniform_is_a_pure_function_of_seed_step_and_key():
    keys = np.arange(-3, 200)
    u = uniform(12345, 7, keys)
    assert u.dtype == np.float64 and (u >= 0).all() and (u < 1).all()
    np.testing.assert_array_equal(u, uniform(12345, 7, keys))
    assert not np.array_equal(u, uniform(12345, 8, keys)) and not np.array_equal(u, uniform(12346, 7, keys))
    np.testing.assert_array_equal(uniform(12345, 7, keys[5:9]), u[5:9])          # no dependence on the other rows
    # a scalar re-implementation with Python integers
    def fm(x):
        x ^= x >> 33; x = (x * 0xFF51AFD7ED558CCD) & MASK64; x ^= x >> 33; x = (x * 0xC4CEB9FE1A85EC53) & MASK64
        return x ^ (x >> 33)
    for key in (-3, 0, 41, 2 ** 40):
        x = fm((fm((12345 + PHI * 8) & MASK64) + PHI * ((key + 1) & MASK64)) & MASK64)
        assert uniform(12345, 7, [key])[0] == (x >> 11) * 2.0 ** -53


def test_emulated_draw_edge_rows_and_shard_independence():
    vals = np.array([[[3.0, 1.0, -np.inf], [2.0, 2.0, 2.0], [-np.inf] * 3, [np.nan, 1.0, 0.5]]], dtype=np.float32)
    items = np.array([[[7, 9, -1], [4, 2, 8], [-1, -1, -1], [-2, 5, 6]]], dtype=np.int64)
    pick = emulate_sample(vals, items, 1, 0, np.arange(4))
    assert pick[0] in (7, 9) and pick[1] in (2, 4, 8) and pick[2] == -1 and pick[3] == -2
    # k = 1: the draw is the best candidate
    assert emulate_sample(vals[:, :, :1], items[:, :, :1], 5, 3, np.arange(4))[:2].tolist() == [7, 4]
    # the same list split over three shards (shuffled inside each) draws the same items
    rng = np.random.default_rng(0)
    M, k = 4000, 5
    v = rng.standard_normal((M, 3 * k)).astype(np.float32)
    it = np.stack([rng.permutation(10_000)[: 3 * k] + 1 for _ in range(M)])
    v[:, 1] = v[:, 0]                                                          # exact ties: the lower id goes first
    one = emulate_sample(*[a[None, :, :] for a in _best_k(v, it, k)], 99, 2, np.arange(M))
    shards = np.stack([v[:, g * k:(g + 1) * k] for g in range(3)]), np.stack([it[:, g * k:(g + 1) * k] for g in range(3)])
    perm = rng.permutation(k)
    three = emulate_sample(shards[0][:, :, perm], shards[1][:, :, perm], 99, 2, np.arange(M))
    np.testing.assert_array_equal(one, three)
    # the draws follow the softmax of the survivors (coarse check; the GPU test has the chi-square)
    vv = np.tile(np.array([[[2.0, 1.0, 0.0]]], dtype=np.float32), (1, 60_000, 1))
    ii = np.tile(np.array([[[1, 2, 3]]]), (1, 60_000, 1))
    freq = np.bincount(emulate_sample(vv, ii, 3, 0, np.arange(60_000)), minlength=4)[1:] / 60_000
    np.testing.assert_allclose(freq, np.exp([2.0, 1.0, 0.0]) / np.exp([2.0, 1.0, 0.0]).sum(), atol=0.01)


def _best_k(v, it, k):
    order = np.lexsort((it, -v), axis=1)[:, :k]
    return np.take_along_axis(v, order, 1), np.take_along_axis(it, order, 1)


def test_null_arguments_are_rejected_without_a_gpu():
    from influentialrs_b200.build import build
    build()
    from influentialrs_b200._lib import lib
    l = lib()
    E_BADARG = -1
    assert l.irs_topk_sample(None, None, 1, 4, 3, 0, 0, None, None, None) == E_BADARG
    # non-null but never dereferenced: the shape checks come before any launch
    p = 16
    assert l.irs_topk_sample(p, p, 1, 4, 3, 0, 0, None, p, None) == E_BADARG
    assert l.irs_topk_sample(p, p, 1, 4, 3, 0, 0, p, None, None) == E_BADARG
    assert l.irs_topk_sample(p, p, 0, 4, 3, 0, 0, p, p, None) == E_BADARG
    assert l.irs_topk_sample(p, p, 1, 4, 0, 0, 0, p, p, None) == E_BADARG
    assert l.irs_topk_sample(p, p, 5, 4, 1000, 0, 0, p, p, None) == l.irs_topk_sample(p, p, 1, 4, 4097, 0, 0, p, p, None)
    assert b"shape" in l.irs_error_string(l.irs_topk_sample(p, p, 1, 4, 4097, 0, 0, p, p, None)).lower()


# ---- sampled sharded generation over gloo --------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


N, L, H, P, TILE = 997, 12, 2, 4, 4
N_LOC = [7, 3]                         # tiles of 4 users: rank 0 -> 4 + 3, rank 1 -> 3 + 0 (empty in the last tile)


def _problem():
    sd = O.synth_irn_state(N, 20, L, 32, 2, 64, seed=13)
    sd["project.weight"][500] = sd["project.weight"][10]          # exact tie straddling the shard boundary (ids 11, 501)
    sd["project.bias"][500] = sd["project.bias"][10] = 2.0        # ... and high enough to sit in most rows' top k
    g = torch.Generator().manual_seed(6)
    B = sum(N_LOC)
    seqs = torch.zeros((B, L), dtype=torch.long)
    for b in range(B):
        n = L if b % 2 == 0 else int(torch.randint(3, L + 1, (1,), generator=g))
        seqs[b, L - n:] = torch.randperm(N, generator=g)[:n] + 1
    users = torch.randint(0, 20, (B,), generator=g)
    return sd, seqs, users


def _decode(sd, win, us):
    """Decoder row L-2, one window at a time: the same bits whatever batch a row is decoded in."""
    rows = [O.irn_decoding(sd, win[b:b + 1], us[b:b + 1], H, fold_cross=True)[0][:, L - 2] for b in range(win.shape[0])]
    h = torch.cat(rows) if rows else torch.zeros((0, sd["project.weight"].shape[1]))
    return torch.nan_to_num(h)                                      # an all-PAD pad window decodes to NaN; it is dropped


def _scores(h, W, b):
    """fp64 scores, each an independent sum over d: identical rows of W give identical scores in any shard."""
    return (h.double()[:, None, :] * W.double()[None]).sum(-1) + b.double()


def _replay(sd, seqs, users, k, seed):
    """Single-process sampled generation over the whole batch: full-catalog top-k, emulated draw with key = row index."""
    temp = seqs.clone()
    B = temp.shape[0]
    paths = torch.zeros((B, P))
    for i in range(P):
        s = _scores(_decode(sd, temp, users), sd["project.weight"], sd["project.bias"])
        vals, items = O.topk_excluding(s, temp[:, : L - 1], k)
        nxt = sample_fn_emulated(vals.float().unsqueeze(0), items.unsqueeze(0), seed, i, torch.arange(B))
        paths[:, i] = nxt.float()
        temp = torch.cat([temp[:, 1:L - 1], nxt.unsqueeze(1), temp[:, L - 1:]], dim=1)
    return paths.numpy()


def _sample_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from influentialrs_b200.dist import ShardedGenerator, trim_paths
        torch.set_num_threads(1)
        sd, seqs, users = _problem()
        mine = slice(sum(N_LOC[:rank]), sum(N_LOC[:rank + 1]))
        stub = SimpleNamespace(n_item=N, user_tile=TILE, net=SimpleNamespace(project=SimpleNamespace(
            weight=sd["project.weight"], bias=sd["project.bias"])))

        def merge(vals, items):                                     # not used when sampling
            raise AssertionError("merge_fn called on the sampled path")

        def shift(win_all, nxt, paths, step, row0, n):
            win_all[:, :-2] = win_all[:, 1:-1].clone()
            win_all[:, -2] = nxt
            paths[:, step] = nxt[row0:row0 + n].float()

        sg = ShardedGenerator(stub, rank, world, decode_fn=lambda w, u: _decode(sd, w, u), merge_fn=merge,
                              shift_fn=shift, sample_fn=sample_fn_emulated)

        def score(h_all, win_all, k):
            vals, items = O.topk_excluding(_scores(h_all, sg.W, sg.b), win_all[:, :-1], k, item_base=sg.lo + 1)
            return vals.float(), items

        sg.score_fn = score
        res = []
        for k in (3, 20):
            torch.manual_seed(100 + k + 7 * rank)                   # rank 1's generator differs: rank 0's seed must win
            paths, tg, hist, ne = sg.get_seq_in_batch(seqs[mine], users[mine], seqs[mine, -1], max_path_len=P,
                                                      sample=True, sample_k=k)
            torch.manual_seed(100 + k)
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            full = _replay(sd, seqs, users, k, seed)
            want, _, whist, wne = trim_paths(full.copy(), seqs[:, -1].numpy(), seqs[:, :-1].numpy())
            assert paths.shape == (N_LOC[rank], P)
            np.testing.assert_array_equal(paths, want[mine])
            assert [len(x) for x in hist] == [len(x) for x in whist[mine]]
            greedy = _replay(sd, seqs, users, 1, seed)
            res.append(int((full != greedy).any(1).sum()))          # the draw is not the arg-max everywhere
        with pytest.raises(NotImplementedError):
            sg.get_seq_in_batch(seqs[mine], users[mine], seqs[mine, -1], max_path_len=P, gap_len=2, sample=True)
        out.put((rank, "ok", res))
    except Exception:  # pragma: no cover
        import traceback
        out.put((rank, "fail", traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_sharded_sampled_generation_equals_single_process_replay():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sample_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in res:
        assert status == "ok", f"rank {rank}: {info}"
    assert all(n > 0 for _, _, info in res for n in info)
