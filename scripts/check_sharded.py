#!/usr/bin/env python
"""Multi-GPU parity on real GPUs: catalog-sharded, user-data-parallel generation (ShardedGenerator over NCCL) must
produce exactly the paths the single-GPU path (IRSNN.get_seq_in_batch, full catalog) produces for the same users -- greedy,
and sampled (sample=True) under one torch seed -- and the
catalog-sharded rank / log-sum-exp / selected logits / top-k (ShardedScorer) must equal the single-GPU operators -- ranks
and top-k ids as the same integers, with ragged per-rank row counts.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 scripts/check_sharded.py

With --backend gloo the collectives run over gloo and ranks may share GPUs (rank r uses GPU r mod the device count): the
same kernels and host logic at any world size on fewer GPUs.  That checks the results, not NCCL and not the speed.
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from types import SimpleNamespace
import influentialrs_b200 as pkg
from influentialrs_b200.dist import ShardedGenerator, ShardedScorer

world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
backend = sys.argv[sys.argv.index("--backend") + 1] if "--backend" in sys.argv else "nccl"
dev = torch.device("cuda", local % torch.cuda.device_count() if backend == "gloo" else local)
torch.cuda.set_device(dev)
timeout = __import__("datetime").timedelta(seconds=180)
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev, timeout=timeout)
else:
    dist.init_process_group(backend, timeout=timeout)
where = f"{world} GPUs" if backend == "nccl" else f"{world} ranks over {backend} on {torch.cuda.device_count()} GPU(s)"
cfg = SimpleNamespace(n_item=300_007, n_user=1000, max_len=201, n_layers=3, n_heads=4, emb_dim=128, u_emb_dim=10, ffn_dim=256,
                      dropout=0.0, lr1=1e-3)
torch.manual_seed(1234)                                   # same weights on every rank
net = pkg.InfluentialNet(cfg).to(dev).eval()
irn = pkg.IRSNN(cfg, net, dev)
B, P, L = 96, 6, cfg.max_len
g = torch.Generator().manual_seed(99)                     # the same global batch on every rank
seqs = torch.zeros((world * B, L), dtype=torch.long)
for b in range(world * B):
    n = L if b % 3 == 0 else int(torch.randint(30, L + 1, (1,), generator=g))
    seqs[b, L - n:] = torch.randperm(cfg.n_item, generator=g)[:n] + 1
users = torch.randint(0, cfg.n_user, (world * B,), generator=g)
mine = slice(rank * B, (rank + 1) * B)
sg = ShardedGenerator(irn, rank, world)
got, _, _, _ = sg.get_seq_in_batch(seqs[mine].to(dev), users[mine].to(dev), seqs[mine, -1].to(dev), max_path_len=P)
want, _, _, _ = irn.get_seq_in_batch(seqs[mine].to(dev), users[mine].to(dev), seqs[mine, -1].to(dev), max_path_len=P, gap_len=0)
same = torch.tensor([int(np.array_equal(np.asarray(got), np.asarray(want)))], device=dev)
n_diff = torch.tensor([int((np.asarray(got) != np.asarray(want)).any(1).sum())], device=dev)
dist.all_reduce(same, op=dist.ReduceOp.MIN); dist.all_reduce(n_diff)
if rank == 0:
    print(f"sharded ({where}) vs single-GPU paths: {'IDENTICAL' if int(same) else 'DIFFERENT'} "
          f"({world * B} users x {P} steps, rows that differ: {int(n_diff)})")
# ---- sampled paths: under one torch seed, each rank's rows equal the single-GPU sampled paths of the WHOLE global batch
# (the draw keys on the global row), with ragged ranks and user tiles that cut the batches differently on every rank
sizes = [40 + 13 * r for r in range(world)]
r0 = sum(sizes[:rank])
mine_s = slice(r0, r0 + sizes[rank])
seqs_s = seqs[torch.arange(sum(sizes)) % seqs.shape[0]].clone()
users_s = users[torch.arange(sum(sizes)) % users.shape[0]].clone()
irn.user_tile = 32
same_s, diff_s = 1, 0
for ks in (3, 20):
    torch.manual_seed(500 + ks)
    got_s, _, _, _ = sg.get_seq_in_batch(seqs_s[mine_s].to(dev), users_s[mine_s].to(dev), seqs_s[mine_s, -1].to(dev),
                                         max_path_len=P, sample=True, sample_k=ks)
    torch.manual_seed(500 + ks)
    want_s, _, _, _ = irn.get_seq_in_batch(seqs_s.to(dev), users_s.to(dev), seqs_s[:, -1].to(dev), max_path_len=P,
                                           gap_len=0, sample=True, sample_k=ks)
    same_s &= int(np.array_equal(np.asarray(got_s), np.asarray(want_s)[mine_s]))
    diff_s += int((np.asarray(got_s) != np.asarray(want_s)[mine_s]).any(1).sum())
irn.user_tile = 4096
t_same, t_diff = torch.tensor([same_s], device=dev), torch.tensor([diff_s], device=dev)
dist.all_reduce(t_same, op=dist.ReduceOp.MIN); dist.all_reduce(t_diff)
same_s, diff_s = int(t_same), int(t_diff)
if rank == 0:
    print(f"sharded ({where}) vs single-GPU SAMPLED paths (sample_k 3 and 20, one torch seed): "
          f"{'IDENTICAL' if same_s else 'DIFFERENT'} ({sum(sizes)} users, ranks bring {sizes}, {P} steps, "
          f"rows that differ: {diff_s})")
# ---- ShardedScorer: rank / lse + logits / top-k over the sharded catalog vs the single-GPU operators
ops = pkg.ops
W, beta = net.project.weight.detach(), net.project.bias.detach()
sc = ShardedScorer(W, beta, rank, world)
n_rows = 64 + 7 * rank                                    # ragged: every rank brings a different number of rows
gg = torch.Generator().manual_seed(7 + rank)
h = torch.randn((n_rows, cfg.emb_dim), generator=gg).to(dev)
ids = torch.randint(1, cfg.n_item + 1, (n_rows, 40), generator=gg).to(dev)
label = torch.randint(1, cfg.n_item + 1, (n_rows,), generator=gg).to(dev)
label[0] = ids[0, 0]                                      # excluded label -> rank 0
sel = torch.randint(0, cfg.n_item + 1, (n_rows, 2), generator=gg).to(dev)
sel[1, 0] = 0
r_sh = sc.rank(h, label, ids)
r_1 = ops.score_rank(h, W, beta, label, ops.sort_exclusions(ids, cfg.n_item, 1), 1)
lse_sh, lg_sh = sc.lse_gather(h, sel)
lse_1, lg_1 = ops.score_lse_gather(h, W, beta, sel, 1)
v_sh, i_sh = sc.topk(h, 20, ids)
v_1, i_1 = ops.score_topk(h, W, beta, 20, ops.sort_exclusions(ids, cfg.n_item, 1), 1)
ok = torch.tensor([int(torch.equal(r_sh, r_1) and int(r_sh[0]) == 0 and torch.equal(i_sh, i_1) and torch.equal(v_sh, v_1)
                       and float((lg_sh - lg_1).abs().max()) < 1e-5 and float((lse_sh - lse_1).abs().max()) < 1e-4)], device=dev)
dist.all_reduce(ok, op=dist.ReduceOp.MIN)
if rank == 0:
    print(f"sharded scorer ({where}) vs single-GPU rank / lse / logits / top-20: {'IDENTICAL' if int(ok) else 'DIFFERENT'} "
          f"(ragged rows per rank, N={cfg.n_item})")
dist.destroy_process_group()
sys.exit(0 if int(same) and int(ok) and same_s else 1)
