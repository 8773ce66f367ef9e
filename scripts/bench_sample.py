#!/usr/bin/env python
"""Sampled vs greedy influence-path generation at cfg3 (1M items, L = 201, d = 128, 6 layers, 4096 users per GPU), on one
GPU or catalog-sharded over several (torchrun).

Sampled steps (get_seq_in_batch(sample=True, sample_k=3), the reference default: tensor-core top-k pass 1 + select ->
irs_topk_sample) and greedy steps (tensor-core arg-max) alternate in blocks inside one process, on two independent sets
of windows, so that both see the same clocks and neighbours.  Reports ms per step and user-steps/s for both, CUDA-event
times of the top-k call, the sampler and the arg-max scorer inside the timed blocks, and -- from a separate, shorter
torch.profiler run -- the time of every kernel class per step (top-k pass 1 and select apart).

    python scripts/bench_sample.py [--users 4096] [--rounds 6] [--block 5] [--k 3]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29541 scripts/bench_sample.py
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402  (Dist, CFG3, build_irn, synth_batch)

KERNEL_CLASSES = [                       # (class, substring of the kernel name), first match wins
    ("topk_pass1", "score_tc_kernel<3>"),
    ("topk_select", "topk_select_kernel"),
    ("sampler", "topk_sample_kernel"),
    ("argmax", "score_tc_kernel<"),
    ("argmax", "rescore_finalize_kernel"),
    ("argmax", "approx_leader_kernel"),
    ("merge", "topk_merge_kernel"),
    ("exclusions", "exclusions_"),
    ("window_shift", "window_shift_kernel"),
]


def gpu_info(index):
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                       "-i", str(index)], text=True, timeout=20).strip()
    except Exception as e:            # the numbers are still printed; the card's name comes from torch
        out = f"{torch.cuda.get_device_name(index)}, power limit unknown ({e.__class__.__name__})"
    return out


def classify(name):
    for cls, sub in KERNEL_CLASSES:
        if sub in name:
            return cls
    return "other"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--users", type=int, default=4096, help="users per GPU")
    ap.add_argument("--k", type=int, default=3, help="sample_k")
    ap.add_argument("--rounds", type=int, default=6, help="timed (sampled block, greedy block) pairs")
    ap.add_argument("--block", type=int, default=5, help="steps per timed block")
    ap.add_argument("--warmup", type=int, default=2, help="untimed blocks of each kind")
    ap.add_argument("--profile-steps", type=int, default=3, help="steps of each kind under torch.profiler (0: skip)")
    ap.add_argument("--small", action="store_true", help="20k-item catalog, 2 layers (a quick run, not cfg3)")
    args = ap.parse_args()

    D = bench.Dist()
    cfg = dict(bench.SMALL if args.small else bench.CFG3)
    B, k = args.users, args.k
    pkg, c, net, irn = bench.build_irn(cfg, D.device)
    ops = pkg.ops
    gen = torch.Generator(device=D.device).manual_seed(1234 + D.rank)
    seqs, users = bench.synth_batch(B, cfg, gen, D.device)
    n_steps = (args.warmup + args.rounds) * args.block + args.profile_steps
    seed = 20261020
    state = {}
    for mode in ("sample", "greedy"):
        state[mode] = dict(temp=seqs.clone(), paths=torch.zeros((B, n_steps), dtype=torch.float32, device=D.device),
                           excl=None, i=0)
    if D.world > 1:
        from influentialrs_b200.dist import ShardedGenerator
        for mode in state:
            state[mode]["sg"] = ShardedGenerator(irn, D.rank, D.world)
        keys_all = torch.arange(D.world * B, dtype=torch.int64, device=D.device)
    else:
        keys = torch.arange(B, dtype=torch.int64, device=D.device)

    def one_step(mode):
        st = state[mode]
        i = st["i"]
        with torch.no_grad():
            if D.world > 1:
                st["sg"].step(st["temp"], users, st["paths"], i, (k, seed, keys_all) if mode == "sample" else None)
            elif mode == "sample":
                st["excl"] = irn.path_step(st["temp"], users, st["paths"], i, st["excl"], True, k, seed=seed, row_key=keys)
            else:
                st["excl"] = irn.path_step(st["temp"], users, st["paths"], i, st["excl"])
        st["i"] = i + 1

    def block(mode, timed):
        torch.cuda.synchronize()
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.block):
            one_step(mode)
        e1.record()
        torch.cuda.synchronize()
        return D.max(e0.elapsed_time(e1)) / args.block if timed else None

    for _ in range(args.warmup):
        for mode in ("sample", "greedy"):
            block(mode, False)
    ms = {"sample": [], "greedy": []}
    ev = {"sample": {}, "greedy": {}}
    for r in range(args.rounds):
        order = ("sample", "greedy") if r % 2 == 0 else ("greedy", "sample")
        for mode in order:
            ops._timer = {}
            ms[mode].append(block(mode, True))
            timer, ops._timer = ops._timer, None
            for name, recs in timer.items():
                t = sum(sum(x[j].elapsed_time(x[j + 1]) for j in range(0, len(x), 2)) for x in recs)
                ev[mode].setdefault(name, []).append(t / args.block)

    prof = {}
    if args.profile_steps > 0:
        from torch.profiler import ProfilerActivity, profile
        for mode in ("sample", "greedy"):
            torch.cuda.synchronize()
            D.barrier()
            with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as p:
                for _ in range(args.profile_steps):
                    one_step(mode)
                torch.cuda.synchronize()
            per = {}
            for e in p.key_averages():
                t = getattr(e, "device_time_total", 0.0)
                if "CUDA" in str(getattr(e, "device_type", "")) and t > 0:
                    per[classify(e.key)] = per.get(classify(e.key), 0.0) + t / 1e3 / args.profile_steps
            prof[mode] = {n: round(v, 4) for n, v in sorted(per.items(), key=lambda kv: -kv[1])}
            D.barrier()

    # every sampled pick is a catalog item (no -1 / -2 row)
    ok = bool((state["sample"]["paths"][:, :state["sample"]["i"]] >= 1).all())
    ok = D.all_true(ok)
    info = gpu_info(D.local)
    if D.rank == 0:
        med = {m: statistics.median(v) for m, v in ms.items()}
        res = {
            "metric": "sampled vs greedy IRN generation step (cfg3)" if not args.small else "sampled vs greedy (small)",
            "gpu": info, "gpus": D.world, "users_per_gpu": B, "sample_k": k, "n_item": cfg["n_item"],
            "steps_timed_per_mode": args.rounds * args.block,
            "ms_per_step": {m: round(v, 4) for m, v in med.items()},
            "ms_per_step_all_blocks": {m: [round(x, 4) for x in v] for m, v in ms.items()},
            "user_steps_per_s": {m: round(B * D.world / (v / 1e3), 1) for m, v in med.items()},
            "sampled_minus_greedy_ms": round(med["sample"] - med["greedy"], 4),
            "event_ms_per_step_rank0": {m: {n: round(statistics.median(v), 4) for n, v in d.items()} for m, d in ev.items()},
            "profiler_ms_per_step_rank0": prof,
            "picks_valid": ok,
        }
        print(f"# {info}; {D.world} GPU(s), {B} users per GPU, sample_k={k}, N={cfg['n_item']}")
        for m in ("greedy", "sample"):
            print(f"#   {m:6s}: {med[m]:.3f} ms/step  {res['user_steps_per_s'][m]:.0f} user-steps/s  "
                  f"events {res['event_ms_per_step_rank0'][m]}  profiler {prof.get(m)}")
        print(json.dumps(res))
    D.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
