#!/usr/bin/env python
"""bench.py -- the IRN hot path on B200, in BASELINE.json's metric and configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|torch_gpu]
                    [--config cfg3|cfg1|cfg2|cfg4|cfg5|k2] [--variant uniform|zipf|ragged] [--users B]
                    [--dump-outputs DIR]

Default = cfg3, the configuration the headline metric is quoted on (SURVEY.md section 8d): IRN influence-path
generation, synthetic 1M-item catalog, history 200 => window L=201, d=128, 6 layers / 4 heads / ffn 256, reference
default initialisers under torch.manual_seed(1234); users in device tiles of B (default 4096) per GPU.  A *step* is one
pass of the hot path over one tile: PIF + gather+PE -> 6 PIM decoder layers (row L-2 only in the last) -> fused catalog
scoring + window mask + arg-max -> window shift, i.e. B user-steps.  value = user-steps/s over all GPUs.

N>1 (torchrun): users are split data-parallel AND the catalog is row-sharded: every step all-gathers the decoded rows,
each rank scores its catalog shard for all users, candidates are all-gathered and merged.  Per-GPU work is constant as
N grows => "scaling": "weak".

Other configurations of BASELINE.json, same JSON schema (one line on stdout, rank 0):
  cfg1  IRN generation on the shipped MovieLens-1M histories (6040 users, 3415 items, L=50, d=64), all users
  cfg2  SASRec full-catalog next-item top-50 with history filter, ml-1m shape, batch 1024
  cfg4  IRN train_batch incl. Adam (gather + PIM attention fwd/bwd + full-softmax CE + scatter-add), N=500k, batch
        4096 per GPU, data-parallel at N>1
  cfg5  Evaluator measurements of generated paths (SampleNet) + Caser catalog scoring, N=1M, batch 8192
  k2    embedding gather / scatter-add (K1/K2) in GB/s with uniform and Zipf ids

The line carries `roofline` (dominant kernel, timed with CUDA events inside the timed region), `e2e` (same metric
through the public drop-in API with pinned HOST buffers, copies inside), `parity` (GPU results against the reference's
own CPU run of the same inputs), `cpu_baseline` (the reference's own implementation on the host cores, bounded sample;
N=1 only) and `gpu_library_baseline` (the reference's own code on the same B200 through stock torch; cfg3, N=1).

--impl reference   the UNMODIFIED reference (oracle/_ref staged by __graft_entry__.build(), shims D1-D3 only) on the
                   host cores; falls back to the oracle port when the staged tree is absent.
--impl torch_gpu   the same reference code with device='cuda' (cuBLAS/ATen, TF32 off) at the largest batch that fits.

--dump-outputs DIR after the timed steps, writes what the timed path computed in its last step as DIR/<name>.npy.  The
                   inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

KERNEL_NAMES = {
    "attention": "pim_attn_persistent_kernel (tcgen05 PIM attention from operand images)",
    "decoder_chain": "decoder_chain_kernel (fused out_proj+LN1+LN2 -> FFN+LN3 -> next in_proj, tcgen05)",
    "scorer": "score_tc_kernel<0> + rescore_finalize_kernel (fused catalog scorer: one bf16 tcgen05 MMA per K step, rigorous "
              "rounding-error band, exact fp32 re-score of the candidates)",
    "gather": "embed_gather_v4_kernel (item embedding gather + sqrt(d) + PE)",
    "scatter_add": "embed_scatter_add_kernel (warp-aggregated scatter-add into the embedding table)",
    "ce_fwd": "score_tc_kernel<1> + lse_finalize_kernel (tcgen05 log-sum-exp over the catalog + exact target logit)",
    "ce_bwd": "ce_bwd_tc_kernel x2 (tcgen05 softmax-CE backward: d_h pass and d_W/d_bias pass, logits recomputed)",
    "attention_train": "pim_attn_fwd_kernel / pim_attn_bwd_kernel (fp32 PIM attention forward with lse + backward)",
    "rank": "score_tc_kernel<2> + rank_finalize_tc_kernel (tcgen05 rank by counting)",
    "lse": "score_tc_kernel<1> + lse_finalize_kernel (tcgen05 log-sum-exp + selected logits)",
    "topk": "fused catalog top-k scorer (score + history mask + top-k, logits never in HBM)",
}

CFG3 = dict(n_item=1_000_000, n_user=100_000, max_len=201, n_layers=6, n_heads=4, emb_dim=128, u_emb_dim=10,
            ffn_dim=256, dropout=0.0, lr1=1e-3)
SMALL = dict(n_item=20_000, n_user=1_000, max_len=201, n_layers=2, n_heads=4, emb_dim=128, u_emb_dim=10,
             ffn_dim=256, dropout=0.0, lr1=1e-3)


# ----------------------------------------------------------------------------------------------------------------------
# shared plumbing
# ----------------------------------------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, source="fallback")


def traffic_table():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each kernel class, parsed at run time from the committed
    ncu summaries that profiles/traffic.json names (written by scripts/ncu_traffic.py from `ncu --set full` captures)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        return json.load(f)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class Dist:
    """torch.distributed plumbing of one bench process (one process per GPU)."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device: influentialrs_b200 has no CPU path")
        torch.cuda.set_device(self.local)
        self.device = torch.device("cuda", self.local)
        if self.world > 1:
            import datetime
            import torch.distributed as dist
            # a rank that dies must not keep the others (and the GPU box) waiting for NCCL's default 10 minutes
            dist.init_process_group("nccl", device_id=self.device, timeout=datetime.timedelta(seconds=180))

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()

    def max(self, x: float) -> float:
        if self.world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], device=self.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, ok: bool) -> bool:
        return self.max(0.0 if ok else 1.0) == 0.0

    def close(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


def timed_steps(D: Dist, ops, step, steps, warmup, flush=None):
    """W untimed steps, then EXACTLY K steps between barrier + synchronize on both sides, CUDA events on the launching
    stream, max over ranks; clocks sampled during the timed region; per-kernel-class events inside it."""
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    D.barrier()
    sampler = ClockSampler(D.local)
    if D.rank == 0:
        sampler.start()
    ops.launch_count_reset()
    ops._timer = {}
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for i in range(steps):
        step(warmup + i)
    t1.record()
    torch.cuda.synchronize()
    D.barrier()
    ms = t0.elapsed_time(t1)
    launches = ops.launch_count()
    clocks = sampler.stop() if D.rank == 0 else None
    timer, ops._timer = ops._timer, None
    # (ms/launch, launches/step); a record is one or more (start, stop) event pairs (the two-phase sharded scorer has two)
    kms = {k: (sum(sum(x[i].elapsed_time(x[i + 1]) for i in range(0, len(x), 2)) for x in v) / len(v), len(v) / steps)
           for k, v in timer.items()}
    return D.max(ms), launches, clocks, kms


DUMP_BYTES = 64_000_000


def dump_outputs(args, D, arrays):
    """--dump-outputs DIR: ``arrays`` (name -> tensor), what the timed path computed in its last step, as DIR/<name>.npy on
    rank 0 -- float32 and float64 as they are, integer ids as float64 (exact).  All files together stay under 64 MB: an
    array above its share is replaced by a fixed, seeded sample of its rows, whose ids go to DIR/<name>.rows.npy."""
    if not args.dump_outputs or D.rank != 0:
        return
    os.makedirs(args.dump_outputs, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = torch.as_tensor(t).detach()
        t = t.reshape(1) if t.dim() == 0 else t
        dtype = t.dtype if t.dtype in (torch.float32, torch.float64) else torch.float64
        row_bytes = t[0].numel() * dtype.itemsize
        if t.shape[0] * row_bytes > share:
            k = share // (row_bytes + 8)
            rows = np.sort(np.random.default_rng(1234).choice(t.shape[0], k, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
            np.save(os.path.join(args.dump_outputs, name + ".rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(args.dump_outputs, name + ".npy"), t.to(dtype).cpu().numpy())


def roofline_blocks(alg, kms, step_ms, workload="cfg3"):
    """alg: kernel class -> (bound, algorithmic work per launch, note).  Returns (dominant block, all blocks).  ``traffic``
    is reported only when the committed ncu capture was taken on this workload (the bytes of a launch depend on the shape)."""
    pk = peaks()
    tr = {k: v for k, v in traffic_table().items() if v.get("workload", "cfg3") == workload}
    kernels = {}
    for name, (bound, work, note) in alg.items():
        if name not in kms:
            continue
        ms_l, per_step = kms[name]
        peak = pk["tf_sus"] if bound == "tensor" else pk["hbm"]
        ach = work / (ms_l / 1e3) / (1e12 if bound == "tensor" else 1e9)
        t = tr.get(name) or {}
        kernels[name] = {"bound": bound, "achieved": ach, "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                         "frac": ach / peak, "traffic": t.get("bytes_per_launch"), "traffic_source": t.get("source"),
                         "ms_per_launch": ms_l, "launches_per_step": per_step, "share_of_step": ms_l * per_step / step_ms,
                         "algorithmic": note}
    if not kernels:
        return None, {}
    dom = max(kernels, key=lambda k: kernels[k]["share_of_step"])
    roof = dict(kernels[dom], kernel=KERNEL_NAMES.get(dom, dom),
                peak_source=pk["source"] + (" bf16 sustained" if kernels[dom]["bound"] == "tensor" else " HBM copy")
                + " (kernel timed inside the step)")
    return roof, {KERNEL_NAMES.get(k, k): v for k, v in kernels.items()}


def base_line(metric, unit, value, D, args, step_ms, dtype, data, config, scaling="weak"):
    return {"metric": metric, "value": value, "unit": unit, "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": dtype,
            "data": data, "config": config}


def load_ref():
    """The reference's own classes (oracle/_ref staged copy or /root/reference), or None."""
    from oracle.ref_shim import load_reference
    try:
        return load_reference()
    except Exception as e:                                       # pragma: no cover - diagnostic only
        sys.stderr.write(f"bench.py: reference import failed: {e!r}\n")
        return None


# ----------------------------------------------------------------------------------------------------------------------
# cfg3 (headline): IRN influence-path generation at 1M items
# ----------------------------------------------------------------------------------------------------------------------
def synth_batch(B, cfg, gen, device, variant="uniform"):
    """Windows [B,L]: L-1 history ids + the objective item in the last column (SURVEY 8d cfg3).
       uniform: distinct ids, uniform over the catalog (worst-case locality);
       zipf   : ids ~ Zipf(alpha=1) over the catalog (popular items repeat across users; duplicates inside a window allowed);
       ragged : uniform ids, history lengths U[20, L-1], pre-padded with 0."""
    L, N = cfg["max_len"], cfg["n_item"]
    if variant == "zipf":
        u = torch.rand((B, L), generator=gen, device=device, dtype=torch.float64)
        seqs = torch.exp(u * math.log(N)).floor().clamp(1, N).long()           # P(id) ~ 1/id
    else:
        stride = N // L
        base = torch.arange(L, device=device).unsqueeze(0) * stride
        off = torch.randint(0, stride, (B, L), generator=gen, device=device)
        ids = base + off + 1                                                    # distinct by construction
        perm = torch.rand((B, L), generator=gen, device=device).argsort(1)
        seqs = ids.gather(1, perm).contiguous()
    if variant == "ragged":
        n = torch.randint(20, L, (B,), generator=gen, device=device)            # history length
        col = torch.arange(L, device=device).unsqueeze(0)
        seqs = torch.where((col >= (L - 1 - n).unsqueeze(1)), seqs, torch.zeros_like(seqs))
    users = torch.randint(0, cfg["n_user"], (B,), generator=gen, device=device)
    return seqs.contiguous(), users


def build_irn(cfg, device, train=False):
    from types import SimpleNamespace
    import influentialrs_b200 as pkg
    torch.manual_seed(1234)
    c = SimpleNamespace(**cfg)
    net = pkg.InfluentialNet(c)
    net.to(device)
    if not train:
        net.eval()
    return pkg, c, net, pkg.IRSNN(c, net, device)


def reference_generate_cpu(cfg, state, seqs, users, steps, threads):
    """The reference's own IRSNN.get_seq_in_batch on the host cores (shims D1-D3 only), or its oracle port when the staged
    reference tree is absent.  Returns (paths np [B,steps], seconds, kind)."""
    from types import SimpleNamespace
    torch.set_num_threads(threads)
    R = load_ref()
    seqs, users = seqs.cpu(), users.cpu()
    if R is not None:
        net = R.IntendedNet(SimpleNamespace(**cfg))
        net.load_state_dict(state)
        net.eval()
        irn = R.IRSNN(SimpleNamespace(**cfg), net, torch.device("cpu"))
        t0 = time.perf_counter()
        with torch.no_grad():
            p, _, _, _ = irn.get_seq_in_batch(seqs.clone(), users, seqs[:, -1].clone(), max_path_len=steps, gap_len=0)
        return p, time.perf_counter() - t0, "reference"
    from oracle import irn_oracle as O       # bench.py's cpu_baseline / --impl reference legs only
    t0 = time.perf_counter()
    with torch.no_grad():
        p, _, _ = O.generate_paths_faithful(state, seqs, users, seqs[:, -1], cfg["n_heads"], max_path_len=steps)
    return p, time.perf_counter() - t0, "port"


def compare_paths(gpu_paths, ref_paths, targets, margins=None):
    """Picks compared position by position up to (and including) each user's first hit of its target (the reference zeroes
    the path after it, get_seq_in_batch :452-470)."""
    B, P = ref_paths.shape
    n_cmp = n_eq = 0
    bad = []
    for b in range(B):
        for i in range(P):
            n_cmp += 1
            if int(gpu_paths[b, i]) == int(ref_paths[b, i]):
                n_eq += 1
            else:
                bad.append((b, i, int(gpu_paths[b, i]), int(ref_paths[b, i])))
                break
            if int(ref_paths[b, i]) == int(targets[b]):
                break
    out = {"users": B, "steps": P, "decisions": n_cmp, "decisions_equal": n_eq, "equal": n_cmp == n_eq}
    if bad:
        out["first_mismatches"] = bad[:4]
    if margins is not None:
        out["min_margin"] = float(margins.min())
    return out


def cfg3_cpu_legs(cfg, state, seqs, users, gpu_paths, want_baseline, threads):
    """`parity` (always) and `cpu_baseline` (N=1) from the SAME reference CPU runs: 4 users x 2 path steps per batch (the
    reference materialises [B,L,N] logits twice: 1.6 GB per user at cfg3)."""
    from oracle import irn_oracle as O       # checker: fp64-free margins of the decisions compared
    users_n, steps = (4, 2) if cfg["n_item"] >= 500_000 else (16, 2)
    p, dt, kind = reference_generate_cpu(cfg, state, seqs[:users_n], users[:users_n], steps, threads)
    with torch.no_grad():
        _, _, _, _, margins = O.generate_paths(state, seqs[:users_n].cpu(), users[:users_n].cpu(), seqs[:users_n, -1].cpu(),
                                               cfg["n_heads"], steps, return_margins=True, fold_cross=True)
    parity = compare_paths(gpu_paths[:users_n, :steps], p, seqs[:users_n, -1].cpu().numpy(), margins)
    parity["against"] = ("the reference's own IRSNN.get_seq_in_batch on CPU" if kind == "reference"
                         else "oracle.generate_paths_faithful (CPU port)") + ", same weights and windows"
    base = None
    if want_baseline:
        reps, tot = 1, dt
        while tot < 10.0 and reps < 12:
            off = reps * users_n
            _, d2, _ = reference_generate_cpu(cfg, state, seqs[off:off + users_n], users[off:off + users_n], steps, threads)
            tot += d2
            reps += 1
        base = {"value": reps * users_n * steps / tot, "unit": "user-steps/s", "cores": threads, "kind": kind,
                "sample": f"{reps} batches of {users_n} users x {steps} path steps of the same workload (the reference "
                          f"materialises [B,L,N] logits + softmax + per-sample top-100 + window filter), torch CPU fp32, {tot:.1f} s"}
    return parity, base


def torch_gpu_reference(cfg, state, seqs, users, device, steps=2, batch=32):
    """The reference's own IRSNN.get_seq_in_batch with device='cuda' (cuBLAS / ATen, TF32 off): the "library Blackwell
    path" bar of SURVEY 8d, at the largest batch whose [B,L,N] logits (+ softmax copy) fit next to our own buffers."""
    from types import SimpleNamespace
    R = load_ref()
    if R is None:
        return {"unavailable": "reference tree not staged (oracle/_ref missing)"}
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    net = R.IntendedNet(SimpleNamespace(**cfg))
    net.load_state_dict(state)
    net.to(device).eval()
    irn = R.IRSNN(SimpleNamespace(**cfg), net, device)
    out = None
    while batch >= 1:
        try:
            s, u = seqs[:batch].to(device), users[:batch].to(device)
            with torch.no_grad():
                irn.get_seq_in_batch(s.clone(), u, s[:, -1].clone(), max_path_len=1, gap_len=0)      # warm-up
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                p, _, _, _ = irn.get_seq_in_batch(s.clone(), u, s[:, -1].clone(), max_path_len=steps, gap_len=0)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
            out = {"value": batch * steps / dt, "unit": "user-steps/s", "kind": "reference code on cuda (stock torch, TF32 off)",
                   "users": batch, "steps": steps, "seconds": dt, "paths": p}
            break
        except torch.OutOfMemoryError:
            batch //= 2
            torch.cuda.empty_cache()
    del net, irn
    torch.cuda.empty_cache()
    return out or {"unavailable": "out of memory at batch 1"}


def run_cfg3(args, D):
    cfg = dict(SMALL if args.small else CFG3)
    B = args.users or 4096
    device = D.device
    pkg, c, net, irn = build_irn(cfg, device)
    ops = pkg.ops
    stepper = None
    if D.world > 1:
        from influentialrs_b200.dist import ShardedGenerator
        stepper = ShardedGenerator(irn, D.rank, D.world)
    gen = torch.Generator(device=device).manual_seed(1234 + D.rank)
    seqs, users = synth_batch(B, cfg, gen, device, args.variant)
    L = cfg["max_len"]
    p = L - 2
    paths = torch.zeros((B, args.steps + args.warmup), dtype=torch.float32, device=device)
    temp = seqs.clone()
    st = {"excl": None}

    def step(i):
        with torch.no_grad():
            if stepper is not None:
                stepper.step(temp, users, paths, i)
                return
            st["excl"] = irn.path_step(temp, users, paths, i, st["excl"])      # the product's own step (IRSNN.generate_on_device)

    ms, launches, clocks, kms = timed_steps(D, ops, step, args.steps, args.warmup)
    if stepper is None:
        dump_outputs(args, D, {"paths": paths, "windows": temp, "exclusions": st["excl"][0], "exclusion_counts": st["excl"][1]})
    else:
        dump_outputs(args, D, {"paths": paths, "windows": temp})

    # ---- end to end through the public API with HOST buffers (H2D of the batch + D2H of the paths inside)
    P_e2e = args.e2e_path_len
    seqs_h = seqs.cpu().pin_memory()
    users_h = users.cpu().pin_memory()
    tg_h = seqs_h[:, -1].clone().pin_memory()

    def e2e_call():
        s = seqs_h.to(device, non_blocking=True)
        u = users_h.to(device, non_blocking=True)
        t = tg_h.to(device, non_blocking=True)
        if stepper is not None:
            return stepper.get_seq_in_batch(s, u, t, max_path_len=P_e2e)
        return irn.get_seq_in_batch(s, u, t, max_path_len=P_e2e, gap_len=0)
    for _ in range(args.e2e_warm):
        e2e_call()
    torch.cuda.synchronize()
    D.barrier()
    w0 = time.perf_counter()
    out = e2e_call()
    torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - w0)
    h2d = (seqs_h.numel() + users_h.numel() + tg_h.numel()) * 8
    d2h = out[0].size * 4
    # sharded picks must equal the single-GPU picks of the same users: every rank re-generates its first users unsharded
    shard_ok = None
    if stepper is not None:
        nchk = min(64, B)
        with torch.no_grad():
            solo = irn.generate_on_device(seqs[:nchk].contiguous(), users[:nchk].contiguous(), max_path_len=2)
        shard_ok = D.all_true(bool(torch.equal(solo, paths[:nchk, :2])))

    if D.rank != 0:
        if not args.no_parity:
            D.barrier()            # rank 0 runs the CPU parity sample
        return None
    value = B * D.world * args.steps / (ms / 1e3)
    step_ms = ms / args.steps
    d, n_layers = cfg["emb_dim"], cfg["n_layers"]
    n_shard = cfg["n_item"] // D.world
    # ALGORITHMIC work per launch (SURVEY.md section 8d / DESIGN.md section 4); B users per launch
    alg = {
        "attention": ("tensor", ((n_layers - 1) * 4.0 * L * L * d + 4.0 * L * d) / n_layers * B,
                      "4*L^2*d FLOP per user per full layer (QK^T + PV over the full window; the kernel issues 3x that in bf16 MMAs "
                      "minus the causally invisible key blocks), 4*L*d for the one-row last layer; average over the step's launches"),
        "decoder_chain": ("hbm", ((n_layers - 1) * 6.0 + 4.0) / n_layers * L * d * 4 * B,
                          "6*L*d*4 B per user per full launch (attn + x read, x' + q,k,v written, fp32-equivalent), 4*L*d*4 for the "
                          "first layer's in_proj-only launch; average over the step's launches"),
        "scorer": ("tensor", 2.0 * d * n_shard * (B * D.world), "2*d*N FLOP per user-step, issued once in bf16 (hi*hi); fp32-faithful "
                   "winners come from the rigorous error band + exact re-scoring (the three-MMA variant issues 3x this)"),
        "gather": ("hbm", float(L * (8 + 4 * d + 4 * d)) * B, "L*(8 + 4d + 4d) B per user-step: id + table row read + row written"),
    }
    roof, kernels = roofline_blocks(alg, kms, step_ms)
    line = base_line("IRN influence-path generation throughput @1M items" if not args.small else "IRN generation (small)",
                     "user-steps/s", value, D, args, step_ms, "f32", "synthetic",
                     {"workload": ("cfg3: IRN generation, 1M-item catalog, L=201 (history 200 + objective), d=128, 6 layers/4 heads/"
                                   "ffn 256") if not args.small else "small", "variant": args.variant, "users_per_gpu": B,
                      "n_item": cfg["n_item"], "catalog_shards": D.world, "l2_policy": "inputs > L2 (W 512 MB, E 512 MB)",
                      "weights": "reference default init, seed 1234"})
    line["e2e"] = {"value": B * D.world * P_e2e / e2e_s, "unit": "user-steps/s", "h2d_bytes_per_step": h2d / P_e2e,
                   "d2h_bytes_per_step": d2h / P_e2e, "path_len": P_e2e,
                   "api": "IRSNN.get_seq_in_batch" if stepper is None else "ShardedGenerator.get_seq_in_batch"}
    line["gpu_launches"] = int(launches)
    line["roofline"] = roof
    line["roofline_kernels"] = kernels
    line["clocks"] = clocks
    if not args.no_parity:
        state = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        threads = os.cpu_count() or 1
        parity, base = cfg3_cpu_legs(cfg, state, seqs.cpu(), users.cpu(), paths.cpu().numpy(),
                                     want_baseline=(D.world == 1 and not args.no_cpu_baseline), threads=threads)
        if shard_ok is not None:
            parity["sharded_equals_unsharded"] = shard_ok
            parity["sharded_check"] = "first 64 users x 2 steps of every rank, catalog-sharded picks vs the same rank's unsharded picks"
        line["parity"] = parity
        if base is not None:
            line["cpu_baseline"] = base
        if D.world == 1 and not args.no_gpu_baseline and not args.small:
            g = torch_gpu_reference(cfg, state, seqs.cpu(), users.cpu(), device, steps=2, batch=32)
            if "paths" in g:
                pg = g.pop("paths")
                g["paths_equal_ours"] = compare_paths(paths.cpu().numpy()[:pg.shape[0], :2], pg,
                                                      seqs[:pg.shape[0], -1].cpu().numpy())["equal"]
            line["gpu_library_baseline"] = g
        D.barrier()
    return line


# ----------------------------------------------------------------------------------------------------------------------
# cfg1: IRN generation on the shipped MovieLens-1M histories
# ----------------------------------------------------------------------------------------------------------------------
def ml1m_windows(L, gen):
    """Windows of every ml-1m user from the staged fixture (oracle/_ref/data/ml-1m/data_pack.npy: 6040 users, 3415 items);
    synthetic Zipf histories of the same shape when the fixture is absent.  Target = a uniform item not in the history."""
    from influentialrs_b200.data import to_csr, collate_eval_irs
    p = None
    for root in (os.path.join(ROOT, "oracle", "_ref"), "/root/reference"):
        q = os.path.join(root, "data", "ml-1m", "data_pack.npy")
        if os.path.exists(q):
            p = q
            break
    rng = np.random.default_rng(1234)
    if p is not None:
        pack = np.load(p, allow_pickle=True).item()
        hist, n_item, n_user, data = pack["data"], int(pack["item_count"]), int(pack["user_count"]), "MovieLens-1M histories (shipped data_pack.npy), random-init weights"
    else:
        n_item, n_user = 3415, 6040
        hist = [np.minimum(np.exp(rng.random(int(n)) * np.log(n_item)).astype(np.int64) + 1, n_item).tolist()
                for n in rng.integers(18, 400, n_user)]
        data = "synthetic Zipf histories of the ml-1m shape (fixture not staged), random-init weights"
    values, offsets = to_csr(hist)
    targets = rng.integers(1, n_item + 1, n_user)
    rows = np.arange(n_user)
    _, seqs, users, tg, _ = collate_eval_irs(values, offsets, rows, rows, targets, targets, L, 0, pin=False)
    return seqs, users, n_item, n_user, data


def run_cfg1(args, D):
    L = 50
    seqs_h, users_h, n_item, n_user, data = ml1m_windows(L, None)
    cfg = dict(n_item=n_item, n_user=n_user, max_len=L, n_layers=6, n_heads=4, emb_dim=64, u_emb_dim=10, ffn_dim=256,
               dropout=0.0, lr1=1e-3)
    device = D.device
    pkg, c, net, irn = build_irn(cfg, device)
    ops = pkg.ops
    n_loc = (n_user + D.world - 1) // D.world                     # users are independent: replicas over the user axis
    lo = D.rank * n_loc
    seqs, users = seqs_h[lo:lo + n_loc].to(device), users_h[lo:lo + n_loc].to(device)
    B = seqs.shape[0]
    p = L - 2
    paths = torch.zeros((B, args.steps + args.warmup), dtype=torch.float32, device=device)
    temp = seqs.clone()
    st = {"excl": None}

    def step(i):
        with torch.no_grad():
            st["excl"] = irn.path_step(temp, users, paths, i, st["excl"])

    ms, launches, clocks, kms = timed_steps(D, ops, step, args.steps, args.warmup)
    dump_outputs(args, D, {"paths": paths, "windows": temp, "exclusions": st["excl"][0], "exclusion_counts": st["excl"][1]})
    P = args.e2e_path_len
    sp, up = seqs.cpu().pin_memory(), users.cpu().pin_memory()

    def e2e_call():
        s, u = sp.to(device, non_blocking=True), up.to(device, non_blocking=True)
        return irn.get_seq_in_batch(s, u, s[:, -1].contiguous(), max_path_len=P, gap_len=0)
    e2e_call()
    torch.cuda.synchronize(); D.barrier()
    w0 = time.perf_counter()
    out = e2e_call()
    torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - w0)
    if D.rank != 0:
        return None
    step_ms = ms / args.steps
    value = n_user * args.steps / (ms / 1e3)
    d = cfg["emb_dim"]
    alg = {"scorer": ("tensor", 2.0 * d * n_item * B, "2*d*N FLOP per user-step"),
           "gather": ("hbm", float(L * (8 + 8 * d)) * B, "L*(8 + 4d + 4d) B per user-step")}
    roof, kernels = roofline_blocks(alg, kms, step_ms, "cfg1")
    line = base_line("IRN influence-path generation throughput, MovieLens-1M", "user-steps/s", value, D, args, step_ms, "f32", data,
                     {"workload": "cfg1: IRN generation on ml-1m, all 6040 users per step, 3415 items, L=50 (history 49 + objective), "
                                  "d=64, 6 layers/4 heads/ffn 256", "users_per_gpu": B, "n_item": n_item,
                      "l2_policy": "working set < L2 (whole catalog 0.9 MB): L2-resident by nature of the dataset",
                      "weights": "reference default init, seed 1234"}, scaling="strong")
    line["e2e"] = {"value": n_user * P / e2e_s, "unit": "user-steps/s", "h2d_bytes_per_step": (sp.numel() + up.numel()) * 8 / P,
                   "d2h_bytes_per_step": out[0].size * 4 / P, "path_len": P, "api": "IRSNN.get_seq_in_batch"}
    line["gpu_launches"] = int(launches)
    line["roofline"], line["roofline_kernels"], line["clocks"] = roof, kernels, clocks
    if not args.no_parity:
        state = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        threads = os.cpu_count() or 1
        nb, steps = 128, min(args.steps + args.warmup, 20)
        pr, dt, kind = reference_generate_cpu(cfg, state, seqs[:nb].cpu(), users[:nb].cpu(), steps, threads)
        from oracle import irn_oracle as O
        with torch.no_grad():
            _, _, _, _, margins = O.generate_paths(state, seqs[:nb].cpu(), users[:nb].cpu(), seqs[:nb, -1].cpu(), cfg["n_heads"],
                                                   steps, return_margins=True, fold_cross=True)
        par = compare_paths(paths.cpu().numpy()[:nb, :steps], pr, seqs[:nb, -1].cpu().numpy(), margins)
        par["against"] = f"{kind}: IRSNN.get_seq_in_batch on CPU, first {nb} users x {steps} steps"
        par["decisions_with_margin_below_1e-5"] = int((margins < 1e-5).sum())
        line["parity"] = par
        if D.world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = {"value": nb * steps / dt, "unit": "user-steps/s", "cores": threads, "kind": kind,
                                    "sample": f"{nb} users x {steps} path steps (the reference's batch size 128), {dt:.1f} s"}
    return line


# ----------------------------------------------------------------------------------------------------------------------
# cfg2: SASRec next-item scoring
# ----------------------------------------------------------------------------------------------------------------------
def run_cfg2(args, D):
    from types import SimpleNamespace
    import influentialrs_b200 as pkg
    ops = pkg.ops
    device = D.device
    N, B, T, K = 3706, args.users or 1024, 20, 50
    cfg = SimpleNamespace(n_user=6040, n_item=N, hidden_units=120, max_len=T, dropout_rate=0.2, num_blocks=4, num_heads=3)
    torch.manual_seed(1234)
    net = pkg.SAS(cfg, device).to(device).eval()
    g = torch.Generator().manual_seed(1234 + D.rank)
    seqs = torch.randint(1, N + 1, (B, T), generator=g)
    npad = torch.randint(0, 6, (B,), generator=g)
    seqs[torch.arange(T).unsqueeze(0) < npad.unsqueeze(1)] = 0
    rats = (torch.rand((B, T), generator=g) > 0.5).long() * (seqs > 0)
    sd_, rd_ = seqs.to(device), rats.to(device)
    res = {}

    def step(i):
        res["out"] = net.predict_topk(sd_, rd_, top_k=K, hist=sd_)

    ms, launches, clocks, kms = timed_steps(D, ops, step, args.steps, args.warmup)
    dump_outputs(args, D, {"topk_scores": res["out"][0], "topk_items": res["out"][1]})
    sp, rp = seqs.pin_memory(), rats.pin_memory()

    def e2e_call():
        s, r = sp.to(device, non_blocking=True), rp.to(device, non_blocking=True)
        v, it = net.predict_topk(s, r, top_k=K, hist=s)
        return it.cpu()
    e2e_call(); torch.cuda.synchronize(); D.barrier()
    w0 = time.perf_counter()
    reps = 10
    for _ in range(reps):
        it = e2e_call()
    e2e_s = D.max(time.perf_counter() - w0) / reps
    if D.rank != 0:
        return None
    step_ms = ms / args.steps
    C = cfg.hidden_units
    alg = {"topk": ("tensor", 2.0 * C * N * B, "2*C*N FLOP per scored user (catalog scoring; top-50 + history mask fused)")}
    roof, kernels = roofline_blocks(alg, kms, step_ms, "cfg2")
    line = base_line("SASRec full-catalog next-item scoring throughput", "scored users/s", B * D.world / (step_ms / 1e3), D, args,
                     step_ms, "f32", "synthetic",
                     {"workload": f"cfg2: SASRec (model_params.params_sas: T=20, C=120, H=3, 4 blocks), N={N}, batch {B}, top-{K} "
                                  "with history filter", "users_per_gpu": B, "n_item": N,
                      "l2_policy": "working set < L2 (catalog 1.8 MB): launch-bound configuration", "weights": "default init, seed 1234"})
    line["e2e"] = {"value": B * D.world / e2e_s, "unit": "scored users/s", "h2d_bytes_per_step": (sp.numel() + rp.numel()) * 8,
                   "d2h_bytes_per_step": it.numel() * 8, "api": "SAS.predict_topk"}
    line["gpu_launches"] = int(launches)
    line["roofline"], line["roofline_kernels"], line["clocks"] = roof, kernels, clocks
    if not args.no_parity:
        R = load_ref()
        if R is not None:
            threads = os.cpu_count() or 1
            torch.set_num_threads(threads)
            rnet = R.SAS(cfg, torch.device("cpu"))
            rnet.load_state_dict({k: v.detach().cpu() for k, v in net.state_dict().items()})
            rnet.eval()
            t0 = time.perf_counter()
            with torch.no_grad():
                logits = rnet.predict(np.arange(B), seqs.numpy(), rats.numpy())                       # SAS.predict, float logits (D9)
                preds = torch.zeros((B, K), dtype=torch.long)
                for b in range(B):                                                                    # SASNN.predict_next tail
                    _, idx = logits[b].sort(descending=True)
                    preds[b] = R.utils.delete_item_in_history(idx + 1, seqs[b])[:K]
            dt = time.perf_counter() - t0
            ours = res["out"][1].cpu()
            srt = logits.sort(dim=1, descending=True).values
            gap = (srt[:, :-1] - srt[:, 1:])[:, : K + T]
            safe = gap.min(1).values > 1e-5
            line["parity"] = {"users": B, "users_with_margins_above_1e-5": int(safe.sum()),
                              "equal": bool(torch.equal(ours[safe], preds[safe])),
                              "against": "the reference's SAS.predict (float logits, D9) + sort + utils.delete_item_in_history on CPU"}
            if D.world == 1 and not args.no_cpu_baseline:
                line["cpu_baseline"] = {"value": B / dt, "unit": "scored users/s", "cores": threads, "kind": "reference",
                                        "sample": f"one batch of {B} users: SAS.predict + per-user sort + history filter, {dt:.2f} s"}
    return line


# ----------------------------------------------------------------------------------------------------------------------
# cfg4: IRN training step
# ----------------------------------------------------------------------------------------------------------------------
def run_cfg4(args, D):
    small = args.small
    N, B, L, d = (20000, 256, 50, 128) if small else (500_000, args.users or 4096, 50, 128)
    cfg = dict(n_item=N, n_user=100_000, max_len=L, n_layers=6, n_heads=4, emb_dim=d, u_emb_dim=10, ffn_dim=256, dropout=0.0, lr1=1e-3)
    device = D.device
    pkg, c, net, irn = build_irn(cfg, device, train=True)
    ops = pkg.ops
    if D.world > 1:
        from influentialrs_b200.dist import make_data_parallel
        make_data_parallel(irn)
    g = torch.Generator().manual_seed(1234 + D.rank)
    seqs = torch.randint(1, N + 1, (B, L), generator=g)
    if args.variant == "ragged":                                   # ml-1m-like padding (~44 % PAD, pre-padded)
        npad = (torch.rand((B,), generator=g) * 0.88 * L).long()
        seqs[torch.arange(L).unsqueeze(0) < npad.unsqueeze(1)] = 0
    users = torch.randint(0, cfg["n_user"], (B,), generator=g)
    sd_, ud_ = seqs.to(device), users.to(device)
    losses = []

    def step(i):
        losses.append(irn.train_batch(sd_, ud_))

    ms, launches, clocks, kms = timed_steps(D, ops, step, args.steps, args.warmup)
    dump_outputs(args, D, {"loss": torch.tensor(losses[-1], dtype=torch.float64),
                           **{"param." + k: p_ for k, p_ in net.named_parameters()}})
    sp, up = seqs.pin_memory(), users.pin_memory()

    def e2e_call():
        return irn.train_batch(sp.to(device, non_blocking=True), up.to(device, non_blocking=True))    # returns loss.item()
    e2e_call(); torch.cuda.synchronize(); D.barrier()
    w0 = time.perf_counter()
    e2e_call()
    torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - w0)
    in_sync = True
    if D.world > 1:
        import torch.distributed as dist
        cs = torch.stack([p_.detach().double().sum() for p_ in net.parameters()]).sum().reshape(1)
        lo_, hi_ = cs.clone(), cs.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN); dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        in_sync = bool((hi_ - lo_).abs().item() <= 1e-9 * max(1.0, abs(hi_.item())))
    if D.rank != 0:
        return None
    step_ms = ms / args.steps
    M = int((seqs[:, 1:] > 0).sum())
    alg = {"ce_bwd": ("tensor", 2 * 2.0 * M * N * d, "2 x 2*M*N*d FLOP (d_h and d_W; logits recomputed in both passes, bf16x3 issues 3x)"),
           "ce_fwd": ("tensor", 2.0 * M * N * d, "2*M*N*d FLOP (log-sum-exp over the catalog; bf16x3 issues 3x)"),
           "scatter_add": ("hbm", float(B * L) * (8 + 3 * 4 * d), "B*L*(8 + 4d dOut read + 4d RMW read + 4d RMW write)"),
           "gather": ("hbm", float(B * L) * (8 + 8 * d), "B*L*(8 + 4d + 4d)")}
    roof, kernels = roofline_blocks(alg, kms, step_ms, "cfg4")
    line = base_line("IRN training throughput (train_batch incl. Adam)", "train samples/s", B * D.world / (step_ms / 1e3), D, args,
                     step_ms, "f32", "synthetic",
                     {"workload": f"cfg4: IRN train_batch (gather + PIM attention fwd/bwd + full-softmax CE over {N} items + scatter-add + "
                                  f"Adam), L={L}, d={d}, 6 layers/4 heads", "variant": args.variant, "batch_per_gpu": B, "n_item": N,
                      "ce_rows_per_gpu": M, "parallelism": f"dp{D.world}", "l2_policy": "inputs > L2 (E, W 256 MB each + Adam state)",
                      "weights": "reference default init, seed 1234"})
    line["steps_per_s"] = 1e3 / step_ms
    line["e2e"] = {"value": B * D.world / e2e_s, "unit": "train samples/s", "h2d_bytes_per_step": (sp.numel() + up.numel()) * 8,
                   "d2h_bytes_per_step": 4, "api": "IRSNN.train_batch"}
    line["gpu_launches"] = int(launches)
    line["roofline"], line["roofline_kernels"], line["clocks"] = roof, kernels, clocks
    line["loss_first_last"] = [losses[0], losses[-1]]
    line["replicas_in_sync"] = in_sync
    if D.world == 1 and not args.no_cpu_baseline and not args.no_parity:
        R = load_ref()
        if R is not None:
            from types import SimpleNamespace
            threads = os.cpu_count() or 1
            torch.set_num_threads(threads)
            nb = 8                                           # [8,50,500k] logits = 0.8 GB (+ grads): what the host can hold
            torch.manual_seed(1234)
            rnet = R.IntendedNet(SimpleNamespace(**cfg))
            rirn = R.IRSNN(SimpleNamespace(**cfg), rnet, torch.device("cpu"))
            # parity of the first loss: same init (seed) except torch's ISA-dependent normal_ stream -> load OUR initial weights
            pkg2, c2, net2, irn2 = build_irn(cfg, device, train=True)
            rnet.load_state_dict({k: v.detach().cpu() for k, v in net2.state_dict().items()})
            t0 = time.perf_counter()
            l_ref = rirn.train_batch(seqs[:nb], users[:nb])
            dt = time.perf_counter() - t0
            l_our = irn2.train_batch(sd_[:nb], ud_[:nb])
            line["parity"] = {"first_loss_reference": l_ref, "first_loss_ours": l_our, "rel_err": abs(l_ref - l_our) / abs(l_ref),
                              "equal": bool(abs(l_ref - l_our) <= 1e-3 * abs(l_ref)),
                              "against": f"the reference's IRSNN.train_batch on CPU, first {nb} samples, same initial weights"}
            line["cpu_baseline"] = {"value": nb / dt, "unit": "train samples/s", "cores": threads, "kind": "reference",
                                    "sample": f"one train_batch of {nb} samples (materialised [B,L,N] logits), {dt:.1f} s"}
            del net2, irn2
    return line


# ----------------------------------------------------------------------------------------------------------------------
# cfg5: Evaluator measurements + Caser scoring
# ----------------------------------------------------------------------------------------------------------------------
def rank_bands(state, dec, end_fn, targets, n_heads):
    """[lo, hi] bounds of the target's history-filtered rank from the oracle's decoder rows scored in fp64: at N=1M a rank
    counts the items ahead of the label, and the handful of items within fp32 summation noise of the label's score may fall
    on either side in ANY fp32 implementation (the reference's CPU run included), so ranks are compared through the band
    of scores within 2e-5*max|s| of the label's."""
    from oracle import irn_oracle as O
    B = dec.shape[0]
    with torch.no_grad():
        h = O.samplenet_decoding(state, dec, n_heads, fold_cross=True)
    lo, hi = [], []
    W, b = state["project.weight"].double(), state["project.bias"].double()
    for i in range(B):
        end = end_fn(dec[i], targets[i])
        s = h[i, end].double() @ W.t() + b
        live = torch.ones_like(s, dtype=torch.bool)
        ids = dec[i, : end + 1]
        live[ids[ids > 0] - 1] = False
        sl = s[int(targets[i]) - 1]
        eps = 2e-5 * float(s.abs().max())
        lo.append(int((live & (s > sl + eps)).sum()) + 1)
        hi.append(int((live & (s > sl - eps)).sum()))
    return np.array(lo), np.array(hi)


def run_cfg5(args, D):
    from types import SimpleNamespace
    import influentialrs_b200 as pkg
    ops = pkg.ops
    device = D.device
    N, B, L, d, P = (20000, 256, 60, 128, 5) if args.small else (1_000_000, args.users or 8192, 60, 128, 21)
    c = SimpleNamespace(n_item=N, max_len=L, n_layers=6, n_heads=4, emb_dim=d, ffn_dim=256, dropout=0.0, lr1=1e-3)
    torch.manual_seed(1234)
    net = pkg.SampleNet(c).to(device).eval()
    ev = pkg.Evaluator(c, net, device)
    shard = None
    if D.world > 1:
        from influentialrs_b200.dist import ShardedScorer
        shard = ShardedScorer(net.project.weight, net.project.bias, D.rank, D.world)
        ev.scorer = shard
    g = torch.Generator().manual_seed(1234 + D.rank)
    nh = 30
    hist = torch.zeros((B, L), dtype=torch.long)
    new = torch.zeros((B, L), dtype=torch.long)
    # nh history items + P path items + the target, DISTINCT per user by construction (one id per catalog stripe): a target
    # inside its own history makes Evaluator.get_rr_increase_in_batch raise, in the reference as here
    n_ids = nh + P + 1
    stripe = N // n_ids
    ids = (torch.arange(n_ids).unsqueeze(0) * stripe + torch.randint(0, stripe, (B, n_ids), generator=g) + 1)
    ids = ids.gather(1, torch.rand((B, n_ids), generator=g).argsort(1))
    hist[:, :nh] = ids[:, :nh]
    new[:, :nh + P] = ids[:, :nh + P]
    targets = ids[:, nh + P]
    start = torch.full((B,), nh, dtype=torch.long)
    lp = torch.full((B,), P, dtype=torch.long)
    hd, nd, td, sd_, ld_ = hist.to(device), new.to(device), targets.to(device), start.to(device), lp.to(device)
    x = torch.randn((B, 2 * d), generator=g).to(device)                    # Caser features [z, user_emb]
    W2 = (torch.randn((N + 1, 2 * d), generator=g) / (2 * d)).to(device)
    b2 = torch.zeros((N + 1,), device=device)
    res = {}

    def step(i):
        res["pp"] = ev.get_pp_in_batch(nd, sd_, ld_)
        res["rr"] = ev.get_rr_increase_in_batch(hd, nd, td)
        res["caser"] = ops.score_topk_any(x, W2[1:], b2[1:], 50, None, 1)

    ms, launches, clocks, kms = timed_steps(D, ops, step, args.steps, args.warmup)
    dump_outputs(args, D, {"path_probability": np.asarray(res["pp"]), "reciprocal_rank_increase": res["rr"][0],
                           "rank_increase": res["rr"][1], "caser_topk_scores": res["caser"][0],
                           "caser_topk_items": res["caser"][1]})
    t0 = time.perf_counter()
    ev.get_grad_in_batch(hd.clone(), nd, td, sd_, ld_)
    torch.cuda.synchronize()
    grad_s = time.perf_counter() - t0
    hp, np_, tp = hist.pin_memory(), new.pin_memory(), targets.pin_memory()

    def e2e_call():
        h_, n_, t_ = hp.to(device, non_blocking=True), np_.to(device, non_blocking=True), tp.to(device, non_blocking=True)
        a = ev.get_pp_in_batch(n_, sd_, ld_)
        b = ev.get_rr_increase_in_batch(h_, n_, t_)
        return a, b
    e2e_call(); torch.cuda.synchronize(); D.barrier()
    w0 = time.perf_counter()
    e2e_call()
    torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - w0)
    if D.rank != 0:
        return None
    step_ms = ms / args.steps
    n_shard = N // D.world
    alg = {"rank": ("tensor", 2.0 * d * n_shard * B * D.world, "2*d*N FLOP per ranked row (bf16x3 issues 3x)"),
           "lse": ("tensor", 2.0 * d * n_shard * B * P * D.world, "2*d*N FLOP per path row (log-sum-exp; bf16x3 issues 3x)"),
           "topk": ("tensor", 2.0 * 2 * d * N * B, "2*(2d)*N FLOP per Caser user (top-50)")}
    roof, kernels = roofline_blocks(alg, kms, step_ms, "cfg5")
    line = base_line("Evaluator path scoring + Caser catalog scoring throughput", "evaluated users/s", B * D.world / (step_ms / 1e3),
                     D, args, step_ms, "f32", "synthetic",
                     {"workload": f"cfg5: Evaluator.get_pp_in_batch + get_rr_increase_in_batch (SampleNet d={d}, L={L}, 6 layers/4 heads, "
                                  f"path length {P}) + Caser top-50 scoring [B,{2*d}]x[N,{2*d}], N={N}", "users_per_gpu": B, "n_item": N,
                      "catalog_shards": D.world, "l2_policy": "inputs > L2 (W 512 MB, Caser W2 1 GB)", "weights": "default init, seed 1234"})
    line["e2e"] = {"value": B * D.world / e2e_s, "unit": "evaluated users/s", "h2d_bytes_per_step": (hp.numel() + np_.numel() + tp.numel()) * 8,
                   "d2h_bytes_per_step": B * 8 * 3, "api": "Evaluator.get_pp_in_batch + get_rr_increase_in_batch (Caser excluded)"}
    line["gpu_launches"] = int(launches)
    line["roofline"], line["roofline_kernels"], line["clocks"] = roof, kernels, clocks
    line["detail"] = {"get_grad_in_batch_s": grad_s,
                      "per_kernel_ms": {k: v[0] * v[1] for k, v in kms.items()}}
    if D.world == 1 and not args.no_cpu_baseline and not args.no_parity:
        R = load_ref()
        if R is not None:
            threads = os.cpu_count() or 1
            torch.set_num_threads(threads)
            nb = 4                                            # [4,59,1M] logits + log-softmax: 1.9 GB
            rnet = R.SampleNet(c)
            rnet.load_state_dict({k: v.detach().cpu() for k, v in net.state_dict().items()})
            rnet.eval()
            rev = R.Evaluator(c, rnet, torch.device("cpu"))
            t0 = time.perf_counter()
            with torch.no_grad():
                pp_ref = rev.get_pp_in_batch(new[:nb], start[:nb], lp[:nb])
                irr_ref, ir_ref = rev.get_rr_increase_in_batch(hist[:nb], new[:nb], targets[:nb])
            dt = time.perf_counter() - t0
            pp_our = np.array(res["pp"][:nb])
            ir_our = np.asarray(res["rr"][1][:nb])
            ir_ref = np.asarray(ir_ref)
            from oracle import irn_oracle as O
            state = {k: v.detach().cpu() for k, v in net.state_dict().items()}
            b_lo, b_hi = rank_bands(state, hist[:nb, :-1].clone(), lambda row, t: O._first_zero_minus1(row), targets[:nb], c.n_heads)
            e_lo, e_hi = rank_bands(state, new[:nb, :-1].clone(), O._last_path_index, targets[:nb], c.n_heads)
            inside = lambda ir: bool(((ir >= e_lo - b_hi) & (ir <= e_hi - b_lo)).all())
            pp_err = float(np.max(np.abs(pp_our - np.array(pp_ref)) / np.abs(np.array(pp_ref))))
            line["parity"] = {"users": nb, "pp_max_rel_err": pp_err,
                              "rank_increase_identical_to_reference": bool(np.array_equal(ir_ref, ir_our)),
                              "rank_increase_max_abs_diff": int(np.abs(ir_ref - ir_our).max()),
                              "rank_band_width_max": int(max((b_hi - b_lo).max(), (e_hi - e_lo).max())),
                              "ours_inside_fp64_band": inside(ir_our), "reference_inside_fp64_band": inside(ir_ref),
                              "equal": bool(inside(ir_our) and pp_err < 1e-3),
                              "against": "the reference's Evaluator.get_pp_in_batch / get_rr_increase_in_batch on CPU, same weights; "
                                         "ranks at N=1M through the fp64 band of scores within fp32 noise of the target's"}
            line["cpu_baseline"] = {"value": nb / dt, "unit": "evaluated users/s", "cores": threads, "kind": "reference",
                                    "sample": f"{nb} users: get_pp_in_batch + get_rr_increase_in_batch (Caser excluded), {dt:.1f} s"}
    return line


# ----------------------------------------------------------------------------------------------------------------------
# k2: gather / scatter-add bandwidth
# ----------------------------------------------------------------------------------------------------------------------
def run_k2(args, D):
    import influentialrs_b200 as pkg
    ops = pkg.ops
    device = D.device
    N, d, B, L = 1_000_000, 128, args.users or 4096, 201
    g = torch.Generator(device=device).manual_seed(1234)
    E = torch.randn((N + 1, d), generator=g, device=device)
    pe = torch.randn((L, d), generator=g, device=device)
    dE = torch.zeros_like(E)
    dout = torch.randn((B, L, d), generator=g, device=device)
    cfg = dict(max_len=L, n_item=N, n_user=10)
    out = {}
    pk = peaks()
    ops.launch_count_reset()
    for variant in ("uniform", "zipf"):
        ids, _ = synth_batch(B, cfg, g, device, variant)

        def run(fn):
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                last = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.steps, last
        ms_g, gathered = run(lambda: ops.embed_gather_raw(ids, E, pe, math.sqrt(d)))
        ms_s, _ = run(lambda: ops.embed_scatter_add_raw(ids, dout, math.sqrt(d), dE, 0))
        rows = B * L
        gb_g = rows * (8 + 8 * d) / 1e9
        gb_s = rows * (8 + 12 * d) / 1e9
        out[variant] = {"gather_ms": ms_g, "gather_GBps": gb_g / (ms_g / 1e3), "gather_frac": gb_g / (ms_g / 1e3) / pk["hbm"],
                        "scatter_add_ms": ms_s, "scatter_add_GBps": gb_s / (ms_s / 1e3), "scatter_add_frac": gb_s / (ms_s / 1e3) / pk["hbm"],
                        "distinct_ids": int(ids.unique().numel()), "rows": rows}
    dump_outputs(args, D, {"gathered": gathered, "scatter_add_table": dE})
    # correctness of the scatter-add at the measured size: column sums survive (linearity), fp64 check on a sample of rows
    dE.zero_()
    ops.embed_scatter_add_raw(ids, dout, 1.0, dE, 0)
    want = dout.reshape(-1, d).double().sum(0)
    got = dE.double().sum(0)
    ok = bool(((want - got).abs().max() / want.abs().max()) < 1e-5)
    if D.rank != 0:
        return None
    v = out["uniform"]
    line = {"metric": "embedding scatter-add (K2) bandwidth", "value": v["scatter_add_GBps"], "unit": "GB/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": v["scatter_add_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"k2: K1 gather and K2 scatter-add over [B={B}, L={L}] ids into a [{N}+1, {d}] fp32 table, uniform and "
                                   "Zipf(1) ids", "l2_policy": "table 512 MB > L2"},
            "roofline": {"bound": "hbm", "achieved": v["scatter_add_GBps"], "peak": pk["hbm"], "unit": "GB/s", "frac": v["scatter_add_frac"],
                         "traffic": None, "kernel": KERNEL_NAMES["scatter_add"],
                         "algorithmic": "rows*(8 + 4d dOut read + 4d RMW read + 4d RMW write)"},
            "detail": out, "parity": {"equal": ok, "against": "column sums of dOut in fp64 (linearity of the scatter-add)"},
            "gpu_launches": int(ops.launch_count())}
    return line


# ----------------------------------------------------------------------------------------------------------------------
# reference arms
# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own get_seq_in_batch (cfg3) on the box's host cores, all threads, a bounded sample
    per step.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cfg = dict(SMALL if args.small else CFG3)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    users_n, steps = (4, 2) if cfg["n_item"] >= 500_000 else (16, 2)
    from types import SimpleNamespace
    R = load_ref()
    torch.manual_seed(1234)
    if R is not None:
        net = R.IntendedNet(SimpleNamespace(**cfg))
        state = net.state_dict()
    else:
        from oracle import irn_oracle as O
        state = O.synth_irn_state(cfg["n_item"], cfg["n_user"], cfg["max_len"], cfg["emb_dim"], cfg["n_layers"], cfg["ffn_dim"], seed=1234)
    g = torch.Generator().manual_seed(1234)
    seqs, us = synth_batch(users_n * 64, cfg, g, torch.device("cpu"), args.variant)
    kind = "port"
    t_all = []
    n_w = min(args.warmup, 1)
    n = max(1, args.steps)
    for i in range(n_w + n):
        off = (i % 64) * users_n
        _, dt, kind = reference_generate_cpu(cfg, state, seqs[off:off + users_n], us[off:off + users_n], steps, threads)
        if i >= n_w:
            t_all.append(dt)
    dt = sum(t_all) / len(t_all)
    v = users_n * steps / dt
    cb = {"value": v, "unit": "user-steps/s", "cores": threads, "kind": kind,
          "sample": f"{users_n} users x {steps} path step(s) per bench step ({'the reference IRSNN.get_seq_in_batch' if kind == 'reference' else 'oracle port'}), "
                    f"{n} timed steps, torch CPU fp32"}
    print(json.dumps({
        "impl": "reference", "metric": "IRN influence-path generation throughput @1M items", "value": v,
        "unit": "user-steps/s", "n_gpus": world, "steps": n, "warmup": n_w,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "cfg3: IRN generation, 1M-item catalog, L=201 (history 200 + objective), d=128, 6 layers/4 heads/ffn 256"
                   if not args.small else "small", "variant": args.variant, "users_per_gpu": args.users or 4096, "n_item": cfg["n_item"],
                   "catalog_shards": world, "weights": "reference default init, seed 1234",
                   "cpu_sample": f"{users_n} users x {steps} path steps per bench step"},
        "cpu_baseline": cb, "e2e": {"value": v, "unit": "user-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": ("the UNMODIFIED reference (oracle/_ref, shims D1-D3) on the host cores" if kind == "reference"
                 else "reference tree not staged: oracle port of the reference algorithm on the host cores")}))


def run_torch_gpu(args):
    """--impl torch_gpu: the reference's own code on cuda (stock torch kernels).  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from types import SimpleNamespace
    cfg = dict(SMALL if args.small else CFG3)
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    R = load_ref()
    if R is None:
        print(json.dumps({"impl": "torch_gpu", "unavailable": "reference tree not staged (oracle/_ref missing)"}))
        return
    torch.manual_seed(1234)
    state = R.IntendedNet(SimpleNamespace(**cfg)).state_dict()
    g = torch.Generator().manual_seed(1234)
    seqs, us = synth_batch(args.users or 32, cfg, g, torch.device("cpu"), args.variant)
    r = torch_gpu_reference(cfg, state, seqs, us, device, steps=max(1, args.steps), batch=args.users or 32)
    r.pop("paths", None)
    print(json.dumps({"impl": "torch_gpu", "metric": "IRN influence-path generation throughput @1M items", "unit": "user-steps/s",
                      "value": r.get("value"), "n_gpus": 1, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "cfg3 (reference code, device=cuda)", "variant": args.variant}, "detail": r}))


RUNNERS = {"cfg3": run_cfg3, "cfg1": run_cfg1, "cfg2": run_cfg2, "cfg4": run_cfg4, "cfg5": run_cfg5, "k2": run_k2}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"])
    ap.add_argument("--config", default="cfg3", choices=sorted(RUNNERS))
    ap.add_argument("--variant", default="uniform", choices=["uniform", "zipf", "ragged"])
    ap.add_argument("--users", type=int, default=0, help="users per GPU per step (default: the configuration's)")
    ap.add_argument("--small", action="store_true", help="tiny catalog (debug)")
    ap.add_argument("--e2e-path-len", type=int, default=20)
    ap.add_argument("--e2e-warm", type=int, default=1, help="untimed end-to-end calls before the timed one")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"cfg3": 20, "cfg1": 20, "cfg2": 50, "cfg4": 3, "cfg5": 3, "k2": 20}[args.config]
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "torch_gpu":
        return run_torch_gpu(args)
    args.warmup = max(args.warmup, 3)
    D = Dist()
    try:
        line = RUNNERS[args.config](args, D)
        if line is not None:
            print(json.dumps(line))
    finally:
        D.close()


if __name__ == "__main__":
    main()
