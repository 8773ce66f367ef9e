#!/usr/bin/env python
"""Long-window attention: the key-blocked tcgen05 forward against the fp32 resident kernel it replaces, and the models at
windows whose attention no longer fits on chip.  One process, CUDA-event timings after warm-up; prints the card's name and
power limit first.

  1. attention forward, 4096 users x 4 heads: dh = 32 at L = 256, 384, 512 and dh = 64 at L = 256, 320, the blocked
     tcgen05 kernel (irs_pim_attn_fwd_tc_blocked) against the fp32 resident kernel (irs_pim_attn_fwd), outputs compared;
     the tcgen05 kernel alone at L = 1024, 2048; at L = 201 the blocked and the resident tcgen05 kernels.  TFLOP/s is the
     causal algorithmic work (QK^T and PV over the visible (row, key) pairs, the PIM objective column included) over
     kernel time.  q/k/v of every shape exceed the 126 MB L2.
  2. one cfg3-shaped generation step (1M items, 6 layers, d = 128, 4 heads, 4096 users) at L = 512;
  3. one training step (train_batch incl. Adam) at L = 512 with 4 heads of 32, and at L = 201 with 2 heads of 64.

    python scripts/attn_long_bench.py [--reps 20] [--skip-models]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def gpu_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                        "-i", "0"], text=True, timeout=20).strip()
    except Exception as e:
        return f"{torch.cuda.get_device_name(0)}, power limit unknown ({e.__class__.__name__})"


def causal_flops(B, H, L, dh, pim=True):
    """QK^T + PV multiply-adds (2 flops each) over the (row, key) pairs the mask leaves visible."""
    pairs = L * (L + 1) // 2 + ((L - 1) if pim else 0)          # j <= i, plus key L-1 for rows i < L-1 in PIM mode
    return 2 * 2 * dh * pairs * B * H


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def attention(reps):
    from influentialrs_b200 import ops
    from influentialrs_b200._lib import lib, check
    B, H, dev = 4096, 4, "cuda:0"
    flag = ops._error_flag(torch.device(dev))
    rows = []

    def run(fn, qkv, ids, r_u, out, L, dh):
        d = H * dh
        q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
        args = (ops._ptr(q), ops._ptr(k), ops._ptr(v), 3 * d, 3 * d, 3 * d, ops._ptr(ids), ops._ptr(r_u), 0.05, 1.0, 0,
                ops._ptr(out), None, B, L, H, dh, 0, L)
        if "tc" in fn:
            return lambda: check(getattr(lib(), fn)(*args, ops._ptr(flag), ops._stream()), fn)
        return lambda: check(getattr(lib(), fn)(*args, 0.0, 0, ops._stream()), fn)

    shapes = [(32, 256, True), (32, 384, True), (32, 512, True), (64, 256, True), (64, 320, True),
              (32, 1024, False), (32, 2048, False), (32, 201, None)]
    for dh, L, vs_fp32 in shapes:
        g = torch.Generator(device=dev).manual_seed(L + dh)
        d = H * dh
        qkv = torch.randn((B, L, 3 * d), generator=g, device=dev)
        ids = torch.randint(1, 1000, (B, L), generator=g, device=dev)
        ids[: B // 2, : L // 4] = 0                                   # half the windows pre-padded
        r_u = torch.randn(B, generator=g, device=dev)
        fl = causal_flops(B, H, L, dh)
        out_b = torch.empty((B, L, d), device=dev)
        t_b = time_ms(run("irs_pim_attn_fwd_tc_blocked", qkv, ids, r_u, out_b, L, dh), reps)
        row = {"L": L, "dh": dh, "B": B, "H": H, "tc_blocked_ms": round(t_b, 4), "tc_blocked_tflops": round(fl / t_b / 1e9, 2)}
        other = None
        if vs_fp32 is True:
            other = ("fp32_resident", "irs_pim_attn_fwd")
        elif vs_fp32 is None:
            other = ("tc_resident", "irs_pim_attn_fwd_tc")
        if other is not None:
            out_o = torch.empty_like(out_b)
            t_o = time_ms(run(other[1], qkv, ids, r_u, out_o, L, dh), reps)
            diff = float((out_b - out_o).abs().max() / out_o.abs().max())
            row.update({other[0] + "_ms": round(t_o, 4), other[0] + "_tflops": round(fl / t_o / 1e9, 2),
                        "speedup": round(t_o / t_b, 3), "max_rel_diff": diff})
        rows.append(row)
        print(json.dumps({"attention_forward": row}), flush=True)
        del qkv, out_b
        torch.cuda.empty_cache()
    assert int(flag.item()) == 0
    return rows


def generation_step(reps):
    import bench
    cfg = dict(bench.CFG3, max_len=512)
    pkg, c, net, irn = bench.build_irn(cfg, "cuda:0")
    B = 4096
    gen = torch.Generator(device="cuda:0").manual_seed(1234)
    seqs, users = bench.synth_batch(B, cfg, gen, "cuda:0")
    steps = reps + 3
    paths = torch.zeros((B, steps), dtype=torch.float32, device="cuda:0")
    temp = seqs.clone()
    st = {"excl": None, "i": 0}

    def step():
        with torch.no_grad():
            st["excl"] = irn.path_step(temp, users, paths, st["i"], st["excl"])
        st["i"] += 1

    ms = time_ms(step, reps)
    row = {"workload": "cfg3 generation step, 1M items, 6 layers, d=128, 4 heads, L=512", "users": B, "ms_per_step": round(ms, 3)}
    print(json.dumps({"generation": row}), flush=True)
    del net, irn
    torch.cuda.empty_cache()
    return row


def training_step(L, H, reps):
    import bench
    cfg = dict(bench.CFG3, n_item=100_000, max_len=L, n_layers=2, n_heads=H)
    pkg, c, net, irn = bench.build_irn(cfg, "cuda:0", train=True)
    B = 256
    gen = torch.Generator(device="cuda:0").manual_seed(99)
    seqs, users = bench.synth_batch(B, cfg, gen, "cuda:0")
    ms = time_ms(lambda: irn.train_batch(seqs, users), reps)
    row = {"workload": f"train_batch incl. Adam, 100k items, 2 layers, d=128, {H} heads of {128 // H}, L={L}", "users": B,
           "ms_per_step": round(ms, 3)}
    print(json.dumps({"training": row}), flush=True)
    del net, irn
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-models", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attn_long_bench.py measures the GPU: no CUDA device")
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    attention(args.reps)
    if not args.skip_models:
        generation_step(max(3, args.reps // 4))
        training_step(512, 4, max(3, args.reps // 4))
        training_step(201, 2, max(3, args.reps // 4))


if __name__ == "__main__":
    main()
