"""CPU: bench.py's host-side pieces -- synthetic window generators of the cfg3 variants, the path comparison used for the
`parity` block, the traffic table, and the reference arm end to end on the tiny configuration (the unmodified reference when
/root/reference or the staged oracle/_ref is present, else the oracle port)."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_synth_batch_variants():
    cfg = dict(bench.SMALL)
    g = torch.Generator().manual_seed(1)
    L, N = cfg["max_len"], cfg["n_item"]
    s, u = bench.synth_batch(64, cfg, g, torch.device("cpu"), "uniform")
    assert s.shape == (64, L) and s.min() >= 1 and s.max() <= N and u.max() < cfg["n_user"]
    assert all(len(set(r.tolist())) == L for r in s)                      # distinct ids: the target is never in the history
    z, _ = bench.synth_batch(256, cfg, g, torch.device("cpu"), "zipf")
    assert z.min() >= 1 and z.max() <= N
    assert (z <= N // 100).float().mean() > 0.4                           # Zipf(1): about half of the draws in the top 1 %
    r, _ = bench.synth_batch(64, cfg, g, torch.device("cpu"), "ragged")
    hist_len = (r[:, :-1] > 0).sum(1)
    assert (r[:, -1] > 0).all() and hist_len.min() >= 20 and hist_len.max() <= L - 1 and hist_len.float().std() > 10
    first_real = (r[:, :-1] > 0).float().argmax(1)                        # pre-padded: zeros first, then the history
    assert all((r[b, : first_real[b]] == 0).all() and (r[b, first_real[b]:] > 0).all() for b in range(64))


def test_compare_paths_stops_at_the_target_and_reports_mismatches():
    ref = np.array([[5., 7., 0.], [1., 2., 3.], [4., 9., 9.]])             # user 0 hit its target 7 at step 1 (then zeroed)
    gpu = np.array([[5., 7., 8.], [1., 2., 3.], [4., 6., 9.]])             # untrimmed GPU buffer; user 2 differs at step 1
    out = bench.compare_paths(gpu, ref, np.array([7, 99, 99]))
    assert out["decisions"] == 2 + 3 + 2 and out["decisions_equal"] == 2 + 3 + 1 and not out["equal"]
    assert out["first_mismatches"] == [(2, 1, 6, 9)]
    assert bench.compare_paths(ref, ref, np.array([7, 99, 99]))["equal"]


def test_traffic_table_points_at_committed_captures():
    t = bench.traffic_table()
    assert {"decoder_chain", "attention", "scorer", "gather"} <= set(t)
    for v in t.values():
        assert v["bytes_per_launch"] > 0 and os.path.exists(os.path.join(ROOT, v["source"]))


def test_dump_outputs_types_sample_and_size_cap(tmp_path):
    from types import SimpleNamespace
    big = torch.arange(3 << 20, dtype=torch.int64).reshape(-1, 8)         # 24 MB as float64: above its quarter of 64 MB
    arrays = {"ids": torch.tensor([[1, 2], [3, 1 << 40]]), "x": torch.rand(5), "loss": torch.tensor(0.5, dtype=torch.float64),
              "big": big}
    files = {}
    for run in ("a", "b"):
        out = tmp_path / run
        bench.dump_outputs(SimpleNamespace(dump_outputs=str(out)), SimpleNamespace(rank=0), arrays)
        files[run] = {p.name: np.load(p) for p in out.iterdir()}
        assert sum(p.stat().st_size for p in out.iterdir()) <= bench.DUMP_BYTES
    got = files["a"]
    assert set(got) == {"ids.npy", "x.npy", "loss.npy", "big.npy", "big.rows.npy"}
    assert got["ids.npy"].dtype == np.float64 and got["ids.npy"].tolist() == [[1, 2], [3, 1 << 40]]
    assert got["x.npy"].dtype == np.float32 and np.array_equal(got["x.npy"], arrays["x"].numpy())
    assert got["loss.npy"].dtype == np.float64 and got["loss.npy"].tolist() == [0.5]
    rows = got["big.rows.npy"].astype(np.int64)
    assert 0 < len(rows) < big.shape[0] and np.array_equal(got["big.npy"], big.numpy()[rows].astype(np.float64))
    assert all(np.array_equal(got[k], files["b"][k]) for k in got)              # the sample is fixed
    bench.dump_outputs(SimpleNamespace(dump_outputs=str(tmp_path / "r1")), SimpleNamespace(rank=1), arrays)
    assert not (tmp_path / "r1").exists()                                       # rank 0 writes


def test_reference_arm_runs_on_cpu_small():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--small", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "user-steps/s"
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["e2e"]["h2d_bytes_per_step"] == 0
    from oracle.ref_shim import find_reference
    assert (line["cpu_baseline"]["kind"] == "reference") == (find_reference() is not None)
