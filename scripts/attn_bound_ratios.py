"""Largest ratio of observed error to the derived bound (tests/attn_cases.py) for every attention kernel, over the cases of
tests/test_gpu_attention_bounds.py (and N(0,1) controls of the same shapes): how much headroom each bound leaves.
Prints one JSON object; writes nothing."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests import attn_cases as AC
from tests import test_gpu_attention_bounds as T
from influentialrs_b200 import ops

res = {}


def put(k, v):
    res[k] = max(res.get(k, 0.0), v)


for fn, L, dh, mode, B, H in T._fwd_params():
    case = T._case(L, dh, mode, B, H, seed=1000 + L + dh + mode)
    eng, kern = T._engine_and_kernel(fn, L, dh)
    out, lse = T._call(ops, fn, case, 0, L)
    ro, rl, _ = AC.row_ratios(case, out, lse, eng)
    put(kern + " out", float(ro.max())); put(kern + " lse", float(rl.max()))
    c = AC.control_case(B, L, H, dh, mode, seed=7 + L)
    out, lse = T._call(ops, fn, c, 0, L)
    ro, rl, _ = AC.row_ratios(c, out, lse, eng)
    put(kern + " out control", float(ro.max()))
for key in T.IMG_KEYS:
    case = T._img_case(key)
    out = T._img_outputs(ops, case)
    ro, _, _ = AC.row_ratios(case, out, None, "img")
    put("persistent out " + key[0], float(ro.max()))
    for r in (0, 100, case.L - 2):
        out = T._img_outputs(ops, case, r, 1)
        ro, _, _ = AC.row_ratios(case, out, None, "row", rows=torch.tensor([r]))
        put("row kernel out", float(ro.max()))
for kernel, shape in T.BWD_PARAMS:
    for feed in ("fp32", "tc"):
        case, go, run = T._bwd_setup(ops, shape, feed)
        dqkv, dru = run(kernel)
        torch.cuda.synchronize()
        ref = AC.reference(case, go)
        b, bru = AC.backward_bound(case, go, feed)
        put(f"bwd {kernel} fed by {feed} d_qkv", float(AC._ratio((dqkv.cpu().double() - ref["d_qkv"]).abs(), b).max()))
        if case.mode == 0:
            put(f"bwd {kernel} fed by {feed} d_r_u", float(AC._ratio((dru.cpu().double() - ref["d_r_u"]).abs(), bru).max()))
print(json.dumps(res, indent=1, sort_keys=True))
