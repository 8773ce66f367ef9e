"""Every attention entry point against the per-row error bound of tests/attn_cases.py, on hard inputs: the fp32 kernels
(resident and key-blocked), the per-head tcgen05 kernels (resident and key-blocked), the persistent kernel on operand
images (shift-free and exact pass, and its one-row kernel), and the fp32 backward fed by either forward.  A row's
error is compared with that row's own bound, not with the largest value of the tensor; each case is checked to reach
the kernel it names."""
import functools
import math
import os
import subprocess
import sys

import pytest
import torch

from tests import attn_cases as AC

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from influentialrs_b200 import ops as _ops
    return _ops


def _flag_ok(ops):
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0


def _kernels(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type.name == "CUDA"}
    return res, {n.split("(")[0].split("<")[0].replace("void ", "").replace("irs::", "") for n in names if "attn" in n}


def _fp32_resident_fits(L, dh):
    """attn_smem_layout of attention.cu: the resident fp32 forward holds the window on chip."""
    ks = dh | 1
    off_v = (L * ks + 3) & ~3
    off_kb = off_v + ((L * dh + 3) & ~3)
    off_warp = off_kb + ((L + 3) & ~3)
    return (off_warp + 8 * (dh * 4 + L * 4)) * 4 <= 227 * 1024


def _bwd_resident_fits(L, dh):
    """attn_bwd_smem_layout of attention.cu."""
    mat = (L * (dh | 1) + 3) & ~3
    off_warp = 4 * mat + 3 * ((L + 3) & ~3)
    return (off_warp + 8 * (dh * 4 + 2 * L * 4)) * 4 <= 227 * 1024


def _engine_and_kernel(fn, L, dh):
    if fn == "irs_pim_attn_fwd":
        return ("fp32", "pim_attn_fwd_kernel") if _fp32_resident_fits(L, dh) else ("fp32_blocked", "pim_attn_fwd_blocked_kernel")
    if fn == "irs_pim_attn_fwd_blocked":
        return "fp32_blocked", "pim_attn_fwd_blocked_kernel"
    if fn == "irs_pim_attn_fwd_tc":
        return ("tc", "tca::pim_attn_tc_kernel") if L <= 223 else ("tc_blocked", "tcb::pim_attn_tc_blocked_kernel")
    return "tc_blocked", "tcb::pim_attn_tc_blocked_kernel"


def _call(ops, fn, case, q_row0, n_q):
    """One raw forward call (as test_gpu_attention_long._call): (out [B, n_q, d], lse [B, H, n_q]) on the CPU."""
    from influentialrs_b200._lib import lib, check
    B, L, d3 = case.qkv.shape
    d = d3 // 3
    qkv = case.qkv.to(DEV)
    ids, r_u = case.ids.to(DEV), case.r_u.to(DEV)
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    out = torch.full((B, n_q, d), 7.0, device=DEV)
    lse = torch.full((B, case.H, n_q), 7.0, device=DEV)
    args = (ops._ptr(q), ops._ptr(k), ops._ptr(v), d3, d3, d3, ops._ptr(ids), ops._ptr(r_u) if case.mode == 0 else None,
            AC.W_H, AC.W_OBJ, case.mode, ops._ptr(out), ops._ptr(lse), B, L, case.H, case.dh, q_row0, n_q)

    if "_tc" in fn:
        check(getattr(lib(), fn)(*args, ops._ptr(ops._error_flag(qkv.device)), ops._stream()), fn)
    else:
        check(getattr(lib(), fn)(*args, 0.0, 0, ops._stream()), fn)
    torch.cuda.synchronize()
    return out.cpu(), lse.cpu()


def _assert_rows(case, out, lse, engine, rows, what):
    st = AC._stats(case)
    r_out, r_lse, dead = AC.row_ratios(case, out, lse, engine, rows=rows, st=st)
    B, H, dh = case.B, case.H, case.dh
    nan_rows = torch.isnan(out.reshape(B, len(rows), H, dh).transpose(1, 2)).all(-1)
    assert torch.equal(nan_rows, dead), f"{what}: NaN rows differ from the reference's"
    if lse is not None:
        assert torch.equal(torch.isnan(lse), dead), f"{what}: lse of rows that see no key"
    worst = float(r_out.max())
    assert worst <= 1.0, f"{what}: out error {worst:.3g} x its row bound (window, head, row {_argmax(r_out)})"
    if r_lse is not None:
        wl = float(r_lse.max())
        assert wl <= 1.0, f"{what}: lse error {wl:.3g} x its row bound (window, head, row {_argmax(r_lse)})"
    return worst


def _argmax(r):
    i = int(r.reshape(-1).argmax())
    return tuple(int(x) for x in torch.unravel_index(torch.tensor(i), r.shape))


@functools.lru_cache(maxsize=None)
def _case(L, dh, mode, B, H, seed):
    return AC.hard_case(B, L, H, dh, mode, seed=seed)


LS = (1, 2, 31, 32, 33, 50, 127, 128, 129, 201, 223, 224, 600, 2048)
FP32_DH = (5, 16, 32, 64, 128)
TC_DH = (32, 16, 64)


def _bh(L):
    return (7, 2) if L <= 256 else ((3, 1) if L <= 600 else (2, 1))


def _fwd_params():
    ps = []
    for n, L in enumerate(LS):
        B, H = _bh(L)
        ps.append(("irs_pim_attn_fwd", L, FP32_DH[n % 5], n % 3, B, H))
        ps.append(("irs_pim_attn_fwd_blocked", L, FP32_DH[(n + 2) % 5], (n + 1) % 3, B, H))
        ps.append(("irs_pim_attn_fwd_tc", L, TC_DH[n % 3], (n + 2) % 3, B, H))
        ps.append(("irs_pim_attn_fwd_tc_blocked", L, TC_DH[(n + 1) % 3], n % 3, B, H))
    # the cfg4 training shape (L = 50, 4 heads of 32) and the cfg3 decoder shape (L = 201, 4 x 32) on every entry point
    for fn in ("irs_pim_attn_fwd", "irs_pim_attn_fwd_blocked", "irs_pim_attn_fwd_tc", "irs_pim_attn_fwd_tc_blocked"):
        ps.append((fn, 50, 32, 0, 7, 4))
        ps.append((fn, 201, 32, 0, 7, 4))
    return ps


@pytest.mark.parametrize("fn,L,dh,mode,B,H", _fwd_params())
def test_forward_entry_point_inside_row_bound(ops, fn, L, dh, mode, B, H):
    case = _case(L, dh, mode, B, H, seed=1000 + L + dh + mode)
    engine, _ = _engine_and_kernel(fn, L, dh)
    out, lse = _call(ops, fn, case, 0, L)
    _assert_rows(case, out, lse, engine, torch.arange(L), f"{fn} L={L} dh={dh} mode={mode}")
    if L > 2:
        # a row subset across a 128-row tile boundary (the generation reads one row)
        r0 = min(max(L - 5, 0), 126)
        n = min(5, L - r0)
        out, lse = _call(ops, fn, case, r0, n)
        _assert_rows(case, out, lse, engine, torch.arange(r0, r0 + n), f"{fn} rows {r0}..{r0 + n - 1}")
    _flag_ok(ops)


# ---------------------------------------------------------------------------------------------- persistent kernel
@functools.lru_cache(maxsize=None)
def _img_case(key):
    if key[0] == "threshold":
        return AC.threshold_case()
    _, L, mode = key
    return AC.hard_case(38, L, 4, 32, mode, seed=2000 + L + mode)           # 152 items: more than one per SM


IMG_KEYS = [("threshold",), ("hard", 201, 0), ("hard", 201, 1), ("hard", 129, 2), ("hard", 223, 0)]


def _img_outputs(ops, case, q_row0=0, n_q=None):
    B, L, d3 = case.qkv.shape
    d = d3 // 3
    qkv = case.qkv.to(DEV)
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    images = torch.zeros((ops.lib().irs_qkv_images_bytes(B, L, case.H, 32),), dtype=torch.uint8, device=DEV)
    ops.qkv_to_images(q, k, v, (d3, d3, d3), B, L, case.H, case.mode, images)
    ids, r_u = case.ids.to(DEV), case.r_u.to(DEV)
    out = ops.pim_attention_img(images, ids, r_u if case.mode == 0 else None, B, L, case.H, case.mode, AC.W_H, AC.W_OBJ,
                                q_row0, L if n_q is None else n_q)
    torch.cuda.synchronize()
    return out.cpu()


def _exact_arm(key, path):
    """Child process body: the same case through the persistent kernel with the row-max pass forced on every item."""
    from influentialrs_b200 import ops
    out = _img_outputs(ops, _img_case(key))
    assert int(ops._error_flag(torch.device(DEV)).item()) == 0
    torch.save(out, path)


@pytest.mark.parametrize("key", IMG_KEYS, ids=lambda k: "-".join(str(x) for x in k))
def test_persistent_kernel_shift_free_and_exact_pass_inside_row_bound(ops, key, tmp_path):
    case = _img_case(key)
    L = case.L
    out = _img_outputs(ops, case)
    _assert_rows(case, out, None, "img", torch.arange(L), f"persistent {case.name}")
    # the forced exact pass (IRS_ATTN_EXACT_MAX is read once per process: a child process, waited for)
    path = str(tmp_path / "exact.pt")
    env = dict(os.environ, IRS_ATTN_EXACT_MAX="1")
    code = (f"import sys; sys.path.insert(0, {ROOT!r}); from tests.test_gpu_attention_bounds import _exact_arm; "
            f"_exact_arm({key!r}, {path!r})")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stderr[-3000:]
    exact = torch.load(path)
    _assert_rows(case, exact, None, "img", torch.arange(L), f"persistent {case.name}, exact pass")
    # items the producer's bound puts at or above the limit take the exact pass in both arms: bit-equal
    n_exact = 0
    for it in range(case.B * case.H):
        b, h = divmod(it, case.H)
        if AC.item_bound(case, b, h) > AC.NO_SHIFT_SAFE:
            sl = slice(h * 32, (h + 1) * 32)
            assert torch.equal(out[b, :, sl].view(torch.int32), exact[b, :, sl].view(torch.int32)), f"item {it}"
            n_exact += 1
    if case.shift_free is not None:
        assert n_exact == int((~case.shift_free).sum()) and n_exact < case.B * case.H
    _flag_ok(ops)


@pytest.mark.parametrize("key", IMG_KEYS[:3], ids=lambda k: "-".join(str(x) for x in k))
def test_persistent_one_row_kernel_inside_row_bound(ops, key):
    case = _img_case(key)
    L = case.L
    for r in (0, 1, 100, L - 2, L - 1):
        out = _img_outputs(ops, case, r, 1)
        _assert_rows(case, out, None, "row", torch.tensor([r]), f"one-row kernel {case.name} row {r}")
    _flag_ok(ops)


# ---------------------------------------------------------------------------------------------- backward
def _bwd_longest_resident(dh):
    L = 1
    while _bwd_resident_fits(L + 1, dh):
        L += 1
    return L


BWD_SHAPES = {"cfg4": (5, 50, 4, 32, 0), "long_resident": (2, _bwd_longest_resident(32), 2, 32, 1),
              "long_blocked": (1, 2048, 1, 32, 0)}


@functools.lru_cache(maxsize=None)
def _bwd_case(shape):
    B, L, H, dh, mode = BWD_SHAPES[shape]
    return AC.hard_case(B, L, H, dh, mode, seed=3000 + L, train=True)


def _bwd_setup(ops, shape, feed):
    """The forward (fp32 or tcgen05) of a training case and a closure that launches the backward entry point on its out
    and lse: run(kernel) -> (d_qkv [B, L, 3d], d_r_u [B]) on the device."""
    from influentialrs_b200._lib import lib, check
    case = _bwd_case(shape)
    B, L, H, dh, mode = BWD_SHAPES[shape]
    d = H * dh
    d3 = 3 * d
    qkv = case.qkv.to(DEV)
    ids, r_u = case.ids.to(DEV), case.r_u.to(DEV)
    q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
    rp = ops._ptr(r_u) if mode == 0 else None
    out = torch.empty((B, L, d), device=DEV)
    lse = torch.empty((B, H, L), device=DEV)
    base = (ops._ptr(q), ops._ptr(k), ops._ptr(v), d3, d3, d3, ops._ptr(ids), rp, AC.W_H, AC.W_OBJ, mode)
    if feed == "tc":
        check(lib().irs_pim_attn_fwd_tc(*base, ops._ptr(out), ops._ptr(lse), B, L, H, dh, 0, L,
                                        ops._ptr(ops._error_flag(qkv.device)), ops._stream()), "fwd_tc")
    else:
        check(lib().irs_pim_attn_fwd(*base, ops._ptr(out), ops._ptr(lse), B, L, H, dh, 0, L, 0.0, 0, ops._stream()), "fwd")
    go = torch.randn((B, L, d), generator=torch.Generator().manual_seed(L))
    g_dev = go.to(DEV)
    torch.cuda.synchronize()

    keep = (qkv, ids, r_u, out, lse, g_dev)           # base holds raw pointers: the tensors must outlive every launch

    def run(kernel):
        assert keep
        d_qkv = torch.full_like(qkv, 7.0)
        d_ru = torch.zeros(B, device=DEV)
        dq, dk, dv = d_qkv[..., :d], d_qkv[..., d:2 * d], d_qkv[..., 2 * d:]
        fn = "irs_pim_attn_bwd" if kernel == "resident" else "irs_pim_attn_bwd_blocked"
        check(getattr(lib(), fn)(*base, ops._ptr(out), ops._ptr(lse), ops._ptr(g_dev), ops._ptr(dq), ops._ptr(dk),
                                 ops._ptr(dv), ops._ptr(d_ru) if mode == 0 else None, B, L, H, dh, 0.0, 0,
                                 ops._stream()), fn)
        return d_qkv, d_ru
    return case, go, run


BWD_PARAMS = [("resident", "cfg4"), ("resident", "long_resident"), ("blocked", "cfg4"), ("blocked", "long_blocked")]


@pytest.mark.parametrize("feed", ["fp32", "tc"])
@pytest.mark.parametrize("kernel,shape", BWD_PARAMS)
def test_backward_inside_element_bound(ops, kernel, shape, feed):
    """dq, dk, dv and d r_u of the fp32 backward against float64 autograd, fed by the fp32 forward or, as ops._PimAttention
    does with USE_TC_TRAIN_ATTENTION, by the tcgen05 forward's out and lse."""
    case, go, run = _bwd_setup(ops, shape, feed)
    d_qkv, d_ru = run(kernel)
    torch.cuda.synchronize()
    ref = AC.reference(case, go)
    b_qkv, b_ru = AC.backward_bound(case, go, "tc" if feed == "tc" else "fp32")
    got = d_qkv.cpu().double()
    assert bool(torch.isfinite(got).all())
    r = AC._ratio((got - ref["d_qkv"]).abs(), b_qkv)
    assert float(r.max()) <= 1.0, f"d_qkv error {float(r.max()):.3g} x its bound at {_argmax(r)}"
    if case.mode == 0:
        rr = AC._ratio((d_ru.cpu().double() - ref["d_r_u"]).abs(), b_ru)
        assert float(rr.max()) <= 1.0, f"d_r_u error {float(rr.max()):.3g} x its bound"
    _flag_ok(ops)


# ---------------------------------------------------------------------------------------------- routing
def _route_groups(ops):
    """kernel name -> the calls of this module that must reach it (routing depends on the shape alone)."""
    groups = {}
    for fn, L, dh, mode, B, H in _fwd_params():
        _, kernel = _engine_and_kernel(fn, L, dh)
        case = _case(L, dh, mode, B, H, seed=1000 + L + dh + mode)
        groups.setdefault(kernel, []).append(functools.partial(_call, ops, fn, case, 0, L))
    for key in IMG_KEYS:
        case = _img_case(key)
        groups.setdefault("tcp::pim_attn_persistent_kernel", []).append(functools.partial(_img_outputs, ops, case))
        groups.setdefault("tcp::pim_attn_row_kernel", []).append(functools.partial(_img_outputs, ops, case, case.L - 2, 1))
    for kernel, shape in BWD_PARAMS:
        name = "pim_attn_bwd_kernel" if kernel == "resident" else "pim_attn_bwd_blocked"
        groups.setdefault(name, []).append((kernel, shape))
    return groups


ROUTES = ["pim_attn_fwd_kernel", "pim_attn_fwd_blocked_kernel", "tca::pim_attn_tc_kernel",
          "tcb::pim_attn_tc_blocked_kernel", "tcp::pim_attn_persistent_kernel", "tcp::pim_attn_row_kernel",
          "pim_attn_bwd_kernel", "pim_attn_bwd_blocked"]


@pytest.mark.parametrize("kernel", ROUTES)
def test_every_case_reaches_the_kernel_it_names(ops, kernel):
    """One profiler trace per kernel over all the calls of this module routed to it: they launch that kernel and no other
    attention kernel (the backward calls: no other backward kernel)."""
    calls = _route_groups(ops)[kernel]
    if kernel.startswith("pim_attn_bwd"):
        runs = [(_bwd_setup(ops, shape, "fp32")[2], k) for k, shape in calls]
        _, names = _kernels(lambda: [run(k) for run, k in runs])
        want = {"pim_attn_bwd_kernel"} if kernel == "pim_attn_bwd_kernel" else {"pim_attn_bwd_dq_blocked_kernel",
                                                                                "pim_attn_bwd_dkv_blocked_kernel"}
    else:
        _, names = _kernels(lambda: [c() for c in calls])
        want = {kernel}
    assert names == want, names
    _flag_ok(ops)
