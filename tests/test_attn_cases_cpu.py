"""The attention error model of tests/attn_cases.py on the CPU: the float64 emulator of the persistent tensor-core kernel
stays inside the per-row bound on every case, the hard cases use a stated share of it (and N(0,1) data only a few
percent), every threshold item lands on its intended side of the shift-free limit, and a P.V that keeps only P_hi V_hi
leaves the bound."""
import functools
import math

import pytest
import torch

from tests import attn_cases as AC

L = 201


@functools.lru_cache(maxsize=None)
def _hard(mode):
    return AC.hard_case(8, L, 1, 32, mode, seed=5 + mode)


@functools.lru_cache(maxsize=None)
def _control(mode):
    return AC.control_case(4, L, 1, 32, mode, seed=15 + mode)


@functools.lru_cache(maxsize=None)
def _threshold():
    return AC.threshold_case()


def _sub(case, b0, b1):
    return AC.Case(case.name, case.qkv[b0:b1], case.ids[b0:b1], case.r_u[b0:b1], case.H, case.mode, case.regime[b0:b1],
                   case.window[b0:b1])


def _emulated_ratios(case, fault=None, force_exact=False):
    """{(b, h): (max ratio over the item's rows, shift_free)} of the emulator against the "img" bound."""
    st = AC._stats(case)
    ref = AC.reference(case)
    ob, _ = AC.forward_bound(case, "img", st)
    out = {}
    for b in range(case.B):
        for h in range(case.H):
            o, free = AC.emulate_persistent(case, b, h, force_exact=force_exact, fault=fault)
            ro = ref["out"][b].reshape(case.L, case.H, case.dh)[:, h]
            dead = st["dead"][b, h]
            assert torch.equal(torch.isnan(o).any(-1), dead), f"{case.name} item ({b},{h}): NaN rows"
            err = (o - ro).abs().amax(-1)
            r = AC._ratio(torch.where(dead, torch.zeros_like(err), err), ob[b, h])
            out[(b, h)] = (float(r.max()), free)
    return out


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("force_exact", [False, True])
def test_emulator_inside_the_bound_on_hard_cases(mode, force_exact):
    rat = _emulated_ratios(_hard(mode), force_exact=force_exact)
    worst = max(r for r, _ in rat.values())
    assert worst <= 1.0, f"mode {mode}: emulated error {worst:.3f} x the bound"
    if not force_exact:
        assert any(f for _, f in rat.values()) and not all(f for _, f in rat.values())


def test_emulator_inside_the_bound_on_threshold_items():
    case = _sub(_threshold(), 0, 12)
    for arm in (False, True):
        rat = _emulated_ratios(case, force_exact=arm)
        assert max(r for r, _ in rat.values()) <= 1.0


def test_hard_cases_use_the_bound_and_control_data_does_not():
    """Worst rounding (PIM: two leaders erring in opposite directions) and the threshold items reach a fifth and an
    eighth of the bound; N(0,1) data stays under a tenth (the margin of 2 and the accumulation terms are not reached)."""
    worst = _hard(0)
    rat = _emulated_ratios(worst)
    w = max(r for (b, _), (r, _) in rat.items() if int(worst.window[b]) == AC.WORST)
    assert w >= 0.15, w
    thr = max(r for r, _ in _emulated_ratios(_sub(_threshold(), 0, 4)).values())
    assert thr >= 0.12, thr
    ctl = max(max(r for r, _ in _emulated_ratios(_control(m)).values()) for m in (0, 1, 2))
    assert ctl <= 0.1, ctl
    assert w > 2 * ctl and thr > ctl


def test_threshold_items_land_on_their_side_of_the_limit():
    case = _threshold()
    n = case.B * case.H
    assert n > 4 * AC.NUM_SMS
    bounds = torch.tensor([AC.item_bound(case, it // case.H, it % case.H) for it in range(n)])
    free = case.shift_free
    assert bool((bounds[free] >= 79.0).all() and (bounds[free] <= 79.9).all())
    exact = ~free
    assert bool((bounds[exact] >= 80.1).all())
    assert int(((bounds >= 80.1) & (bounds <= 81.0)).sum()) >= n // 3          # most exact items just above the limit
    assert bool((case.r_u.abs() == 80).any() and (case.r_u.abs() == 40).any())
    # kinds alternate between neighbouring items and, per CTA of a 148-CTA grid, both staging buffers carry both kinds
    k = torch.arange(4 * AC.NUM_SMS)
    assert bool((free[k[:-1]] != free[k[1:]]).float().mean() > 0.9)
    for cta in range(AC.NUM_SMS):
        seq = free[cta::AC.NUM_SMS][:4]
        assert seq[0] != seq[2] and seq[1] != seq[3]
    # and the emulated producer agrees item by item on a sample
    for it in range(0, n, 37):
        b, h = divmod(it, case.H)
        qt, k_, _, _, kb = AC.item_operands(case, b, h)
        assert (AC.producer_bound(AC.bf16_rn(qt), AC.bf16_rn(k_), float(kb[torch.isfinite(kb)].abs().max()))
                <= AC.NO_SHIFT_SAFE) == bool(free[it])


def test_single_mma_pv_leaves_the_bound():
    """P_hi V_hi alone (the lo halves dropped) errs by ~u sum_j w_j |v_j|: far outside the bound, so a precision
    regression in P.V fails the suite."""
    case = _hard(1)
    rat = _emulated_ratios(case, fault="pv_hi_only")
    voff = [r for (b, _), (r, _) in rat.items() if int(case.window[b]) == AC.VOFF]
    assert min(voff) > 2.0, voff
    assert max(r for r, _ in rat.values()) > 10.0


def test_reference_matches_the_mask_semantics():
    """NaN rows exactly where a row sees no key; the objective column is seen by every row in PIM mode."""
    case = AC.hard_case(7, 9, 1, 16, 0, seed=3)
    ref = AC.reference(case)
    mb = AC.mask_bias(case.ids, case.r_u.double(), case.L, 0)
    dead = torch.isinf(mb).all(-1)
    assert torch.equal(torch.isnan(ref["lse"][:, 0]), dead)
    assert torch.equal(torch.isnan(ref["out"]).all(-1), dead)
    live = case.ids[:, -1] != 0
    assert bool(torch.isfinite(mb[live, :, -1]).all())
    assert bool(dead[(case.ids == 0).all(1)].all())
