"""The chain stage cases of tests/chain_cases.py on the float64 emulator (no device): with the kernel's arithmetic, x' stays
well inside the LN3 band of ``ln_cases.chain_bands`` with the accumulator rounded either way, and an FFN or out_proj that
drops lo*hi, or keeps hi*hi alone (a plain bf16 GEMM), leaves it.  So the stage tests of tests/test_gpu_gemm_bounds.py
can tell the kernel from one that loses a term."""
import numpy as np
import pytest

from tests import chain_cases as CC
from tests import gemm_cases as GC
from tests import ln_cases as C


def _ratio(stage, mode="rn", terms=("lohi", "hilo", "hihi")):
    attn, x, P, kinds = CC.stage_case(stage)
    want, band, _, _ = C.chain_bands(attn, x, P)
    r = C.row_err(CC.emulate_chain_x(attn, x, P, mode, terms), want) / band
    hard = np.asarray(kinds) == ("worst+" if stage == "out_proj" else stage)
    return r, hard


@pytest.mark.parametrize("stage", CC.STAGES)
def test_kernel_arithmetic_inside_the_stage_band(stage):
    for mode in ("rn", "rz"):
        r, _ = _ratio(stage, mode)
        assert r.max() <= 1.0 / GC.MARGIN, (mode, float(r.max()))


@pytest.mark.parametrize("terms", [("hilo", "hihi"), ("hihi",)])
@pytest.mark.parametrize("stage", CC.STAGES)
def test_dropped_terms_leave_the_stage_band(stage, terms):
    r, hard = _ratio(stage, "rn", terms)
    assert hard.any()
    assert r[hard].min() > 2.0, float(r[hard].min())


def test_stage_inputs_are_pinned():
    """g2 = 0 stages: y is b2 for every row; the linear2 stage's relu output is exactly its worst-rounding bf1."""
    attn, x, P, _ = CC.stage_case("linear2")
    assert not P["W1"].any() and (P["bf1"] > 0).all() and not P["g2"].any()
    attn, x, P, _ = CC.stage_case("linear1+")
    assert (np.abs(P["W2"]).sum(1) == 1).all() and not P["g2"].any()
