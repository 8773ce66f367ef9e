"""CPU: the attention entry points' window bound (IRS_ATTN_MAX_L = 2048) is checked before any device work."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from influentialrs_b200.build import build
    build()
    from influentialrs_b200._lib import lib as _lib
    return _lib()


def test_tensor_core_forward_covers_windows_up_to_2048(lib):
    for dh in (16, 32, 48, 64):
        assert lib.irs_pim_attn_tc_supported(1, dh) == 1
        assert lib.irs_pim_attn_tc_supported(224, dh) == 1
        assert lib.irs_pim_attn_tc_supported(2048, dh) == 1
        assert lib.irs_pim_attn_tc_supported(2049, dh) == 0
    assert lib.irs_pim_attn_tc_supported(512, 8) == 0 and lib.irs_pim_attn_tc_supported(512, 128) == 0


def test_windows_longer_than_2048_are_a_shape_error(lib):
    # CAUSAL mode needs no ids / r_u; the pointers are never dereferenced because the shape is rejected first
    p = 256
    fwd = (p, p, p, 96, 96, 96, None, None, 0.05, 1.0, 2, p, None, 1, 2049, 1, 32, 0, 2049)
    assert lib.irs_pim_attn_fwd(*fwd, 0.0, 0, None) == -2
    assert lib.irs_pim_attn_fwd_blocked(*fwd, 0.0, 0, None) == -2
    assert lib.irs_pim_attn_fwd_tc(*fwd, None, None) == -2
    assert lib.irs_pim_attn_fwd_tc_blocked(*fwd, None, None) == -2
    bwd = (p, p, p, 96, 96, 96, None, None, 0.05, 1.0, 2, p, p, p, p, p, p, None, 1, 2049, 1, 32, 0.0, 0, None)
    assert lib.irs_pim_attn_bwd(*bwd) == -2
    assert lib.irs_pim_attn_bwd_blocked(*bwd) == -2
    # head sizes beyond the blocked fp32 kernels' 256, at a window only they could take
    big = (p, p, p, 3 * 257, 3 * 257, 3 * 257, None, None, 0.05, 1.0, 2, p, None, 1, 1000, 1, 257, 0, 1000)
    assert lib.irs_pim_attn_fwd(*big, 0.0, 0, None) == -2
