"""CPU: every entry point that takes a workspace returns IRS_E_WORKSPACE for a workspace one byte smaller than its
``*_workspace_bytes`` query, and IRS_E_BADARG for a null required pointer, before it touches the device.

The device pointers are dummies that are never dereferenced, so the file is skipped wherever a CUDA device is visible:
a check that ever moved behind a launch must not run a kernel on them."""
import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="dummy device pointers: run only without a GPU")

IRS_E_BADARG, IRS_E_WORKSPACE = -1, -3
M, N, D, K, N_SEL = 4, 1000, 64, 5, 2
# distinct 256-byte aligned dummy device addresses
h, W, bias, prep, label, lscore, out_f, out_i, lse, sel, lead, excl_flag, ws = (0x7f0000000000 + (i << 20) for i in range(1, 14))


def _cases(l):
    """name -> (workspace query, call(h, workspace, workspace_bytes)); shapes and every other argument valid."""
    return {
        "topk_k1": (l.irs_score_topk_workspace_bytes(M, N, D, 1),
                    lambda h, w, n: l.irs_score_topk(h, D, W, bias, 1, None, None, 0, 1, out_f, out_i, M, N, D, w, n, None)),
        "topk": (l.irs_score_topk_workspace_bytes(M, N, D, K),
                 lambda h, w, n: l.irs_score_topk(h, D, W, bias, 1, None, None, 0, K, out_f, out_i, M, N, D, w, n, None)),
        "argmax_tc": (l.irs_score_argmax_tc_workspace_bytes(M, N, D),
                      lambda h, w, n: l.irs_score_argmax_tc(h, D, W, prep, bias, 1, None, None, 0, out_f, out_i, M, N, D, 2,
                                                            w, n, None)),
        "argmax_tc_phase1": (l.irs_score_argmax_tc_workspace_bytes(M, N, D),
                             lambda h, w, n: l.irs_score_argmax_tc_phase1(h, D, W, prep, bias, 1, None, None, 0, lead, M, N, D,
                                                                          2, w, n, None)),
        "argmax_tc_phase2": (l.irs_score_argmax_tc_workspace_bytes(M, N, D),
                             lambda h, w, n: l.irs_score_argmax_tc_phase2(h, D, W, prep, bias, 1, None, None, 0, lead, out_f,
                                                                          out_i, M, N, D, 2, w, n, None)),
        "topk_tc": (l.irs_score_topk_tc_workspace_bytes(M, N, D, K),
                    lambda h, w, n: l.irs_score_topk_tc(h, D, W, prep, bias, 1, None, None, 0, K, out_f, out_i, M, N, D, w, n,
                                                        None)),
        "lse_gather": (l.irs_score_lse_gather_workspace_bytes(M, N, D, N_SEL),
                       lambda h, w, n: l.irs_score_lse_gather(h, D, W, bias, 1, sel, N_SEL, lse, out_f, M, N, D, w, n, None)),
        "lse_gather_tc": (l.irs_score_lse_gather_tc_workspace_bytes(M, N, D),
                          lambda h, w, n: l.irs_score_lse_gather_tc(h, D, W, prep, bias, 1, sel, N_SEL, lse, out_f, M, N, D,
                                                                    w, n, None)),
        "rank": (l.irs_score_rank_workspace_bytes(M, N, D),
                 lambda h, w, n: l.irs_score_rank(h, D, W, bias, 1, label, None, None, 0, out_i, M, N, D, w, n, None)),
        "rank_tc": (l.irs_score_rank_tc_workspace_bytes(M, N, D),
                    lambda h, w, n: l.irs_score_rank_tc(h, D, W, prep, bias, 1, label, None, None, 0, out_i, M, N, D, w, n,
                                                        None)),
        "count_ahead": (l.irs_score_count_ahead_workspace_bytes(M, N, D),
                        lambda h, w, n: l.irs_score_count_ahead(h, D, W, bias, 1, label, lscore, None, None, 0, out_i,
                                                                excl_flag, M, N, D, w, n, None)),
        "count_ahead_tc": (l.irs_score_rank_tc_workspace_bytes(M, N, D),
                           lambda h, w, n: l.irs_score_count_ahead_tc(h, D, W, prep, bias, 1, label, lscore, None, None, 0,
                                                                      out_i, excl_flag, M, N, D, w, n, None)),
        "ce_bwd_tc": (l.irs_score_ce_bwd_tc_workspace_bytes(M, N, D),
                      lambda h, w, n: l.irs_score_ce_bwd_tc(h, D, W, bias, label, lse, 1.0, out_f, None, None, M, N, D, w, n,
                                                            None)),
    }


NAMES = ["topk_k1", "topk", "argmax_tc", "argmax_tc_phase1", "argmax_tc_phase2", "topk_tc", "lse_gather", "lse_gather_tc",
         "rank", "rank_tc", "count_ahead", "count_ahead_tc", "ce_bwd_tc"]


@pytest.fixture(scope="module")
def cases():
    from influentialrs_b200.build import build
    from influentialrs_b200._lib import lib
    build()
    c = _cases(lib())
    assert sorted(c) == sorted(NAMES)
    return c


@pytest.mark.parametrize("name", NAMES)
def test_workspace_one_byte_short_is_rejected(cases, name):
    need, call = cases[name]
    assert need > 0
    assert call(h, ws, need - 1) == IRS_E_WORKSPACE


@pytest.mark.parametrize("name", NAMES)
def test_null_required_pointer_is_rejected(cases, name):
    need, call = cases[name]
    assert call(None, ws, need) == IRS_E_BADARG          # h
    assert call(h, None, need) == IRS_E_BADARG           # workspace
