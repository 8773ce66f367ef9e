"""Shared test helpers: golden loading and tolerances (tests only)."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# north_star: logits / attention outputs / gradients within 1e-3 relative error.  Element-wise
# relative error is meaningless next to zero (SURVEY.md section 7 "hard parts"), so the bound used
# everywhere is  |a-b| <= RTOL * max|ref|  over the compared tensor (row-max for logits).
RTOL = 1e-3


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    rest = {k: z[k] for k in z.files if not k.startswith(("sd.", "rows."))}
    if "sd_fingerprint" in z.files:
        return seeded_state(z), rest
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    return sd, rest


def seeded_state(z):
    """Rebuild the weights of a fixture stored by oracle/make_golden.py::seeded_weights: the reference's default
    initialisers under the stored seed, through the drop-in InfluentialNet (it creates the same torch.nn modules in the
    same order), every tensor checked bit for bit against the fingerprint the reference-side generator stored.  The two
    normal_-initialised embedding tables come from the fixture (torch's CPU normal_ stream depends on the host's vector
    ISA): the rows the fixture reads, NaN in every other row, so that a read of one shows in the results."""
    from oracle.ref_shim import irn_config
    from influentialrs_b200.irn import InfluentialNet
    cfg = irn_config(*[int(x) for x in z["cfg"][:7]], u_emb_dim=int(z["cfg"][7]))
    torch.manual_seed(int(z["seed"]))
    sd = {k: v.detach().clone() for k, v in InfluentialNet(cfg).state_dict().items()}
    keys = [str(k) for k in z["sd_keys"]]
    assert sorted(sd.keys()) == keys
    for i, k in enumerate(keys):
        if "rows." + k in z.files:
            sd[k] = torch.full_like(sd[k], float("nan"))
            sd[k][torch.from_numpy(z["rows." + k])] = torch.from_numpy(z["sd." + k])
            continue
        bits = sd[k].contiguous().reshape(-1).view(torch.int32).to(torch.int64)
        w = torch.arange(bits.numel(), dtype=torch.int64) % 8191 + 1
        got = (int(bits.sum()), int((bits * w).sum()), bits.numel())
        assert got == tuple(int(x) for x in z["sd_fingerprint"][i]), f"weights of {k} differ from the reference's"
    return sd


def max_rel(a, b):
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    denom = b.abs().max().clamp_min(1e-30)
    return float((a - b).abs().max() / denom)


def assert_close_rel(a, b, rtol=RTOL, what=""):
    r = max_rel(a, b)
    assert r <= rtol, f"{what}: max|a-b|/max|ref| = {r:.3e} > {rtol:g}"


def baseline_tail_scores(g, name):
    """Score matrix [B,N] (fp64) each classical baseline's predict_next sorts (model/baselines.py), from the stored factors."""
    T = lambda k: torch.from_numpy(g[k]).double()
    hist, users = torch.from_numpy(g["hist"]), torch.from_numpy(g["users"])
    last = hist[:, -1] - 1
    if name == "pop":
        return T("pop_counts").unsqueeze(0).expand(hist.shape[0], -1)
    if name == "mc":
        return (T("mc_gam").float() @ T("mc_eta").float()).double()[last]
    if name == "fpmc":
        a = (T("fpmc_gamU").float() @ T("fpmc_gamI").float())
        b = (T("fpmc_kap").float() @ T("fpmc_eta").float())
        return (a[users] + b[last]).double()
    if name == "tr":
        H, R, r, beta = T("tr_H").float(), T("tr_R").float(), T("tr_r").float(), T("tr_beta").float()
        l = torch.square(H[last].unsqueeze(1) + r.view(1, 1, -1) + R[users].unsqueeze(1) - H.unsqueeze(0))
        return (-l.sum(2) - beta.unsqueeze(0)).double()
    if name == "bpr":
        return (T("bpr_W").float()[users] @ T("bpr_H").float().t()).double()
    raise KeyError(name)


def assert_same_topk_up_to_ties(got, want, scores, hist=None, h=50):
    """Two top-k id lists [B,k] over the same score matrix [B,N] are the same answer up to the order INSIDE groups of
    equal scores: the reference sorts with torch's default (unstable) sort, so the order of tied items -- and which of
    them make a cut that falls inside a tie group -- is implementation-defined there (SURVEY D7 pins 'lower id first'
    here).  Checks: same score sequence position by position, no excluded item, no duplicates, and every item scoring
    strictly above the k-th score present in both."""
    got, want = torch.as_tensor(got).long(), torch.as_tensor(want).long()
    s = torch.as_tensor(scores)
    sg, sw = s.gather(1, got - 1), s.gather(1, want - 1)
    assert torch.equal(sg, sw), "score sequences differ"
    for b in range(got.shape[0]):
        gb, wb = got[b].tolist(), want[b].tolist()
        assert len(set(gb)) == len(gb)
        if hist is not None:
            ex = set(hist[b, -h:].tolist())
            assert not (set(gb) & ex)
        kth = float(sg[b, -1])
        assert {i for i, v in zip(gb, sg[b].tolist()) if v > kth} == {i for i, v in zip(wb, sw[b].tolist()) if v > kth}
