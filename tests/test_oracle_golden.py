"""CPU: the oracle restatement (oracle/irn_oracle.py) against vectors produced by the reference
itself (oracle/make_golden.py -> tests/golden/*.npz).  This is what pins the oracle."""
import numpy as np
import pytest
import torch

from oracle import irn_oracle as O
from tests.helpers import load_golden, assert_close_rel

TIGHT = 2e-5   # two fp32 implementations of the same formulas (measured ~2e-6)


@pytest.mark.parametrize("name", ["irn_small", "irn_d30", "irn_ml1m"])
def test_irn_forward_matches_reference(name):
    sd, g = load_golden(name)
    H = int(g["cfg"][4])
    seqs, users = torch.from_numpy(g["seqs"]), torch.from_numpy(g["users"])
    h, r_u = O.irn_decoding(sd, seqs, users, H)
    rows = torch.from_numpy(g["h_rows"])
    assert_close_rel(h[:, rows], g["h"], TIGHT, "h")
    assert_close_rel(r_u, g["r_u"], 1e-6, "r_u")
    logits = h[:, rows] @ sd["project.weight"].t() + sd["project.bias"]
    assert_close_rel(logits, g["logits"], TIGHT, "logits")
    # constant-folded cross attention is the same function
    h2, _ = O.irn_decoding(sd, seqs, users, H, fold_cross=True)
    assert_close_rel(h2, h, TIGHT, "fold_cross")
    assert abs(float(O.irn_loss(sd, seqs, users, H)) - float(g["eval_loss"])) < 1e-5


@pytest.mark.parametrize("name", ["irn_small", "irn_d30", "irn_ml1m"])
def test_irn_generation_matches_reference(name):
    sd, g = load_golden(name)
    H = int(g["cfg"][4])
    seqs, users = torch.from_numpy(g["seqs"]), torch.from_numpy(g["users"])
    P = g["paths"].shape[1]
    paths, tg, hist, ne, margins = O.generate_paths(sd, seqs, users, torch.from_numpy(g["targets"]), H, P,
                                                    return_margins=True)
    assert margins.min() > 1e-5, "fixture contains a near-tie decision"
    np.testing.assert_array_equal(paths, g["paths"])
    np.testing.assert_array_equal(tg, g["targets"])
    assert ne == int(g["n_early"])
    np.testing.assert_array_equal([len(x) for x in hist], g["hist_lens"])


@pytest.mark.parametrize("name", ["irn_small", "irn_d30"])
def test_irn_generation_faithful_loop(name):
    sd, g = load_golden(name)
    H = int(g["cfg"][4])
    seqs, users = torch.from_numpy(g["seqs"]), torch.from_numpy(g["users"])
    paths, _, ne = O.generate_paths_faithful(sd, seqs, users, torch.from_numpy(g["targets"]), H, g["paths"].shape[1])
    np.testing.assert_array_equal(paths, g["paths"])
    assert ne == int(g["n_early"])


def test_irn_accuracy_metrics():
    sd, g = load_golden("irn_small")
    H = int(g["cfg"][4])
    seqs, users = torch.from_numpy(g["seqs"]), torch.from_numpy(g["users"])
    raw = list(torch.split(torch.from_numpy(g["raw_flat"]), g["raw_lens"].tolist()))
    hit, rr = O.accuracy_metrics(sd, raw, seqs, users, torch.from_numpy(g["labels"]), H, top_k=20, gap_len=0)
    assert hit == int(g["acc_hit"])
    np.testing.assert_allclose(rr, g["acc_rr"], rtol=0, atol=0)


@pytest.mark.parametrize("name", ["irn_small", "irn_d30"])
def test_irn_train_gradients(name):
    sd, g = load_golden(name)
    H = int(g["cfg"][4])
    seqs, users = torch.from_numpy(g["seqs"]), torch.from_numpy(g["users"])
    loss, grads = O.irn_loss_and_grads(sd, seqs, users, H)
    assert abs(float(loss) - float(g["train_loss"])) < 1e-5
    for k, gr in grads.items():
        ref = g["grad." + k]
        if np.abs(ref).max() == 0:
            assert float(gr.abs().max()) < 1e-7, k     # cross-attention in_proj weights: exactly 0
        else:
            assert_close_rel(gr, ref, 2e-4, "grad " + k)
    # folded cross attention gives the same gradients for everything it touches
    _, g2 = O.irn_loss_and_grads(sd, seqs, users, H, fold_cross=True)
    for k in ("item_embedder.weight", "project.weight", "user_embedder.weight",
              "decoder.layers.0.multihead_attn.out_proj.weight", "decoder.layers.0.multihead_attn.in_proj_bias"):
        assert_close_rel(g2[k], g["grad." + k], 2e-4, "fold grad " + k)


def test_evaluator_matches_reference():
    sd, g = load_golden("evaluator_small")
    H = int(g["cfg"][3])
    hist, new = torch.from_numpy(g["histories"]), torch.from_numpy(g["new_seqs"])
    tg, sp, lp = torch.from_numpy(g["targets"]), torch.from_numpy(g["start_pos"]), torch.from_numpy(g["l_path"])
    assert_close_rel(O.samplenet_forward(sd, new[:, :-1], H), g["logits_new"], TIGHT, "logits")
    np.testing.assert_allclose(O.evaluator_pp(sd, new, sp, lp, H), g["pp"], atol=2e-5)
    irr, ir = O.evaluator_rr_increase(sd, hist, new, tg, H)
    np.testing.assert_array_equal(ir, g["ir"])
    np.testing.assert_allclose(irr, g["irr"], atol=1e-12)
    tp, pp, avg, ioi = O.evaluator_grad(sd, hist.clone(), new, tg, sp, lp, H)
    np.testing.assert_allclose(tp, g["t_probs"], atol=3e-5)
    np.testing.assert_allclose(pp, g["p_probs"], atol=3e-5)
    np.testing.assert_allclose(avg, g["avg_ps"], atol=3e-5)
    np.testing.assert_allclose(ioi, g["iois"], atol=3e-5)
    assert abs(float(O.samplenet_loss(sd, new, H)) - float(g["eval_loss"])) < 1e-5


def test_sas_predict_matches_reference():
    sd, g = load_golden("sas_small")
    H = int(g["cfg"][4])
    seqs, rats = torch.from_numpy(g["seqs"]), torch.from_numpy(g["rats"])
    assert_close_rel(O.sas_log2feats(sd, seqs, rats, H), g["feats"], TIGHT, "feats")
    assert_close_rel(O.sas_predict(sd, seqs, rats, H), g["logits"], TIGHT, "logits")


def test_caser_scores_match_reference():
    _, g = load_golden("caser_small")
    s = O.caser_scores(torch.from_numpy(g["x"]), torch.from_numpy(g["W2"]), torch.from_numpy(g["b2"]))
    assert_close_rel(s, g["scores"], TIGHT, "caser scores")


def test_embed_is_two_rounded_ops():
    """x*sqrt(d) then +pe, each rounded to fp32 (the bit-exact contract of K1)."""
    sd, g = load_golden("irn_small")
    seqs = torch.from_numpy(g["seqs"])
    x = O.embed(seqs, sd["item_embedder.weight"], sd["pos_embedder.pe"][0])
    E = sd["item_embedder.weight"].numpy()
    pe = sd["pos_embedder.pe"][0].numpy()
    d = E.shape[1]
    want = (E[g["seqs"]] * np.float32(np.sqrt(np.float64(d)))).astype(np.float32) + pe[None, : seqs.shape[1]]
    np.testing.assert_array_equal(x.numpy(), want)
    np.testing.assert_array_equal(O.positional_table(12, d).numpy(), pe)


def test_topk_rank_tiebreak():
    s = torch.tensor([[1.0, 3.0, 3.0, 2.0, 3.0]])
    v, it = O.topk_excluding(s, torch.tensor([[2, 0]]), 3)
    assert it.tolist() == [[3, 5, 4]]                     # item 2 excluded; ties -> lower id
    assert O.rank_excluding(s, torch.tensor([5]), torch.tensor([[2]])).tolist() == [2]
    assert O.rank_excluding(s, torch.tensor([2]), torch.tensor([[2]])).tolist() == [0]
    assert O.rank_excluding(s, torch.tensor([4]), None).tolist() == [4]


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_batched_generation_equals_per_sample_loop_on_random_ragged_windows(seed):
    """The batched restatement (row L-2, raw-logit arg-max outside the window, shift) is the specification the CUDA path
    implements; the per-sample loop is how the reference writes it.  On random synthetic weights with ragged pre-padded
    histories -- including a one-item history and an objective that the model is steered to reach early -- both must give
    the same paths wherever the decision margin is above fp32 noise."""
    L, N, d, H, P = 14, 400, 16, 2, 6
    sd = O.synth_irn_state(N, 20, L, d, 2, 32, seed=seed)
    g = torch.Generator().manual_seed(100 + seed)
    B = 7
    seqs = torch.zeros((B, L), dtype=torch.long)
    for b in range(B):
        n = [L, 2, 5, L - 1, 9, 3, L][b]                      # history + objective; row 1: a single history item
        seqs[b, L - n:] = torch.randperm(N, generator=g)[:n] + 1
    users = torch.randint(0, 20, (B,), generator=g)
    targets = seqs[:, -1].clone()
    # steer row 0 to its objective: a large bias on that item makes it the first pick -> an early success
    sd = dict(sd)
    sd["project.bias"] = sd["project.bias"].clone()
    sd["project.bias"][int(targets[0]) - 1] += 50.0
    got, tg, hist, ne, margins = O.generate_paths(sd, seqs, users, targets, H, P, return_margins=True)
    want, _, ne2 = O.generate_paths_faithful(sd, seqs, users, targets, H, P)
    # a row is comparable up to its first near-tie decision (later windows may legitimately differ after a flip)
    for b in range(B):
        tie = np.where(margins[b] <= 1e-5)[0]
        upto = int(tie[0]) if len(tie) else P
        np.testing.assert_array_equal(got[b, :upto], want[b, :upto])
    assert got[0, 0] == float(targets[0]) and (got[0, 1:] == 0).all()      # trimmed after the early success
    assert ne >= 1 and (ne == ne2 or (margins <= 1e-5).any())
    assert [len(x) for x in hist] == [L - 1, 1, 4, L - 2, 8, 2, L - 1]


def test_irn_cfg3_decoder_shape_matches_reference():
    """The BASELINE cfg3 decoder shape (L=201, d=128, 4 heads, ffn 256, SIX layers; 6000-item catalog), full and ragged
    windows, weights = reference default init under seed 1234 (rebuilt here, fingerprint-checked): oracle decoder rows
    (a fixed sample of the non-PAD rows), generation-row logits, loss and generated paths against the reference's own
    outputs."""
    sd, g = load_golden("irn_cfg3_shape")
    seqs, users = torch.from_numpy(g["seqs"]), torch.from_numpy(g["users"])
    H, L = int(g["cfg"][4]), seqs.shape[1]
    h, r_u = O.irn_decoding(sd, seqs, users, H, fold_cross=True)
    rows = torch.from_numpy(g["h_index"])
    assert_close_rel(h.reshape(-1, h.shape[-1])[rows], g["h"], TIGHT, "h at the cfg3 decoder shape")
    assert_close_rel(r_u, g["r_u"], 1e-6, "r_u")
    logits = h[:, L - 2] @ sd["project.weight"].t() + sd["project.bias"]
    assert_close_rel(logits, g["logits_row"], TIGHT, "generation-row logits")
    assert abs(float(O.irn_loss(sd, seqs, users, H, fold_cross=True)) - float(g["eval_loss"])) < 1e-4
    P = g["paths"].shape[1]
    paths, tg, _, ne, margins = O.generate_paths(sd, seqs, users, torch.from_numpy(g["targets"]), H, P,
                                                 return_margins=True, fold_cross=True)
    assert margins.min() > 1e-5, "fixture contains a near-tie decision"
    np.testing.assert_array_equal(paths, g["paths"])
    assert ne == int(g["n_early"])


@pytest.mark.parametrize("name", ["pop", "mc", "fpmc", "tr", "bpr"])
def test_predict_next_tail_matches_reference_baselines(name):
    """oracle.predict_next_tail against predict_next of the reference's own POP / MC / FPMC / TransRec / BPR."""
    from tests.helpers import baseline_tail_scores
    _, g = load_golden("baseline_tails")
    scores = baseline_tail_scores(g, name)
    hist = torch.from_numpy(g["hist"])
    want = torch.from_numpy(g[name + "_preds"]).long()
    got = O.predict_next_tail(scores, hist, int(g["top_k"]))
    if name == "pop":
        # popularity counts are tie-heavy and the reference's torch.sort is unstable: equal up to the order inside ties
        from tests.helpers import assert_same_topk_up_to_ties
        assert_same_topk_up_to_ties(got, want, scores, hist)
        assert not torch.equal(got, want), "the fixture is meant to contain reference-side tie reordering"
    else:
        # fp32 sort of the reference vs fp64 scores here: identical unless two scores collide in fp32
        s32 = scores.float()
        srt = s32.sort(dim=1, descending=True).values
        assert (srt[:, :-1] - srt[:, 1:]).min() > 0, "fixture has an fp32 tie"
        assert torch.equal(got, want)
