"""Generate tests/golden/*.npz by running the UNMODIFIED reference (via oracle/ref_shim.py).

TEST INFRASTRUCTURE.  Run in the dev container (which has /root/reference but no GPU):

    python oracle/make_golden.py

The reference is Python and cannot travel to the GPU box, so its outputs are committed as small
fixtures next to this script.  Every array in a fixture is produced by the reference's own code
path (class / method named in the key comment); weights are stored as ``sd.<state_dict key>``.
"""
from __future__ import annotations

import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_shim import load_reference, irn_config  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def sd_arrays(net):
    return {"sd." + k: v.detach().cpu().clone().numpy() for k, v in net.state_dict().items()}


def prepadded(B, L, n_item, g, min_len=3, full_rows=1):
    """[0..0, history, target] rows, lengths ragged, ids without replacement per row."""
    seqs = torch.zeros((B, L), dtype=torch.long)
    for b in range(B):
        n = L if b < full_rows else int(torch.randint(min_len, L + 1, (1,), generator=g))
        seqs[b, L - n:] = torch.randperm(n_item, generator=g)[:n] + 1
    return seqs


def postpadded(B, L, n_item, g, min_len=3, max_fill=None):
    seqs = torch.zeros((B, L), dtype=torch.long)
    hi = L if max_fill is None else max_fill
    for b in range(B):
        n = int(torch.randint(min_len, hi + 1, (1,), generator=g))
        seqs[b, :n] = torch.randperm(n_item, generator=g)[:n] + 1
    return seqs


def irn_case(R, name, cfg, seqs, users, P, raw=None, labels=None, keep_rows=None, train=True, seeded=False):
    torch.manual_seed(1234)
    net = R.IntendedNet(cfg)
    net.eval()
    irn = R.IRSNN(cfg, net, torch.device("cpu"))
    out = dict(sd_arrays(net))
    out["cfg"] = np.array([cfg.n_item, cfg.n_user, cfg.max_len, cfg.n_layers, cfg.n_heads, cfg.emb_dim,
                           cfg.ffn_dim, cfg.u_emb_dim])
    out["seqs"], out["users"] = seqs.numpy(), users.numpy()
    targets = seqs[:, -1].clone()
    with torch.no_grad():
        h, r = net.decoding(seqs.clone(), users, return_pi=True)          # InfluentialNet.decoding
        logits = net.forward(seqs.clone(), users)                         # InfluentialNet.forward
        rows = slice(None) if keep_rows is None else keep_rows
        out["h"] = h[:, rows].numpy()
        out["logits"] = logits[:, rows].numpy()
        out["h_rows"] = np.arange(seqs.shape[1])[rows]
        out["r_u"] = irn.get_pif_in_batch(seqs, users)                    # IRSNN.get_pif_in_batch
        out["eval_loss"] = np.array(irn.get_loss_on_eval_data(seqs, users))   # IRSNN.get_loss_on_eval_data
        p, t, hist, ne = irn.get_seq_in_batch(seqs, users, targets, max_path_len=P, gap_len=0)  # IRSNN.get_seq_in_batch
        out["paths"], out["targets"], out["n_early"] = p, t, np.array(ne)
        out["hist_lens"] = np.array([len(x) for x in hist])
        if raw is not None:
            hit, rr = irn.get_accuracy_metrics_in_batch(raw, seqs, users, targets, labels, top_k=20, gap_len=0, use_h=True)
            out["acc_hit"], out["acc_rr"] = np.array(hit), rr             # IRSNN.get_accuracy_metrics_in_batch
            out["labels"] = labels.numpy()
            out["raw_lens"] = np.array([len(x) for x in raw])
            out["raw_flat"] = torch.cat(raw).numpy()
    if train:
        loss = irn.train_batch(seqs, users)                               # IRSNN.train_batch (dropout=0)
        out["train_loss"] = np.array(loss)
        for k, p_ in net.named_parameters():
            g = p_.grad
            out["grad." + k] = (torch.zeros_like(p_) if g is None else g).numpy()
        for k in ("item_embedder.weight", "project.weight", "project.bias", "user_mask_layer.weight",
                  "decoder.layers.0.self_attn.in_proj_weight", "decoder.layers.0.norm2.bias"):
            out["post." + k] = net.state_dict()[k].numpy().copy()         # after one Adam step
    if seeded:
        out = seeded_weights(out, 1234)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, {k: v.shape for k, v in out.items() if not k.startswith(("sd.", "grad.", "post."))})


def weight_fingerprint(sd):
    """Per-tensor exact integer checksums of the fp32 bit patterns (int64 wrap-around sums: independent of summation order,
    thread count and vector ISA): [sum bits, sum bits*(1 + index mod 8191), numel].  The cfg3-shape fixture stores these next
    to the two embedding tables; the tests rebuild the other weights from the seed and must reproduce them bit for bit."""
    keys = sorted(sd.keys())
    fp = np.zeros((len(keys), 3), dtype=np.int64)
    for i, k in enumerate(keys):
        bits = sd[k].detach().contiguous().reshape(-1).view(torch.int32).to(torch.int64)
        w = torch.arange(bits.numel(), dtype=torch.int64) % 8191 + 1
        fp[i] = (int(bits.sum()), int((bits * w).sum()), bits.numel())
    return keys, fp


def seeded_weights(out, seed):
    """Replace the state dict of an IRN fixture (``sd.<key>``, default initialisers under torch.manual_seed(seed)) by what
    rebuilds it: the seed, a fingerprint of every tensor, and the two normal_-initialised embedding tables -- torch's CPU
    normal_ stream depends on the host's vector ISA, so those cannot be rebuilt from the seed on another machine; the
    uniform_-initialised tensors can.  Of the tables only the rows the fixture reads are kept (``rows.<key>`` ids,
    ``sd.<key>`` values): the window items, the generated picks and PAD; the fixture's users.  That keeps fixtures at
    catalog scale under 1 MB."""
    sd = {k[3:]: torch.from_numpy(out.pop(k)) for k in [k for k in out if k.startswith("sd.")]}
    keys, fp = weight_fingerprint(sd)
    out.update(seed=np.array(seed), sd_keys=np.array(keys), sd_fingerprint=fp)
    read = {"item_embedder.weight": np.union1d(np.union1d(out["seqs"], out["paths"].astype(np.int64)), [0]),
            "user_embedder.weight": np.unique(out["users"])}
    for k, ids in read.items():
        out["rows." + k], out["sd." + k] = ids, sd[k][torch.from_numpy(ids)].numpy()
    return out


def sample_h_rows(out, n, seed):
    """Keep a fixed, seeded sample of n decoder rows [B,L,d] at non-PAD positions: ``h_index`` (sorted flat b*L + position)
    and ``h`` [n,d]."""
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(np.flatnonzero(out["seqs"].reshape(-1) != 0), n, replace=False))
    out["h_index"], out["h"] = idx, out["h"].reshape(-1, out["h"].shape[-1])[idx]
    return out


def irn_cfg3_shape_case(R, name):
    """The BASELINE cfg3 decoder shape: window L=201 (200 history + objective), d=128, 4 heads, ffn 256, SIX layers;
    catalog 6000 items so that the fixture stays small.  Weights = the reference's default initialisers under
    torch.manual_seed(1234) (what bench.py uses at N=1M), stored as ``seeded_weights``.  Full and ragged windows; 320 of
    the 1048 non-PAD decoder rows, all generation-row logits."""
    cfg = irn_config(n_item=6000, n_user=50, max_len=201, n_layers=6, n_heads=4, emb_dim=128, ffn_dim=256)
    g = torch.Generator().manual_seed(21)
    B, L, P = 8, 201, 4
    seqs = prepadded(B, L, cfg.n_item, g, min_len=20, full_rows=3)
    users = torch.randint(0, cfg.n_user, (B,), generator=g)
    torch.manual_seed(1234)
    net = R.IntendedNet(cfg)
    net.eval()
    irn = R.IRSNN(cfg, net, torch.device("cpu"))
    out = dict(sd_arrays(net))
    out.update(cfg=np.array([cfg.n_item, cfg.n_user, cfg.max_len, cfg.n_layers, cfg.n_heads, cfg.emb_dim,
                             cfg.ffn_dim, cfg.u_emb_dim]), seqs=seqs.numpy(), users=users.numpy())
    targets = seqs[:, -1].clone()
    with torch.no_grad():
        h, r = net.decoding(seqs.clone(), users, return_pi=True)          # InfluentialNet.decoding
        logits = net.forward(seqs.clone(), users)                         # InfluentialNet.forward
        out["h"] = h.numpy()                                              # [B,L,d], sampled below
        out["logits_row"] = logits[:, L - 2].numpy()                      # the row generation reads [B,N]
        out["r_u"] = r.numpy()
        out["eval_loss"] = np.array(irn.get_loss_on_eval_data(seqs, users))   # IRSNN.get_loss_on_eval_data
        p, t, hist, ne = irn.get_seq_in_batch(seqs, users, targets, max_path_len=P, gap_len=0)  # IRSNN.get_seq_in_batch
        out["paths"], out["targets"], out["n_early"] = p, t, np.array(ne)
    out = sample_h_rows(seeded_weights(out, 1234), 320, seed=21)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, {k: v.shape for k, v in out.items()})


def evaluator_case(R, name):
    g = torch.Generator().manual_seed(7)
    cfg = SimpleNamespace(n_item=70, max_len=14, n_layers=2, n_heads=2, emb_dim=32, ffn_dim=48, dropout=0.0, lr1=1e-3)
    torch.manual_seed(4321)
    net = R.SampleNet(cfg)
    net.eval()
    ev = R.Evaluator(cfg, net, torch.device("cpu"))
    out = dict(sd_arrays(net))
    out["cfg"] = np.array([cfg.n_item, cfg.max_len, cfg.n_layers, cfg.n_heads, cfg.emb_dim, cfg.ffn_dim])
    B, seq_len = 6, 13
    # histories / paths / targets as pipeline.evaluate_prob builds them (DatasetEvalNN1, data_provider.py:716-754)
    hists, paths, targets = [], [], []
    for b in range(B):
        perm = (torch.randperm(cfg.n_item, generator=g) + 1).numpy()
        nh = [3, 5, 9, 12, 13, 16][b]          # includes histories longer than seq_len
        npth = [2, 4, 3, 5, 4, 3][b]
        hists.append(perm[:nh].astype(np.float64))
        pth = np.zeros(6)
        pth[:npth] = perm[nh:nh + npth]
        tgt = perm[nh + npth + 1]
        if b == 2:                              # early success: the path already contains the target
            pth[npth - 1] = tgt
        paths.append(pth)
        targets.append(int(tgt))
    ds = R.data_provider.DatasetEvalNN1(hists, np.array(paths), np.array(targets), seq_len=seq_len)
    dl = R.data_provider.DataLoaderEvalNN1(dataset=ds, batch_size=B, shuffle=False, num_workers=0)
    histories, new_seqs, tg, start_pos, l_path = next(iter(dl))
    out.update(histories=histories.numpy(), new_seqs=new_seqs.numpy(), targets=tg.numpy(),
               start_pos=start_pos.numpy(), l_path=l_path.numpy())
    with torch.no_grad():
        out["logits_new"] = net.forward(new_seqs[:, :-1]).numpy()                       # SampleNet.forward
        out["pp"] = np.array(ev.get_pp_in_batch(new_seqs, start_pos, l_path))           # Evaluator.get_pp_in_batch
        irr, ir = ev.get_rr_increase_in_batch(histories, new_seqs, tg)                  # Evaluator.get_rr_increase_in_batch
        out["irr"], out["ir"] = irr, ir
        tp, pp_, avg, ioi = ev.get_grad_in_batch(histories.clone(), new_seqs, tg, start_pos, l_path)  # Evaluator.get_grad_in_batch
        out["t_probs"], out["p_probs"], out["avg_ps"], out["iois"] = tp, pp_, np.array(avg), np.array(ioi)
        out["eval_loss"] = np.array(ev.get_loss_on_eval_data(new_seqs))                  # Evaluator.get_loss_on_eval_data
        hit, rr = ev.get_accuracy_metrics_in_batch(new_seqs, top_k=5, use_h=True)        # Evaluator.get_accuracy_metrics_in_batch
        out["acc_hit"], out["acc_rr"] = np.array(hit), rr
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "ok")


def sas_case(R, name):
    g = torch.Generator().manual_seed(11)
    cfg = SimpleNamespace(n_user=9, n_item=90, hidden_units=24, max_len=10, dropout_rate=0.2, num_blocks=2, num_heads=3)
    torch.manual_seed(99)
    net = R.SAS(cfg, torch.device("cpu"))
    net.eval()
    B = 7
    seqs = torch.zeros((B, cfg.max_len), dtype=torch.long)
    for b in range(B):
        n = int(torch.randint(2, cfg.max_len + 1, (1,), generator=g))
        seqs[b, cfg.max_len - n:] = torch.randperm(cfg.n_item, generator=g)[:n] + 1
    rats = (torch.rand((B, cfg.max_len), generator=g) > 0.5).long() * (seqs > 0)
    out = dict(sd_arrays(net))
    out["cfg"] = np.array([cfg.n_item, cfg.hidden_units, cfg.max_len, cfg.num_blocks, cfg.num_heads])
    out["seqs"], out["rats"] = seqs.numpy(), rats.numpy()
    with torch.no_grad():
        out["feats"] = net.log2feats(seqs.numpy(), rats.numpy()).numpy()                 # SAS.log2feats
        out["logits"] = net.predict(np.arange(B), seqs.numpy(), rats.numpy()).numpy()    # SAS.predict
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "ok")


def caser_case(R, name):
    g = torch.Generator().manual_seed(13)
    args = SimpleNamespace(max_len=5, d=16, nh=4, nv=2, drop=0.5, ac_conv="relu", ac_fc="relu")
    n_users, n_items = 8, 75
    torch.manual_seed(77)
    net = R.Caser(n_users, n_items, args)
    net.eval()
    with torch.no_grad():
        net.b2.weight.copy_(torch.randn(net.b2.weight.shape, generator=g) * 0.1)   # b2 is zero-initialised; make it matter
        net.b2.weight[0] = 0
    captured = {}
    net.fc1.register_forward_hook(lambda m, i, o: captured.__setitem__("fc1", o.detach()))
    B = 4
    xs, scores, seqs_all = [], [], []
    items = (torch.arange(n_items) + 1).long()
    with torch.no_grad():
        for b in range(B):
            seq = (torch.randperm(n_items, generator=g)[: args.max_len] + 1).unsqueeze(0)
            rat = (torch.rand((1, args.max_len), generator=g) > 0.5).long()
            user = torch.tensor([[b]])
            s = net(seq, rat, user, items, for_pred=True)                            # Caser.forward(for_pred=True)
            z = torch.relu(captured["fc1"])
            xs.append(torch.cat([z, net.user_embeddings(user).squeeze(1)], 1)[0].numpy())
            scores.append(s.numpy())
            seqs_all.append(seq[0].numpy())
    out = {"W2": net.W2.weight.detach().numpy(), "b2": net.b2.weight.detach().numpy(),
           "x": np.stack(xs), "scores": np.stack(scores), "seqs": np.stack(seqs_all)}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "ok")


def baseline_tails_case(R, name):
    """predict_next of the reference's classical baselines (model/baselines.py: POP :57-71, MC :165-179, FPMC :280-298,
    TransRec :411-428, BPR :527-550) on freshly constructed (random-initialised) models: score -> sort -> +1 ->
    utils.delete_item_in_history(last 50) -> [:top_k].  Inputs (factors / counts / histories) and the reference's preds."""
    import model.baselines as MB
    g = torch.Generator().manual_seed(31)
    n_item, n_user, B, k = 300, 11, 9, 12
    seqs = []
    for b in range(B):
        n = int(torch.randint(1, 71, (1,), generator=g))           # up to 70 > h=50: only the last 50 entries count
        seqs.append((torch.randperm(n_item, generator=g)[:n] + 1).tolist())
    users = torch.randint(0, n_user, (B,), generator=g).tolist()
    Lh = max(len(s) for s in seqs)
    hist = np.zeros((B, Lh), dtype=np.int64)
    for b, s_ in enumerate(seqs):
        hist[b, Lh - len(s_):] = s_
    out = {"hist": hist, "users": np.array(users), "top_k": np.array(k), "n_item": np.array(n_item)}
    base = dict(n_item=n_item, n_user=n_user, lam=0.1, lr=0.01, max_iter=1, earlystop_threshold=1e-3, dataset="x", method="y")
    torch.manual_seed(5)
    pop = MB.POP(n_item)
    pop.train([[int(x) for x in (torch.randint(0, 40, (30,), generator=g) + 1)] for _ in range(40)])   # heavy ties
    out["pop_counts"] = pop.item.numpy().copy()
    out["pop_preds"] = pop.predict_next(seqs, users, top_k=k).numpy()
    mc = MB.MC(SimpleNamespace(K=8, **base))
    out["mc_gam"], out["mc_eta"] = mc.gam.numpy().copy(), mc.eta.numpy().copy()
    out["mc_preds"] = mc.predict_next(seqs, users, top_k=k).numpy()
    fp = MB.FPMC(SimpleNamespace(K1=6, K2=7, **base))
    out["fpmc_gamU"], out["fpmc_gamI"] = fp.gamU.numpy().copy(), fp.gamI.numpy().copy()
    out["fpmc_kap"], out["fpmc_eta"] = fp.kap.numpy().copy(), fp.eta.numpy().copy()
    out["fpmc_preds"] = fp.predict_next(seqs, users, top_k=k).numpy()
    tr = MB.TransRec(SimpleNamespace(K=8, bias_lam=0.1, reg_lam=0.1, **base))
    tr.R = torch.rand(tr.R.shape) - 0.5
    tr.r = torch.rand(tr.r.shape) - 0.5
    tr.beta = torch.rand(tr.beta.shape) - 0.5
    out["tr_H"], out["tr_R"], out["tr_r"], out["tr_beta"] = tr.H.numpy().copy(), tr.R.numpy().copy(), tr.r.numpy().copy(), tr.beta.numpy().copy()
    out["tr_preds"] = tr.predict_next(seqs, users, top_k=k).numpy()
    bpr = MB.BPR(SimpleNamespace(dim=10, weight_decay=0.0, n_epochs=1, batch_size=4, **base))
    with torch.no_grad():
        out["bpr_W"], out["bpr_H"] = bpr.W.numpy().copy(), bpr.H.numpy().copy()
        out["bpr_preds"] = bpr.predict_next(seqs, users, top_k=k).numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "ok")


def collate_case(R, name):
    """DataLoaderEvalIRS._collate_fn (data_provider.py:591-617) and DataLoaderIRS._collate_fn (:568-575) run on ragged
    histories (single-item, longer than the window) for (seq_len, gap_len) in ((60,0),(60,20),(201,0))."""
    rng = np.random.default_rng(3)
    n = 40
    hist = [rng.integers(1, 500, size=int(m)).tolist() for m in rng.integers(1, 90, size=n)]
    hist[0] = hist[0][:1]
    hist[1] = rng.integers(1, 500, size=300).tolist()
    users, targets, labels = rng.integers(0, 50, n), rng.integers(1, 500, n), rng.integers(1, 500, n)
    out = {"hist_flat": np.concatenate([np.asarray(h_, dtype=np.int64) for h_ in hist]),
           "hist_lens": np.array([len(h_) for h_ in hist]), "users": users, "targets": targets, "labels": labels}
    data = [(np.array(hist[i]), int(users[i]), int(targets[i]), int(labels[i])) for i in range(n)]
    for seq_len, gap_len in ((60, 0), (60, 20), (201, 0)):
        rows = rng.permutation(n)[:17]
        dl = R.data_provider.DataLoaderEvalIRS(seq_len, gap_len, dataset=[data[i] for i in rows], batch_size=17,
                                               shuffle=False, num_workers=0)
        raw, seqs, us, tg, lb = next(iter(dl))
        tag = f"L{seq_len}_g{gap_len}"
        out[tag + "_rows"] = rows
        out[tag + "_seqs"], out[tag + "_users"], out[tag + "_targets"], out[tag + "_labels"] = \
            seqs.numpy(), us.numpy(), tg.numpy(), lb.numpy()
        out[tag + "_raw_flat"] = torch.cat(raw).numpy()
        out[tag + "_raw_lens"] = np.array([len(x) for x in raw])
    # train collate on float64 pre-padded windows (the dtype irs_valid_seq.npy stores)
    w = np.zeros((5, 12))
    for b in range(5):
        m = int(rng.integers(2, 13))
        w[b, 12 - m:] = rng.integers(1, 500, size=m)
    ds = R.data_provider.DatasetNN(np.array([[w[b], int(users[b])] for b in range(5)], dtype=object))
    seqs, us = next(iter(R.data_provider.DataLoaderIRS(ds, batch_size=5, shuffle=False, num_workers=0)))
    out["train_windows"], out["train_seqs"], out["train_users"] = w, seqs.numpy(), us.numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "ok")


def get_path_case(R, name):
    """main_baselines.get_path (main_baselines.py:93-121) cannot be imported as a module (it parses argv and imports a
    missing ``params`` module at import time), so the function itself is lifted from the reference source with ast and
    executed unmodified, with the reference's utils.cal_fv_dist and the reference's POP / BPR predict_next as providers."""
    import ast
    import model.baselines as MB
    src = open(os.path.join(R.path, "main_baselines.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "get_path"][0]
    ns = {"np": np, "cal_fv_dist": R.utils.cal_fv_dist}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "main_baselines.get_path", "exec"), ns)
    get_path = ns["get_path"]
    g = torch.Generator().manual_seed(41)
    rng = np.random.default_rng(41)
    n_item, n_user, B, k_c, P = 120, 7, 6, 5, 8
    fv = (rng.random((n_item + 1, 18)) < 0.3).astype(int)                      # binary genre vectors (ml-1m style)
    fv_dict = {i: fv[i] for i in range(1, n_item + 1)}
    seqs = [(torch.randperm(n_item, generator=g)[: int(torch.randint(3, 30, (1,), generator=g))] + 1).numpy() for _ in range(B)]
    users = torch.randint(0, n_user, (B,), generator=g).tolist()
    targets = [int(x) for x in (torch.randint(1, n_item + 1, (B,), generator=g))]
    out = {"fv": fv, "users": np.array(users), "targets": np.array(targets), "k_c": np.array(k_c), "P": np.array(P),
           "seq_flat": np.concatenate(seqs), "seq_lens": np.array([len(x) for x in seqs]), "n_item": np.array(n_item)}
    base = dict(n_item=n_item, n_user=n_user, lr=0.01, earlystop_threshold=1e-3, dataset="x", method="y")
    torch.manual_seed(6)
    bpr = MB.BPR(SimpleNamespace(dim=10, weight_decay=0.0, n_epochs=1, batch_size=4, **base))
    with torch.no_grad():
        out["bpr_W"], out["bpr_H"] = bpr.W.numpy().copy(), bpr.H.numpy().copy()
        # make two users succeed early: their target is one of the first step's candidates (distance 0 to itself)
        first = bpr.predict_next([seqs[0], seqs[1]], users[:2], top_k=k_c)
        targets[0], targets[1] = int(first[0][2]), int(first[1][4])
        out["targets"] = np.array(targets)
        paths, n_succ = get_path([x.copy() for x in seqs], users, targets, bpr, k_c=k_c, max_path_len=P, fv_dict=fv_dict, binary=True)
    out["bpr_paths"], out["bpr_success"] = paths, np.array(n_succ)
    # Euclidean variant (embedding feature vectors, binary=False)
    fv2 = rng.standard_normal((n_item + 1, 6))
    with torch.no_grad():
        paths2, n2 = get_path([x.copy() for x in seqs], users, targets, bpr, k_c=k_c, max_path_len=P,
                              fv_dict={i: fv2[i] for i in range(1, n_item + 1)}, binary=False)
    out["fv_real"], out["bpr_paths_real"], out["bpr_success_real"] = fv2, paths2, np.array(n2)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "ok")


def main():
    R = load_reference()
    assert R is not None, "reference tree not found"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    only = set(sys.argv[1:])            # python oracle/make_golden.py [case ...]; no argument = every case
    if only:
        cases = {"irn_cfg3_shape": lambda: irn_cfg3_shape_case(R, "irn_cfg3_shape"),
                 "baseline_tails": lambda: baseline_tails_case(R, "baseline_tails"),
                 "collate": lambda: collate_case(R, "collate"),
                 "get_path": lambda: get_path_case(R, "get_path")}
        for c in sorted(only):
            cases[c]()
        return

    # --- IRN, tiny synthetic (every row of h / logits kept; train step with gradients)
    g = torch.Generator().manual_seed(1)
    cfg = irn_config(n_item=150, n_user=12, max_len=12, n_layers=2, n_heads=2, emb_dim=32, ffn_dim=64)
    B, L = 6, 12
    seqs = prepadded(B, L, cfg.n_item, g)
    users = torch.randint(0, cfg.n_user, (B,), generator=g)
    raw = [torch.randperm(cfg.n_item, generator=g)[: 5 + b] + 1 for b in range(B)]
    labels = torch.randint(1, cfg.n_item + 1, (B,), generator=g)
    labels[0] = raw[0][0]                          # a label inside the raw history: skipped by the reference
    irn_case(R, "irn_small", cfg, seqs, users, P=6, raw=raw, labels=labels)

    # --- IRN, reference default hyper-parameters (d=30, 6 heads of 5, dropout off), L < max_len
    g = torch.Generator().manual_seed(2)
    cfg = irn_config(n_item=160, n_user=20, max_len=20, n_layers=3, n_heads=6, emb_dim=30, ffn_dim=256)
    seqs = prepadded(5, 16, cfg.n_item, g)
    users = torch.randint(0, cfg.n_user, (5,), generator=g)
    irn_case(R, "irn_d30", cfg, seqs, users, P=4)

    # --- IRN on the shipped MovieLens-1M fixture (cfg1 shape: 3415 items, 6040 users, d=64)
    arr = np.load(os.path.join(R.path, "data", "ml-1m", "irs_valid_seq.npy"), allow_pickle=True)
    Bm = 48
    ds = R.data_provider.DatasetNN(arr[:Bm])
    dl = R.data_provider.DataLoaderIRS(ds, batch_size=Bm, shuffle=False, num_workers=0)
    seqs, users = next(iter(dl))                   # DataLoaderIRS collate (data_provider.py:568-575)
    cfg = irn_config(n_item=3415, n_user=6040, max_len=60, n_layers=2, n_heads=2, emb_dim=64, ffn_dim=128)
    irn_case(R, "irn_ml1m", cfg, seqs, users, P=20, keep_rows=slice(58, 59), train=False, seeded=True)

    evaluator_case(R, "evaluator_small")
    sas_case(R, "sas_small")
    caser_case(R, "caser_small")
    irn_cfg3_shape_case(R, "irn_cfg3_shape")
    baseline_tails_case(R, "baseline_tails")
    collate_case(R, "collate")
    get_path_case(R, "get_path")


if __name__ == "__main__":
    main()
