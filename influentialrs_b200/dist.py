"""Multi-GPU paths (one process per GPU, torch.distributed over NCCL/NVLink; SURVEY.md section 8e).

Generation  -- users are split data-parallel AND the catalog (``project`` rows) is sharded: rank g owns
               item ids [lo_g+1, hi_g].  Per path step every rank decodes its own users, the decoded
               rows are all-gathered (B*d floats per rank), each rank runs the fused arg-max over ITS
               catalog shard for ALL users (window mask applied in-kernel with item_base = lo_g+1; on the
               tensor cores in two phases around a MAX all-reduce of the per-row shard leaders, so that only
               the shard that can hold a row's winner re-scores it exactly), the per-shard (score, item)
               candidates are all-gathered (one collective) and merged by (score desc, item id asc) with
               irs_topk_merge, and every rank shifts every user's window (so windows never have to be
               exchanged again).  Two small collectives per step, three on the tensor cores.
               Sampled generation: every shard sends its k best per row through the same one all-gather and every
               rank draws the pick with irs_topk_sample, a pure function of (seed, step, global row) and of the
               merged list -- the same picks on every rank, and the same as on one GPU, with no further collective.
Scoring     -- ShardedScorer: rank, log-sum-exp and top-k over a row-sharded catalog for data-parallel rows.
Training    -- plain data parallelism: local mean-CE gradients are rescaled by the local/global row
               counts and all-reduced in one flat bucket, so the update equals the single-GPU one.

The reference has only nn.DataParallel (pipeline.py:43-44), which gathers [B,L,N] logits on GPU 0.

The collective plumbing is torch.distributed.  The compute callables default to the dispatching scorer ops of ops.py,
which choose the engine (tcgen05 or fp32 CUDA cores) by the same rules as on one GPU and keep the weight image of each
shard in the same process-wide cache.  They can be injected, which is how tests/test_dist_cpu.py drives the same host
logic on CPU over gloo (ops loads the CUDA library only at the first kernel call).
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import ops


def shard_bounds(n_item: int, rank: int, world: int):
    """Catalog columns [lo, hi) owned by ``rank`` (item ids lo+1 .. hi)."""
    return rank * n_item // world, (rank + 1) * n_item // world


def _all_gather_cat(t: torch.Tensor, world: int, group=None) -> torch.Tensor:
    out = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t.contiguous(), group=group)
    return out


def pack_candidates(vals: torch.Tensor, items: torch.Tensor) -> torch.Tensor:
    """(fp32 scores [..], int64 items [..]) -> int64 [.., 2]: the score's bit pattern rides in the low half of word 0, so that
    both travel in ONE all-gather.  Bit-exact for every float, -inf, -0.0 and NaN payloads included."""
    return torch.stack([vals.contiguous().view(torch.int32).to(torch.int64), items.to(torch.int64)], dim=-1)


def unpack_candidates(packed: torch.Tensor):
    """Inverse of ``pack_candidates``: int64 [.., 2] -> (fp32 [..], int64 [..])."""
    return packed[..., 0].to(torch.int32).view(torch.float32), packed[..., 1].contiguous()


class ShardedGenerator:
    """Catalog-sharded, user-data-parallel influence-path generation (a7 across GPUs).

    Compute callables (injectable): ``decode_fn(windows, users) -> h``; ``score_fn(h_all, windows_all[, k])`` -> (vals,
    items) [G*B, 1] of this shard (the arg-max), or its k best when sampling passes ``k``; ``merge_fn(vals, items)`` ->
    best (vals, items) of the [G, G*B, k] candidates; ``sample_fn(vals, items, seed, step, row_key)`` -> one pick [G*B]
    per row (irs_topk_sample); ``shift_fn(windows_all, nxt_all, paths_local, step, row0, n_local)``."""

    def __init__(self, irn, rank: int, world: int, group=None, decode_fn: Optional[Callable] = None,
                 score_fn: Optional[Callable] = None, merge_fn: Optional[Callable] = None,
                 shift_fn: Optional[Callable] = None, sample_fn: Optional[Callable] = None):
        self.irn, self.rank, self.world, self.group = irn, rank, world, group
        self.n_item = irn.n_item
        self.lo, self.hi = shard_bounds(self.n_item, rank, world)
        W, b = irn.net.project.weight, irn.net.project.bias
        self.W = W.detach()[self.lo:self.hi]            # a deployment loads only these rows
        self.b = b.detach()[self.lo:self.hi]
        self._excl = None                               # sorted exclusion lists of every window for MY catalog shard
        self._all = None                                # every user's window, kept in step on every rank
        self.decode_fn = decode_fn or self._decode_cuda
        self.score_fn = score_fn or self._score_cuda
        self.merge_fn = merge_fn or self._merge_cuda
        self.shift_fn = shift_fn or self._shift_cuda
        self.sample_fn = sample_fn or self._sample_cuda

    # ---- default CUDA operators -------------------------------------------------------------------
    def _decode_cuda(self, windows, users):
        return self.irn.net.decoding(windows, users, last_row=windows.shape[1] - 2)

    def _score_cuda(self, h_all, windows_all, k=None):
        if self._excl is None:          # first step of a generation; afterwards the lists are updated incrementally (step())
            self._excl = ops.sort_exclusions(windows_all[:, :-1], self.hi - self.lo, self.lo + 1)
        if k is not None:               # sampling: the k best of my shard for every row
            return ops.score_topk_any(h_all, self.W, self.b, k, self._excl, self.lo + 1)
        reduce_lead = None if self.world == 1 else (lambda t: dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group))
        return ops.score_argmax(h_all, self.W, self.b, self._excl, self.lo + 1, reduce_lead)

    def _merge_cuda(self, vals, items):
        return ops.topk_merge(vals, items)

    def _sample_cuda(self, vals, items, seed, step, row_key):
        return ops.topk_sample(vals, items, seed, step, row_key)

    def _shift_cuda(self, windows_all, nxt_all, paths_local, step, row0, n_local):
        if self._excl is not None:      # the id that slides out leaves the list, the pick enters (instead of a re-sort)
            ops.exclusions_update(self._excl, windows_all[:, 0], nxt_all, self.hi - self.lo, self.lo + 1)
        ops.window_shift(windows_all, nxt_all, None, 0)
        if paths_local is not None:
            paths_local[:, step] = nxt_all[row0:row0 + n_local].float()

    def invalidate_prepared(self):
        """Forget every cached weight image (after editing project.weight through ``.data``)."""
        ops.invalidate_prepared()

    # ---- one path step ------------------------------------------------------------------------------
    def begin(self, windows_local: torch.Tensor):
        """All-gather the windows once; afterwards every rank advances all of them itself.  Every rank must bring the
        same number of users (all_gather_into_tensor and the row0 = rank*B slicing assume it): a ragged last batch is
        detected here -- one tiny MAX/MIN all-reduce per generation -- instead of hanging or mis-slicing in NCCL.
        ``generate`` pads ragged batches itself."""
        if self.world > 1:
            n = torch.tensor([windows_local.shape[0], -windows_local.shape[0]], dtype=torch.int64, device=windows_local.device)
            dist.all_reduce(n, op=dist.ReduceOp.MAX, group=self.group)
            if int(n[0]) != -int(n[1]):
                raise ValueError(f"ShardedGenerator: ranks hold different numbers of users (max {int(n[0])}, min {-int(n[1])}); "
                                 "pad the last batch (ShardedGenerator.generate does) or drop it")
        self._all = _all_gather_cat(windows_local, self.world, self.group)
        self._excl = None

    def step(self, windows_local, users_local, paths_local, step: int, sample=None):
        """Advance every user by one path position.  ``windows_local`` is updated in place.  ``sample`` = (k, seed,
        row_key [G*B] int64 of every rank's rows) draws each pick from the softmax over the k best of the whole catalog
        (irs_topk_sample on the gathered per-shard lists: every rank computes the same picks) instead of the arg-max."""
        B = windows_local.shape[0]
        if self._all is None or self._all.shape[0] != B * self.world:
            self.begin(windows_local)
        row0 = self.rank * B
        mine = self._all[row0:row0 + B]
        h = self.decode_fn(mine, users_local)                                   # [B,d]
        h_all = _all_gather_cat(h, self.world, self.group)                      # exchange 1
        if sample is None:
            vals, items = self.score_fn(h_all, self._all)                       # [G*B,1] over my shard
        else:
            vals, items = self.score_fn(h_all, self._all, sample[0])            # [G*B,k] over my shard
        # exchange 2: (score, item) of every user from every shard in ONE collective -- the fp32 scores travel as the
        # low halves of int64 words next to the item ids ([G, G*B, k, 2] int64)
        packed_all = _all_gather_cat(pack_candidates(vals, items).unsqueeze(0), self.world, self.group)
        vals_all, items_all = unpack_candidates(packed_all)                     # [G, G*B, k] each
        if sample is None:
            _, best = self.merge_fn(vals_all, items_all)
            nxt_all = best[:, 0].contiguous()
        else:
            nxt_all = self.sample_fn(vals_all, items_all, sample[1], step, sample[2]).contiguous()
        self.shift_fn(self._all, nxt_all, paths_local, step, row0, B)
        windows_local.copy_(self._all[row0:row0 + B])

    def generate(self, seqs_local, users_local, max_path_len=20, sample=None):
        """Paths [B_local, P] of this rank's users.  Ranks may hold different numbers of users (a ragged last batch):
        every rank pads to the largest local batch with copies of its first row (or an all-PAD window when it holds no
        user at all) and the pad rows are dropped from the result.  ``sample`` = (k, seed, first_key): sampled picks,
        rank r's row i drawing with the key first_key[r] + i (a sequence of G ints, the same on every rank)."""
        n_local = seqs_local.shape[0]
        n_max = n_local
        if self.world > 1:
            t = torch.tensor([n_local], dtype=torch.int64, device=seqs_local.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            n_max = int(t.item())
        windows = seqs_local.clone()
        if n_max > n_local:
            fill_w = windows[:1] if n_local > 0 else torch.zeros((1, seqs_local.shape[1]), dtype=seqs_local.dtype, device=seqs_local.device)
            fill_u = users_local[:1] if n_local > 0 else torch.zeros((1,), dtype=users_local.dtype, device=users_local.device)
            windows = torch.cat([windows, fill_w.expand(n_max - n_local, -1)]).contiguous()
            users_local = torch.cat([users_local, fill_u.expand(n_max - n_local)]).contiguous()
        paths = torch.zeros((n_max, max_path_len), dtype=torch.float32, device=seqs_local.device)
        step_sample = None
        if sample is not None:
            k, seed, first_key = sample
            first = torch.tensor(list(first_key), dtype=torch.int64, device=seqs_local.device)
            keys = (first.view(-1, 1) + torch.arange(n_max, dtype=torch.int64, device=seqs_local.device)).reshape(-1)
            step_sample = (k, seed, keys)
        self._all = None
        with torch.no_grad():
            for i in range(max_path_len):
                self.step(windows, users_local, paths, i, step_sample)
        self._all = None
        return paths[:n_local]

    def get_seq_in_batch(self, seqs, users, targets, max_path_len=20, gap_len=0, sample=False, sample_k=3):
        """Same contract as IRSNN.get_seq_in_batch (model/influentialRS.py:392-470) for this rank's users.

        ``sample``: every rank draws one seed from torch's CPU generator (as IRSNN does, so the generators stay in step)
        and rank 0's is used; every row draws with its index in the batch of all ranks together (the ranks' local batches
        in rank order).  So the paths equal those of IRSNN.get_seq_in_batch(sample=True) over that whole batch under the
        same torch seed on rank 0, whatever the number of ranks."""
        if gap_len != 0:
            raise NotImplementedError("sharded generation implements the gap_len=0 path (SURVEY D6)")
        # device tiles of irn.user_tile users per rank (activation memory), the same number of tiles on every rank
        tile = int(getattr(self.irn, "user_tile", 4096))
        n_local = seqs.shape[0]
        n_max = n_local
        if sample:
            # one collective per call: every rank's batch size (-> global row keys) and rank 0's seed
            from .irn import _draw_seed
            mine = torch.tensor([[n_local, _draw_seed()]], dtype=torch.int64, device=seqs.device)
            info = _all_gather_cat(mine, self.world, self.group).cpu() if self.world > 1 else mine.cpu()
            sizes, seed = info[:, 0].tolist(), int(info[0, 1])
            offsets = [sum(sizes[:r]) for r in range(len(sizes))]
            n_max = max(sizes)
        elif self.world > 1:
            t = torch.tensor([n_local], dtype=torch.int64, device=seqs.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            n_max = int(t.item())
        parts = []
        for t0 in range(0, max(n_max, 1), tile):
            tile_sample = (int(sample_k), seed, [o + t0 for o in offsets]) if sample else None
            parts.append(self.generate(seqs[t0:t0 + tile], users[t0:t0 + tile], max_path_len, tile_sample))
        paths = torch.cat(parts).cpu().numpy()
        return trim_paths(paths, targets.detach().cpu().numpy(), seqs[:, :-1].detach().cpu().numpy())


class ShardedScorer:
    """Catalog-sharded scoring for the rank / log-probability / top-k consumers: Evaluator (model/evaluator.py:245-323),
    IRSNN accuracy metrics (model/influentialRS.py:340-390), SASRec / Caser next-item top-k (model/sas.py:357-388,
    model/caser.py:273-299) -- SURVEY 8e row 3.  The reference's only multi-GPU route is nn.DataParallel, which gathers full
    [B,L,N] logits on GPU 0 (pipeline.py:43-44, evaluator_pipeline.py:46-47,137-138).

    Rank g owns catalog rows [lo_g, hi_g) (item ids lo_g+1 .. hi_g); users are data-parallel.  Every call all-gathers the
    callers' local rows (d floats per row + ids), every rank scores ITS shard for ALL rows, and the per-shard results are
    combined exactly:
      rank     label's exact score = MAX over shards of irs_score_select (-inf outside the owning shard);
               rank = 0 if any shard excludes the label else 1 + SUM over shards of irs_score_count_ahead
      lse      log-sum-exp merge of the per-shard lse (mathematically the (max, sum exp) merge); selected logits as above
      top-k    per-shard top-k, one packed all-gather, irs_topk_merge (score desc, id asc)
    Compute callables are injectable (tests/test_dist_cpu.py drives the same host logic on CPU over gloo)."""

    def __init__(self, W, bias, rank: int, world: int, group=None, select_fn=None, count_fn=None, lse_fn=None,
                 topk_fn=None, merge_fn=None):
        self.rank_id, self.world, self.group = rank, world, group
        self.n_item = W.shape[0]
        self.lo, self.hi = shard_bounds(self.n_item, rank, world)
        self.W = W.detach()[self.lo:self.hi]            # a deployment loads only these rows
        self.b = None if bias is None else bias.detach()[self.lo:self.hi]
        self.select_fn = select_fn or self._select_cuda
        self.count_fn = count_fn or self._count_cuda
        self.lse_fn = lse_fn or self._lse_cuda
        self.topk_fn = topk_fn or self._topk_cuda
        self.merge_fn = merge_fn or self._merge_cuda

    # ---- default CUDA operators -------------------------------------------------------------------
    def invalidate_prepared(self):
        """Forget every cached weight image (after editing the catalog weights through ``.data``)."""
        ops.invalidate_prepared()

    def _excl(self, ids_all):
        return None if ids_all is None else ops.sort_exclusions(ids_all, self.hi - self.lo, self.lo + 1)

    def _select_cuda(self, h_all, sel_all):
        return ops.score_select(h_all, self.W, self.b, sel_all, self.lo + 1)

    def _count_cuda(self, h_all, label_all, score_all, ids_all):
        return ops.score_count_ahead(h_all, self.W, self.b, label_all, score_all, self._excl(ids_all), self.lo + 1)

    def _lse_cuda(self, h_all):
        sel0 = torch.zeros((h_all.shape[0], 1), dtype=torch.int64, device=h_all.device)
        return ops.score_lse_gather(h_all, self.W, self.b, sel0, self.lo + 1)[0]

    def _topk_cuda(self, h_all, k, ids_all):
        return ops.score_topk_any(h_all, self.W, self.b, k, self._excl(ids_all), self.lo + 1)

    def _merge_cuda(self, vals, items):
        return ops.topk_merge(vals, items)

    # ---- plumbing ------------------------------------------------------------------------------------
    def _gather_rows(self, *tensors):
        """All-gather row-aligned local tensors (None passes through); ranks may bring different row counts: every rank
        pads to the largest.  Returns (gathered tensors, row slices of this rank inside them, padded local count)."""
        n = tensors[0].shape[0]
        n_max = n
        if self.world > 1:
            t = torch.tensor([n], dtype=torch.int64, device=tensors[0].device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            n_max = int(t.item())
        out = []
        for x in tensors:
            if x is None:
                out.append(None)
                continue
            if n_max > n:
                pad = torch.zeros((n_max - n,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
                x = torch.cat([x, pad])
            out.append(_all_gather_cat(x, self.world, self.group) if self.world > 1 else x.contiguous())
        row0 = self.rank_id * n_max
        return out, slice(row0, row0 + n), n_max

    def any_rank(self, flag: bool, device) -> bool:
        """True on every rank iff ``flag`` is true on at least one: lets a data error be raised by ALL ranks together
        (a rank that raises alone leaves the others waiting in the next collective)."""
        if self.world == 1:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return bool(int(t.item()))

    # ---- the three consumers --------------------------------------------------------------------------
    def rank(self, h, label, excl_ids=None):
        """1-based rank [B] of ``label`` (global item ids) among the non-excluded items, 0 where the label itself is in the
        row's exclusion list ``excl_ids`` [B,Lx] (raw ids, 0 = pad).  Same integers as ops.score_rank over the full catalog."""
        (h_all, lab_all, ids_all), mine, _ = self._gather_rows(h, label.reshape(-1).long(), excl_ids)
        s = self.select_fn(h_all, lab_all.view(-1, 1)).reshape(-1)
        if self.world > 1:
            dist.all_reduce(s, op=dist.ReduceOp.MAX, group=self.group)
        cnt, flag = self.count_fn(h_all, lab_all, s, ids_all)
        both = torch.stack([cnt.to(torch.int64), flag.to(torch.int64)])
        if self.world > 1:
            dist.all_reduce(both, op=dist.ReduceOp.SUM, group=self.group)
        valid = (both[1] == 0) & (lab_all >= 1) & (lab_all <= self.n_item)
        r = torch.where(valid, both[0] + 1, torch.zeros_like(both[0]))
        return r[mine].contiguous()

    def lse_gather(self, h, sel):
        """(lse [B], logit [B,s]) over the full catalog: logit[m,t] = exact score of item sel[m,t] (0.0 for an id outside
        1 .. n_item, PAD included)."""
        sel = sel.reshape(h.shape[0], -1).long()
        (h_all, sel_all), mine, _ = self._gather_rows(h, sel)
        lse_loc = self.lse_fn(h_all)
        logit = self.select_fn(h_all, sel_all)
        if self.world > 1:
            lse_all = _all_gather_cat(lse_loc.unsqueeze(0), self.world, self.group)      # [G, M]
            dist.all_reduce(logit, op=dist.ReduceOp.MAX, group=self.group)
        else:
            lse_all = lse_loc.unsqueeze(0)
        lse = torch.logsumexp(lse_all.double(), dim=0).float()
        # ids outside the catalog (0 = PAD, negative, > n_item) select 0.0, as score_lse_gather does
        logit = torch.where((sel_all < 1) | (sel_all > self.n_item), torch.zeros_like(logit), logit)
        return lse[mine].contiguous(), logit[mine].contiguous()

    def topk(self, h, k: int, excl_ids=None):
        """Best k (score desc, item id asc) per row among non-excluded items of the whole catalog."""
        (h_all, ids_all), mine, _ = self._gather_rows(h, excl_ids)
        vals, items = self.topk_fn(h_all, k, ids_all)
        if self.world > 1:
            packed = _all_gather_cat(pack_candidates(vals, items).unsqueeze(0), self.world, self.group)
            vals_all, items_all = unpack_candidates(packed)
            vals, items = self.merge_fn(vals_all, items_all)
        return vals[mine].contiguous(), items[mine].contiguous()


def trim_paths(paths: np.ndarray, targets: np.ndarray, histories: np.ndarray):
    """Host tail of get_seq_in_batch (model/influentialRS.py:452-470): zero each path after the first
    occurrence of its target, count early successes, strip PAD from the histories."""
    hit = paths == targets[:, None].astype(paths.dtype)
    has = hit.any(1)
    first = hit.argmax(1)
    after = np.arange(paths.shape[1])[None, :] > first[:, None]
    paths[has[:, None] & after] = 0
    keep = histories != 0                                   # one masked gather, then B views of it
    flat = histories[keep]
    ends = np.cumsum(keep.sum(1)).tolist()
    actual = [flat[a:b] for a, b in zip([0] + ends[:-1], ends)]
    return paths, targets, actual, int(has.sum())


def make_data_parallel(irn, group=None):
    """Data-parallel training (cfg4): installs ``irn.grad_sync`` so that IRSNN.train_batch all-reduces
    gradients before the (identical, dense) Adam step on every rank.  The loss is a mean over the
    non-pad rows, so local gradients are weighted by local_rows/global_rows before the sum."""
    params = [p for p in irn.net.parameters() if p.requires_grad]

    def sync():
        rows = torch.tensor([float(getattr(irn, "last_ce_rows", 1))], device=params[0].device)
        total = rows.clone()
        dist.all_reduce(total, group=group)
        scale = (rows / total.clamp_min(1.0)).item()       # total == 0: no rank had a target row, all gradients are zero
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in params]
        flat = torch._utils._flatten_dense_tensors(grads)
        flat.mul_(scale)
        dist.all_reduce(flat, group=group)
        for p, g in zip(params, torch._utils._unflatten_dense_tensors(flat, grads)):
            if p.grad is None:
                p.grad = g.clone()
            else:
                p.grad.copy_(g)

    irn.grad_sync = sync
    return irn
