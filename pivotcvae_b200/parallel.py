"""Multi-GPU plumbing for the slate-generation path (SURVEY §8e).

Two ways the path shards, both one process per GPU over torch.distributed:

* batch data-parallel — rows are independent, the (<= 320 MB) table is replicated,
  inference needs NO collective (bench.py --gpus N, weak scaling);
* vocab-parallel — each rank owns a contiguous, 128-aligned row range of the item
  table; every rank runs the tiny MLPs redundantly on identical inputs/noise, the
  fused score+select runs on the local shard, and ONE small collective per scoring
  step merges the per-row partial winners (val f32, global idx) with the reference's
  tie rule (largest value, equal values -> lowest global index): on GPUs an
  all-reduce(MAX) of order-preserving int64 keys, on the gloo test path an
  all-gather + merge.  The opt-in no-repeat selection adds one all-gather of
  every shard's top-L lists for the slates whose picks repeat an item
  (no_repeat_exchange).

The host logic here is backend-agnostic so that the gloo/CPU tests can exercise the
exchange + merge with a stand-in local scorer.
"""
import torch
import torch.distributed as dist

SHARD_ALIGN = 128  # the tensor-core select's TMA tiles stay aligned across shards


def shard_stride(n_rows, world, align=SHARD_ALIGN):
    """Rows per shard of shard_bounds (the last shard may be shorter, or empty)."""
    per = -(-n_rows // world)
    return -(-per // align) * align


def shard_bounds(n_rows, world, rank, align=SHARD_ALIGN):
    """Contiguous [lo, hi) row range of `rank`; every boundary but the last is a multiple of align."""
    per = shard_stride(n_rows, world, align)
    lo = min(rank * per, n_rows)
    hi = min(lo + per, n_rows)
    return lo, hi


def merge_partials(vals, idx):
    """vals/idx: [G, M] partial winners in shard order (torch tensors, any device).
    Winner = largest value, equal values -> lowest global index.  Pure torch: the merge of the
    backend-agnostic all-gather path (gloo / CPU tests); CUDA partials merge by all-reduce(MAX) of packed keys."""
    G, M = vals.shape
    best_v, best_i = vals[0].clone(), idx[0].clone()
    for g in range(1, G):
        take = (vals[g] > best_v) | ((vals[g] == best_v) & (idx[g] < best_i))
        best_v = torch.where(take, vals[g], best_v)
        best_i = torch.where(take, idx[g], best_i)
    return best_i, best_v


def all_gather_rows(t, group=None):
    """[rows/world, C] on every rank -> [rows, C] in rank order (one NCCL all-gather, capturable in a CUDA graph)."""
    world = dist.get_world_size(group)
    t = t.contiguous()
    out = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t, group=group)
    return out


def exchange_owned_rows(t, group=None):
    """In place on `t` ([N, C], the same shape on every rank): rows shard_bounds(N, world, rank) of each rank replace
    every other rank's copy of them, so that `t` ends byte-identical on every rank.  ONE all-gather through a padded
    [world * stride, C] buffer (the last shard may be short or empty); capturable in a CUDA graph with NCCL, and it
    runs over gloo too.

    Vocab-parallel table training: a rank's table gradient is exact on the rows it owns only (the catalog
    cross-entropy's term is computed there alone), and the MLP gathers' scatter-add runs with atomics, so the
    replicas' Adam steps stay identical only after this exchange."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n = t.shape[0]
    per = shard_stride(n, world)
    lo, hi = shard_bounds(n, world, rank)
    send = t.new_zeros((per,) + tuple(t.shape[1:]))
    send[:hi - lo] = t[lo:hi]
    out = t.new_empty((world * per,) + tuple(t.shape[1:]))
    dist.all_gather_into_tensor(out, send, group=group)
    t.copy_(out[:n])


def merge_ce_partials(recs, W_full, Q, targets):
    """recs: [G, M, 2 + D] shard records {m, l, acc[D]} (see include/pcv_b200.h pcv_ce_partials).
    -> (loss_rows[M], lse[M], dq[M, D]).  Pure torch restatement of pcv_ce_vp_merge for the CPU / gloo tests."""
    m, l, acc = recs[..., 0], recs[..., 1], recs[..., 2:]
    mx = m.max(0).values
    w = torch.exp(m - mx)
    Lsum = (l * w).sum(0)
    lse = mx + torch.log(Lsum)
    wt = W_full[targets]
    xt = (Q * wt).sum(1)
    dq = (acc * w.unsqueeze(-1)).sum(0) / Lsum.unsqueeze(1) - wt
    return lse - xt, lse, dq


def local_ce_partials(W_shard, Q):
    """Torch stand-in of pcv_ce_partials for one row shard (CPU tests of the exchange): {m, l, acc[D]}."""
    x = Q @ W_shard.t()
    m = x.max(1).values
    e = torch.exp(x - m.unsqueeze(1))
    return torch.cat([m.unsqueeze(1), e.sum(1, keepdim=True), e @ W_shard], 1)


class VocabParallelSelector:
    """score+select over a catalog sharded across the ranks of `group`.

    local_select(Q) -> (idx_global int64[M], val f32[M]) scores the local shard; on a B200 it is
    ops.score_select on a Table built with row_offset=lo."""

    def __init__(self, local_select, group=None):
        self.local_select = local_select
        self.group = group

    def __call__(self, Q):
        idx, val = self.local_select(Q)
        world = dist.get_world_size(self.group)
        if world == 1:
            return idx, val
        if val.is_cuda:
            # ONE collective per scoring step and nothing else: (val, idx) -> order-preserving int64 key,
            # all-reduce(MAX) over NVLink (in-switch where NCCL picks NVLS), key -> (idx, val).  Capturable
            # in the step's CUDA graph.
            from . import ops
            keys = ops.vp_pack_keys(val, idx)
            dist.all_reduce(keys, op=dist.ReduceOp.MAX, group=self.group)
            return ops.vp_unpack_keys(keys)
        M = idx.shape[0]
        # backend-agnostic path (gloo / CPU tests): all-gather of (val, idx) packed in one int64 buffer + merge
        packed = torch.empty(2, M, dtype=torch.int64, device=idx.device)
        packed[0] = val.view(torch.int32).to(torch.int64)
        packed[1] = idx
        flat = torch.empty(world * 2, M, dtype=torch.int64, device=idx.device)
        dist.all_gather_into_tensor(flat, packed, group=self.group)
        out = flat.view(world, 2, M)
        vals = out[:, 0].to(torch.int32).view(torch.float32)
        idxs = out[:, 1].contiguous()
        return merge_partials(vals.contiguous(), idxs)


def no_repeat_exchange(local_partials, items, L, group=None, merge=None):
    """Vocab-parallel no-repeat selection, in place on `items` ([B*L] global top-1 picks, identical on every rank).

    local_partials(items) -> int64 [B*L, L] this rank's shard lists (ops.slate_no_repeat_partials on a B200).  ONE
    all-gather of them (B*L*L*8 bytes per rank, capturable in a CUDA graph), then every rank runs the same merge:
    ops.slate_no_repeat_merge on CUDA tensors, merge_no_repeat_partials otherwise."""
    keys = local_partials(items).contiguous()
    world = dist.get_world_size(group)
    gathered = torch.empty((world * keys.shape[0], keys.shape[1]), dtype=keys.dtype, device=keys.device)
    dist.all_gather_into_tensor(gathered, keys, group=group)
    if merge is None:
        if keys.is_cuda:
            from . import ops
            merge = ops.slate_no_repeat_merge
        else:
            merge = merge_no_repeat_partials
    return merge(gathered.view(world, keys.shape[0], keys.shape[1]), items, L)


KEY_NONE = -(1 << 63)   # empty entry of a shard list (include/pcv_b200.h pcv_slate_no_repeat_partials)


def merge_no_repeat_partials(keys, items, L):
    """keys: [G, B*L, L] shard lists of order-preserving int64 keys (larger key = larger score, equal scores -> lower
    global index; index = 0xffffffff - low 32 bits).  In place on `items`: every slate holding a duplicate is
    re-selected slot by slot, slot l taking its best item slots 0..l-1 have not taken.  Pure torch restatement of
    pcv_slate_no_repeat_merge for the CPU / gloo tests."""
    G, M, _ = keys.shape
    sl = items.view(-1, L)
    for b in range(sl.shape[0]):
        if len(set(sl[b].tolist())) == L:
            continue
        taken = []
        for l in range(L):
            cand = keys[:, b * L + l].reshape(-1)
            cand = cand[cand != KEY_NONE].sort(descending=True).values
            for k in cand.tolist():
                j = 0xffffffff - (k & 0xffffffff)
                if j not in taken:
                    taken.append(j)
                    sl[b, l] = j
                    break
    return items


def shard_table(ops, weight, group=None):
    """Build the local ops.Table for this rank's shard of `weight` ([N, D] on this rank's GPU)."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, hi = shard_bounds(weight.shape[0], world, rank)
    return ops.Table(weight[lo:hi].contiguous(), row_offset=lo), lo, hi
