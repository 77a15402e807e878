"""CPU: the vocab-parallel no-repeat exchange over gloo at world size 2 — a numpy stand-in for the shard partials
(pcv_slate_no_repeat_partials), ONE all-gather, and merge_no_repeat_partials — equals the no-repeat selection over
the unsharded catalog."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pack_keys(vals, idx):
    """numpy restatement of the library's order-preserving (score, global index) int64 key."""
    b = np.ascontiguousarray(vals, dtype=np.float32).view(np.uint32)
    b = np.where(b & np.uint32(0x80000000), ~b, b | np.uint32(0x80000000)).astype(np.uint64)
    k = (b << np.uint64(32)) | (np.uint64(0xffffffff) - idx.astype(np.uint64))
    return (k ^ np.uint64(1 << 63)).view(np.int64)


def _shard_partials(W, lo, hi, Q, items, L):
    """numpy stand-in for pcv_slate_no_repeat_partials on rows [lo, hi): this shard's top-L of every row of the
    slates whose picks hold a duplicate, as keys by row; everything else empty."""
    import oracle
    from pivotcvae_b200.parallel import KEY_NONE
    keys = np.full((Q.shape[0], L), KEY_NONE, dtype=np.int64)
    for b, slate in enumerate(items.reshape(-1, L)):
        if len(set(slate.tolist())) == L:
            continue
        rows = slice(b * L, (b + 1) * L)
        ti, tv = oracle.score_topk(W[lo:hi], Q[rows], L)
        n = ti.shape[1]
        keys[rows, :n] = _pack_keys(tv, ti + lo)
    return torch.from_numpy(keys)


def _worker(rank, world, port, tmpdir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import oracle
    from pivotcvae_b200.parallel import no_repeat_exchange, shard_bounds
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(13)          # identical on every rank (replicated inputs)
    n_items, B, L, D = 1000, 30, 5, 8
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    W[900] = W[100]                          # exact tie across the two shards: the lower global index goes first
    Q = rng.standard_normal((B, L, D)).astype(np.float32)
    Q[::3, 1] = Q[::3, 0]                    # duplicated picks
    Q[1::7] = Q[1::7, :1]                    # every slot identical: the full top-L of the union
    Q[2] = W[100]
    Q = Q.reshape(-1, D)
    lo, hi = shard_bounds(n_items, world, rank)
    items = torch.from_numpy(oracle.score_select(W, Q)[0])     # global top-1, as the sharded select delivers it
    out = no_repeat_exchange(lambda it: _shard_partials(W, lo, hi, Q, it.numpy(), L), items.clone(), L)
    want = oracle.slate_no_repeat(W, Q, L)[0]
    ok = (np.array_equal(out.numpy(), want) and list(out.numpy()[2 * L:2 * L + 2]) == [100, 900]
          and not np.array_equal(items.numpy(), want))
    open(os.path.join(tmpdir, "nr_ok%d" % rank), "w").write("1" if ok else "0")
    dist.barrier()
    dist.destroy_process_group()


def test_vp_no_repeat_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "nr_ok0").read_text() == "1" and (tmp_path / "nr_ok1").read_text() == "1"
