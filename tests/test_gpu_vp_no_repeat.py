"""-m gpu: the no-repeat slate selection on a vocab-parallel catalog, with G row shards on one device.

Each shard is an ops.Table(W[lo:hi], row_offset=lo) over parallel.shard_bounds; its partials are stacked in shard
order (what the all-gather delivers) and merged.  The result must be bit-identical to the selection over the whole
catalog: the oracle and ops.score_select(..., no_repeat=L)."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from gpu_util import N, T

pytestmark = pytest.mark.gpu

KEY_NONE = -(1 << 63)


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _problem(n_items, B, L, D, G, seed):
    """Unit catalog + slot queries with forced duplicates, all-identical slates and an exact tie across shards."""
    from pivotcvae_b200.parallel import shard_bounds
    rng = np.random.default_rng(seed)
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = rng.standard_normal((B, L, D)).astype(np.float32)
    Q[::3, 1] = Q[::3, 0]
    Q[::3, L - 1] = Q[::3, 0]
    Q[1::7] = Q[1::7, :1]                       # every slot identical: needs the full top-L of the union
    # copies of item 5 in the last shard and (G > 2) a middle one: equal scores, the lowest global index wins
    for g in range(1, G):
        lo, hi = shard_bounds(n_items, G, g)
        W[hi - 1] = W[5]
    Q[2] = 2 * W[5]
    return W, Q.reshape(-1, D)


def _sharded(ops, W, Qf, items, L, G, vals=None):
    from pivotcvae_b200.parallel import shard_bounds
    Wt = T(W)
    keys = []
    for g in range(G):
        lo, hi = shard_bounds(W.shape[0], G, g)
        keys.append(ops.slate_no_repeat_partials(ops.Table(Wt[lo:hi], row_offset=lo), Qf, items, L))
    keys = torch.stack(keys)
    return keys, ops.slate_no_repeat_merge(keys, items.clone(), L, vals=vals)


def _check(ops, W, Qf, L, G, engine="simt"):
    B = Qf.shape[0] // L
    whole = ops.Table(T(W))
    plain_i, plain_v = ops.score_select(whole, T(Qf), "greedy", engine=engine)
    ref_i, ref_v = ops.score_select(whole, T(Qf), "greedy", engine=engine, no_repeat=L)
    oi, ov = oracle.slate_no_repeat(W, Qf, L)
    vals = plain_v.clone()
    keys, idx = _sharded(ops, W, T(Qf), plain_i, L, G, vals=vals)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(vals), ov)
    assert torch.equal(idx, ref_i) and torch.equal(vals, ref_v)
    sl = N(idx).reshape(B, L)
    assert all(len(set(r)) == L for r in sl)
    pl = N(plain_i).reshape(B, L)
    clean = np.array([len(set(r)) == L for r in pl])
    assert (~clean).sum() >= B // 3
    assert np.array_equal(sl[clean], pl[clean])                             # clean slates untouched
    assert np.array_equal(N(vals).reshape(B, L)[clean], N(plain_v).reshape(B, L)[clean])
    k = N(keys).reshape(G, B, L, L)
    assert (k[:, clean] == KEY_NONE).all()                                  # clean slates hold no lists
    return keys, idx


@pytest.mark.parametrize("L", [2, 5, 16])
@pytest.mark.parametrize("D", [8, 16, 64, 128])
@pytest.mark.parametrize("G", [1, 2, 3, 4])
def test_vp_no_repeat_small_last_shard(ops, G, D, L):
    """Shards of 256 rows and (G > 1) a last shard with fewer than L rows."""
    from pivotcvae_b200.parallel import shard_bounds
    tail = max(1, L - 2)
    n_items = 256 * (G - 1) + tail if G > 1 else 700
    W, Qf = _problem(n_items, 40, L, D, G, seed=G * 100 + D + L)
    keys, idx = _check(ops, W, Qf, L, G)
    if G > 1:
        lo, hi = shard_bounds(n_items, G, G - 1)
        assert hi - lo == tail < L
        last = N(keys[G - 1]).reshape(-1, L)
        flagged = (last != KEY_NONE).any(1)
        assert flagged.any() and (last[flagged, tail:] == KEY_NONE).all() and (last[flagged, :tail] != KEY_NONE).all()
    # the exact tie of item 5 and its copies, one per later shard: slate 2 takes them in global index order
    copies = [5] + [shard_bounds(n_items, G, g)[1] - 1 for g in range(1, G)]
    m = min(L, len(copies))
    assert list(N(idx)[2 * L:2 * L + m]) == copies[:m]


@pytest.mark.parametrize("n_items,G,D,L,engine", [(50000, 2, 8, 5, "tcgen05"), (20011, 3, 16, 10, "auto"),
                                                  (9001, 4, 64, 16, "simt"), (6007, 4, 128, 5, "auto")])
def test_vp_no_repeat_many_splits(ops, n_items, G, D, L, engine):
    """Shards large enough for several catalog splits each (the per-shard merge), top-1 from the tc engines."""
    W, Qf = _problem(n_items, 64, L, D, G, seed=n_items + L)
    _check(ops, W, Qf, L, G, engine)


def test_vp_no_repeat_graph_capture(ops):
    """Partials + merge are captured in a CUDA graph; replays equal the eager run and follow new inputs."""
    from pivotcvae_b200.parallel import shard_bounds
    G, L, D, n_items, B = 3, 5, 8, 5000, 96
    W, Qf = _problem(n_items, B, L, D, G, seed=3)
    Wt, whole = T(W), ops.Table(T(W))
    tables = [ops.Table(Wt[lo:hi], row_offset=lo) for lo, hi in (shard_bounds(n_items, G, g) for g in range(G))]
    Qs = T(Qf).clone()
    items = torch.empty(B * L, dtype=torch.int64, device=Qs.device)

    def step():
        items.copy_(ops.score_select(whole, Qs, "greedy", engine="simt", want_val=False)[0])
        keys = torch.stack([ops.slate_no_repeat_partials(t, Qs, items, L) for t in tables])
        return ops.slate_no_repeat_merge(keys, items, L)

    eager = step().clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step()
    items.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    assert np.array_equal(N(out), oracle.slate_no_repeat(W, Qf, L)[0])
    # new queries through the same graph
    Q2 = Qf[::-1].copy()
    Qs.copy_(T(Q2))
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(N(out), oracle.slate_no_repeat(W, Q2, L)[0])


def test_vp_no_repeat_argument_errors(ops):
    from pivotcvae_b200 import _lib as L_
    lib = L_.load()
    W = T(np.eye(8, dtype=np.float32).repeat(32, 0))
    tab = ops.Table(W[128:], row_offset=128)
    B, L = 4, 5
    Q = torch.zeros(B * L, 8, device=W.device)
    items = torch.zeros(B * L, dtype=torch.int64, device=W.device)
    keys = torch.full((2, B * L, L), KEY_NONE, dtype=torch.int64, device=W.device)
    ws = tab.workspace("topk", B * L)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def partials(th=tab.handle, q=p(Q), b=B, l=L, it=p(items), k=p(keys), w=p(ws)):
        return lib.pcv_slate_no_repeat_partials(th, q, b, l, it, k, w, ws.numel(), s)

    def merge(k=p(keys), g=2, b=B, l=L, it=p(items)):
        return lib.pcv_slate_no_repeat_merge(k, g, b, l, it, None, s)

    ERR = -1
    for rc in (partials(l=0), partials(l=17), partials(th=None), partials(q=None), partials(it=None), partials(k=None),
               partials(b=0), partials(b=(1 << 31) // L + 1),
               merge(l=0), merge(l=17), merge(g=0), merge(g=33), merge(k=None), merge(it=None), merge(b=0),
               merge(b=(1 << 31) // L + 1)):
        assert rc == ERR and lib.pcv_last_error()
    assert merge(g=33) == ERR and b"[1, 32]" in lib.pcv_last_error()
    torch.cuda.synchronize()
    with pytest.raises(L_.PcvError):
        ops.slate_no_repeat_merge(keys, items[:-1], L)
    with pytest.raises(L_.PcvError):
        ops.slate_no_repeat_partials(tab, Q[:-1], items[:-1], L)
    # the valid calls still work on these buffers
    assert partials() == 0 and merge() == 0
    torch.cuda.synchronize()
