"""-m gpu: the item-table gradient on a vocab-parallel catalog (row shards of pcv_ce_table_grad and
pcv_cand_ce_table_grad), and table training behind enable_vocab_parallel(train_tables=True).

1. G row shards (parallel.shard_bounds, G = 2, 3, 5) on one device, each with the whole catalog's lse, concatenated in
   shard order == the whole-table gradient: bit for bit on the tf32 path, and on the exact pass where both plans cut
   the query rows the same way (elsewhere, and for the Philox mask and candidates, within the error model of
   test_gpu_table_grad.py).  Every mode is also checked against its float64 autograd reference on the shard's rows.
   N = 1025, 5000, 100003 (and 262144 for the exact pass) give short last shards, shards straddling 1024-column
   Philox blocks and very small shards.
2. Argument errors.
3. The model: the opt-in guard; a world-size-1 NCCL group trains eagerly and through GraphedTrainStep exactly as the
   model without vocab-parallel; candidate mode runs on a vocab-parallel model with frozen tables.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

import oracle
from gpu_util import T
from test_gpu_table_grad import U, _bound, _check, _problem, _ref, _unpack

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _bounds(n_items, G):
    from pivotcvae_b200.parallel import shard_bounds
    return [b for b in (shard_bounds(n_items, G, g) for g in range(G)) if b[1] > b[0]]


def _rows_per_split(n_rows, M):
    """The exact pass's row split (csrc/ce.cu tg_plan): equal splits sum every item's rows in the same order."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    item_ctas, row_tiles = -(-n_rows // 128), -(-M // 32)
    ns = max(1, min(-(-(4 * sm) // item_ctas), 64, row_tiles))
    return -(-row_tiles // ns)


def _cols(bitmask, lo, hi):
    return None if bitmask is None else bitmask[:, lo // 32:-(-hi // 32)]


@pytest.mark.parametrize("mode", ["dense", "bitmask"])
@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
@pytest.mark.parametrize("n_items", [1025, 5000, 100003, 262144])
def test_shards_exact(ops, mode, D, n_items):
    M = 200
    W, Q, tg, rs = _problem(n_items, M, D, 31 * D + n_items, rep_targets=True)
    keep_prob, bm, keep = 1.0, None, None
    if mode == "bitmask":
        rng = np.random.default_rng(D + n_items)
        kb = rng.random((M, n_items)) < 0.1
        kb[:3] = False                                   # rows where only the target is kept
        bm, keep, keep_prob = T(oracle.pack_bitmask(kb).view(np.int32)), torch.from_numpy(kb).cuda(), 0.1
    whole = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(whole, Q, tg, keep_prob, bitmask=bm, want_dq=False)
    full = ops.ce_table_grad(whole, Q, tg, lse, rs, keep_prob, bitmask=bm)
    want, S = _ref(W, Q, tg, rs, keep)
    bound = _bound(S, M)
    same_plans = 0
    for G in (2, 3, 5):
        parts = []
        for lo, hi in _bounds(n_items, G):
            sh = ops.Table(W[lo:hi], row_offset=lo)
            dW = ops.ce_shard_table_grad(sh, Q, tg, lse, rs, keep_prob, bitmask=_cols(bm, lo, hi))
            if _rows_per_split(hi - lo, M) == _rows_per_split(n_items, M):
                assert torch.equal(dW, full[lo:hi]), (G, lo, hi)
                same_plans += 1
            _check("%s D=%d G=%d [%d, %d)" % (mode, D, G, lo, hi), dW, want[lo:hi], bound[lo:hi])
            parts.append(dW)
        assert torch.cat(parts).shape == full.shape
    if n_items == 262144:
        assert same_plans >= 2          # G = 2: both shards and the whole table have a single row split
    _check("%s D=%d whole" % (mode, D), full, want, bound)


@pytest.mark.parametrize("D", [8, 16, 32, 64, 128])
@pytest.mark.parametrize("n_items", [1025, 5000, 100003])
def test_shards_tf32(ops, D, n_items):
    """A shard's 128-item slabs are the whole table's: every row is the whole table's, bit for bit.  The float64
    bound is that of test_gpu_table_grad.py test_table_grad_tf32_engine."""
    M = 130
    W, Q, tg, rs = _problem(n_items, M, D, 7 * D + n_items, rep_targets=True)
    whole = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(whole, Q, tg, 1.0, want_dq=False, engine="tf32")
    full = ops.ce_table_grad(whole, Q, tg, lse, rs, 1.0, engine="tf32")
    want, _ = _ref(W, Q, tg, rs)
    with torch.no_grad():
        X = Q.double() @ W.double().t()
        lse64 = torch.logsumexp(X, 1)
        p = torch.exp(X - lse64[:, None])
        p[torch.arange(M), tg] += 1.0
        rel = (torch.expm1(2.0 ** -9 * Q.double().norm(dim=1)) + (lse.double() - lse64).abs() + 2.0 ** -9 + 2e-5
               + 2 * M * U)
        S = (p * (rs.double().abs() * rel)[:, None]).t() @ Q.double().abs()
    for G in (2, 3, 5):
        for lo, hi in _bounds(n_items, G):
            dW = ops.ce_shard_table_grad(ops.Table(W[lo:hi], row_offset=lo), Q, tg, lse, rs, 1.0, engine="tf32")
            assert torch.equal(dW, full[lo:hi]), (G, lo, hi)
            _check("tf32 D=%d G=%d [%d, %d)" % (D, G, lo, hi), dW, want[lo:hi], 2 * S[lo:hi] + 1e-30)


@pytest.mark.parametrize("D", [4, 8, 32, 128])
@pytest.mark.parametrize("n_items,keep", [(1025, 0.5), (5000, 0.1), (100003, 0.025)])
def test_shards_philox(ops, D, n_items, keep):
    """Each shard walks only the 1024-column blocks it overlaps and keeps exactly the forward's columns there."""
    M = 64
    W, Q, tg, rs = _problem(n_items, M, D, 13 * D + n_items, rep_targets=True)
    tg[M - 8:] = torch.arange(8, device="cuda") * (n_items // 8)     # targets spread over every shard
    whole = ops.Table(W)
    seed, off = 77 + D, 3
    _, lse, _ = ops.ce_fwd_bwd(whole, Q, tg, keep, seed=seed, offset=off, want_dq=False)
    full = ops.ce_table_grad(whole, Q, tg, lse, rs, keep, seed=seed, offset=off)
    want, S = _ref(W, Q, tg, rs, _unpack(oracle.bernoulli_bitmask(seed, off, M, n_items, keep), n_items))
    bound = _bound(S, M)
    for G in (2, 3, 5):
        parts = []
        for lo, hi in _bounds(n_items, G):
            dW = ops.ce_shard_table_grad(ops.Table(W[lo:hi], row_offset=lo), Q, tg, lse, rs, keep, seed=seed, offset=off)
            _check("philox D=%d G=%d [%d, %d)" % (D, G, lo, hi), dW, want[lo:hi], bound[lo:hi])
            parts.append(dW)
        cat = torch.cat(parts)
        assert torch.equal((cat != 0).any(1), (full != 0).any(1)), G
        _check("philox D=%d G=%d vs whole" % (D, G), cat, full.double(), 2 * bound)


@pytest.mark.parametrize("D", [4, 8, 32, 128])
@pytest.mark.parametrize("n_items", [1025, 5000, 100003])
def test_shards_candidates(ops, D, n_items):
    import torch.nn.functional as F
    M, nC = 70, 100
    W, Q, _, rs = _problem(n_items, M, D, 19 * D + n_items)
    g = torch.Generator(device="cuda").manual_seed(D + n_items)
    cand = torch.randint(0, n_items, (M, nC), device="cuda", generator=g)
    cand[:, 1] = cand[:, 0]                                     # duplicates within a row
    cand[:, 2] = n_items - 1                                    # the last (short) shard's last row
    tpos = torch.randint(0, nC, (M,), device="cuda", generator=g)
    whole = ops.Table(W)
    _, lse, _, _ = ops.cand_ce_fwd_bwd(whole, Q, cand, tpos, want_dq=False)
    full = ops.cand_ce_table_grad(whole, Q, cand, tpos, lse, rs)
    W64 = W.double().requires_grad_()
    X = torch.bmm(W64[cand], Q.double()[:, :, None]).squeeze(2)
    (F.cross_entropy(X, tpos, reduction="none") * rs.double()).sum().backward()
    with torch.no_grad():
        P = torch.softmax(X, 1)
        P[torch.arange(M), tpos] += 1.0
        S = torch.zeros_like(W64).index_add_(0, cand.reshape(-1),
                                             ((P * rs.double().abs()[:, None])[:, :, None] * Q.double().abs()[:, None, :])
                                             .reshape(-1, D))
    bound = 2 * (2e-5 + (M * nC) * U) * S + 1e-30            # test_gpu_table_grad.py test_cand_table_grad
    for G in (2, 3, 5):
        parts = []
        for lo, hi in _bounds(n_items, G):
            dW = ops.cand_ce_table_grad(ops.Table(W[lo:hi], row_offset=lo), Q, cand, tpos, lse, rs)
            _check("cand D=%d G=%d [%d, %d)" % (D, G, lo, hi), dW, W64.grad[lo:hi], bound[lo:hi])
            parts.append(dW)
        cat = torch.cat(parts)
        assert torch.equal((cat != 0).any(1), (full != 0).any(1)), G
        _check("cand D=%d G=%d vs whole" % (D, G), cat, full.double(), 2 * bound)


def test_shard_argument_errors(ops):
    """Row shards at the C ABI: row_offset must be a multiple of 128 (the 32-item mask words and 128-item tf32 slabs
    stay aligned with the whole table's), PCV_ERR_ARG otherwise; tf32 at D = 4 stays PCV_ERR_UNSUPPORTED on a shard."""
    from pivotcvae_b200 import _lib as L
    lib = L.load()
    p = ops._ptr
    W, Q, tg, rs = _problem(500, 16, 8, 3)
    _, lse, _ = ops.ce_fwd_bwd(ops.Table(W), Q, tg, 1.0, want_dq=False)
    mask = L.CeMask(1.0)
    cand = torch.randint(0, 500, (16, 4), device="cuda")
    tp = torch.zeros(16, dtype=torch.int64, device="cuda")
    bad = ops.Table(W[64:], row_offset=64)
    dWb = torch.zeros(bad.n_rows, 8, device="cuda")
    wsb = bad.workspace("ce_tgrad", 16)
    assert lib.pcv_ce_table_grad(bad.handle, p(Q), p(tg), 16, ctypes.byref(mask), p(lse), p(rs), p(dWb), p(wsb),
                                 wsb.numel(), None) == -1
    assert b"128" in lib.pcv_last_error()
    assert lib.pcv_cand_ce_table_grad(bad.handle, p(Q), p(cand), p(tp), 16, 4, p(lse), p(rs), p(dWb), None) == -1
    assert b"128" in lib.pcv_last_error()
    good = ops.Table(W[128:], row_offset=128)
    assert ops.ce_shard_table_grad(good, Q, tg, lse, rs, 1.0).shape == (372, 8)
    assert ops.cand_ce_table_grad(good, Q, cand, tp, lse, rs).shape == (372, 8)
    with pytest.raises(L.PcvError, match="ce_shard_table_grad"):      # the whole-table wrapper names the shard one
        ops.ce_table_grad(good, Q, tg, lse, rs, 1.0)
    with pytest.raises(L.PcvError, match="n_rows, dim"):              # `out` must be the shard's rows
        ops.ce_shard_table_grad(good, Q, tg, lse, rs, 1.0, out=torch.empty(500, 8, device="cuda"))
    W4, Q4, tg4, rs4 = _problem(500, 16, 4, 4)
    shard4 = ops.Table(W4[128:], row_offset=128)
    m4 = L.CeMask(1.0)
    m4.engine = 1
    d4 = torch.zeros(shard4.n_rows, 4, device="cuda")
    ws4 = shard4.workspace("ce_tgrad", 16)
    assert lib.pcv_ce_table_grad(shard4.handle, p(Q4), p(tg4), 16, ctypes.byref(m4), p(lse), p(rs4), p(d4), p(ws4),
                                 ws4.numel(), None) == -5


# ============================================================ model level
def test_vp_train_tables_opt_in(golden):
    from pivotcvae_b200 import _lib as L
    from test_gpu_table_grad import _build_list
    m = _build_list(golden("list_small_user"))
    with pytest.raises(L.PcvError, match="fine_tune.*train_tables"):
        m.enable_vocab_parallel()


def _worker(rank, port, out):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        torch.save(_world1_checks(), out)
    finally:
        dist.destroy_process_group()


def _world1_checks():
    """{name: (ok, detail)}: vocab-parallel over a world-size-1 NCCL group against the same model without it."""
    from test_gpu_table_refresh import _batch, _list_model

    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.train_generative import get_gen_loss
    n_items, n_users, B, L = 3001, 40, 64, 5
    M = B * L
    res = {}

    def build(vp, engine, fine_tune=True):
        m = _list_model(8, n_items, n_users, 21, engine)
        if not fine_tune:
            for w in m.trainable_tables():
                w.requires_grad_(False)
        if vp:
            m.enable_vocab_parallel(train_tables=fine_tune)
        m.noise.reseed(99)
        return m

    def close(a, b, rtol, atol):
        return bool(torch.allclose(a, b, rtol=rtol, atol=atol)), float((a - b).abs().max())

    batch = _batch(5, n_items, n_users, B)
    g = torch.Generator(device="cuda").manual_seed(8)
    nC = 50
    cand = torch.randint(0, n_items, (M, nC), device="cuda", generator=g)
    tpos = torch.randint(0, nC, (M,), device="cuda", generator=g)
    cand[torch.arange(M), tpos] = batch["slates"].reshape(-1)
    bits = (torch.rand(M, -(-n_items // 32) * 32, device="cuda", generator=g) < 0.1).cpu().numpy()
    bitmask = T(oracle.pack_bitmask(bits[:, :n_items]).view(np.int32))
    modes = {"exact": ("exact", n_items), "tf32": ("tf32", n_items), "bitmask": ("exact", 300),
             "philox": ("exact", 300), "candidate": ("exact", n_items)}
    for mode, (engine, n_neg) in modes.items():
        for fine_tune in ((True, False) if mode == "candidate" else (True,)):
            tag = mode + ("" if fine_tune else " frozen")
            losses, grads = [], []
            for vp in (False, True):
                m = build(vp, engine, fine_tune)
                opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2)
                bt = dict(batch, sample_candidates=cand, sample_targets=tpos) if mode == "candidate" else batch
                m.candidateFlag = mode == "candidate"
                ls = []
                for step in range(3):
                    if mode == "bitmask":
                        m.noise.push("mask", bitmask)
                    opt.zero_grad(set_to_none=True)
                    loss, _, _ = get_gen_loss(bt, m, None, 0.01, n_neg=n_neg)
                    loss.backward()
                    if step == 0:
                        grads.append({k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None})
                    opt.step()
                    ls.append(float(loss))
                losses.append(ls)
            l0, l1 = losses
            res[tag + " loss"] = (abs(l0[0] - l1[0]) <= 1e-5 * abs(l0[0]), (l0[0], l1[0]))
            res[tag + " steps"] = (all(abs(a - b) <= 1e-4 * abs(a) for a, b in zip(l0, l1)), (l0, l1))
            res[tag + " grad names"] = (sorted(grads[0]) == sorted(grads[1]), sorted(grads[1]))
            for k in grads[0]:
                res[tag + " grad " + k] = close(grads[1][k], grads[0][k], 1e-3, 1e-6)
    # GraphedTrainStep(train_tables=True): the shard handle (and the full one in masked mode) refreshed per replay
    for mode, (engine, n_neg) in (("exact", ("exact", n_items)), ("tf32", ("tf32", n_items)),
                                  ("philox", ("exact", 300))):
        losses, params = [], []
        for vp in (False, True):
            m = build(vp, engine)
            opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2, capturable=True)
            step = GraphedTrainStep(m, opt, B, 0.01, n_neg, train_tables=True)
            if vp:
                res["graph %s handles" % mode] = (step._table is m.item_table() and step._table.row_offset == 0 and
                                                  (step._full is not None) == (n_neg < n_items), None)
            losses.append([float(step(batch)[0]) for _ in range(3)])
            params.append({k: p.detach().clone() for k, p in m.named_parameters()})
        l0, l1 = losses
        res["graph %s steps" % mode] = (all(abs(a - b) <= 1e-4 * abs(a) for a, b in zip(l0, l1)), (l0, l1))
        for k in params[0]:
            res["graph %s param %s" % (mode, k)] = close(params[1][k], params[0][k], 1e-3, 1e-4)
    return res


def test_vp_train_tables_world1(tmp_path):
    import torch.multiprocessing as mp
    port = 35500 + (os.getpid() % 2000)
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(port, out), nprocs=1, join=True)
    res = torch.load(out)
    bad = {k: v for k, v in res.items() if not v[0]}
    assert not bad, bad
    assert "candidate frozen loss" in res and "graph philox steps" in res
