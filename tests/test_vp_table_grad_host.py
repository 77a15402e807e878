"""CPU: the row exchange that keeps vocab-parallel table replicas identical (enable_vocab_parallel(train_tables=True)),
over gloo at world size 2.

Each rank gives both tables a different local gradient; after backward every rank's .grad must hold, in each row, the
gradient of the rank that owns the row (parallel.shard_bounds), byte-identical on both ranks.  The catalog has an
uneven last shard (300 rows: 256 + 44) and the user table an empty one (100 rows: 100 + 0).  Two backwards before a
step accumulate, and a pickled model carries no hook."""
import os
import pickle
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_ITEMS, N_USERS, D = 300, 100, 8


def _model():
    """A BaseCVAE with its two tables on the CPU (the constructor insists on CUDA; the exchange does not need it)."""
    from torch import nn

    from pivotcvae_b200.models.cvae import BaseCVAE
    m = BaseCVAE.__new__(BaseCVAE)
    nn.Module.__init__(m)
    g = torch.Generator().manual_seed(0)
    m.docEmbed = nn.Embedding(N_ITEMS, D)
    m.userEmbed = nn.Embedding(N_USERS, D)
    with torch.no_grad():
        m.docEmbed.weight.copy_(torch.randn(N_ITEMS, D, generator=g))
        m.userEmbed.weight.copy_(torch.randn(N_USERS, D, generator=g))
    m.noUser = False
    m._table = m._full = m._vp = None
    m._vp_train, m._vp_hooks = False, []
    return m


def _local(rank, step):
    """This rank's own gradients of (docEmbed, userEmbed) in backward `step`: different on every rank."""
    g = torch.Generator().manual_seed(1000 * step + rank)
    return torch.randn(N_ITEMS, D, generator=g), torch.randn(N_USERS, D, generator=g)


def _backward(m, rank, step):
    rd, ru = _local(rank, step)
    ((m.docEmbed.weight * rd).sum() + (m.userEmbed.weight * ru).sum()).backward()


def _owned(world, steps):
    """Expected .grad: row j summed over the steps as its owner computes it."""
    from pivotcvae_b200.parallel import shard_bounds
    out = []
    for k, n in enumerate((N_ITEMS, N_USERS)):
        want = torch.zeros(n, D)
        for r in range(world):
            lo, hi = shard_bounds(n, world, r)
            acc = None
            for s in range(steps):
                x = _local(r, s)[k][lo:hi]
                acc = x if acc is None else acc + x
            want[lo:hi] = acc
        out.append(want)
    return out


def _worker(rank, world, port, tmpdir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from pivotcvae_b200 import _lib as L
    from pivotcvae_b200.parallel import shard_bounds
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    checks = {}
    assert shard_bounds(N_ITEMS, world, 1) == (256, 300) and shard_bounds(N_USERS, world, 1) == (100, 100)
    m = _model()
    try:
        m.enable_vocab_parallel()
        checks["refused"] = False
    except L.PcvError as e:
        checks["refused"] = "fine_tune" in str(e) and "train_tables" in str(e)
    m.enable_vocab_parallel(train_tables=True)
    m.enable_vocab_parallel(train_tables=True)          # a second call replaces the hooks: one exchange per table
    checks["two_hooks"] = len(m._vp_hooks) == 2
    _backward(m, rank, 0)
    want = _owned(world, 1)
    checks["one"] = torch.equal(m.docEmbed.weight.grad, want[0]) and torch.equal(m.userEmbed.weight.grad, want[1])
    torch.save([m.docEmbed.weight.grad.clone(), m.userEmbed.weight.grad.clone()], os.path.join(tmpdir, "g1_%d" % rank))
    _backward(m, rank, 1)                                # accumulates into .grad
    want = _owned(world, 2)
    checks["two"] = torch.equal(m.docEmbed.weight.grad, want[0]) and torch.equal(m.userEmbed.weight.grad, want[1])
    torch.save([m.docEmbed.weight.grad.clone(), m.userEmbed.weight.grad.clone()], os.path.join(tmpdir, "g2_%d" % rank))
    # whole-model pickling drops the vocab-parallel state and the hooks: the reloaded model's backward is local
    m2 = pickle.loads(pickle.dumps(m))
    checks["state"] = m2._vp is None and m2._vp_hooks == [] and not m2._vp_train
    checks["no_hook"] = all(not w._post_accumulate_grad_hooks for w in (m2.docEmbed.weight, m2.userEmbed.weight))
    m2.zero_grad(set_to_none=True)
    _backward(m2, rank, 2)
    rd, ru = _local(rank, 2)
    checks["local"] = torch.equal(m2.docEmbed.weight.grad, rd) and torch.equal(m2.userEmbed.weight.grad, ru)
    torch.save(checks, os.path.join(tmpdir, "ok_%d" % rank))
    dist.barrier()
    dist.destroy_process_group()


def test_vp_table_grad_exchange_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        checks = torch.load(tmp_path / ("ok_%d" % r))
        assert all(checks.values()), (r, checks)
    for tag in ("g1", "g2"):
        a, b = torch.load(tmp_path / (tag + "_0")), torch.load(tmp_path / (tag + "_1"))
        for x, y in zip(a, b):                           # byte-identical replicas
            assert torch.equal(x.view(torch.int32), y.view(torch.int32)), tag
