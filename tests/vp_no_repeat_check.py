"""Vocab-parallel no-repeat slates on N GPUs == single-GPU no-repeat slates, bit for bit (run under torchrun on a
multi-GPU box):
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/vp_no_repeat_check.py

PivotCVAE (gt_pi, gt_spi) and ListCVAE with model.no_repeat = True, in three settings: parity-mode eps (MLP rows
unsharded), Philox noise with the MLP rows sharded, and a GraphedSlateGenerator replay.  A tiny last slate-completion
layer makes the slot queries nearly identical, so the plain top-1 picks really repeat items.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_ITEMS, N_USERS, L, D, Z, B = 5000, 300, 5, 8, 16, 256


def make_model(kind, env, dev):
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    from pivotcvae_b200.models.pivotcvae import PIVOTCVAE_MODELS
    torch.manual_seed(1)
    if kind == "listcvae":
        m = UserListCVAEWithPrior(env.docEmbed, env.userEmbed, L, D, Z, L + 1, [L * D + L + 1 + D, 64, 64],
                                  [Z + L + 1 + D, 64, 64, L * D], [L + 1 + D, 32, 32], False, dev)
        last, n_slots = m.dec_3, L
    else:
        m = PIVOTCVAE_MODELS[kind](env.docEmbed, env.userEmbed, L, D, Z, L + 1, [54, 64, 64], [30, 64, 8],
                                   [38, 64, 32], [14, 32, 32], False, dev)
        last, n_slots = m.scm_2, L - 1
    with torch.no_grad():   # every slot query (nearly) the same direction -> duplicated top-1 picks
        last.weight.mul_(1e-3)
        v = torch.randn(D, generator=torch.Generator().manual_seed(7)).to(dev)
        last.bias.copy_(v.repeat(n_slots))
    m.no_repeat = True
    return m


def dup_slates(items):
    return sum(len(set(r)) < L for r in items.reshape(-1, L).tolist())


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    from pivotcvae_b200.env.response_model import UserResponseModel_MLP
    from pivotcvae_b200.graphs import GraphedSlateGenerator
    dev = "cuda:%d" % torch.cuda.current_device()
    torch.manual_seed(0)
    env = UserResponseModel_MLP(N_ITEMS - 1, N_USERS - 1, D, L, [48, 64, 5], dev, False).to(dev)
    g = torch.Generator().manual_seed(3)
    users = torch.randint(0, N_USERS, (B,), generator=g).to(dev)
    ctx = torch.randint(0, 2, (B, L), generator=g).float().to(dev)
    eps = torch.randn(B, Z, generator=g).to(dev)
    ok = True

    def report(what, single, sharded):
        nonlocal ok
        same = np.array_equal(single, sharded)
        clean = dup_slates(sharded) == 0 and dup_slates(single) == 0
        ok = ok and same and clean
        if rank == 0:
            print("no_repeat vocab-parallel x%d, %s: %s, every slate duplicate-free: %s" % (
                world, what, "bit-identical to one GPU" if same else "MISMATCH", clean))

    for kind in ("pivotcvae_gt_pi", "pivotcvae_gt_spi", "listcvae"):
        # 1. parity-mode eps: the MLP rows stay unsharded, only the catalog is
        outs = []
        for vp in (False, True):
            m = make_model(kind, env, dev)
            if vp:
                m.enable_vocab_parallel()
            m.noise.reseed(2024)
            m.noise.push("eps", eps)
            outs.append(m.recommend(ctx, users, return_item=True)[0].cpu().numpy())
        plain = make_model(kind, env, dev)
        plain.no_repeat = False
        plain.noise.reseed(2024)
        plain.noise.push("eps", eps)
        n_dup = dup_slates(plain.recommend(ctx, users, return_item=True)[0].cpu().numpy())
        ok = ok and n_dup > 0
        if rank == 0:
            print("%s: %d of %d slates repeat an item without no_repeat" % (kind, n_dup, B))
        report("%s parity eps" % kind, *outs)
        # 2. Philox noise: the MLP rows are sharded over the ranks too
        outs = []
        for vp in (False, True):
            m = make_model(kind, env, dev)
            m.noise.reseed(2024)
            if vp:
                m.enable_vocab_parallel()
                assert world == 1 or m._vp_row_slice(B) is not None
            outs.append(m.recommend(ctx, users, return_item=True)[0].cpu().numpy())
        report("%s Philox, rows sharded" % kind, *outs)
        # 3. CUDA-graph replays
        outs = []
        for vp in (False, True):
            m = make_model(kind, env, dev)
            m.noise.reseed(2024)
            if vp:
                m.enable_vocab_parallel()
            gen = GraphedSlateGenerator(m, env, B)
            reps = []
            for _ in range(2):
                items, _ = gen(ctx, users)
                reps.append(items.cpu().numpy().copy())
            outs.append(np.concatenate(reps))
        report("%s GraphedSlateGenerator replays" % kind, *outs)
    t = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    sys.exit(0 if int(t) == 1 else 1)


if __name__ == "__main__":
    main()
