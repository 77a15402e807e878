"""Vocab-parallel fine_tune training on N GPUs == single-GPU training (run under torchrun on a multi-GPU box):
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/vp_fine_tune_check.py

UserListCVAEWithPrior(fine_tune=True) on the list_small_user fixture and on a synthetic 100 k-item catalog, in five
training modes (dense exact, dense tf32, bitmask, Philox, candidates), with enable_vocab_parallel(train_tables=True):
  - one step: the loss and every gradient, tables included, match the single-GPU run (the tolerances of
    vp_gpu_check.py: loss 1e-5 relative, gradients rtol 1e-3 / atol 1e-6);
  - 5 Adam steps, eager and (the modes a static batch can carry: exact, tf32, Philox) as a
    GraphedTrainStep(train_tables=True): every parameter byte-identical across the ranks after every step, per-step
    losses within 1e-4 of the single-GPU run.
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import load_golden  # noqa: E402


class _Emb:
    def __init__(self, w):
        self.weight = w


def _problem(name, dev):
    """-> (build(fine_tune) -> model, batch, n_items)"""
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    if name == "list_small_user":
        fx = load_golden(name)
        cfg, sd = fx.cfg, fx.sub("sd/")
        L, D, Z, H, PH = cfg["L"], cfg["D"], cfg["Z"], cfg["hidden"], cfg["phidden"]
        import gpu_util
        doc, usr = _Emb(torch.from_numpy(sd["docEmbed.weight"])), _Emb(torch.from_numpy(sd["userEmbed.weight"]))

        def build():
            m = UserListCVAEWithPrior(doc, usr, L, D, Z, L + 1, [L * D + L + 1 + D, H, H], [Z + L + 1 + D, H, H, L * D],
                                      [L + 1 + D, PH, PH], False, dev, fine_tune=True)
            return gpu_util.load_sd(m, sd)
        batch = {"slates": torch.from_numpy(fx["in/slates"]).to(dev), "users": torch.from_numpy(fx["in/users"]).to(dev),
                 "responses": torch.from_numpy(fx["in/resp"]).to(dev)}
        return build, batch, cfg["n_items"]
    n_items, n_users, B, L, D, Z, H, PH = 100000, 6041, 256, 5, 8, 16, 256, 128
    g = torch.Generator(device=dev).manual_seed(4)
    doc = _Emb(torch.randn(n_items, D, device=dev, generator=g))
    usr = _Emb(torch.randn(n_users, D, device=dev, generator=g))

    def build():
        torch.manual_seed(4)
        return UserListCVAEWithPrior(doc, usr, L, D, Z, L + 1, [L * D + L + 1 + D, H, H], [Z + L + 1 + D, H, H, L * D],
                                     [L + 1 + D, PH, PH], False, dev, fine_tune=True)
    batch = {"slates": torch.randint(0, n_items, (B, L), device=dev, generator=g),
             "users": torch.randint(0, n_users, (B, 1), device=dev, generator=g),
             "responses": (torch.rand(B, L, device=dev, generator=g) < 0.3).float()}
    return build, batch, n_items


def _identical_across_ranks(m):
    flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).view(torch.int32)
    ref = flat.clone()
    dist.broadcast(ref, 0)
    ok = torch.tensor([int(torch.equal(flat, ref))], device=flat.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return bool(ok.item())


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    import gpu_util
    gpu_util.dev = lambda: torch.device("cuda:%d" % torch.cuda.current_device())
    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.train_generative import get_gen_loss
    dev = "cuda:%d" % torch.cuda.current_device()
    ok = True

    def report(what, good, detail=""):
        nonlocal ok
        ok = ok and good
        if rank == 0:
            print("vocab-parallel x%d fine_tune %s: %s %s" % (world, what, "ok" if good else "MISMATCH", detail), flush=True)

    for name in ("list_small_user", "synthetic100k"):
        build, batch, n_items = _problem(name, dev)
        M = batch["slates"].numel()
        g = torch.Generator(device=dev).manual_seed(6)
        nC = 100
        cand = torch.randint(0, n_items, (M, nC), device=dev, generator=g)
        tpos = torch.randint(0, nC, (M,), device=dev, generator=g)
        cand[torch.arange(M), tpos] = batch["slates"].reshape(-1)
        n_words = -(-n_items // 32)
        bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (M, n_words), dtype=torch.int32, device=dev, generator=g)
        bits &= torch.randint(-2 ** 31, 2 ** 31 - 1, (M, n_words), dtype=torch.int32, device=dev, generator=g)
        bits &= torch.randint(-2 ** 31, 2 ** 31 - 1, (M, n_words), dtype=torch.int32, device=dev, generator=g)  # ~1/8
        n_neg = min(1000, n_items // 4)
        modes = {"exact": ("exact", n_items), "tf32": ("tf32", n_items), "bitmask": ("exact", n_neg),
                 "philox": ("exact", n_neg), "candidates": ("exact", n_items)}
        for mode, (engine, nn) in modes.items():
            bt = dict(batch, sample_candidates=cand, sample_targets=tpos) if mode == "candidates" else batch
            runs = []
            for vp in (False, True):
                m = build()
                m.ce_engine, m.candidateFlag = engine, mode == "candidates"
                if vp:
                    m.enable_vocab_parallel(train_tables=True)
                m.noise.reseed(31)
                opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2)
                losses, grads, same = [], None, True
                for step in range(5):
                    if mode == "bitmask":
                        m.noise.push("mask", bits)
                    opt.zero_grad(set_to_none=True)
                    loss, _, _ = get_gen_loss(bt, m, None, 0.01, n_neg=nn)
                    loss.backward()
                    if step == 0:
                        grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
                    opt.step()
                    losses.append(float(loss))
                    if vp:
                        same = same and _identical_across_ranks(m)
                runs.append((losses, grads, same))
            (l0, g0, _), (l1, g1, same) = runs
            good = abs(l0[0] - l1[0]) <= 1e-5 * abs(l0[0]) and sorted(g0) == sorted(g1)
            worst = 0.0
            for k in g0:
                good = good and bool(torch.allclose(g1[k], g0[k], rtol=1e-3, atol=1e-6))
                worst = max(worst, float((g1[k] - g0[k]).abs().max()))
            report("%s %s one step" % (name, mode), good, "loss %.7f vs %.7f, grads max diff %.2e" % (l1[0], l0[0], worst))
            report("%s %s 5 eager steps" % (name, mode), same and all(abs(a - b) <= 1e-4 * abs(a) for a, b in zip(l0, l1)),
                   "replicas identical: %s, losses %s vs %s" % (same, l1, l0))
            if mode in ("bitmask", "candidates"):
                continue                    # a static batch carries neither a pushed mask nor candidate lists
            runs = []
            for vp in (False, True):
                m = build()
                m.ce_engine = engine
                if vp:
                    m.enable_vocab_parallel(train_tables=True)
                m.noise.reseed(31)
                opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2, capturable=True)
                step = GraphedTrainStep(m, opt, batch["slates"].shape[0], 0.01, nn, train_tables=True)
                losses, same = [], True
                for _ in range(5):
                    losses.append(float(step(batch)[0]))
                    if vp:
                        same = same and _identical_across_ranks(m)
                runs.append((losses, same))
            (l0, _), (l1, same) = runs
            report("%s %s 5 graphed steps" % (name, mode),
                   same and all(abs(a - b) <= 1e-4 * abs(a) for a, b in zip(l0, l1)),
                   "replicas identical: %s, losses %s vs %s" % (same, l1, l0))
    t = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    sys.exit(0 if int(t) == 1 else 1)


if __name__ == "__main__":
    main()
