"""Times of the item-table gradient on a vocab-parallel catalog (fine_tune=True under enable_vocab_parallel).

    python profiles/sweep_vp_table_grad.py [--out FILE]                                  # one GPU: per-rank kernels
    python -m torch.distributed.run --nproc-per-node G profiles/sweep_vp_table_grad.py [--out FILE]   # training steps

One GPU: the CUDA-event time of one rank's table gradient, i.e. of the first row shard of parallel.shard_bounds for a
1/G split, G = 1, 2, 4, 8, at the C3 shape (100 k items x 20 480 query rows), D = 8 and 32: exact dense, tf32 dense,
Philox n_neg = 1000 and candidates n_cand = 1000, each with the whole catalog's lse.  Under torchrun: the ListCVAE C3
fine_tune step (B = 4096, slate 5, D = 8, full-catalog exact CE), eager and as a GraphedTrainStep(train_tables=True),
with and without vocab-parallel, and the time of the row exchange of one [100 k, 8] gradient.  The card's name and
power limit are printed first; the L2 (126 MB) is overwritten between timed calls with a 256 MB write, outside the
timed window.
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pivotcvae_b200 import ops  # noqa: E402
from pivotcvae_b200.parallel import shard_bounds  # noqa: E402

N_ITEMS, M = 100000, 20480
_FLUSH = None


def flush_l2():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device="cuda")
    _FLUSH.fill_(1.0)


def timed(fn, iters=10, warm=2):
    for _ in range(warm):
        fn()
    total = 0.0
    for _ in range(iters):
        flush_l2()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        total += s.elapsed_time(e)
    return total / iters


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        out = "nvidia-smi unavailable (%s)" % e
    return "%s | %s" % (torch.cuda.get_device_name(), out)


def kernels(log):
    g = torch.Generator(device="cuda").manual_seed(0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rs = torch.full((M,), 1.0 / M, device="cuda")
    log("per-rank table gradient, shard 0 of G (C3: 100k items x 20480 rows), ms; %d SMs" % sms)
    log("%-4s %-3s %8s %6s %9s %9s %11s %11s" % ("D", "G", "rows", "slabs", "exact", "tf32", "philox1000", "cand1000"))
    for D in (8, 32):
        W = F.normalize(torch.randn(N_ITEMS, D, device="cuda", generator=g), dim=1)
        Q = torch.randn(M, D, device="cuda", generator=g) * 0.5
        tg = torch.randint(0, N_ITEMS, (M,), device="cuda", generator=g)
        cand = torch.randint(0, N_ITEMS, (M, 1000), device="cuda", generator=g)
        tpos = torch.randint(0, 1000, (M,), device="cuda", generator=g)
        whole = ops.Table(W)
        keep = 1000.0 / N_ITEMS
        lse = {e: ops.ce_fwd_bwd(whole, Q, tg, 1.0, engine=e)[1] for e in ("exact", "tf32")}
        lse_p = ops.ce_fwd_bwd(whole, Q, tg, keep, seed=1, offset=0)[1]
        lse_c = ops.cand_ce_fwd_bwd(whole, Q, cand, tpos)[1]
        for G in (1, 2, 4, 8):
            lo, hi = shard_bounds(N_ITEMS, G, 0)
            sh = ops.Table(W[lo:hi], row_offset=lo)
            t = [timed(lambda: ops.ce_shard_table_grad(sh, Q, tg, lse["exact"], rs, 1.0)),
                 timed(lambda: ops.ce_shard_table_grad(sh, Q, tg, lse["tf32"], rs, 1.0, engine="tf32")),
                 timed(lambda: ops.ce_shard_table_grad(sh, Q, tg, lse_p, rs, keep, seed=1, offset=0)),
                 timed(lambda: ops.cand_ce_table_grad(sh, Q, cand, tpos, lse_c, rs))]
            log("%-4d %-3d %8d %6d %9.3f %9.3f %11.3f %11.3f" % (D, G, hi - lo, -(-(hi - lo) // 128), *t))
            del sh


class _Emb:
    def __init__(self, w):
        self.weight = w


def train_steps(log, steps=20):
    """Under torchrun: every rank runs the same steps; rank 0 logs."""
    import torch.distributed as dist

    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    from pivotcvae_b200.parallel import exchange_owned_rows
    from pivotcvae_b200.train_generative import get_gen_loss
    world = dist.get_world_size()
    g = torch.Generator(device="cuda").manual_seed(0)
    B, L, D, Z, H, PH, U = 4096, 5, 8, 16, 256, 128, 6041
    doc = _Emb(torch.randn(N_ITEMS, D, generator=g, device="cuda"))
    usr = _Emb(torch.randn(U, D, generator=g, device="cuda"))
    batch = {"slates": torch.randint(0, N_ITEMS, (B, L), device="cuda", generator=g),
             "users": torch.randint(0, U, (B, 1), device="cuda", generator=g),
             "responses": (torch.rand(B, L, device="cuda", generator=g) < 0.3).float()}
    for vp in (False, True):
        for graphed in (False, True):
            torch.manual_seed(0)
            m = UserListCVAEWithPrior(doc, usr, L, D, Z, L + 1, [L * D + L + 1 + D, H, H], [Z + L + 1 + D, H, H, L * D],
                                      [L + 1 + D, PH, PH], False, "cuda", fine_tune=True)
            if vp:
                m.enable_vocab_parallel(train_tables=True)
            opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-3, capturable=graphed)
            if graphed:
                gs = GraphedTrainStep(m, opt, B, 0.01, N_ITEMS, train_tables=True)
                step = lambda: gs(batch)        # noqa: E731
            else:
                def step():
                    opt.zero_grad()
                    loss, _, _ = get_gen_loss(batch, m, None, 0.01, n_neg=N_ITEMS)
                    loss.backward()
                    opt.step()
            for _ in range(3):
                step()
            dist.barrier()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(steps):
                step()
            e.record()
            torch.cuda.synchronize()
            log("ListCVAE C3 fine_tune step, world %d, vocab-parallel=%-5s %-7s %8.3f ms/step" % (
                world, vp, "graphed" if graphed else "eager", s.elapsed_time(e) / steps))
    grad = torch.randn(N_ITEMS, D, device="cuda", generator=g)
    log("row exchange of a [100000, 8] gradient, world %d        %8.3f ms" % (
        world, timed(lambda: exchange_owned_rows(grad), iters=20)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    distributed = "WORLD_SIZE" in os.environ
    rank = 0
    if distributed:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl")
        rank = dist.get_rank()
    lines = []

    def log(s):
        if rank == 0:
            print(s, flush=True)
            lines.append(s)
    log("card: " + card())
    if distributed:
        train_steps(log)
        dist.destroy_process_group()
    else:
        kernels(log)
    if args.out and rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
