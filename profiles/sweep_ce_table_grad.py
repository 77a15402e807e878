"""Kernel and step times of the item-table gradient (fine_tune=True) at the C3 shape: 100 k items x 20 480 query rows.

    python profiles/sweep_ce_table_grad.py [--out FILE]

Prints the card and its power limit, then per D the CUDA-event time of pcv_ce_fwd_bwd (exact and tf32 engines) and of
pcv_ce_table_grad on the same inputs, the Philox path (n_neg = 1000, D = 8) and candidate mode (n_cand = 1000, D = 8),
and an eager ListCVAE training step (B = 4096, slate 5, D = 8, full catalog, exact CE) with fine_tune off and on.  The
L2 (126 MB) is overwritten between timed calls with a 256 MB write, which is outside the timed window.
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pivotcvae_b200 import ops  # noqa: E402

DEV = "cuda:0"
N_ITEMS, M = 100000, 20480
G = torch.Generator(device=DEV).manual_seed(0)
_FLUSH = None


def flush_l2():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=DEV)
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
    return "%s | %s" % (torch.cuda.get_device_name(0), out)


def kernels(log):
    log("%-34s %10s" % ("call (C3: 100k items x 20480 rows)", "ms"))
    rs = torch.full((M,), 1.0 / M, device=DEV)
    for D in (4, 8, 16, 32, 64, 128):
        W = F.normalize(torch.randn(N_ITEMS, D, device=DEV, generator=G), dim=1)
        Q = torch.randn(M, D, device=DEV, generator=G) * 0.5
        tg = torch.randint(0, N_ITEMS, (M,), device=DEV, generator=G)
        tab = ops.Table(W)
        engines = ("exact",) if D == 4 else ("exact", "tf32")
        for eng in engines:
            _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, 1.0, engine=eng)
            t_f = timed(lambda: ops.ce_fwd_bwd(tab, Q, tg, 1.0, engine=eng))
            t_g = timed(lambda: ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0, engine=eng))
            log("D=%-3d %-5s ce_fwd_bwd            %10.3f" % (D, eng, t_f))
            log("D=%-3d %-5s ce_table_grad         %10.3f" % (D, eng, t_g))
        if D == 8:
            keep = 1000.0 / N_ITEMS
            _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, keep, seed=1, offset=0)
            log("D=8   philox ce_fwd_bwd n_neg=1000   %10.3f" % timed(lambda: ops.ce_fwd_bwd(tab, Q, tg, keep, seed=1, offset=0)))
            log("D=8   philox ce_table_grad n_neg=1000 %9.3f" % timed(
                lambda: ops.ce_table_grad(tab, Q, tg, lse, rs, keep, seed=1, offset=0)))
            cand = torch.randint(0, N_ITEMS, (M, 1000), device=DEV, generator=G)
            tpos = torch.randint(0, 1000, (M,), device=DEV, generator=G)
            _, lse, _, _ = ops.cand_ce_fwd_bwd(tab, Q, cand, tpos)
            log("D=8   cand_ce_fwd_bwd n_cand=1000    %10.3f" % timed(lambda: ops.cand_ce_fwd_bwd(tab, Q, cand, tpos)))
            log("D=8   cand_ce_table_grad n_cand=1000 %10.3f" % timed(
                lambda: ops.cand_ce_table_grad(tab, Q, cand, tpos, lse, rs)))
        del tab


class _Emb:
    def __init__(self, w):
        self.weight = w


def train_steps(log, steps=20):
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    from pivotcvae_b200.train_generative import get_gen_loss
    B, L, D, Z, H, PH, U = 4096, 5, 8, 16, 256, 128, 6041
    doc = _Emb(torch.randn(N_ITEMS, D, generator=G, device=DEV))
    usr = _Emb(torch.randn(U, D, generator=G, device=DEV))
    batch = {"slates": torch.randint(0, N_ITEMS, (B, L), device=DEV, generator=G),
             "users": torch.randint(0, U, (B, 1), device=DEV, generator=G),
             "responses": (torch.rand(B, L, device=DEV, generator=G) < 0.3).float()}
    for ft in (False, True):
        torch.manual_seed(0)
        m = UserListCVAEWithPrior(doc, usr, L, D, Z, L + 1, [L * D + L + 1 + D, H, H], [Z + L + 1 + D, H, H, L * D],
                                  [L + 1 + D, PH, PH], False, DEV, fine_tune=ft)
        opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-3)

        def step():
            opt.zero_grad()
            loss, _, _ = get_gen_loss(batch, m, None, 0.01, n_neg=N_ITEMS)
            loss.backward()
            opt.step()
            m.item_table()      # the handle re-creation after the step (fine_tune: the table changed) is part of it
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            step()
        e.record()
        torch.cuda.synchronize()
        log("ListCVAE C3 eager train step, fine_tune=%-5s %8.3f ms/step" % (ft, s.elapsed_time(e) / steps))
        # where the device time of a step goes: torch.profiler over 5 steps (a separate, slower run), top entries
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                step()
            torch.cuda.synchronize()
        dev_us = lambda r: getattr(r, "device_time_total", None) or getattr(r, "cuda_time_total", 0.0)
        rows = sorted(prof.key_averages(), key=lambda r: -dev_us(r))[:12]
        for r in rows:
            log("    device %-60s %8.3f ms/step  (%d calls/step)" % (r.key[:60], dev_us(r) / 5e3, r.count // 5))
    t = timed(lambda: ops.Table(m.docEmbed.weight.detach()), iters=10)
    log("table handle re-creation (100k x 8)           %8.3f ms" % t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log("card: " + card())
    kernels(log)
    train_steps(log)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
