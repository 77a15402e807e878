"""In-place refresh of the item-table handle (pcv_table_refresh) and the fine_tune training step it enables.

    python profiles/sweep_table_refresh.py [--out FILE]

Prints the card and its power limit, then
  - the CUDA-event time of Table.refresh() at 100 k x D for D in 4..128 (with and without the tf32 CE's transposed
    image built) and at 1 M x 8 and 10 M x 8, with the bytes it moves (W read once, every image written) over that
    time against the 7.7 TB/s data-sheet HBM bandwidth; the L2 (126 MB) is overwritten between timed calls with a
    256 MB write outside the timed window;
  - an eager ListCVAE C3 training step with fine_tune (B = 4096, slate 5, D = 8, 100 k items, full catalog, exact and
    tf32 CE) that re-creates the table handle after every optimizer step (what item_table() did before the refresh
    existed) and one that refreshes it;
  - the same step captured by GraphedTrainStep(train_tables=True).
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pivotcvae_b200 import ops  # noqa: E402

DEV = "cuda:0"
G = torch.Generator(device=DEV).manual_seed(0)
HBM_TBS = 7.7
_FLUSH = None


def flush_l2():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=DEV)
    _FLUSH.fill_(1.0)


def timed(fn, iters=20, warm=3):
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


def refresh_bytes(n, D, with_t):
    """W read once + every image written (include/pcv_b200.h, csrc/table_images.cuh)."""
    b = n * D * 4                                   # W
    if D in (8, 16, 32, 64, 128):
        b += n * D * 4                              # pre-swizzled tf32 image
        if D == 8:
            b += n * 32                             # f16 image (unit-norm rows: it exists)
        if with_t:
            b += n * D * 4                          # transposed image (its zero rows at D = 8 are not rewritten)
    return b


def refresh_sweep(log):
    log("%-34s %10s %10s %12s" % ("Table.refresh()", "us", "MB moved", "TB/s (of 7.7)"))
    cases = [(100000, D, t) for D in (4, 8, 16, 32, 64, 128) for t in (False, True)]
    cases += [(1000000, 8, False), (1000000, 8, True), (10000000, 8, False), (10000000, 8, True)]
    for n, D, with_t in cases:
        if with_t and D not in (8, 16, 32, 64, 128):
            continue
        W = torch.nn.functional.normalize(torch.randn(n, D, device=DEV, generator=G), dim=1)
        tab = ops.Table(W)
        if with_t:   # one tf32 CE call builds the transposed image
            Q = torch.randn(128, D, device=DEV, generator=G)
            ops.ce_fwd_bwd(tab, Q, torch.zeros(128, dtype=torch.int64, device=DEV), engine="tf32")
        ms = timed(tab.refresh)
        b = refresh_bytes(n, D, with_t)
        log("%9d x %-3d %-20s %10.2f %10.2f %12.3f" % (n, D, "with transposed" if with_t else "", ms * 1e3, b / 1e6,
                                                       b / (ms * 1e-3) / 1e12))
        del tab, W
        torch.cuda.empty_cache()


class _Emb:
    def __init__(self, w):
        self.weight = w


def train_steps(log, steps=20):
    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    from pivotcvae_b200.train_generative import get_gen_loss
    N_ITEMS = 100000
    B, L, D, Z, H, PH, U = 4096, 5, 8, 16, 256, 128, 6041
    doc = _Emb(torch.randn(N_ITEMS, D, generator=G, device=DEV))
    usr = _Emb(torch.randn(U, D, generator=G, device=DEV))
    batch = {"slates": torch.randint(0, N_ITEMS, (B, L), device=DEV, generator=G),
             "users": torch.randint(0, U, (B, 1), device=DEV, generator=G),
             "responses": (torch.rand(B, L, device=DEV, generator=G) < 0.3).float()}

    def model(engine):
        torch.manual_seed(0)
        m = UserListCVAEWithPrior(doc, usr, L, D, Z, L + 1, [L * D + L + 1 + D, H, H], [Z + L + 1 + D, H, H, L * D],
                                  [L + 1 + D, PH, PH], False, DEV, fine_tune=True)
        m.ce_engine = engine
        return m

    def window(step):
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            step()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / steps

    for engine in ("exact", "tf32"):
        res = {}
        for rnd in range(2):    # the two eager variants alternate, twice
            for how in ("re-create", "refresh"):
                m = model(engine)
                opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-3)

                def step():
                    opt.zero_grad()
                    loss, _, _ = get_gen_loss(batch, m, None, 0.01, n_neg=N_ITEMS)
                    loss.backward()
                    opt.step()
                    if how == "re-create":
                        m._table = None     # what item_table() did after every optimizer step before the refresh
                    m.item_table()
                res.setdefault(how, []).append(window(step))
        for how, v in res.items():
            log("ListCVAE C3 eager fine_tune step, %-5s CE, handle %-9s %8.3f ms/step  (runs: %s)"
                % (engine, how, min(v), " ".join("%.3f" % x for x in v)))
        m = model(engine)
        opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-3, capturable=True)
        g = GraphedTrainStep(m, opt, B, 0.01, N_ITEMS, train_tables=True)
        log("ListCVAE C3 GraphedTrainStep(train_tables=True), %-5s CE  %8.3f ms/step  (%d launches/step)"
            % (engine, window(lambda: g(batch)), g.launches_per_step))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log("card: " + card())
    refresh_sweep(log)
    train_steps(log)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
