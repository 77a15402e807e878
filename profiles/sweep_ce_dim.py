"""Embedding-dimension sweep of the full-catalog soft-max CE, forward + backward (`ops.ce_fwd_bwd`, dense mask): the
tensor-core (tf32) engine and the exact SIMT engine at D in {8, 16, 32, 64, 128}.  N x M from the command line
(default 100000 items x 20480 rows, the C3 shape); an optional third argument picks the engines ("tf32,exact") and a
fourth the dims ("8,128").  Every timed call follows an L2 flush and is timed alone with CUDA events.  Prints ms per
call, logits/s and the contraction TFLOP/s, counting 4 D N M operations: the scores plus the gradient."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pivotcvae_b200 import ops  # noqa: E402

N, M = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (100000, 20480)
ENGINES = sys.argv[3].split(",") if len(sys.argv) > 3 else ["tf32", "exact"]
DIMS = [int(d) for d in sys.argv[4].split(",")] if len(sys.argv) > 4 else [8, 16, 32, 64, 128]
WARMUP, CALLS = 3, 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name()


ops.device_ok()
print("# %s" % card())
print("# N=%d items x M=%d rows, CE forward + backward, L2 flushed before every call, %d calls" % (N, M, CALLS))
g = torch.Generator(device="cuda").manual_seed(0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for D in DIMS:
    W = torch.nn.functional.normalize(torch.rand(N, D, generator=g, device="cuda") * 2 - 1, dim=1)
    Q = torch.randn(M, D, generator=g, device="cuda") * (0.5 * (8.0 / D) ** 0.5)
    tg = torch.randint(0, N, (M,), generator=g, device="cuda")
    tab = ops.Table(W)
    for engine in ENGINES:
        for _ in range(WARMUP):
            ops.ce_fwd_bwd(tab, Q, tg, 1.0, engine=engine)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(CALLS)]
        for s, e in ev:
            flush.zero_()
            s.record()
            ops.ce_fwd_bwd(tab, Q, tg, 1.0, engine=engine)
            e.record()
        torch.cuda.synchronize()
        ms = sorted(s.elapsed_time(e) for s, e in ev)
        med = ms[len(ms) // 2]
        print("D=%3d %-6s %.4f ms/call (min %.4f)  %.3f T logits/s  %.1f TFLOP/s" % (
            D, engine, med, ms[0], N * M / med / 1e9, 4.0 * D * N * M / med / 1e9), flush=True)
    del tab
