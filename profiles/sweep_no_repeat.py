"""Cost of the opt-in no-repeat selection (`model.no_repeat = True`) on bench.py's C4 synthetic model (PivotCVAE gt_pi,
1 M items, B = 4096, L = 5, D = 8).

    python profiles/sweep_no_repeat.py [K]                                            # one GPU
    python -m torch.distributed.run --nproc-per-node G profiles/sweep_no_repeat.py [K]   # vocab-parallel over G GPUs

Each arm is a GraphedSlateGenerator step (recommend + response score, bench.py's timed step) over K distinct input
batches; every step is timed alone with CUDA events after an L2 flush (256 MiB write), and the off / on arms alternate
over REPS windows.  Prints the median ms per step of each arm.  On one GPU it also prints the fraction of slates whose
top-1 picks hold a duplicate (the slates the no-repeat pass re-scores) and the time of the no-repeat pass alone
(`ops.slate_no_repeat` through ops.KernelTimer, L2 flushed before each call) against the step."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pivotcvae_b200 import ops  # noqa: E402
from pivotcvae_b200.graphs import GraphedSlateGenerator  # noqa: E402

K = int(sys.argv[1]) if len(sys.argv) > 1 else 100
REPS = 3


def card(index):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(index)


def main():
    D = bench.Dist()
    D.start()
    w = bench.WORKLOADS["c4"]
    B, L = w["B"], w["L"]
    vp = D.world > 1
    sd, env_sd = bench.make_weights(w, "pivot")
    ctx, usr = zip(*[bench.make_inputs(w, B, i) for i in range(K)])
    ctx, usr = [c.to(D.device) for c in ctx], [u.to(D.device) for u in usr]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=D.device)
    if D.rank == 0:
        print("# %s" % card(D.local))
        print("# C4 greedy: %d items, B=%d, L=%d, D=%d; %s; %d steps per window, %d windows per arm, L2 flushed "
              "before every step" % (w["n_items"], B, L, w["D"], "vocab-parallel over %d GPUs" % D.world if vp else "one GPU",
                                     K, REPS), flush=True)
    gens = {}
    for nr in (False, True):
        model, env = bench.build_gpu(w, sd, env_sd, "greedy", D.device)
        model.noise.reseed(1234)
        model.no_repeat = nr
        if vp:
            model.enable_vocab_parallel()
        gens[nr] = GraphedSlateGenerator(model, env, B, warmup=3)
    times = {False: [], True: []}
    for _ in range(REPS):
        for nr in (False, True):
            gen = gens[nr]
            times[nr].append(bench.timed_steps(D, lambda i: gen(ctx[i], usr[i]), K, 3, flush) / K)
    med = {nr: sorted(t)[len(t) // 2] for nr, t in times.items()}
    if D.rank == 0:
        for nr in (False, True):
            print("%s no_repeat=%-5s %.4f ms/step (windows: %s)" % ("vocab-parallel x%d" % D.world if vp else "one GPU",
                  nr, med[nr], ", ".join("%.4f" % t for t in times[nr])))
        print("no_repeat adds %.4f ms/step (%.1f %%)" % (med[True] - med[False], 100.0 * (med[True] / med[False] - 1)))
    if not vp:
        # duplicate-holding slates among the top-1 picks of the same K batches
        flagged = 0
        for i in range(K):
            items, _ = gens[False](ctx[i], usr[i])
            flagged += sum(len(set(r)) < L for r in items.view(B, L).tolist())
        print("flagged slates: %d of %d (%.3f %%)" % (flagged, K * B, 100.0 * flagged / (K * B)))
        # the no-repeat pass alone on the decoder's slot queries of the same batches
        model = gens[True].model
        tab = model.item_table()
        qs = []
        for i in range(K):
            model.noise.reseed(99 + i)
            rx, _ = model.recommend(ctx[i], usr[i], return_item=False)
            qs.append(rx.reshape(-1, w["D"]).contiguous())
        picks = [ops.score_select(tab, q, "greedy", want_val=False)[0] for q in qs]
        for i in range(3):
            ops.slate_no_repeat(tab, qs[i], picks[i].clone(), L)
        with ops.KernelTimer() as kt:
            for i in range(K):
                it = picks[i].clone()
                flush.zero_()
                ops.slate_no_repeat(tab, qs[i], it, L)
        s = kt.summary()["slate_no_repeat_M%d" % (B * L)]
        print("no-repeat pass (flag + top-L re-score of the flagged rows + resolve): %.4f ms/call over %d calls, "
              "%.1f %% of the no_repeat=True step" % (s["ms_avg"], s["calls"], 100.0 * s["ms_avg"] / med[True]))
        print("vocab-parallel step time: not measured (one GPU in this run; run under torchrun with G > 1)")
    elif D.rank == 0:
        print("exchange per step: one all-gather of B*L*L int64 = %d bytes per rank" % (B * L * L * 8))
    D.stop()


if __name__ == "__main__":
    main()
