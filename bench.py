#!/usr/bin/env python
"""bench.py — generated slates/sec (greedy + sampled) and train samples/sec of the PivotCVAE hot path on B200.

One generation "step" = one batch of users through recommend(return_item=True) (prior MLP -> reparameterise ->
PSM MLP -> pivot pick over the catalog -> SCM MLP -> per-slot arg-max over the catalog) + the response-model
score of the generated slates.  One training "step" = get_gen_loss (fused catalog CE + KL) -> backward -> Adam.

    python bench.py [--gpus N] [--steps K] [--warmup W]        # default workload: C4 (1 M items, B = 4096)
    python bench.py --workload c2|c1|c3|c4|c5 --mode greedy|sampled|list|train ...
    python bench.py --impl reference ...     # CPU arm: the unmodified reference (baseline/_ref) on the host cores

N>1 is launched by the driver through torch.distributed.run (one rank per GPU).  Prints ONE JSON line (rank 0):
the headline (C4 greedy: `value` device-resident, `e2e` through host buffers), its `roofline`, `cpu_baseline`,
`gpu_library_baseline`, a `vp` block at N>1 (the 1 M-item catalog sharded vocab-parallel, strong scaling) and, at
N=1, an `also` array with the sampled / C2 / C1 / training sub-results.  See DESIGN.md "Measurement".

Timing: after W warm-up steps, exactly K timed steps (per-step CUDA-event pairs, L2 flushed between steps, summed),
bracketed by barrier + synchronize, max over ranks.  K defaults to the workload's `steps`, about 0.5 s of timed work.

--dump-outputs DIR writes what the timed path returned in its last timed step as DIR/<name>.npy (float32 / float64).
Weights, inputs and noise seeds are fixed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "c1": dict(n_items=3707, n_users=6041, L=5, D=8, Z=16, H=256, PH=128, no_user=False, B=64, steps=4500,
               desc="C1 ML-1M shape: 3707 items, 6041 users, slate 5, dim 8, with user, B=64"),
    "c2": dict(n_items=50000, n_users=1, L=10, D=8, Z=16, H=256, PH=128, no_user=True, B=1024, steps=3500,
               desc="C2 Yoochoose shape: 50k items, slate 10, dim 8, nouser, B=1024"),
    "c3": dict(n_items=100000, n_users=6041, L=5, D=8, Z=16, H=256, PH=128, no_user=False, B=4096, steps=400,
               desc="C3: PivotCVAE gt training, fused full-catalog soft-max CE + KL, 100k items, slate 5, dim 8, B=4096"),
    "c4": dict(n_items=1000000, n_users=6041, L=5, D=8, Z=16, H=256, PH=128, no_user=False, B=4096, steps=400,
               desc="C4: 1M items, slate 5, dim 8, with user, B=4096, PivotCVAE + response MLP"),
    "c5": dict(n_items=10000000, n_users=1024, L=5, D=8, Z=16, H=256, PH=128, no_user=False, B=65536, samples_per_user=64, steps=4,
               desc="C5 variation-control sweep: 10M items, slate 5, dim 8, 1024 users x 64 sampled slates = 65536 rows "
                    "(gt_spi: sampled pivot + fresh z per sample), coverage + ILS of the result"),
}
# steps: the default --steps of a workload, about 0.5 s of timed steps on one B200 (C4: 1.55 ms per step, C2: 0.13-0.17 ms,
# C1: 0.12 ms, C3 training: 1.3 ms, C5: 176 ms); the `also` sub-results of the default run time half of that.
# The CPU reference arm (--impl reference) defaults to REFERENCE_STEPS: at C4 one of its steps takes about 0.5 s.
REFERENCE_STEPS = 20
MODEL_OF_MODE = {"greedy": "PivotCVAE gt_pi", "sampled": "PivotCVAE gt_spi (sampled pivot)", "list": "ListCVAE", "train": "PivotCVAE gt"}


def structs(w):
    L, D, Z, H, PH = w["L"], w["D"], w["Z"], w["H"], w["PH"]
    C, ud = L + 1, (0 if w["no_user"] else D)
    return dict(enc=[L * D + C + ud, H, H], psm=[Z + C + ud, H, H, D], scm=[Z + C + D + ud, H, H, (L - 1) * D],
                dec=[Z + C + ud, H, H, L * D], prior=[C + ud, PH, PH], resp=[(L + (0 if w["no_user"] else 1)) * D, H, H, L])


def make_weights(w, model_kind):
    """Synthetic weights with the reference's initialisers, built on the CPU so every arm shares them:
    tables uniform(-a, a), a = sqrt(2/D) (env/response_model.py:29-37), then row-normalised by the
    model (cvae.py:31); hidden layers kaiming_uniform_, heads default nn.Linear init (pivotcvae.py:108-152)."""
    g = torch.Generator().manual_seed(20211)
    a = (2.0 / w["D"]) ** 0.5
    doc = (torch.rand(w["n_items"], w["D"], generator=g) * 2 - 1) * a
    usr = (torch.rand(w["n_users"], w["D"], generator=g) * 2 - 1) * a
    torch.manual_seed(0)
    st = structs(w)
    sd, env_sd = {}, {}

    def mlp(prefix, dims, out):
        for i in range(len(dims) - 1):
            lin = torch.nn.Linear(dims[i], dims[i + 1])
            torch.nn.init.kaiming_uniform_(lin.weight)
            out["%s_%d.weight" % (prefix, i + 1)] = lin.weight.detach().numpy().copy()
            out["%s_%d.bias" % (prefix, i + 1)] = lin.bias.detach().numpy().copy()

    def head(name, n_in, out):
        lin = torch.nn.Linear(n_in, w["Z"])
        out[name + ".weight"], out[name + ".bias"] = lin.weight.detach().numpy().copy(), lin.bias.detach().numpy().copy()

    mlp("enc", st["enc"], sd)
    head("encmu", st["enc"][-1], sd)
    head("enclogvar", st["enc"][-1], sd)
    if model_kind == "list":
        mlp("dec", st["dec"], sd)
    else:
        mlp("psm", st["psm"], sd)
        mlp("scm", st["scm"], sd)
    mlp("prior", st["prior"], sd)
    head("priorMu", st["prior"][-1], sd)
    head("priorLogvar", st["prior"][-1], sd)
    nd = torch.nn.functional.normalize(doc, p=2, dim=1)
    sd["docEmbed.weight"] = nd.numpy().copy()
    env_sd["docEmbed.weight"] = doc.numpy().copy()
    if not w["no_user"]:
        sd["userEmbed.weight"] = torch.nn.functional.normalize(usr, p=2, dim=1).numpy().copy()
        env_sd["userEmbed.weight"] = usr.numpy().copy()
    mlp("mlp", st["resp"], env_sd)
    return sd, env_sd


def make_inputs(w, B, step, seed=1234):
    """Eval-loop inputs (train_generative.py:177-184): uniform users, context = first k responses set.
    C5: 1024 users x 64 samples — every user id repeated 64 times (variation-control sweep)."""
    g = torch.Generator().manual_seed(seed + step)
    spu = w.get("samples_per_user", 1)
    if spu > 1 and B % spu == 0:
        users = torch.randint(0, w["n_users"], (B // spu,), generator=g).repeat_interleave(spu)
    else:
        users = torch.randint(0, w["n_users"], (B,), generator=g)
    k = step % w["L"] + 1
    ctx = torch.zeros(B, w["L"])
    ctx[:, :k] = 1
    return ctx, users


def make_train_batch(w, B, step, seed=4321):
    """Synthetic (slate, user, response) rows: uniform items/users, Bernoulli(0.5) responses (SURVEY d2)."""
    g = torch.Generator().manual_seed(seed + step)
    slates = torch.randint(0, w["n_items"], (B, w["L"]), generator=g)
    users = torch.randint(0, w["n_users"], (B, 1), generator=g)
    resp = (torch.rand(B, w["L"], generator=g) < 0.5).float()
    return {"slates": slates, "users": users, "responses": resp}


class Emb:
    def __init__(self, wt):
        self.weight = torch.from_numpy(wt)


def build_gpu(w, sd, env_sd, mode, device):
    from pivotcvae_b200.env.response_model import UserResponseModel_MLP
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    from pivotcvae_b200.models.pivotcvae import PIVOTCVAE_MODELS
    st = structs(w)
    L, D, Z = w["L"], w["D"], w["Z"]
    uemb = None if w["no_user"] else Emb(env_sd["userEmbed.weight"])
    if mode == "list":
        m = UserListCVAEWithPrior(Emb(env_sd["docEmbed.weight"]), uemb, L, D, Z, L + 1, st["enc"], st["dec"], st["prior"],
                                  w["no_user"], device)
    else:
        key = "pivotcvae_gt_spi" if mode == "sampled" else "pivotcvae_gt_pi"
        m = PIVOTCVAE_MODELS[key](Emb(env_sd["docEmbed.weight"]), uemb, L, D, Z, L + 1, st["enc"], st["psm"], st["scm"],
                                  st["prior"], w["no_user"], device)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    env = UserResponseModel_MLP(w["n_items"] - 1, w["n_users"] - 1, D, L, st["resp"], device, w["no_user"])
    env.load_state_dict({k: torch.from_numpy(v) for k, v in env_sd.items()})
    env.to(device)
    return m, env


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, busy_sm, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                if float(r[7]) > 0:
                    busy_sm.append(float(r[0]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        load = busy_sm or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(busy_sm)}


# ------------------------------------------------------------------ distributed helpers
class Dist:
    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = "cuda:%d" % self.local
        self.started = False

    def start(self):
        torch.cuda.set_device(self.local)
        if self.world > 1 and not self.started:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device(self.device))
            self.started = True

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_(self, values):
        t = torch.tensor(values, device=self.device, dtype=torch.float64)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def stop(self):
        if self.started:
            import torch.distributed as dist
            dist.destroy_process_group()
            self.started = False


def timed_steps(D, step, K, W, flush):
    """W warm-up steps, then exactly K timed steps; step(i) runs step i on the current stream.  Per-step CUDA-event
    pairs (L2 flushed outside the pairs) are summed; the K steps are bracketed by barrier + synchronize and the MAX
    over ranks is taken.  -> ms of the K steps."""
    for i in range(W):
        step(i % K)
    D.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for i in range(K):
        flush.zero_()
        ev[i][0].record()
        step(i)
        ev[i][1].record()
    D.barrier()
    return D.max_([sum(a.elapsed_time(b) for a, b in ev)])[0]


DUMP_LIMIT = 64 * 10 ** 6      # bytes of all files written by dump_outputs
NPY_HEADER = 256               # bytes allowed per .npy header (numpy writes 128 for these shapes)


def dump_outputs(path, arrays):
    """Write {name: tensor} as path/<name>.npy: floats of 32 bits or fewer as float32, everything else (item ids,
    float64) as float64.  When the files would exceed DUMP_LIMIT bytes in all, every array keeps the same fraction of
    its rows, a sorted sample drawn with a fixed seed, and the kept row indices go to <name>.rows.npy."""
    os.makedirs(path, exist_ok=True)
    out = {}
    for k, v in arrays.items():
        a = v.detach().cpu().numpy()
        out[k] = a.astype(np.float32 if a.dtype.kind == "f" and a.itemsize <= 4 else np.float64)
    budget = DUMP_LIMIT - 2 * NPY_HEADER * len(out)      # an array and its row indices: two files, two headers
    total = sum(a.nbytes + 8 * len(a) for a in out.values() if a.ndim)
    fixed = sum(a.nbytes for a in out.values() if not a.ndim)
    for k, a in out.items():
        if a.ndim and total + fixed > budget:
            keep = int(len(a) * (budget - fixed) / total)
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            np.save(os.path.join(path, k + ".rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(path, k + ".npy"), a)


# ------------------------------------------------------------------ CPU arms
def cpu_port_step(oracle, w, sd, env_sd, mode, ctx, users, eps, noise=None):
    if mode == "list":
        out = oracle.list_recommend(sd, ctx, users, eps, w["no_user"])
    else:
        out = oracle.pivot_recommend(sd, ctx, users, eps, w["no_user"], "sample" if mode == "sampled" else "max", noise)
    resp = oracle.resp_mlp(env_sd, out["items"].reshape(ctx.shape[0], -1), users, w["no_user"])
    return out["items"], resp


def time_cpu_port(w, sd, env_sd, mode, B, min_seconds, warmup=1, max_steps=2000):
    """The oracle's C restatement of the reference (kind "port") on all host threads."""
    import oracle
    threads = os.cpu_count() or 1
    oracle.set_threads(threads)
    rng = np.random.default_rng(0)
    times, i = [], 0
    while True:
        ctx, users = make_inputs(w, B, i)
        eps = rng.standard_normal((B, w["Z"])).astype(np.float32)
        noise = rng.exponential(size=(B, w["n_items"])).astype(np.float32) if mode == "sampled" else None
        t0 = time.perf_counter()
        cpu_port_step(oracle, w, sd, env_sd, mode, ctx.numpy(), users.numpy(), eps, noise)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        i += 1
        if (sum(times) >= min_seconds and len(times) >= 3) or len(times) >= max_steps:
            break
    oracle.set_threads(1)
    return B / float(np.mean(times)), threads, len(times)


def cpu_sample_batch(w, mode):
    """Rows per CPU step: a bounded sample of the workload's batch (the reference is batch-linear there)."""
    per_row = w["n_items"] * w["L"] * (3 if mode == "sampled" else 1)
    return int(max(16, min(w["B"], 256, (1 << 28) // per_row * 4)))


def cpu_baselines(w, sd, env_sd, mode, seconds):
    """-> (cpu_baseline dict, cpu_port dict): the unmodified reference on the host cores when baseline/_ref
    travelled with the repo (kind "reference"), and the oracle's C port beside it."""
    cb = cpu_sample_batch(w, mode)
    pv, threads, n = time_cpu_port(w, sd, env_sd, mode, cb, seconds * 0.4)
    port = {"value": pv, "unit": "slates/s", "cores": threads, "kind": "port",
            "sample": "%d steps of %d slates of the same workload (oracle/pcv_oracle.c, pthreads x%d)" % (n, cb, threads)}
    from baseline import ref_runner
    if not ref_runner.available():
        return port, port
    torch.set_num_threads(os.cpu_count() or 1)
    v, n, b = ref_runner.time_generate(w, structs(w), sd, env_sd, mode, "cpu", lambda i: make_inputs(w, cb, i), seconds * 0.6)
    ref = {"value": v, "unit": "slates/s", "cores": torch.get_num_threads(), "kind": "reference",
           "sample": "%d steps of %d slates of the same workload: the unmodified reference classes (baseline/_ref) on "
                     "torch CPU, %d threads" % (n, b, torch.get_num_threads())}
    return ref, port


def gpu_library_baseline(w, sd, env_sd, mode, device, seconds):
    """The unmodified reference classes on the B200 through stock PyTorch (cuBLAS sgemm + ATen max / multinomial):
    the GPU-library baseline of SURVEY §8 d5.  The (B*L, N) logits it materialises bound the batch."""
    from baseline import ref_runner
    if not ref_runner.available():
        return None
    rows = max(1, int((6 << 30) // (w["n_items"] * 4 * (4 if mode == "sampled" else 1))))   # <= 6 GiB of logits
    B = int(max(16, min(w["B"], rows // w["L"])))
    try:
        v, n, b = ref_runner.time_generate(w, structs(w), sd, env_sd, mode, device, lambda i: make_inputs(w, B, i), seconds, warmup=2)
    except Exception as e:     # noqa: BLE001 - reported, never fatal for the bench
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
    finally:
        gc.collect()
        torch.cuda.empty_cache()
    return {"value": v, "unit": "slates/s", "impl": "unmodified reference classes, device=%s, stock PyTorch %s" % (device, torch.__version__),
            "sample": "%d steps of %d slates (host inputs, .cpu() of the scores: the reference's own eval loop)" % (n, b)}


def parity_check(w, sd, env_sd, mode, model, env, device):
    """GPU slates == CPU-arm slates on one shared batch (same weights, inputs and eps), with the engines of the timed
    region.  -> (ok, detail).  With the FFMA MLP engine everything is bit-identical.  The tcgen05 MLP engine is fp32-grade
    but not bit-identical to the FMA chain: response scores are held to north_star's 1e-4, and a slot that differs is
    reported with the CPU arm's own score gap between its pick and the GPU's pick (a near-tie when ~1e-6)."""
    import oracle
    rows = int(max(8, min(64, (1 << 26) // w["n_items"])))
    oracle.set_threads(os.cpu_count() or 1)
    ctx, users = make_inputs(w, rows, 0, seed=777)
    eps = np.random.default_rng(5).standard_normal((rows, w["Z"])).astype(np.float32)
    noise = np.random.default_rng(6).exponential(size=(rows, w["n_items"])).astype(np.float32) if mode == "sampled" else None
    if mode == "list":
        ref = oracle.list_recommend(sd, ctx.numpy(), users.numpy(), eps, w["no_user"])
    else:
        ref = oracle.pivot_recommend(sd, ctx.numpy(), users.numpy(), eps, w["no_user"], "sample" if mode == "sampled" else "max", noise)
    items_cpu = ref["items"]
    resp_cpu = oracle.resp_mlp(env_sd, items_cpu.reshape(rows, -1), users.numpy(), w["no_user"])
    oracle.set_threads(1)
    tc = getattr(model, "mlp_engine", None) in ("tc", "auto")
    saved = model.mlp_engine, env.mlp_engine
    if tc:
        model.mlp_engine = env.mlp_engine = "tc"       # "auto" would pick the FFMA engine for this small batch
    try:
        model.noise.push("eps", torch.from_numpy(eps).to(device))
        if noise is not None:
            model.noise.push("race", torch.from_numpy(noise).to(device))
        items, _ = model.recommend(ctx.to(device), None if w["no_user"] else users.to(device), return_item=True)
        resp = env(torch.from_numpy(items_cpu).to(device).view(rows, -1), users.to(device))
    finally:
        model.mlp_engine, env.mlp_engine = saved
    items = items.cpu().numpy()
    same = bool(np.array_equal(items, items_cpu))
    detail = {"rows": rows, "slots": int(items.size), "mismatching_slots": int((items != items_cpu).sum()),
              "mlp_engine": "tc" if tc else "exact"}
    if not same:
        W = sd["docEmbed.weight"]
        q = ref["rx"].reshape(-1, W.shape[1]).astype(np.float64)
        bad = np.nonzero(items != items_cpu)[0]
        gaps = [float(q[i] @ W[items_cpu[i]].astype(np.float64) - q[i] @ W[items[i]].astype(np.float64)) for i in bad[:64]]
        detail["cpu_score_gap_of_mismatches_max"] = max(gaps)
    if tc:
        ok = same and bool(np.allclose(resp.cpu().numpy(), resp_cpu, rtol=1e-4, atol=1e-5))
        detail["resp_max_abs_diff"] = float(np.abs(resp.cpu().numpy() - resp_cpu).max())
    else:
        ok = same and bool(np.array_equal(resp.cpu().numpy(), resp_cpu))
    return ok, detail


# ------------------------------------------------------------------ generation measurement
def measure_generate(D, args, wname, mode, vp=False, full=True, cpu_seconds=0.0, dump=None, steps=None):
    """One (workload, mode) measurement -> dict with value / e2e / roofline (/ cpu_baseline when cpu_seconds > 0).
    dump: directory for rank 0's slates, z_mu and response scores of the last timed step.  steps: timed steps
    (default --steps)."""
    from pivotcvae_b200 import ops
    from pivotcvae_b200.graphs import GraphedSlateGenerator
    w = WORKLOADS[wname]
    device, world, rank = D.device, D.world, D.rank
    B, K, W = (args.batch or w["B"]), (steps or args.steps), args.warmup
    sd, env_sd = make_weights(w, "list" if mode == "list" else "pivot")
    model, env = build_gpu(w, sd, env_sd, mode, device)
    model.noise.reseed(1234 + (0 if vp else rank))   # vocab-parallel ranks replicate inputs AND noise
    model.select_engine = args.engine
    model.mlp_engine = env.mlp_engine = args.mlp_engine
    no_user = w["no_user"]
    parity = None
    if full and not vp and rank == 0:
        parity, parity_detail = parity_check(w, sd, env_sd, mode, model, env, device)
    if vp:
        model.enable_vocab_parallel()

    ctxs, userss = zip(*[make_inputs(w, B, i, seed=1234 + (0 if vp else 7919 * rank)) for i in range(K)])
    ctx_d, usr_d = [c.to(device) for c in ctxs], [u.to(device) for u in userss]
    ctx_h, usr_h = [c.pin_memory() for c in ctxs], [u.pin_memory() for u in userss]
    items_h = torch.empty(B * w["L"], dtype=torch.int64).pin_memory()
    resp_h = torch.empty(B, w["L"], dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)  # > 126 MB L2

    vp_equal = None
    if vp:      # the sharded result must be the 1-GPU result: same batch, same noise, unsharded model on this rank
        ref_model, _ = build_gpu(w, sd, env_sd, mode, device)
        ref_model.noise.reseed(4321)
        model.noise.reseed(4321)
        a, _ = model.recommend(ctx_d[0], None if no_user else usr_d[0], return_item=True)
        b_, _ = ref_model.recommend(ctx_d[0], None if no_user else usr_d[0], return_item=True)
        vp_equal = bool(torch.equal(a, b_))
        del ref_model, a, b_
        model.noise.reseed(1234)
    # the whole step (recommend + response score) is one CUDA graph over static buffers; the Philox row counter
    # lives on the device, so every replay draws fresh noise.  Vocab-parallel: the NCCL all-reduces are captured too.
    gen = GraphedSlateGenerator(model, env, B, warmup=3)

    ms = timed_steps(D, lambda i: gen(ctx_d[i], usr_d[i]), K, W, flush)
    if dump and rank == 0:
        dump_outputs(dump, {"items": gen.items, "z_mu": gen.z_mu, "resp": gen.resp})

    def e2e_step(i):
        items, resp = gen(ctx_h[i], usr_h[i])      # pinned host -> static device buffers
        items_h.copy_(items, non_blocking=True)
        resp_h.copy_(resp, non_blocking=True)
    ms_e2e = timed_steps(D, e2e_step, K, min(W, 3), flush)

    total = B * (1 if vp else world) * K      # vocab-parallel: all ranks work on the SAME batch (strong scaling)
    out = {"workload": wname, "mode": mode, "model": MODEL_OF_MODE[mode], "metric": "generated slates/sec (%s)" % mode,
           "value": total / (ms / 1e3), "unit": "slates/s", "ms_per_step": ms / K, "batch_per_gpu": B, "steps": K,
           "timed_region_s": ms / 1e3,
           "e2e": {"value": total / (ms_e2e / 1e3), "unit": "slates/s", "h2d_bytes_per_step": int(B * w["L"] * 4 + B * 8),
                   "d2h_bytes_per_step": int(B * w["L"] * 8 + B * w["L"] * 4), "ms_per_step": ms_e2e / K},
           "launches_per_step": gen.launches_per_step, "gpu_launches": int(gen.launches_per_step * K)}
    if parity is not None:
        out["parity_check"] = parity
        out["parity_detail"] = parity_detail
    if vp:
        out["slates_equal_1gpu"] = vp_equal
        out["scaling"] = "strong"
        out["parallelism"] = ("vp%d (per-slot scoring: catalog rows sharded, one all-reduce(MAX) of int64 keys; MLP blocks, pivot pick "
                              "and response model: batch rows sharded, one all-gather of [rx | z_mu] and one of the scores; "
                              "3 NCCL collectives per step, all inside the step graph)" % world)

    # ---- roofline of the dominant kernel: the per-slot score+select over the catalog.  Events cannot sit inside
    # a graph replay, so the call alone (its kernels, on the decoder's own queries) is captured as its own graph
    # and replayed between event pairs with the L2 flushed; per-call times of the rest come from eager launches.
    if rank == 0 or vp:
        KP = min(K, 20)
        with ops.KernelTimer() as kt:
            for i in range(KP):
                flush.zero_()
                gen.load_inputs(ctx_d[i], usr_d[i])
                gen._step()
        D.barrier() if vp else torch.cuda.synchronize()
        ksum = kt.summary()
        L_, Dm = w["L"], w["D"]
        N = model.item_table().n_rows
        key = "score_select_greedy_M%d" % (B * L_)
        dom_ms, eager_ms = None, ksum.get(key, {}).get("ms_avg")
        if not vp:
            seen = {}
            orig_select = model._select

            def spy(q, mode="greedy", **kw):
                if mode == "greedy" and q.shape[0] == B * L_:
                    seen["q"] = q.detach().clone()
                return orig_select(q, mode, **kw)
            model._select = spy
            try:
                gen._step()
            finally:
                model._select = orig_select
            if "q" in seen:
                torch.cuda.synchronize()
                sg = torch.cuda.CUDAGraph()
                with torch.cuda.graph(sg):
                    seen["out"] = orig_select(seen["q"])
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KP)]
                for a, b in evs:
                    flush.zero_()
                    a.record()
                    sg.replay()
                    b.record()
                torch.cuda.synchronize()
                dom_ms = sum(a.elapsed_time(b) for a, b in evs) / KP
        if dom_ms is None:
            dom_ms = eager_ms or float("nan")
        pk = peaks()
        peak_tf = pk.get("bf16_tflops", 1590.0)
        flops = 2.0 * Dm * N * (B * L_)
        ach = flops / (dom_ms * 1e-3) / 1e12
        tc = args.engine in ("auto", "tcgen05", "tcgen05_f16") and N >= 2048
        f16 = tc and Dm == 8 and args.engine != "tcgen05"
        kname = (("score_select_tc_kernel (tcgen05 kind::%s filter) + tc_refine_kernel (exact fp32)" % ("f16, f16 accumulators" if f16 else "tf32"))
                 if tc else "score_select_kernel<D=%d> (exact fp32 SIMT) + finalize" % Dm)
        out["roofline"] = {
            "bound": "tensor", "kernel": "%s, M=%d rows x N=%d items, D=%d" % (kname, B * L_, N, Dm),
            "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
            "peak_source": (("MEASURED_PEAKS.json bf16_tflops (burst, cuBLAS bf16; %s)" % (
                                "the kernel is kind::f16 with K = 16, of which D = 8 are real dimensions" if f16 else
                                "the kernel is kind::tf32 whose nominal peak is half of bf16's"))
                            if pk else "fallback 1590 (B200_PROFILING.md)"),
            "traffic": traffic_of(wname, B * L_, N) if not vp else None,
            "algorithmic_bytes": N * Dm * 4 + B * L_ * (Dm * 4 + 8), "ms_avg_launch": dom_ms,
            "logits_per_s": (B * L_) * N / (dom_ms * 1e-3),
            # at D = 8 the consumer of the logits bounds the kernel (SURVEY H2).  Measured (profiles/micro/tmem_f16.cu): a
            # 128 x 256 tile is read from TMEM in 277 cycles as fp32 and in 142 cycles as packed f16; the MMA that makes it takes 128
            "epilogue_roofline": {"note": "TMEM read of the accumulators, measured: 128x256 logits per %d cycles per SM (%s); the MMA "
                                          "producing them takes 128" % ((142, "f16, .pack::16b") if f16 else (277, "fp32")),
                                  "peak_logits_per_s": 32768 / (142.0 if f16 else 277.0) * 148 * 1.965e9,
                                  "frac": (B * L_) * N / (dom_ms * 1e-3) / (32768 / (142.0 if f16 else 277.0) * 148 * 1.965e9)},
            "share_of_step": dom_ms / (ms / K),
            "timing": "CUDA events around a graph replay of the call alone on the decoder's queries, L2 flushed, %d replays after "
                      "the timed region (eager launch of the same call: %s ms)" % (KP, "%.4f" % eager_ms if eager_ms else "n/a"),
            "per_call_ms": {k: round(v["ms_avg"], 4) for k, v in ksum.items()}}
    if cpu_seconds > 0 and rank == 0 and not vp:
        out["cpu_baseline"], out["cpu_port"] = cpu_baselines(w, sd, env_sd, mode, cpu_seconds)
    del gen, model, env, flush
    gc.collect()
    torch.cuda.empty_cache()
    return out, (w, sd, env_sd)


def traffic_of(wname, M, N):
    """dram bytes per launch of the dominant kernel from the ncu capture of THIS build (profiles/traffic.json
    carries the source digest of the build it was captured on); null when the capture is of another build."""
    try:
        from pivotcvae_b200 import build as b
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        e = t.get(wname)
        if e and e.get("M") == M and e.get("N") == N and t.get("kernel_digest") == b.kernel_digest("score_select_tc.cu"):
            return e["bytes"]
    except Exception:
        pass
    return None


# ------------------------------------------------------------------ training measurement
def measure_train(D, args, wname, n_neg_arg, ce_engine, cpu_seconds=0.0, dump=None, steps=None):
    """train samples/sec: get_gen_loss (prior + encoder + decoder + fused catalog CE + KL) -> backward -> Adam.step.
    dump: directory for rank 0's loss, recLoss, KLD and trained parameters after the last timed step.  steps: timed
    steps (default --steps)."""
    import torch.distributed as dist
    from pivotcvae_b200 import ops
    from pivotcvae_b200.train_generative import get_gen_loss
    w = WORKLOADS[wname]
    device, world, rank = D.device, D.world, D.rank
    B, K, W = (args.batch or w["B"]), (steps or args.steps), args.warmup
    sd, env_sd = make_weights(w, "pivot")
    model, _ = build_gpu(w, sd, env_sd, "greedy", device)
    model.noise.reseed(99 + rank)
    model.ce_engine = ce_engine
    n_neg = w["n_items"] if n_neg_arg <= 0 else n_neg_arg
    tf32 = ce_engine == "tf32" and n_neg >= w["n_items"]
    # the reduced-precision training config also runs the MLP-gradient GEMMs in one tf32 pass (own tcgen05 GEMMs,
    # csrc/gemm_tc.cu); the fp32 config uses the same kernels with the 3xTF32 split
    from pivotcvae_b200 import autograd as _ag
    _ag.MLP_BWD_ENGINE = "tc" if tf32 else "tc3"
    # Adam stays torch's (SURVEY K18); fused=True = ONE multi-tensor kernel per step instead of ~15 foreach launches
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, capturable=(world == 1), fused=True)
    params = [p for p in model.parameters() if p.requires_grad]
    batches = [make_train_batch(w, B, i, seed=4321 + 7919 * rank) for i in range(K)]
    dev_batches = [{k: v.to(device) for k, v in b.items()} for b in batches]
    pin_batches = [{k: v.pin_memory() for k, v in b.items()} for b in batches]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()

    def eager_step(batch):
        opt.zero_grad(set_to_none=True)
        loss, rec, kld = get_gen_loss(batch, model, None, 0.001, n_neg=n_neg)
        loss.backward()
        if world > 1:      # data-parallel: one all-reduce of the (~270k fp32) MLP gradients per step
            flat = torch.cat([p.grad.reshape(-1) for p in params if p.grad is not None])
            dist.all_reduce(flat)
            flat /= world
            o = 0
            for p in params:
                if p.grad is not None:
                    n = p.grad.numel()
                    p.grad.copy_(flat[o:o + n].view_as(p.grad))
                    o += n
        opt.step()
        return loss, rec, kld

    graphed = None
    if world == 1:     # single GPU: the whole step is one CUDA graph (the DP arm keeps the eager NCCL all-reduce)
        from pivotcvae_b200.graphs import GraphedTrainStep
        graphed = GraphedTrainStep(model, opt, B, 0.001, n_neg)
        run = graphed
    else:
        run = eager_step
    last, step_launches = {}, []

    def step(i):
        l0 = ops.launch_count()
        last["out"] = run(dev_batches[i])
        step_launches.append(ops.launch_count() - l0)
    ms = timed_steps(D, step, K, W, flush)
    # a graph replay launches no kernel from the host: its count is the one taken at capture
    launches = graphed.launches_per_step * K if graphed else sum(step_launches[-K:])
    if dump and rank == 0:
        loss, rec, kld = last.pop("out")
        dump_outputs(dump, dict({"loss": loss, "rec_loss": rec, "kld": kld},
                                **{"param." + k: v for k, v in model.named_parameters() if v.requires_grad}))

    def e2e_step(i):
        if graphed:
            loss = run(pin_batches[i])[0]
        else:
            loss = run({k: v.to(device, non_blocking=True) for k, v in pin_batches[i].items()})[0]
        loss_h.copy_(loss.detach(), non_blocking=True)
    ms_e2e = timed_steps(D, e2e_step, K, min(W, 3), flush)

    # per-kernel CUDA-event timing of the same step launched eagerly (roofline of the dominant kernel)
    with ops.KernelTimer() as kt:
        for i in range(min(K, 10)):
            flush.zero_()
            if graphed:
                for k_, v_ in graphed.static.items():
                    v_.copy_(dev_batches[i][k_].reshape(v_.shape))
                graphed._step()
            else:
                eager_step(dev_batches[i])
    D.barrier()
    ksum = kt.summary()
    total = B * world * K
    L_, Dm, N = w["L"], w["D"], w["n_items"]
    dom = ksum.get("ce_fwd_bwd", {"ms_avg": float("nan"), "calls": 0})
    peak_tf = peaks().get("bf16_tflops", 1590.0)
    keep = n_neg / N
    flops = (2.0 * Dm * N * B * L_ + 2.0 * Dm * N * B * (L_ - 1)) * keep   # logits + dq accumulation over kept items
    ach = flops / (dom["ms_avg"] * 1e-3) / 1e12
    out = {"workload": wname, "mode": "train", "model": MODEL_OF_MODE["train"],
           "metric": "train samples/sec (PivotCVAE gt, fused catalog CE + KL, fwd+bwd+Adam)", "value": total / (ms / 1e3),
           "unit": "samples/s", "ms_per_step": ms / K, "batch_per_gpu": B, "steps": K, "timed_region_s": ms / 1e3,
           "dtype": ("tf32 operands (logits, MLP gradient GEMMs), f32 accumulate" if tf32 else "f32"),
           "n_neg": n_neg, "beta": 0.001, "ce_engine": ce_engine,
           "e2e": {"value": total / (ms_e2e / 1e3), "unit": "samples/s",
                   "h2d_bytes_per_step": int(B * L_ * 8 + B * 8 + B * L_ * 4), "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K},
           "launches_per_step": graphed.launches_per_step if graphed else None, "gpu_launches": int(launches),
           "roofline": {"bound": "tensor", "kernel": "catalog CE fwd+bwd (%s engine, + finalize), M=%d rows x N=%d items, keep=%.4f" % (ce_engine, B * L_, N, keep),
                        "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": None,
                        "ms_avg_launch": dom["ms_avg"], "share_of_step": dom["ms_avg"] / (ms / K) if dom["calls"] else None,
                        "per_call_ms": {k: round(v["ms_avg"], 4) for k, v in ksum.items()}}}
    if cpu_seconds > 0 and rank == 0:
        from baseline import ref_runner
        if ref_runner.available():
            cb = 64
            torch.set_num_threads(os.cpu_count() or 1)

            def nb(i):
                b = make_train_batch(w, cb, i)
                return {"slates": b["slates"].numpy(), "users": b["users"].numpy(), "responses": b["responses"].numpy().astype(np.float64)}
            v, n, b = ref_runner.time_train(w, structs(w), sd, env_sd, "cpu", nb, n_neg, 0.001, cpu_seconds)
            out["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "reference",
                                   "sample": "%d steps of %d samples: unmodified reference get_gen_loss + backward + Adam (baseline/_ref), "
                                             "torch CPU %d threads" % (n, b, torch.get_num_threads())}
            gb = max(16, min(B, int((8 << 30) // (N * 4 * 8 * L_))))
            try:
                def gbatch(i):
                    b2 = make_train_batch(w, gb, i)
                    return {"slates": b2["slates"].numpy(), "users": b2["users"].numpy(), "responses": b2["responses"].numpy().astype(np.float64)}
                v, n, b = ref_runner.time_train(w, structs(w), sd, env_sd, device, gbatch, n_neg, 0.001, min(cpu_seconds, 3.0), warmup=2)
                out["gpu_library_baseline"] = {"value": v, "unit": "samples/s", "impl": "unmodified reference, device=%s, stock PyTorch" % device,
                                               "sample": "%d steps of %d samples" % (n, b)}
            except Exception as e:   # noqa: BLE001
                out["gpu_library_baseline"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
    del graphed, model, opt, flush
    gc.collect()
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------ arms
def base_config(args, w):
    return {"workload": w["desc"], "batch": args.batch or w["B"], "mode": args.mode, "model": MODEL_OF_MODE[args.mode]}


def run_reference(args, w):
    """CPU arm: the unmodified reference on the box's host cores (baseline/_ref; the oracle's C port only when
    the copy did not travel), all host threads, each step a bounded sample of the workload's batch."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from baseline import ref_runner
    mode = args.mode
    sd, env_sd = make_weights(w, "list" if mode == "list" else "pivot")
    threads = os.cpu_count() or 1
    K, W = args.steps, args.warmup
    if mode == "train":
        n_neg = w["n_items"] if args.n_neg <= 0 else args.n_neg
        cb = 64
        torch.set_num_threads(threads)

        def nb(i):
            b = make_train_batch(w, cb, i)
            return {"slates": b["slates"].numpy(), "users": b["users"].numpy(), "responses": b["responses"].numpy().astype(np.float64)}
        val, n, _ = ref_runner.time_train(w, structs(w), sd, env_sd, "cpu", nb, n_neg, 0.001, 1e9, warmup=W, max_steps=K)
        kind, unit, metric = "reference", "samples/s", "train samples/sec (PivotCVAE gt, fused catalog CE + KL, fwd+bwd+Adam)"
        sample = "%d steps of %d samples: unmodified reference (baseline/_ref), torch CPU %d threads" % (n, cb, threads)
    else:
        cb = cpu_sample_batch(w, mode)
        unit, metric = "slates/s", "generated slates/sec (%s)" % mode
        if ref_runner.available():
            torch.set_num_threads(threads)
            val, n, _ = ref_runner.time_generate(w, structs(w), sd, env_sd, mode, "cpu", lambda i: make_inputs(w, cb, i), 1e9,
                                                 warmup=W, max_steps=K)
            kind = "reference"
            sample = "%d steps of %d slates: unmodified reference classes (baseline/_ref), torch CPU %d threads" % (n, cb, threads)
        else:
            val, threads, n = time_cpu_port(w, sd, env_sd, mode, cb, 1e9, warmup=W, max_steps=K)
            kind = "port"
            sample = "%d steps of %d slates (oracle/pcv_oracle.c, pthreads x%d; baseline/_ref did not travel)" % (n, cb, threads)
    line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": cb / val * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": base_config(args, w),
            "cpu_baseline": {"value": val, "unit": unit, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


ALSO_GENERATE = [("c4", "sampled"), ("c2", "greedy"), ("c2", "sampled"), ("c2", "list"), ("c1", "greedy")]
ALSO_TRAIN = [("c3", 0, "tf32"), ("c3", 1000, "exact")]


def run_ours(args, w):
    from pivotcvae_b200 import ops
    D = Dist()
    D.start()
    ops.device_ok(D.local)
    clocks = ClockSampler(D.local)
    if D.rank == 0:
        clocks.start()
    is_default = not args.no_also and args.mode == "greedy" and args.workload == "c4" and not args.batch
    if args.mode == "train":
        main = measure_train(D, args, args.workload, args.n_neg, args.ce_engine,
                             cpu_seconds=0 if args.no_cpu else 8.0, dump=args.dump_outputs)
        wsd = None
    else:
        main, wsd = measure_generate(D, args, args.workload, args.mode, vp=(args.parallel == "vp" and D.world > 1),
                                     cpu_seconds=0 if (args.no_cpu or D.world > 1) else 12.0, dump=args.dump_outputs)
    clk = clocks.stop() if D.rank == 0 else None
    extra = {}
    if args.mode != "train" and args.parallel != "vp":
        if D.world > 1 and not args.no_vp:
            # the 1 M-item catalog sharded vocab-parallel over the same N GPUs (strong scaling on ONE batch)
            vpres, _ = measure_generate(D, args, args.workload, args.mode, vp=True, full=False)
            extra["vp"] = {k: vpres[k] for k in ("value", "unit", "ms_per_step", "batch_per_gpu", "e2e", "slates_equal_1gpu",
                                                 "scaling", "parallelism", "launches_per_step") if k in vpres}
            if "roofline" in vpres:
                extra["vp"]["per_call_ms"] = vpres["roofline"]["per_call_ms"]
        if D.world == 1 and D.rank == 0 and wsd is not None and not args.no_cpu:
            extra["gpu_library_baseline"] = gpu_library_baseline(wsd[0], wsd[1], wsd[2], args.mode, D.device, 3.0)
        if D.world == 1 and is_default:
            also = []
            for wn, md in ALSO_GENERATE:
                try:
                    r, s = measure_generate(D, args, wn, md, cpu_seconds=0 if args.no_cpu else 4.0, steps=WORKLOADS[wn]["steps"] // 2)
                    r["config"] = {"workload": WORKLOADS[wn]["desc"], "batch": WORKLOADS[wn]["B"], "mode": md, "model": MODEL_OF_MODE[md]}
                    if (wn, md) == ("c2", "greedy") and not args.no_cpu:
                        r["gpu_library_baseline"] = gpu_library_baseline(s[0], s[1], s[2], md, D.device, 2.0)
                    also.append(r)
                except Exception as e:     # noqa: BLE001 - a failed sub-result is reported, the headline stands
                    also.append({"workload": wn, "mode": md, "error": "%s: %s" % (type(e).__name__, str(e)[:300])})
            for wn, nn, eng in ALSO_TRAIN:
                try:
                    r = measure_train(D, args, wn, nn, eng, cpu_seconds=0 if args.no_cpu else 4.0, steps=WORKLOADS[wn]["steps"] // 2)
                    r["config"] = {"workload": WORKLOADS[wn]["desc"], "batch": WORKLOADS[wn]["B"], "mode": "train", "n_neg": r["n_neg"]}
                    also.append(r)
                except Exception as e:     # noqa: BLE001
                    also.append({"workload": wn, "mode": "train", "error": "%s: %s" % (type(e).__name__, str(e)[:300])})
            # the same headline config with the other engine of the MLP blocks: FFMA chain (bit-identical to the oracle) vs
            # tcgen05 3xTF32 (csrc/mlp_tc.cu: fp32-grade, gated on the reference fixtures and the parity check below)
            other = "tc" if args.mlp_engine == "exact" else "exact"
            saved_engine = args.mlp_engine
            try:
                args.mlp_engine = other
                r, _ = measure_generate(D, args, args.workload, args.mode, cpu_seconds=0, steps=w["steps"] // 2)
                also.append({"workload": args.workload, "mode": args.mode, "mlp_engine": other, "value": r["value"], "unit": r["unit"],
                             "ms_per_step": r["ms_per_step"], "steps": r["steps"], "parity_check": r.get("parity_check"),
                             "parity_detail": r.get("parity_detail"), "per_call_ms": r.get("roofline", {}).get("per_call_ms")})
            except Exception as e:     # noqa: BLE001
                also.append({"workload": args.workload, "mode": args.mode, "mlp_engine": other, "error": "%s: %s" % (type(e).__name__, str(e)[:300])})
            finally:
                args.mlp_engine = saved_engine
            extra["also"] = also
    D.stop()
    if D.rank != 0:
        return
    vp_main = args.parallel == "vp" and D.world > 1
    config = base_config(args, w)
    config.update({"parallelism": main.get("parallelism", "dp%d (replicated table, independent batches per GPU)" % D.world),
                   "batch_per_gpu": main["batch_per_gpu"],
                   "mlp_engine": ({"tc": "tcgen05 3xTF32, fp32-grade (csrc/mlp_tc.cu)", "exact": "FFMA chain, bit-identical to the oracle",
                                   "auto": "tcgen05 3xTF32 (csrc/mlp_tc.cu) for batches >= 2048 rows, FFMA chain below"}[args.mlp_engine])
                                 if args.mode != "train" else "training engine (saves activations)",
                   "l2": "flushed between steps (256 MiB write, outside the event pairs)",
                   "timing": "per-step CUDA-event pairs summed over the %d timed steps after %d warm-up steps, max over ranks"
                             % (args.steps, args.warmup),
                   "launch": "one CUDA graph replay per step (%s kernels of libpcv_b200)" % main.get("launches_per_step")})
    line = {"metric": main["metric"], "value": main["value"], "unit": main["unit"], "n_gpus": D.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "timed_region_s": main["timed_region_s"],
            "higher_is_better": True, "scaling": "strong" if vp_main else "weak", "vs_baseline": None,
            "dtype": main.get("dtype", "f32"), "data": "synthetic", "config": config, "e2e": main["e2e"],
            "gpu_launches": main["gpu_launches"], "roofline": main.get("roofline"), "cpu_baseline": main.get("cpu_baseline"),
            "clocks": clk}
    for k in ("cpu_port", "parity_check", "parity_detail", "slates_equal_1gpu", "gpu_library_baseline"):
        if k in main:
            line[k] = main[k]
    line.update(extra)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: the workload's, about 0.5 s on one B200; --impl reference: %d)" % REFERENCE_STEPS)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="greedy", choices=["greedy", "sampled", "list", "train"])
    ap.add_argument("--n-neg", type=int, default=0, help="train mode: negatives per row (0 = the whole catalog)")
    ap.add_argument("--ce-engine", default="tf32", choices=["exact", "tf32"],
                    help="train mode, full catalog: CE logits in exact fp32 (SIMT) or tf32 on the tensor cores (C3 is a reduced-precision config)")
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tcgen05", "tcgen05_f16"],
                    help="score+select engine: auto = tensor cores (dim 8: the f16 filter, else tf32) with the exact fp32 refine")
    ap.add_argument("--mlp-engine", default="auto", choices=["exact", "tc", "auto"],
                    help="fused MLP blocks at inference: tc = tcgen05 3xTF32 (fp32-grade), exact = FFMA chain bit-identical to the oracle, "
                         "auto = tc for batches of >= 2048 rows")
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--parallel", default="dp", choices=["dp", "vp"], help="N>1 headline: batch data-parallel (default) or vocab-parallel")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU / GPU-library baselines")
    ap.add_argument("--no-also", action="store_true", help="skip the sub-results of the default run")
    ap.add_argument("--no-vp", action="store_true", help="N>1: skip the vocab-parallel block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the slates, z_mu and response scores (train: loss terms and parameters) of the last timed step "
                         "of the headline measurement as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    w = WORKLOADS[args.workload]
    if args.workload == "c5" and args.mode == "greedy":
        args.mode = "sampled"      # C5 is the sampled-slates sweep
    if args.workload == "c3" and args.mode != "train":
        args.mode = "train"
    if args.steps is None:
        args.steps = REFERENCE_STEPS if args.impl == "reference" else w["steps"]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
