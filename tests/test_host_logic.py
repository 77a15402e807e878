"""CPU-only tests: the C ABI surface, ctypes struct layouts, host-side logic, the drop-in
import aliases and the world_size-2 (gloo) vocab-parallel exchange."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pcv_b200.h")


def _header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pcv_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from pivotcvae_b200 import _lib
    lib = _lib.load()           # loads without a GPU; no compute call is made here
    names = _header_functions()
    assert len(names) >= 22
    for n in names:
        assert hasattr(lib, n), "libpcv_b200.so does not export %s" % n
        assert n in _lib.EXPORTS, "%s is declared in the header but has no ctypes prototype" % n
    assert set(_lib.EXPORTS) == set(names)
    assert lib.pcv_abi_version() == 2
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (pcv_[a-z0-9_]+)", out))
    assert exported == set(names), exported ^ set(names)


def test_ctypes_structs_match_the_c_header(tmp_path):
    """sizeof/offsetof of every descriptor struct, compiled from the real header with gcc."""
    from pivotcvae_b200 import _lib
    checks = {"pcv_select_opts": (_lib.SelectOpts, ["mode", "engine", "noise", "seed", "offset", "no_repeat", "offset_dev"]),
              "pcv_linear": (_lib.Linear, ["W", "b", "n_in", "n_out", "act"]),
              "pcv_segment": (_lib.Segment, ["kind", "ptr", "idx", "width", "count", "norm"]),
              "pcv_mlp_desc": (_lib.MlpDesc, ["n_segments", "seg", "n_layers", "layer", "out", "out_ld", "out_col0",
                                              "copy_seg", "x0", "acts", "latent", "eps", "seed", "offset", "z", "eps_out", "offset_dev"]),
              "pcv_ce_mask": (_lib.CeMask, ["keep_prob", "bitmask", "seed", "offset", "offset_dev", "engine"]),
              "pcv_urm_desc": (_lib.UrmDesc, ["variant", "doc_table", "user_table", "item_bias", "user_bias", "pos_bias",
                                              "pos_dep", "mr_factor", "L", "D"])}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "pcv_b200.h"', "int main(void){"]
    for cname, (_, fields) in checks.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for f in fields:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, f, cname, f))
    lines.append("return 0;}")
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines())
    for cname, (cls, fields) in checks.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for f in fields:
            assert int(got["%s.%s" % (cname, f)]) == getattr(cls, f).offset, (cname, f)


def test_no_cpu_fallback_anywhere():
    """The product path must fail loudly without CUDA; nothing under pivotcvae_b200/ touches oracle/."""
    from pivotcvae_b200 import _lib, ops
    with pytest.raises(_lib.PcvError):
        ops.Table(torch.zeros(16, 8))
    with pytest.raises(_lib.PcvError):
        ops.score_logits(None, torch.zeros(4, 8))
    for dirpath, _, files in os.walk(os.path.join(ROOT, "pivotcvae_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "libpcv_oracle" not in txt, f
    if not torch.cuda.is_available():
        from pivotcvae_b200.models.pivotcvae import UserPivotCVAE
        emb = type("E", (), {"weight": torch.randn(50, 8)})()
        with pytest.raises(Exception):
            UserPivotCVAE(emb, emb, 5, 8, 16, 6, [54, 32, 32], [30, 32, 32, 8], [38, 32, 32, 32], [14, 16, 16], False, "cuda:0")


def test_dropin_aliases_and_registry():
    import pivotcvae_b200
    pivotcvae_b200.install_dropin()
    from models.pivotcvae import PIVOTCVAE_MODELS
    from models.listcvae import UserListCVAEWithPrior  # noqa: F401
    from env.response_model import URM_P_MR, UserResponseModel_MLP, sample_users  # noqa: F401
    import train_generative
    assert sorted(PIVOTCVAE_MODELS) == sorted(["pivotcvae_gt_pi", "pivotcvae_pt_pi", "pivotcvae_spt_pi", "pivotcvae_sgt_pi",
                                               "pivotcvae_gt_spi", "pivotcvae_pt_spi", "pivotcvae_spt_spi", "pivotcvae_sgt_spi"])
    picks = {k: (c.train_pick, c.infer_pick) for k, c in PIVOTCVAE_MODELS.items()}
    assert picks["pivotcvae_gt_pi"] == ("gt", "max") and picks["pivotcvae_sgt_spi"] == ("sample_gt", "sample")
    assert picks["pivotcvae_pt_spi"] == ("max", "sample") and picks["pivotcvae_spt_pi"] == ("sample", "max")
    for name in ("downsample", "get_gen_loss", "train_on_dataset", "get_model", "add_gen_model_parse", "main"):
        assert hasattr(train_generative, name)
    import analysis
    assert callable(analysis.get_coverage) and callable(analysis.get_ILS)
    import argparse
    with pytest.raises(ImportError, match="data modules"):      # data IO stays the reference's (out of scope)
        train_generative.main(argparse.Namespace(dataset="sim"))
    # the reference's class names resolve for whole-model pickles (train_generative.py:199)
    import models.pivotcvae as mp
    for cls in ("UserPivotCVAE", "UserPivotCVAE2", "UserPivotCVAE_PrePermute", "UserPivotCVAE_PrePermute2",
                "UserPivotCVAE_PrePermute3", "UserPivotCVAE_PrePermute4", "UserPivotCVAE_PrePermute5",
                "UserPivotCVAE_PrePermute6"):
        assert getattr(mp, cls).__name__ == cls


def test_noise_source_streams_do_not_overlap():
    from pivotcvae_b200.noise import NoiseSource
    ns = NoiseSource(seed=5)
    a = ns.next_stream(100)
    b = ns.next_stream(7)
    c = ns.next_stream(1)
    assert a == (5, 0) and b == (5, 100) and c == (5, 107)
    ns.push("eps", "E1")
    ns.push("eps", "E2")
    assert ns.pop("eps") == "E1" and ns.pop("eps") == "E2" and ns.pop("eps") is None and ns.pop("race") is None
    ns.reseed(9)
    assert ns.next_stream(3) == (9, 0)


def test_downsample_semantics():
    """pred * (onehot(target) U Bernoulli): masked-out logits are 0, targets always kept (SURVEY F7)."""
    from pivotcvae_b200.train_generative import downsample
    torch.manual_seed(0)
    pred = torch.randn(64, 200) + 3.0
    tgt = torch.randint(0, 200, (64,))
    out = downsample(pred, tgt, n_neg=20)
    kept = out != 0
    assert bool(kept[torch.arange(64), tgt].all())
    assert torch.equal(out[kept], pred[kept])
    assert 0.05 < kept.float().mean() < 0.2
    full = downsample(pred, tgt, n_neg=200)
    assert torch.equal(full, pred)


def test_shard_bounds_cover_and_align():
    from pivotcvae_b200.parallel import shard_bounds
    for n in (1, 127, 128, 129, 50000, 1000000, 10_000_019):
        for world in (1, 2, 4, 8):
            spans = [shard_bounds(n, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for (lo, hi), (lo2, _) in zip(spans, spans[1:]):
                assert hi == lo2 and lo <= hi
            assert all(lo % 128 == 0 for lo, hi in spans if hi > lo)


def test_merge_partials_tie_rule():
    from pivotcvae_b200.parallel import merge_partials
    vals = torch.tensor([[1.0, 5.0, 2.0, -0.0], [1.0, 4.0, 3.0, 0.0], [0.5, 5.0, 3.0, -1.0]])
    idx = torch.tensor([[10, 11, 12, 13], [110, 111, 112, 113], [210, 211, 212, 213]])
    mi, mv = merge_partials(vals, idx)
    assert mi.tolist() == [10, 11, 112, 13] and mv.tolist() == [1.0, 5.0, 3.0, 0.0]


def _vp_worker(rank, world, port, tmpdir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import oracle
    from pivotcvae_b200.parallel import VocabParallelSelector, shard_bounds
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(7)          # identical on every rank (replicated inputs)
    n_items, M, D = 1000, 37, 8
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    W[900] = W[100]                          # exact tie across shards: lowest global index must win
    Q = rng.standard_normal((M, D)).astype(np.float32)
    Q[0] = W[100]
    lo, hi = shard_bounds(n_items, world, rank)

    def local(q):                            # stand-in for ops.score_select on the local shard
        i, v = oracle.score_select(W[lo:hi], q.numpy())
        return torch.from_numpy(i + lo), torch.from_numpy(v)

    idx, val = VocabParallelSelector(local)(torch.from_numpy(Q))
    fi, fv = oracle.score_select(W, Q)
    ok = np.array_equal(idx.numpy(), fi) and np.array_equal(val.numpy(), fv) and int(idx[0]) == 100
    open(os.path.join(tmpdir, "ok%d" % rank), "w").write("1" if ok else "0")
    dist.barrier()
    dist.destroy_process_group()


def test_vocab_parallel_gloo_world2(tmp_path):
    """N>1 path on CPU: 2 ranks, gloo, one all-gather per scoring step, merged == one-shot."""
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_vp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").read_text() == "1" and (tmp_path / "ok1").read_text() == "1"


def _vp_ce_worker(rank, world, port, tmpdir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import oracle
    from pivotcvae_b200.parallel import local_ce_partials, merge_ce_partials, shard_bounds
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(11)
    n_items, M, D = 777, 23, 8
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = (2.0 * rng.standard_normal((M, D))).astype(np.float32)
    tgt = rng.integers(0, n_items, M)
    lo, hi = shard_bounds(n_items, world, rank)
    rec = local_ce_partials(torch.from_numpy(W[lo:hi]), torch.from_numpy(Q))        # stand-in for pcv_ce_partials
    recs = torch.empty(world * rec.shape[0], rec.shape[1])
    dist.all_gather_into_tensor(recs, rec)                                          # the ONE collective of the step
    recs = recs.view(world, rec.shape[0], rec.shape[1])
    loss, lse, dq = merge_ce_partials(recs, torch.from_numpy(W), torch.from_numpy(Q), torch.from_numpy(tgt))
    ol, olse, odq = oracle.ce(W, Q, tgt)
    ok = (np.allclose(loss.numpy(), ol, rtol=1e-4, atol=1e-5) and np.allclose(lse.numpy(), olse, rtol=1e-4, atol=1e-5)
          and np.allclose(dq.numpy(), odq, rtol=1e-3, atol=1e-5))
    open(os.path.join(tmpdir, "ce_ok%d" % rank), "w").write("1" if ok else "0")
    dist.barrier()
    dist.destroy_process_group()


def test_vocab_parallel_ce_gloo_world2(tmp_path):
    """Vocab-parallel training exchange on CPU: 2 ranks, gloo, one all-gather of {m, l, acc[D]} records, merged
    loss / lse / dq == the unsharded oracle CE (1e-4)."""
    import torch.multiprocessing as mp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_vp_ce_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ce_ok0").read_text() == "1" and (tmp_path / "ce_ok1").read_text() == "1"


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the unmodified reference from baseline/_ref on the host cores when that copy
    exists, else the oracle port) prints the contract line, with the SAME config dict as the GPU arm would."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    have_ref = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "models", "pivotcvae.py"))
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["config"] == {"workload": line["config"]["workload"], "batch": 64, "mode": "greedy", "model": "PivotCVAE gt_pi"}
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["unit"] == "slates/s"


def test_bench_dump_outputs_dtypes_and_size_limit(tmp_path, monkeypatch):
    """bench.dump_outputs: item ids as float64, scores as float32, scalars whole; past DUMP_LIMIT every array keeps the
    same fixed sample of its rows, stored beside it as <name>.rows.npy."""
    import bench
    arrays = {"items": torch.arange(5000, dtype=torch.int64).view(1000, 5) * 977, "resp": torch.randn(1000, 5),
              "loss": torch.tensor(0.25, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    items, resp, loss = (np.load(tmp_path / "all" / (k + ".npy")) for k in ("items", "resp", "loss"))
    assert items.dtype == np.float64 and np.array_equal(items, arrays["items"].numpy())
    assert resp.dtype == np.float32 and np.array_equal(resp, arrays["resp"].numpy())
    assert loss.dtype == np.float64 and loss == 0.25
    assert sorted(os.listdir(tmp_path / "all")) == ["items.npy", "loss.npy", "resp.npy"]
    monkeypatch.setattr(bench, "DUMP_LIMIT", 30000)
    for run in ("cut", "cut_again"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    for k in ("items", "resp"):
        rows = np.load(tmp_path / "cut" / (k + ".rows.npy"))
        got = np.load(tmp_path / "cut" / (k + ".npy"))
        assert 0 < len(rows) < 1000 and (np.diff(rows) > 0).all()
        assert np.array_equal(got, arrays[k].numpy()[rows.astype(np.int64)].astype(got.dtype))
        assert np.array_equal(rows, np.load(tmp_path / "cut_again" / (k + ".rows.npy")))
    assert sum(f.stat().st_size for f in (tmp_path / "cut").iterdir()) <= 30000
    assert np.load(tmp_path / "cut" / "loss.npy") == 0.25


def test_bench_times_exactly_k_steps(monkeypatch):
    """bench.timed_steps: the W warm-up steps run before the first event; then exactly K steps, each alone between the
    two events of its pair, and the result is the sum of the K pairs."""
    import bench
    log = []

    class Event:
        def __init__(self, enable_timing=False):
            self.id = len([e for e in log if e[0] == "new"])
            log.append(("new", self.id))

        def record(self):
            log.append(("record", self.id))

        def elapsed_time(self, end):
            return 1.5

    class Dist:
        def barrier(self):
            log.append(("barrier",))

        def max_(self, values):
            return values

    class Flush:
        def zero_(self):
            log.append(("flush",))

    monkeypatch.setattr(torch.cuda, "Event", Event)
    K, W = 7, 3
    ms = bench.timed_steps(Dist(), lambda i: log.append(("step", i)), K, W, Flush())
    assert ms == 1.5 * K
    first = log.index(next(e for e in log if e[0] == "record"))
    assert [e for e in log[:first] if e[0] == "step"] == [("step", i % K) for i in range(W)]
    timed = [e for e in log[first:] if e[0] != "flush"]
    assert timed[:-1] == [x for i in range(K) for x in (("record", 2 * i), ("step", i), ("record", 2 * i + 1))]
    assert timed[-1] == ("barrier",)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(argv):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and "error" in out.stderr


def test_mlp_engine_policy_is_validated_and_scoped():
    """ops.mlp_engine: context manager over the process default; unknown names are rejected; the library default is the
    bit-exact FFMA engine and the model classes default to it (mlp_engine = None)."""
    from pivotcvae_b200 import ops
    from pivotcvae_b200.models.cvae import BaseCVAE
    from pivotcvae_b200.env.response_model import UserResponseModel_MLP
    assert ops.MLP_ENGINE == "exact" and BaseCVAE.mlp_engine is None and UserResponseModel_MLP.mlp_engine is None
    with ops.mlp_engine("tc"):
        assert ops.MLP_ENGINE == "tc"
        with ops.mlp_engine("auto"):
            assert ops.MLP_ENGINE == "auto"
        assert ops.MLP_ENGINE == "tc"
    assert ops.MLP_ENGINE == "exact"
    with pytest.raises(ValueError):
        ops.mlp_engine("bf16")


def test_f16_filter_error_bound_in_numpy():
    """The band of the f16 select filter (csrc/score_select_tc.cu) rests on |a~ - (s' + 1)| <= 2^-9 for
    a~ = f16(sum_k f16(q'_k) f16(w_k) + 1), q' = q * 0.99 / (|q| max|w| 1.003): operands rounded to nearest (2^-11 each),
    products and the 9-term sum exact in the tensor core, ONE final conversion of a value in (0, 2) to f16 (truncation
    assumed: the worse case).  Emulated here in float64 / float16 over random and adversarial rows; also: the shifted
    scores are strictly positive and below 2, so their f16 bit patterns order like unsigned integers."""
    rng = np.random.default_rng(0)

    def trunc_f16(x):      # round toward zero to float16 (positive inputs)
        h = x.astype(np.float16)
        too_big = h.astype(np.float64) > x
        return np.where(too_big, np.nextafter(h, np.float16(0)), h).astype(np.float16)

    worst = 0.0
    for trial in range(40):
        n = 4000
        W = rng.standard_normal((n, 8)) * rng.uniform(0.01, 30.0)
        if trial % 3 == 0:
            W /= np.linalg.norm(W, axis=1, keepdims=True)
        W = W.astype(np.float32)
        q = (rng.standard_normal(8) * 10.0 ** rng.uniform(-6, 6)).astype(np.float32)
        if trial % 5 == 0:
            q = (W[rng.integers(n)] * rng.uniform(0.1, 50)).astype(np.float32)       # parallel to an item: score at the ceiling
        if trial % 7 == 0:
            q = (-W[rng.integers(n)] * rng.uniform(0.1, 50)).astype(np.float32)      # anti-parallel: shifted score near 0
        wmax = float(np.linalg.norm(W.astype(np.float64), axis=1).max()) * 1.000001 * 1.003
        c = np.float32(0.99) / np.float32(np.sqrt(np.float32((q.astype(np.float64) ** 2).sum())) * np.float32(wmax))
        qs = (q * c).astype(np.float32)
        exact = W.astype(np.float64) @ qs.astype(np.float64) + 1.0                  # s' + 1
        approx = W.astype(np.float16).astype(np.float64) @ qs.astype(np.float16).astype(np.float64) + 1.0
        assert approx.min() > 0.0 and approx.max() < 2.0
        a16 = trunc_f16(approx)
        assert (a16.view(np.uint16) > 0).all() and (a16.astype(np.float64) < 2.0).all()
        worst = max(worst, float(np.abs(a16.astype(np.float64) - exact).max()))
        # unsigned order of the bit patterns == order of the values
        order = np.argsort(a16.astype(np.float64), kind="stable")
        assert (np.diff(a16.view(np.uint16)[order].astype(np.int64)) >= 0).all()
    assert worst <= 2.0 ** -9, worst
    assert 2.0 * 1.25 * 2.0 ** -9 >= 2.0 * worst        # the band the kernel uses (TC_H_BAND)
