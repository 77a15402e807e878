"""The throughput-mode sampled pivot (csrc/sampler.cu): exact rejection sampling from
Categorical(sigmoid(scores)) (pivotcvae.py:349-351).  CPU legs check the oracle restatement's DISTRIBUTION
against the exact probabilities (chi-square) and its edge cases; GPU legs check the CUDA kernel bit for bit
against the oracle, and the model-level path."""
import numpy as np
import pytest
import torch

import oracle


def _table(rng, n, D):
    W = rng.standard_normal((n, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    return W


def _chi2_ok(counts, probs, z=5.0):
    """Pearson chi-square against `probs` within z sigmas of its expectation (dof = k-1, var = 2 dof)."""
    n = counts.sum()
    exp = probs * n
    chi2 = ((counts - exp) ** 2 / exp).sum()
    dof = len(probs) - 1
    return abs(chi2 - dof) <= z * np.sqrt(2 * dof) + 1e-9, chi2, dof


@pytest.mark.parametrize("scale", [0.5, 3.0, 8.0])
def test_oracle_sampler_distribution(scale):
    rng = np.random.default_rng(17)
    W = _table(rng, 37, 8)
    q = (scale * rng.standard_normal(8) / np.sqrt(8)).astype(np.float32).reshape(1, 8)
    M = 200000
    idx, iters = oracle.sigmoid_categorical(W, np.repeat(q, M, 0), seed=1234, offset=77)
    p = 1.0 / (1.0 + np.exp(-(W.astype(np.float64) @ q[0].astype(np.float64))))
    ok, chi2, dof = _chi2_ok(np.bincount(idx, minlength=37).astype(np.float64), p / p.sum())
    assert ok, (chi2, dof)
    assert (iters > 0).all()
    # ~ sigma_b / mean(p) proposals per row
    assert iters.mean() < 1.05 * (1.0 / (1.0 + np.exp(-np.linalg.norm(q) * 1.0002))) / p.mean() + 0.1


def test_oracle_sampler_streams_and_fallback():
    rng = np.random.default_rng(3)
    W = _table(rng, 1000, 8)
    Q = rng.standard_normal((64, 8)).astype(np.float32)
    a, _ = oracle.sigmoid_categorical(W, Q, seed=5, offset=0)
    b, _ = oracle.sigmoid_categorical(W, Q, seed=5, offset=0)
    c, _ = oracle.sigmoid_categorical(W, Q, seed=5, offset=64)
    d, _ = oracle.sigmoid_categorical(W, Q, seed=6, offset=0)
    assert np.array_equal(a, b) and not np.array_equal(a, c) and not np.array_equal(a, d)
    # rows 32.. of a call at offset 0 are rows 0.. of a call at offset 32 (row counter = row + offset)
    e, _ = oracle.sigmoid_categorical(W, Q[32:], seed=5, offset=32)
    assert np.array_equal(a[32:], e)
    # pathological acceptance rate: every item opposite to a huge q except one aligned -> sigma_b = 1,
    # mean sigmoid ~ 1/N: most rows exhaust 1024 proposals and take the inverse-CDF fallback, which must pick item 0
    Wp = np.tile(-np.eye(8, dtype=np.float32)[0], (400, 1))
    Wp[0] = np.eye(8, dtype=np.float32)[0]
    q = (60 * np.eye(8, dtype=np.float32)[0]).reshape(1, 8)
    idx, iters = oracle.sigmoid_categorical(Wp, np.repeat(q, 50, 0), seed=9, offset=0)
    assert (idx == 0).all() and (iters == -1).sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("n_items,M,D", [(5003, 300, 8), (50000, 1024, 8), (1000, 64, 16), (2000, 40, 64)])
def test_gpu_sampler_bitexact_vs_oracle(n_items, M, D):
    from gpu_util import N, T
    from pivotcvae_b200 import ops
    rng = np.random.default_rng(n_items + D)
    W = _table(rng, n_items, D)
    Q = (rng.standard_normal((M, D)) * 1.5).astype(np.float32)
    tab = ops.Table(T(W))
    seed, off = 0xABCDEF0123, 4242
    idx, iters = ops.sigmoid_categorical(tab, T(Q), seed=seed, offset=off, want_iters=True)
    oi, oit = oracle.sigmoid_categorical(W, Q, seed=seed, offset=off)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(iters), oit)
    # device-side counter (CUDA-graph replays): offset = host offset + *offset_dev
    ctr = torch.tensor([off - 42], dtype=torch.int64, device="cuda:0")
    idx2 = ops.sigmoid_categorical(tab, T(Q), seed=seed, offset=42, offset_dev=ctr)
    assert torch.equal(idx, idx2)


@pytest.mark.gpu
def test_gpu_sampler_fallback_and_distribution():
    from gpu_util import N, T
    from pivotcvae_b200 import ops
    Wp = np.tile(-np.eye(8, dtype=np.float32)[0], (400, 1))
    Wp[0] = np.eye(8, dtype=np.float32)[0]
    q = (60 * np.eye(8, dtype=np.float32)[0]).reshape(1, 8)
    Q = np.repeat(q, 50, 0)
    idx, iters = ops.sigmoid_categorical(ops.Table(T(Wp)), T(Q), seed=9, offset=0, want_iters=True)
    oi, oit = oracle.sigmoid_categorical(Wp, Q, seed=9, offset=0)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(iters), oit) and (oit == -1).any()
    rng = np.random.default_rng(11)
    W = _table(rng, 6, 8)
    q = (3 * W[2]).reshape(1, 8)
    M = 200000
    idx = ops.sigmoid_categorical(ops.Table(T(W)), T(np.repeat(q, M, 0)), seed=99, offset=0)
    p = 1 / (1 + np.exp(-(W.astype(np.float64) @ q[0].astype(np.float64))))
    ok, chi2, dof = _chi2_ok(np.bincount(N(idx), minlength=6).astype(np.float64), p / p.sum())
    assert ok, (chi2, dof)


@pytest.mark.gpu
def test_model_sampled_pivot_uses_the_sampler_and_matches_the_oracle(golden):
    """recommend() of a *_spi model without caller noise: pivot = the sampler's draw on the PSM output; external
    noise still takes the parity path."""
    from gpu_util import N, T, build_pivot
    fx = golden("pivot_c1")
    m = build_pivot(fx, "pivotcvae_gt_spi")
    cfg, sd, tag = fx.cfg, fx.sub("sd/"), "rec_spi_k2/"
    m.noise.reseed(31337)
    m.noise.push("eps", T(fx[tag + "eps"]))
    items, _ = m.recommend(T(fx[tag + "ctx"]), T(fx["in/users"]), return_item=True)
    # oracle: same eps; the pivot comes from the restated sampler (row counter starts at 0 after reseed)
    ref0 = oracle.pivot_recommend(sd, fx[tag + "ctx"], fx["in/users"], fx[tag + "eps"], cfg["no_user"], "max")
    pidx, _ = oracle.sigmoid_categorical(sd["docEmbed.weight"], ref0["pivot_out"], seed=31337, offset=0)
    W = sd["docEmbed.weight"]
    uemb = sd["userEmbed.weight"][fx["in/users"]]
    parts = [ref0["z"], oracle.condition(fx[tag + "ctx"]), W[pidx], uemb]
    out = oracle.mlp(np.concatenate(parts, 1), sd, "scm", oracle.ACT_NONE)
    rx = np.concatenate([W[pidx].reshape(cfg["B"], 1, -1), out.reshape(cfg["B"], cfg["L"] - 1, -1)], 1)
    want, _ = oracle.score_select(W, rx.reshape(-1, cfg["D"]), "greedy")
    assert np.array_equal(N(items), want)
    m.noise.push("eps", T(fx[tag + "eps"]))
    m.noise.push("race", T(fx[tag + "noise"]))
    items_par, _ = m.recommend(T(fx[tag + "ctx"]), T(fx["in/users"]), return_item=True)
    assert np.array_equal(N(items_par), fx[tag + "items"])       # identical RNG stream -> the reference's slates
