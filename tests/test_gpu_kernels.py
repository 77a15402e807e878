"""-m gpu: every CUDA entry point of libpcv_b200.so against the CPU oracle
(bit-exact for indices / integer work / the fp32 FMA-chain paths; stated
tolerances for the soft-max and transcendental paths)."""
import numpy as np
import pytest
import torch

import oracle
from gpu_util import N, T, dev

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


# ------------------------------------------------------------------ score + select
@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
def test_select_greedy_golden(ops, golden, D):
    fx = golden("dims")
    W, Q = fx["d%d/W" % D], fx["d%d/Q" % D]
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine="simt")
    assert np.array_equal(N(idx), fx["d%d/idx" % D])       # the reference's torch.max indices
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(val), ov)   # bitwise vs the oracle
    p = ops.score_logits(tab, T(Q))
    assert np.array_equal(N(p), oracle.score_logits(W, Q))
    if D == 8:
        assert np.array_equal(N(p)[:4], fx["d8/p_rows"])  # bitwise == reference torch.mm (SURVEY F3)


@pytest.mark.parametrize("n_items,M,D", [(1, 3, 8), (31, 1, 8), (129, 70, 8), (5000, 333, 8), (70001, 257, 8),
                                         (4097, 65, 16), (3000, 17, 32), (999, 9, 64), (777, 5, 128), (2048, 64, 4)])
def test_select_greedy_ragged(ops, n_items, M, D):
    rng = np.random.default_rng(n_items + M)
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = rng.standard_normal((M, D)).astype(np.float32)
    if n_items > 40:  # exact ties at both ends of the catalog and across split boundaries
        W[n_items - 1] = W[7]
        W[n_items // 2] = W[7]
        Q[0] = 2 * W[7]
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine="simt")
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi)
    assert np.array_equal(N(val), ov)
    if n_items > 40:
        assert N(idx)[0] == 7


def test_select_all_equal_scores_returns_first(ops):
    W = np.tile(np.array([[0.5, 0.5, 0.5, 0.5, 0, 0, 0, 0]], dtype=np.float32), (3000, 1))
    Q = np.ones((5, 8), dtype=np.float32)
    idx, _ = ops.score_select(ops.Table(T(W)), T(Q), "greedy", engine="simt")
    assert np.array_equal(N(idx), np.zeros(5, dtype=np.int64))


@pytest.mark.parametrize("name,tag", [("pivot_small", "rec_spi_k2/"), ("pivot_c1", "rec_spi_k2/")])
def test_select_exprace_external_noise(ops, golden, name, tag):
    """Sampled pivot (pivotcvae.py:389-391) with the reference's own Exp(1) draws."""
    fx = golden(name)
    sd, cfg = fx.sub("sd/"), fx.cfg
    ref = oracle.pivot_recommend(sd, fx[tag + "ctx"], fx["in/users"], fx[tag + "eps"], cfg["no_user"], "sample",
                                 noise=fx[tag + "noise"])
    tab = ops.Table(T(sd["docEmbed.weight"]))
    idx, val = ops.score_select(tab, T(ref["pivot_out"]), "exprace", noise=T(fx[tag + "noise"]))
    oi, ov = oracle.score_select(sd["docEmbed.weight"], ref["pivot_out"], "exprace", fx[tag + "noise"])
    assert np.array_equal(N(idx), oi) and np.array_equal(N(val), ov)
    assert np.array_equal(N(idx), ref["pivot"])


def test_select_exprace_philox(ops):
    rng = np.random.default_rng(5)
    n_items, M, D = 5003, 77, 8
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = rng.standard_normal((M, D)).astype(np.float32)
    tab = ops.Table(T(W))
    seed, off = 0x1234ABCD5678, 1000
    E = ops.philox_exponential(seed, off, M, n_items, dev())
    u = oracle.exprace_uniform(seed, off, M, n_items)
    np.testing.assert_allclose(N(E), -np.log(u.astype(np.float64)), rtol=2e-6, atol=1e-7)  # integer stream exact
    a, av = ops.score_select(tab, T(Q), "exprace", seed=seed, offset=off)
    b, bv = ops.score_select(tab, T(Q), "exprace", noise=E)
    assert torch.equal(a, b) and torch.equal(av, bv)          # fused Philox == external noise path
    oi, _ = oracle.score_select(W, Q, "exprace", N(E))
    assert np.array_equal(N(a), oi)
    # a different offset gives different draws; the same one is reproducible
    c, _ = ops.score_select(tab, T(Q), "exprace", seed=seed, offset=off + M)
    assert not torch.equal(a, c)
    d, _ = ops.score_select(tab, T(Q), "exprace", seed=seed, offset=off)
    assert torch.equal(a, d)


def test_exprace_is_sigmoid_categorical(ops):
    """Distribution check: P(pick j) ∝ sigmoid(score_j) (pivotcvae.py:349-350)."""
    rng = np.random.default_rng(11)
    W = rng.standard_normal((6, 8)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    q = (3 * W[2]).reshape(1, 8)
    M = 40000
    idx, _ = ops.score_select(ops.Table(T(W)), T(np.repeat(q, M, 0)), "exprace", seed=99, offset=0)
    freq = np.bincount(N(idx), minlength=6) / M
    p = 1 / (1 + np.exp(-(W @ q[0])))
    np.testing.assert_allclose(freq, p / p.sum(), atol=0.01)


def test_vp_merge(ops):
    """Vocab-parallel shards + merge == one-shot (SURVEY §8e), incl. ties across shards."""
    rng = np.random.default_rng(3)
    n_items, M, D, G = 4096, 100, 8, 4
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    W[3000] = W[100]
    W[1500] = W[100]
    Q = rng.standard_normal((M, D)).astype(np.float32)
    Q[0] = W[100]
    Wd = T(W)
    full_i, full_v = ops.score_select(ops.Table(Wd), T(Q), "greedy", engine="simt")
    vals, idxs = [], []
    per = n_items // G
    for g in range(G):
        t = ops.Table(Wd[g * per:(g + 1) * per], row_offset=g * per)
        i, v = ops.score_select(t, T(Q), "greedy", engine="simt")
        vals.append(v)
        idxs.append(i)
    mi, mv = ops.vp_merge_select(torch.stack(vals), torch.stack(idxs))
    assert torch.equal(mi, full_i) and torch.equal(mv, full_v)
    assert int(mi[0]) == 100


# ------------------------------------------------------------------ MLP blocks
def _mlp_case(ops, rng, B, dims, acts, n_seg):
    import pivotcvae_b200._lib as L
    x_parts, segs = [], []
    Ls = 5
    r = (rng.random((B, Ls)) < 0.5).astype(np.float32)
    tab = rng.standard_normal((50, 8)).astype(np.float32)
    idx = rng.integers(0, 50, (B, 3))
    z = rng.standard_normal((B, dims[0] - (Ls + 1) - 24)).astype(np.float32)
    segs = [ops.Dense(T(z)), ops.OneHot(T(r)), ops.Gather(T(tab), T(idx))]
    x = np.concatenate([z, oracle.condition(r), tab[idx.reshape(-1)].reshape(B, -1)], 1)
    layers, ref = [], x
    for i in range(len(dims) - 1):
        Wm = (rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32)
        b = rng.standard_normal(dims[i + 1]).astype(np.float32) * 0.1
        layers.append((T(Wm), T(b), acts[i]))
        ref = oracle.linear(ref, Wm, b, acts[i])
    return segs, layers, x, ref


@pytest.mark.parametrize("B", [1, 15, 64, 1000, 5000])
@pytest.mark.parametrize("dims", [(54, 256, 256, 32), (38, 64, 8), (47, 300, 512, 40), (33, 16)])
def test_mlp_block_bitexact(ops, B, dims):
    rng = np.random.default_rng(B + sum(dims))
    acts = [1] * (len(dims) - 2) + [0]
    segs, layers, x, ref = _mlp_case(ops, rng, B, dims, acts, 3)
    res = ops.mlp_forward(segs, layers, B, save=True)
    assert np.array_equal(N(res["x0"]), x)
    assert np.array_equal(N(res["out"]), ref)     # same FMA chain as the oracle: bitwise
    h = x
    for i, a in enumerate(res["acts"]):
        h = oracle.linear(h, N(layers[i][0]), N(layers[i][1]), acts[i])
        assert np.array_equal(N(a), h)


@pytest.mark.parametrize("B", [1, 15, 64, 1000, 1300, 5000])
@pytest.mark.parametrize("dims", [(54, 256, 256, 32), (38, 64, 8), (47, 300, 512, 40), (33, 16), (62, 256, 72)])
def test_mlp_packed_engine_bitexact(ops, B, dims):
    """Inference (save=False) runs the packed-weight TMA engine: bit-identical to the oracle and to the
    streaming engine (save=True), also after the weights change in place (cache re-pack on the version counter)."""
    rng = np.random.default_rng(B + sum(dims))
    acts = [1] * (len(dims) - 2) + [0]
    segs, layers, x, ref = _mlp_case(ops, rng, B, dims, acts, 3)
    got = ops.mlp_forward(segs, layers, B)
    assert np.array_equal(N(got["out"]), ref)
    plain = ops.mlp_forward(segs, layers, B, save=True)
    assert torch.equal(got["out"], plain["out"])
    layers[0][0].mul_(0.5)                          # in-place update -> version bump -> re-pack
    h = x
    for i, (W, b, a) in enumerate(layers):
        h = oracle.linear(h, N(W), N(b), a)
    assert np.array_equal(N(ops.mlp_forward(segs, layers, B)["out"]), h)


def test_mlp_packed_chain_and_reparam(ops):
    """Two chained blocks (prior -> z -> next block) on the packed engine == two separate launches."""
    rng = np.random.default_rng(5)
    B, Z = 777, 16
    r = (rng.random((B, 5)) < 0.5).astype(np.float32)
    eps = rng.standard_normal((B, Z)).astype(np.float32)
    mk = lambda o, i: (T((rng.standard_normal((o, i)) / np.sqrt(i)).astype(np.float32)), T(rng.standard_normal(o).astype(np.float32) * 0.1))
    pl = [mk(128, 6) + (1,), mk(128, 128) + (1,), mk(2 * Z, 128) + (0,)]
    nl = [mk(256, Z + 6) + (1,), mk(256, 256) + (1,), mk(8, 256) + (0,)]
    cond = ops.OneHot(T(r))
    first = ([cond], pl, dict(latent=Z, eps=T(eps)))
    ra, rb = ops.mlp_forward_chain(first, lambda res: ([ops.Dense(res["z"]), cond], nl, {}), B)
    h = oracle.condition(r)
    for (W, b, a) in pl:
        h = oracle.linear(h, N(W), N(b), a)
    z = oracle.reparam(h[:, :Z], h[:, Z:], eps)
    assert np.array_equal(N(ra["out"]), h) and np.array_equal(N(ra["z"]), z)
    g = np.concatenate([z, oracle.condition(r)], 1)
    for (W, b, a) in nl:
        g = oracle.linear(g, N(W), N(b), a)
    assert np.array_equal(N(rb["out"]), g)


def test_mlp_reparam_and_relu(ops):
    rng = np.random.default_rng(0)
    B, Z = 100, 16
    x = rng.standard_normal((B, 20)).astype(np.float32)
    W1 = rng.standard_normal((64, 20)).astype(np.float32) * 0.2
    b1 = rng.standard_normal(64).astype(np.float32) * 0.1
    W2 = rng.standard_normal((2 * Z, 64)).astype(np.float32) * 0.2
    b2 = rng.standard_normal(2 * Z).astype(np.float32) * 0.1
    eps = rng.standard_normal((B, Z)).astype(np.float32)
    res = ops.mlp_forward([ops.Dense(T(x))], [(T(W1), T(b1), 2), (T(W2), T(b2), 0)], B, latent=Z, eps=T(eps))
    h = oracle.linear(oracle.linear(x, W1, b1, oracle.ACT_RELU), W2, b2, 0)
    assert np.array_equal(N(res["out"]), h)
    assert np.array_equal(N(res["z"]), oracle.reparam(h[:, :Z], h[:, Z:], eps))   # portable exp: bitwise
    # Philox normals: reproducible, ~N(0,1)
    big = ops.mlp_forward([ops.Dense(T(np.zeros((20000, 20), np.float32)))], [(T(W1), T(b1), 2), (T(W2 * 0), T(b2 * 0), 0)],
                          20000, latent=Z, seed=7, offset=3)
    e = N(big["eps"])
    assert abs(e.mean()) < 0.01 and abs(e.std() - 1) < 0.01
    assert np.array_equal(N(big["z"]), e)       # mu = 0, logvar = 0 -> z = eps
    again = ops.mlp_forward([ops.Dense(T(np.zeros((20000, 20), np.float32)))], [(T(W1), T(b1), 2), (T(W2 * 0), T(b2 * 0), 0)],
                            20000, latent=Z, seed=7, offset=3)
    assert torch.equal(big["eps"], again["eps"])


def test_normalize_rows(ops):
    rng = np.random.default_rng(1)
    W = rng.standard_normal((1000, 8)).astype(np.float32)
    W[5] = 0
    assert np.array_equal(N(ops.normalize_rows(T(W))), oracle.normalize_rows(W))
    ref = torch.nn.functional.normalize(torch.from_numpy(W), p=2, dim=1).numpy()
    np.testing.assert_allclose(N(ops.normalize_rows(T(W))), ref, rtol=3e-7, atol=0)


# ------------------------------------------------------------------ CE / KL
@pytest.mark.parametrize("n_items,M,D", [(500, 37, 8), (5000, 130, 8), (40000, 64, 8), (3000, 50, 16), (1000, 33, 32),
                                         (1500, 41, 64), (900, 19, 128)])      # --dim is free in the reference
@pytest.mark.parametrize("mode", ["dense", "bitmask", "philox"])
def test_ce_fwd_bwd(ops, n_items, M, D, mode):
    rng = np.random.default_rng(n_items + M)
    W = rng.standard_normal((n_items, D)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = rng.standard_normal((M, D)).astype(np.float32) * 2
    tg = rng.integers(0, n_items, M)
    tab = ops.Table(T(W))
    if mode == "dense":
        loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0)
        rl, rlse, rdq = oracle.ce(W, Q, tg, None)
    elif mode == "bitmask":
        bits = oracle.pack_bitmask(rng.random((M, n_items)) < 0.1)
        loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 0.1, bitmask=T(bits.view(np.int32)))
        rl, rlse, rdq = oracle.ce(W, Q, tg, bits)
    else:
        keep = 0.07
        loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), keep, seed=42, offset=9)
        bits = oracle.bernoulli_bitmask(42, 9, M, n_items, keep)   # integer Philox stream: exact
        rl, rlse, rdq = oracle.ce(W, Q, tg, bits)
    # fp32 soft-max path: north_star tolerance 1e-4 relative
    np.testing.assert_allclose(N(loss), rl, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(N(lse), rlse, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(N(dq), rdq, rtol=1e-3, atol=2e-6)


def test_kl(ops):
    rng = np.random.default_rng(2)
    a = [rng.standard_normal((300, 16)).astype(np.float32) * 0.5 for _ in range(4)]
    out, g = ops.kl_fwd_bwd(*[T(x) for x in a])
    ref, rg = oracle.kl(*a, grads=True)
    np.testing.assert_allclose(float(out), ref, rtol=1e-5)
    for x, y in zip(g, rg):
        np.testing.assert_allclose(N(x), y, rtol=1e-4, atol=1e-6)


# ------------------------------------------------------------------ response models
def test_urm_variants(ops, golden):
    fx = golden("env_small")
    slates, users = fx["in/slates"], fx["in/users"]
    for v, name in enumerate(["urm", "urm_p", "urm_p_mr"]):
        sd = fx.sub(name + "/sd/")
        kw = {}
        if v >= 1:
            kw = dict(pos_bias=T(fx[name + "/posBias"]), pos_dep=T(fx[name + "/posDependentBias"]))
        if v == 2:
            kw["mr_factor"] = float(fx[name + "/mrFactor"])
        out = ops.urm_forward(v, T(sd["docEmbed.weight"]), T(sd["userEmbed.weight"]), T(sd["itemBias.weight"]),
                              T(sd["userBias.weight"]), T(slates), T(users), **kw)
        np.testing.assert_allclose(N(out), fx[name + "/out"], rtol=1e-5, atol=1e-6)   # reference output


def test_errors_are_loud(ops):
    import pivotcvae_b200._lib as L
    with pytest.raises(L.PcvError):
        ops.Table(torch.zeros(10, 8))            # CPU tensor: no fallback
    with pytest.raises(L.PcvError):
        ops.Table(torch.zeros(10, 7, device=dev()))   # dim not a multiple of 4
    tab = ops.Table(torch.zeros(10, 8, device=dev()))
    with pytest.raises(L.PcvError):
        ops.score_select(tab, torch.zeros(4, 16, device=dev()))
    before = ops.launch_count()
    ops.score_select(tab, torch.zeros(4, 8, device=dev()))
    assert ops.launch_count() >= before + 2


@pytest.mark.parametrize("n_items,M", [(2048, 128), (5000, 130), (100000, 300), (40001, 1000)])
def test_ce_tensor_core_engine(ops, n_items, M):
    """Opt-in tf32 engine of the dense catalog CE (logits on tcgen05): reduced-precision tolerance
    (north_star: 1e-2; observed ~1e-4 on the loss, ~1e-3 on dq)."""
    rng = np.random.default_rng(n_items + M)
    W = rng.standard_normal((n_items, 8)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = rng.standard_normal((M, 8)).astype(np.float32) * rng.uniform(0.2, 1.0, (M, 1)).astype(np.float32)
    tg = rng.integers(0, n_items, M)
    tab = ops.Table(T(W))
    loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="tf32")
    rl, rlse, rdq = oracle.ce(W, Q, tg, None)
    np.testing.assert_allclose(N(loss), rl, rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(lse), rlse, rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(dq), rdq, rtol=1e-2, atol=1e-3)
    el, _, edq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="exact")
    np.testing.assert_allclose(N(loss), N(el), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("n_items,M,G,engine", [(5000, 130, 2, "exact"), (40000, 300, 4, "exact"), (40000, 300, 4, "tf32"),
                                                 (100003, 515, 8, "tf32"), (3000, 64, 3, "exact")])
def test_ce_vocab_parallel_partials_merge(ops, n_items, M, G, engine):
    """pcv_ce_partials over G row shards + pcv_ce_vp_merge == the unsharded CE (and the oracle): what the ranks of a
    vocab-parallel training step compute around their one all-gather (SURVEY 8e), here on one GPU."""
    from pivotcvae_b200.parallel import merge_ce_partials, shard_bounds
    rng = np.random.default_rng(n_items + G)
    W = rng.standard_normal((n_items, 8)).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = (3.0 * rng.standard_normal((M, 8))).astype(np.float32)
    tgt = rng.integers(0, n_items, M)
    tgt[0], tgt[1] = 0, n_items - 1
    Wt, Qt, tt = T(W), T(Q), T(tgt)
    recs = []
    for g in range(G):
        lo, hi = shard_bounds(n_items, G, g)
        shard = ops.Table(Wt[lo:hi], row_offset=lo)
        recs.append(ops.ce_partials(shard, Qt, tt, engine=engine))
    recs = torch.stack(recs)
    loss, lse, dq = ops.ce_vp_merge(recs, Wt, Qt, tt)
    full = ops.Table(Wt)
    l1, s1, d1 = ops.ce_fwd_bwd(full, Qt, tt, engine=engine)
    tol = dict(rtol=2e-4, atol=2e-5) if engine == "tf32" else dict(rtol=1e-5, atol=1e-6)
    assert np.allclose(N(loss), N(l1), **tol) and np.allclose(N(lse), N(s1), **tol)
    assert np.allclose(N(dq), N(d1), rtol=1e-3 if engine == "tf32" else 1e-4, atol=2e-5)
    ol, olse, odq = oracle.ce(W, Q, tgt)
    # |q| ~ 8.5 here: the tf32 logits carry ~2^-10 |q| of absolute error, so the reduced-precision engine is held
    # to 1e-3 against the fp32 oracle (the sharded-vs-unsharded comparison above is the vocab-parallel claim)
    lt = 1e-3 if engine == "tf32" else 1e-4
    assert np.allclose(N(loss), ol, rtol=lt, atol=1e-4) and np.allclose(N(dq), odq, rtol=5e-3 if engine == "tf32" else 2e-3, atol=1e-3 if engine == "tf32" else 2e-4)
    # the torch restatement used by the gloo CPU test agrees with the kernel
    pl, ps, pd = merge_ce_partials(recs, Wt, Qt, tt)
    assert np.allclose(N(pl), N(loss), rtol=1e-5, atol=1e-5) and np.allclose(N(pd), N(dq), rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("D", [16, 64, 128])
def test_urm_metrics_and_candidate_ce_other_dims(ops, D):
    """--dim other than 8 (train_generative.py:302 leaves it free): URM variants, slate metrics and the candidate CE
    against the oracle restatements."""
    from pivotcvae_b200 import _lib as L
    from pivotcvae_b200 import analysis
    rng = np.random.default_rng(D)
    n_items, n_users, B, Ls = 700, 90, 257, 5
    doc = rng.standard_normal((n_items, D)).astype(np.float32)
    usr = rng.standard_normal((n_users, D)).astype(np.float32)
    ib = (0.1 * rng.standard_normal(n_items)).astype(np.float32)
    ub = (0.1 * rng.standard_normal(n_users)).astype(np.float32)
    pb = rng.standard_normal(Ls).astype(np.float32)
    pd = rng.standard_normal((Ls, D)).astype(np.float32)
    slates = rng.integers(0, n_items, (B, Ls))
    users = rng.integers(0, n_users, B)
    got = ops.urm_forward(L.URM_P_MR, T(doc), T(usr), T(ib), T(ub), T(slates), T(users), pos_bias=T(pb), pos_dep=T(pd), mr_factor=0.3)
    want = oracle.urm(L.URM_P_MR, doc, usr, ib, ub, slates, users, pos_bias=pb, pos_dep=pd, mr_factor=0.3)
    np.testing.assert_allclose(N(got), want, rtol=1e-5, atol=1e-6)
    ils, _ = analysis._metrics(T(slates), T(doc), True, False)
    np.testing.assert_allclose(N(ils), oracle.ils(doc, slates), rtol=1e-4, atol=1e-6)
    W = doc / np.linalg.norm(doc, axis=1, keepdims=True)
    Q = rng.standard_normal((B, D)).astype(np.float32)
    cand = rng.integers(0, n_items, (B, 50))
    tp = rng.integers(0, 50, B)
    loss, lse, dq, p = ops.cand_ce_fwd_bwd(ops.Table(T(W)), T(Q), T(cand), T(tp), want_logits=True)
    rl, rdq, rp = oracle.cand_ce(W, Q, cand, tp)
    np.testing.assert_allclose(N(loss), rl, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(N(dq), rdq, rtol=1e-3, atol=2e-6)
    assert np.array_equal(N(p), rp)
