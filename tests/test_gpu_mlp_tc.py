"""-m gpu: the tcgen05 engine of the fused MLP blocks (csrc/mlp_tc.cu, ops.MLP_ENGINE = "tc").

It is NOT bit-identical to the oracle's sequential FMA chain (3xTF32 products, tensor-core summation order), so it is
held to (a) a float64 restatement of the block with an fp32-grade bound, (b) the distance the exact engine itself has
from float64, (c) the reference fixtures: logits within north_star's 1e-4 and identical slates
(tests/test_big_parity.py repeats (c) at the BASELINE sizes)."""
import numpy as np
import pytest
import torch

import oracle
from conftest import load_golden
from gpu_util import N, T, build_list, build_pivot

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _act64(v, a):
    if a == 1:
        return np.where(v > 0, v, 0.01 * v)
    if a == 2:
        return np.maximum(v, 0)
    return v


def _case(ops, rng, B, dims, acts, normalize=False):
    """[dense z | one-hot | gather] -> layers; returns segments, layers, float64 outputs and the fp32-grade error scale
    sum_k |x_k||w_k| + |b| propagated through the layers."""
    Ls = 5
    r = (rng.random((B, Ls)) < 0.5).astype(np.float32)
    tab = rng.standard_normal((50, 8)).astype(np.float32)
    idx = rng.integers(0, 50, (B, 3))
    nz = dims[0] - (Ls + 1) - 24
    z = rng.standard_normal((B, nz)).astype(np.float32)
    segs = [ops.Dense(T(z)), ops.OneHot(T(r)), ops.Gather(T(tab), T(idx), normalize=normalize)]
    g = tab[idx.reshape(-1)].reshape(B, -1).astype(np.float64)
    if normalize:
        g = g / np.maximum(np.sqrt((g * g).sum(1, keepdims=True)), 1e-12)
    x = np.concatenate([z.astype(np.float64), oracle.condition(r).astype(np.float64), g], 1)
    layers, h, scale = [], x, np.zeros((B, 1))
    for i in range(len(dims) - 1):
        Wm = (rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32)
        b = (rng.standard_normal(dims[i + 1]) * 0.1).astype(np.float32)
        layers.append((T(Wm), T(b), acts[i]))
        W64 = Wm.astype(np.float64)
        scale = np.abs(h) @ np.abs(W64.T) + np.abs(b) + scale.max(1, keepdims=True) * np.abs(W64).sum(1)[None, :]
        h = _act64(h @ W64.T + b, acts[i])
    return segs, layers, h, scale


SHAPES = [(54, 256, 256, 32), (38, 64, 8), (46, 256, 256, 5), (33, 16), (62, 256, 72), (44, 128, 128, 32), (35, 100, 200, 24, 7),
          (100, 256, 80), (128, 48, 10)]


@pytest.mark.parametrize("B", [1, 100, 128, 129, 1000, 4096])
@pytest.mark.parametrize("dims", SHAPES)
def test_mlp_tc_block_fp32_grade(ops, B, dims):
    rng = np.random.default_rng(B * 7 + sum(dims))
    acts = [1] * (len(dims) - 2) + [0]
    segs, layers, want, scale = _case(ops, rng, B, dims, acts)
    with ops.mlp_engine("tc"):
        ops.mlp_forward(segs, layers, B)              # packs the weights (one launch per layer, cached)
        before = ops.launch_count()
        got = N(ops.mlp_forward(segs, layers, B)["out"]).astype(np.float64)
        assert ops.launch_count() - before == 1
    exact = N(ops.mlp_forward(segs, layers, B)["out"]).astype(np.float64)
    err_tc = np.abs(got - want) / scale
    err_ex = np.abs(exact - want) / scale
    # 3xTF32 products are good to ~2^-21 of sum|x||w|; fp32 accumulation adds ~sqrt(K) 2^-24.  The exact engine's own
    # distance from float64 is printed next to it.
    print("dims %s B %d: tc %.2e  exact %.2e (max |err| / sum|x||w|)" % (dims, B, err_tc.max(), err_ex.max()))
    assert err_tc.max() < 2e-6
    # two-pass MMA order (csrc/mlp_tc.cu): the truncating tensor-core accumulator must not cost more than a few times
    # the error of the sequential fp32 chain (measured ~3x with the two-pass order; a single interleaved pass was ~6x)
    rms_tc, rms_ex = np.sqrt((err_tc ** 2).mean()), np.sqrt((err_ex ** 2).mean())
    print("   rms: tc %.2e exact %.2e ratio %.2f" % (rms_tc, rms_ex, rms_tc / rms_ex))
    if B >= 100:      # (a handful of outputs is too small a sample for an rms ratio)
        assert rms_tc < 5.0 * rms_ex + 1e-12
    assert np.allclose(got, exact, rtol=1e-4, atol=1e-5)


def test_mlp_tc_differs_from_exact_engine_only_in_rounding(ops):
    """Guards against a silent fall-through to the FFMA engine: the tc engine must have run (one launch, results not
    bit-identical to the sequential chain on a wide block) — and for a block it does not fit, the exact engine runs."""
    rng = np.random.default_rng(3)
    segs, layers, want, _ = _case(ops, rng, 512, (54, 256, 256, 32), [1, 1, 0])
    exact = ops.mlp_forward(segs, layers, 512)["out"]
    with ops.mlp_engine("tc"):
        got = ops.mlp_forward(segs, layers, 512)["out"]
    assert not torch.equal(got, exact)
    assert torch.allclose(got, exact, rtol=1e-4, atol=1e-5)
    segs, layers, want, _ = _case(ops, rng, 64, (47, 300, 512, 40), [1, 1, 0])     # wider than 256: exact engine
    exact = ops.mlp_forward(segs, layers, 64)["out"]
    with ops.mlp_engine("tc"):
        got = ops.mlp_forward(segs, layers, 64)["out"]
    assert torch.equal(got, exact)


def test_mlp_tc_normalised_gather_relu_and_repack(ops):
    """Response-MLP shaped block (response_model.py:76-87): whole-segment L2 normalise, ReLU; weights updated in place
    are re-packed through the version counter."""
    rng = np.random.default_rng(11)
    B = 700
    tab = rng.standard_normal((300, 8)).astype(np.float32)
    idx = rng.integers(0, 300, (B, 6))
    W1 = (rng.standard_normal((256, 48)) / 7).astype(np.float32)
    b1 = (rng.standard_normal(256) * 0.1).astype(np.float32)
    W2 = (rng.standard_normal((256, 256)) / 16).astype(np.float32)
    b2 = (rng.standard_normal(256) * 0.1).astype(np.float32)
    W3 = (rng.standard_normal((5, 256)) / 16).astype(np.float32)
    b3 = (rng.standard_normal(5) * 0.1).astype(np.float32)
    layers = [(T(W1), T(b1), 2), (T(W2), T(b2), 2), (T(W3), T(b3), 0)]
    segs = [ops.Gather(T(tab), T(idx), normalize=True)]

    def ref():
        g = tab[idx.reshape(-1)].reshape(B, -1).astype(np.float64)
        h = g / np.maximum(np.sqrt((g * g).sum(1, keepdims=True)), 1e-12)
        for (W, b, a) in layers:
            h = _act64(h @ N(W).astype(np.float64).T + N(b), a)
        return h

    with ops.mlp_engine("tc"):
        got = N(ops.mlp_forward(segs, layers, B)["out"])
        assert np.allclose(got, ref(), rtol=2e-5, atol=2e-6)
        layers[1][0].mul_(0.5)
        got = N(ops.mlp_forward(segs, layers, B)["out"])
        assert np.allclose(got, ref(), rtol=2e-5, atol=2e-6)


def test_mlp_tc_chain_reparam_and_copy_seg(ops):
    """prior -> z -> PSM in one launch (pivotcvae.py:279-291, 204-210) and the pivot row copied to slot 0."""
    rng = np.random.default_rng(5)
    B, Z = 777, 16
    r = (rng.random((B, 5)) < 0.5).astype(np.float32)
    eps = rng.standard_normal((B, Z)).astype(np.float32)
    mk = lambda o, i: (T((rng.standard_normal((o, i)) / np.sqrt(i)).astype(np.float32)), T(rng.standard_normal(o).astype(np.float32) * 0.1))
    pl = [mk(128, 6) + (1,), mk(128, 128) + (1,), mk(2 * Z, 128) + (0,)]
    nl = [mk(256, Z + 6) + (1,), mk(256, 256) + (1,), mk(8, 256) + (0,)]
    cond = ops.OneHot(T(r))
    first = ([cond], pl, dict(latent=Z, eps=T(eps)))
    ea, eb = ops.mlp_forward_chain(first, lambda res: ([ops.Dense(res["z"]), cond], nl, {}), B)
    with ops.mlp_engine("tc"):
        ops.mlp_forward_chain(first, lambda res: ([ops.Dense(res["z"]), cond], nl, {}), B)   # packs the weights
        before = ops.launch_count()
        ra, rb = ops.mlp_forward_chain(first, lambda res: ([ops.Dense(res["z"]), cond], nl, {}), B)
        assert ops.launch_count() - before == 1
        # Philox eps: the same stream as the exact engine
        pa = ops.mlp_forward([cond], pl, B, latent=Z, seed=9, offset=5)
    assert torch.allclose(ra["out"], ea["out"], rtol=1e-4, atol=1e-5) and torch.allclose(ra["z"], ea["z"], rtol=1e-4, atol=2e-5)
    assert torch.allclose(rb["out"], eb["out"], rtol=1e-4, atol=2e-5)
    assert not torch.equal(rb["out"], eb["out"])
    pe = ops.mlp_forward([cond], pl, B, latent=Z, seed=9, offset=5)
    assert torch.equal(pa["eps"], pe["eps"]) and torch.allclose(pa["z"], pe["z"], rtol=1e-4, atol=2e-5)
    # copy_seg: rx = [pivot row | block output]
    piv = rng.standard_normal((B, 8)).astype(np.float32)
    sl = [mk(64, 8 + 6) + (1,), mk(32, 64) + (0,)]
    with ops.mlp_engine("tc"):
        out = ops.mlp_forward([ops.Dense(T(piv)), cond], sl, B, out_ld=40, out_col0=8, copy_seg=0)["out"]
    ex = ops.mlp_forward([ops.Dense(T(piv)), cond], sl, B, out_ld=40, out_col0=8, copy_seg=0)["out"]
    assert torch.equal(out[:, :8], T(piv)) and torch.allclose(out, ex, rtol=1e-4, atol=1e-5)


def test_tc_policy_runs_blocks_it_does_not_fit_bit_exact(ops):
    """Under "tc", a block with a 17-click one-hot and a chain whose second block is 86 wide ([z 16 | one-hot 6 |
    user 64]) do not fit the tc engine: they run on the FFMA cluster engine, bit-identical to the oracle."""
    rng = np.random.default_rng(17)
    B, Z = 777, 16
    mk = lambda o, i: (T((rng.standard_normal((o, i)) / np.sqrt(i)).astype(np.float32)), T(rng.standard_normal(o).astype(np.float32) * 0.1))
    r17 = (rng.random((B, 17)) < 0.5).astype(np.float32)
    layers = [mk(128, 18) + (1,), mk(8, 128) + (0,)]
    with ops.mlp_engine("tc"):
        out = ops.mlp_forward([ops.OneHot(T(r17))], layers, B)["out"]
    h = oracle.condition(r17)
    for (W, b, a) in layers:
        h = oracle.linear(h, N(W), N(b), a)
    assert np.array_equal(N(out), h)

    r = (rng.random((B, 5)) < 0.5).astype(np.float32)
    user = rng.standard_normal((B, 64)).astype(np.float32)
    eps = rng.standard_normal((B, Z)).astype(np.float32)
    pl = [mk(128, 6) + (1,), mk(2 * Z, 128) + (0,)]
    nl = [mk(256, Z + 6 + 64) + (1,), mk(8, 256) + (0,)]
    cond = ops.OneHot(T(r))
    with ops.mlp_engine("tc"):
        ra, rb = ops.mlp_forward_chain(([cond], pl, dict(latent=Z, eps=T(eps))),
                                       lambda res: ([ops.Dense(res["z"]), cond, ops.Dense(T(user))], nl, {}), B)
    h = oracle.condition(r)
    for (W, b, a) in pl:
        h = oracle.linear(h, N(W), N(b), a)
    z = oracle.reparam(h[:, :Z], h[:, Z:], eps)
    assert np.array_equal(N(ra["out"]), h) and np.array_equal(N(ra["z"]), z)
    g = np.concatenate([z, oracle.condition(r), user], 1)
    for (W, b, a) in nl:
        g = oracle.linear(g, N(W), N(b), a)
    assert np.array_equal(N(rb["out"]), g)


@pytest.mark.parametrize("name", ["pivot_c1", "pivot_small", "pivot_small_nouser"])
def test_tc_engine_recommend_matches_reference_fixtures(ops, name):
    """recommend() with the tc engine against the UNMODIFIED reference's outputs (tests/golden/make_golden.py):
    identical greedy slates, z_mu / rx within north_star's 1e-4."""
    fx = load_golden(name)
    m = build_pivot(fx)
    m.mlp_engine = "tc"
    cfg = fx.cfg
    users = None if cfg["no_user"] else T(fx["in/users"])
    for k in (1, cfg["L"]):
        tag = "rec_pi_k%d/" % k
        m.noise.push("eps", T(fx[tag + "eps"]))
        items, zmu = m.recommend(T(fx[tag + "ctx"]), users, return_item=True)
        assert np.array_equal(N(items), fx[tag + "items"])          # == reference slates
        np.testing.assert_allclose(N(zmu), fx[tag + "z_mu"], rtol=1e-4, atol=1e-5)
        m.noise.push("eps", T(fx[tag + "eps"]))
        rx, _ = m.recommend(T(fx[tag + "ctx"]), users, return_item=False)
        np.testing.assert_allclose(N(rx), fx[tag + "rx"], rtol=1e-4, atol=1e-5)
        m.mlp_engine = None
        m.noise.push("eps", T(fx[tag + "eps"]))
        rx_exact, _ = m.recommend(T(fx[tag + "ctx"]), users, return_item=False)
        m.mlp_engine = "tc"
        assert not torch.equal(rx, rx_exact)                        # the tc engine really ran


@pytest.mark.parametrize("name", ["list_small", "list_small_user"])
def test_tc_engine_list_recommend(ops, name):
    fx = load_golden(name)
    m = build_list(fx)
    m.mlp_engine = "tc"
    users = None if fx.cfg["no_user"] else T(fx["in/users"])
    for k in (1, 3):
        tag = "rec_k%d/" % k
        m.noise.push("eps", T(fx[tag + "eps"]))
        items, zmu = m.recommend(T(fx[tag + "ctx"]), users, return_item=True)
        assert np.array_equal(N(items), fx[tag + "items"])
        np.testing.assert_allclose(N(zmu), fx[tag + "z_mu"], rtol=1e-4, atol=1e-5)


def test_tc_engine_response_model(ops):
    """UserResponseModel_MLP.forward (response_model.py:76-87) with the tc engine vs the reference fixture."""
    from pivotcvae_b200.env.response_model import UserResponseModel_MLP
    fx = load_golden("env_small")
    n_items, n_users, L, D, B = [int(v) for v in fx["cfg"]]
    for tag, nu in (("mlp_user/", False), ("mlp_nouser/", True)):
        e = UserResponseModel_MLP(n_items - 1, n_users - 1, D, L, [(L + (0 if nu else 1)) * D, 64, 48, L], "cuda:0", nu)
        e.load_state_dict({k: torch.from_numpy(v) for k, v in fx.sub(tag + "sd/").items()})
        e.to("cuda:0")
        exact = e(T(fx["in/slates"]), T(fx["in/users"]))
        e.mlp_engine = "tc"
        out = e(T(fx["in/slates"]), T(fx["in/users"]))
        np.testing.assert_allclose(N(out), fx[tag + "out"], rtol=1e-4, atol=1e-5)
        assert not torch.equal(out, exact)
