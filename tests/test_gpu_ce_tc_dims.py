"""-m gpu: the tensor-core (tf32) full-catalog CE engine at embedding dims 16 to 128 (ce_tc2_kernel<D>), against the
CPU oracle and the exact SIMT engine, through the vocab-parallel records, and through a PivotCVAE training step."""
import numpy as np
import pytest
import torch

import oracle
from gpu_util import N, T, _Emb

pytestmark = pytest.mark.gpu

DIMS = [16, 32, 64, 128]


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _unit_rows(rng, n, D):
    W = rng.standard_normal((n, D)).astype(np.float32)
    return W / np.linalg.norm(W, axis=1, keepdims=True)


def _shapes():
    out = []
    for D in DIMS:
        out += [(D, 2048, 128), (D, 5000, 130), (D, 100003, 1000 if D <= 32 else 257)]
    return out


@pytest.mark.parametrize("D,n_items,M", _shapes())
def test_ce_tf32_engine_dims_vs_oracle(ops, D, n_items, M):
    """Shapes that are not multiples of the tile (BN = 128 / 64 / 32 items) or of the 256-row table tile, targets 0 and
    N - 1 included.  The query rows get the norm distribution of the D = 8 test (|q| ~ U(0.2, 1) x sqrt(8)), so the
    tf32 error per logit (<= 2^-9 sum_k |q_k w_k| <= 2^-9 |q| max|w|) is the same as there, and so are the tolerances:
    loss / lse 1e-3, dq 1e-2 relative."""
    rng = np.random.default_rng(D * 1000 + M)
    W = _unit_rows(rng, n_items, D)
    Q = rng.standard_normal((M, D)).astype(np.float32)
    Q *= (rng.uniform(0.2, 1.0, (M, 1)) * np.sqrt(8.0) / np.linalg.norm(Q, axis=1, keepdims=True)).astype(np.float32)
    tg = rng.integers(0, n_items, M)
    tg[0], tg[1] = 0, n_items - 1
    tab = ops.Table(T(W))
    loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="tf32")
    rl, rlse, rdq = oracle.ce(W, Q, tg, None)
    np.testing.assert_allclose(N(loss), rl, rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(lse), rlse, rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(dq), rdq, rtol=1e-2, atol=1e-3)
    el, else_, edq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="exact")
    np.testing.assert_allclose(N(loss), N(el), rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(lse), N(else_), rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(dq), N(edq), rtol=1e-2, atol=1e-3)


def test_ce_tf32_engine_d128_unscaled_queries(ops):
    """D = 128 with queries whose norm grows with D (entries N(0, 1) x U(0.2, 1): |q| up to ~15).  A tf32 logit
    differs from the fp32 one by at most 2^-9 sum_k |q_k w_k| <= 2^-9 |q| max|w| (each operand keeps 10 of its 23
    mantissa bits), lse moves by no more than the largest logit error, and the target logit is re-derived in fp32: so
    |loss - loss_fp32| <= 2^-9 |q| max|w| per row, plus fp32 summation slack (1e-3).  That is well under the 1e-2
    reduced-precision tolerance, which is asserted as well."""
    rng = np.random.default_rng(128)
    n_items, M, D = 30011, 300, 128
    W = _unit_rows(rng, n_items, D)
    Q = (rng.standard_normal((M, D)) * rng.uniform(0.2, 1.0, (M, 1))).astype(np.float32)
    tg = rng.integers(0, n_items, M)
    tab = ops.Table(T(W))
    loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="tf32")
    rl, rlse, rdq = oracle.ce(W, Q, tg, None)
    bound = 2.0 ** -9 * np.linalg.norm(Q, axis=1) * np.linalg.norm(W, axis=1).max() + 1e-3
    assert np.all(np.abs(N(loss) - rl) <= bound)
    assert np.all(np.abs(N(lse) - rlse) <= bound)
    np.testing.assert_allclose(N(loss), rl, rtol=1e-2)
    np.testing.assert_allclose(N(dq), rdq, rtol=1e-2, atol=2e-3)


@pytest.mark.parametrize("D", DIMS)
def test_ce_tf32_flagged_rows_redone_exactly(ops, D):
    """Rows with |q| max|w| > 140 whose target and first 32 items point away from q fail the reference-exponent test
    of ce_ref_kernel: ce_rowfix_kernel redoes them in exact fp32, so they match the exact engine at its own tolerance.
    The other rows of the same call stay on the tensor cores."""
    rng = np.random.default_rng(7 + D)
    n_items, M, n_bad = 5000, 200, 6
    u0 = rng.standard_normal(D).astype(np.float32)
    u0 /= np.linalg.norm(u0)
    W = _unit_rows(rng, n_items, D)
    head = -u0[None, :] + 0.1 * rng.standard_normal((32, D)).astype(np.float32)
    W[:32] = head / np.linalg.norm(head, axis=1, keepdims=True)
    Q = rng.standard_normal((M, D)).astype(np.float32)
    Q *= (rng.uniform(0.2, 1.0, (M, 1)) * np.sqrt(8.0) / np.linalg.norm(Q, axis=1, keepdims=True)).astype(np.float32)
    bad = rng.choice(M, n_bad, replace=False)
    for r in bad:
        u = u0 + 0.05 * rng.standard_normal(D).astype(np.float32)
        Q[r] = 200.0 * u / np.linalg.norm(u)
    tg = rng.integers(32, n_items, M)
    tg[bad] = 5                                   # far off: one of the items pointing away from q
    ub = np.linalg.norm(Q[bad], axis=1) * 1.01
    lb = (Q[bad] @ W[:32].T).max(axis=1)
    assert np.all(lb < ub - 140.0)                # these rows are flagged
    tab = ops.Table(T(W))
    loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="tf32")
    el, else_, edq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="exact")
    rl, rlse, rdq = oracle.ce(W, Q, tg, None)
    # flagged rows: exact-engine tolerance (as the exact engine is held to against the oracle)
    np.testing.assert_allclose(N(loss)[bad], N(el)[bad], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(N(lse)[bad], N(else_)[bad], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(N(dq)[bad], N(edq)[bad], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(N(loss)[bad], rl[bad], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(N(dq)[bad], rdq[bad], rtol=2e-3, atol=2e-4)
    ok = np.setdiff1d(np.arange(M), bad)
    np.testing.assert_allclose(N(loss)[ok], rl[ok], rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(N(dq)[ok], rdq[ok], rtol=1e-2, atol=1e-3)


@pytest.mark.parametrize("D", [32, 128])
@pytest.mark.parametrize("G", [3, 4])
def test_ce_tf32_vocab_parallel_partials_dims(ops, D, G):
    """pcv_ce_partials over G row shards + pcv_ce_vp_merge == the unsharded tf32 CE and the oracle, with the bounds
    of the D = 8 vocab-parallel test (query rows of the same norm, |q| ~ 8.5)."""
    from pivotcvae_b200.parallel import shard_bounds
    rng = np.random.default_rng(D + G)
    n_items, M = 40000, 300
    W = _unit_rows(rng, n_items, D)
    Q = (3.0 * np.sqrt(8.0 / D) * rng.standard_normal((M, D))).astype(np.float32)
    tgt = rng.integers(0, n_items, M)
    tgt[0], tgt[1] = 0, n_items - 1
    Wt, Qt, tt = T(W), T(Q), T(tgt)
    recs = []
    for g in range(G):
        lo, hi = shard_bounds(n_items, G, g)
        recs.append(ops.ce_partials(ops.Table(Wt[lo:hi], row_offset=lo), Qt, tt, engine="tf32"))
    recs = torch.stack(recs)
    loss, lse, dq = ops.ce_vp_merge(recs, Wt, Qt, tt)
    l1, s1, d1 = ops.ce_fwd_bwd(ops.Table(Wt), Qt, tt, engine="tf32")
    assert np.allclose(N(loss), N(l1), rtol=2e-4, atol=2e-5) and np.allclose(N(lse), N(s1), rtol=2e-4, atol=2e-5)
    assert np.allclose(N(dq), N(d1), rtol=1e-3, atol=2e-5)
    ol, olse, odq = oracle.ce(W, Q, tgt)
    assert np.allclose(N(loss), ol, rtol=1e-3, atol=1e-4) and np.allclose(N(dq), odq, rtol=5e-3, atol=1e-3)


def _pivot_d32(n_items, n_users, seed):
    from pivotcvae_b200.models.pivotcvae import UserPivotCVAE
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    Ls, D, Z = 5, 32, 16
    doc = (0.5 * rng.standard_normal((n_items, D))).astype(np.float32)
    usr = (0.5 * rng.standard_normal((n_users, D))).astype(np.float32)
    m = UserPivotCVAE(_Emb(doc), _Emb(usr), Ls, D, Z, Ls + 1, [Ls * D + Ls + 1 + D, 64, 64], [Z + Ls + 1 + D, 64, D],
                      [Z + Ls + 1 + 2 * D, 64, (Ls - 1) * D], [Ls + 1 + D, 32], False, "cuda:0")
    return m


def _batch(rng, n_items, n_users, B, Ls=5):
    return {"slates": torch.from_numpy(rng.integers(0, n_items, (B, Ls))).cuda(),
            "users": torch.from_numpy(rng.integers(0, n_users, (B, 1))).cuda(),
            "responses": torch.from_numpy(rng.integers(0, 2, (B, Ls)).astype(np.float32)).cuda()}


def test_pivotcvae_d32_full_catalog_tf32_vs_exact():
    """get_gen_loss + backward of a PivotCVAE at D = 32 with n_neg = N (full-catalog soft-max): the tf32 engine against
    the exact one: loss within 1e-3 relative, every parameter gradient within 1e-2 of its max-abs."""
    from pivotcvae_b200.train_generative import get_gen_loss
    n_items, n_users, B = 3001, 50, 64
    rng = np.random.default_rng(3)
    batch = _batch(rng, n_items, n_users, B)
    eps = torch.randn(B, 16, generator=torch.Generator().manual_seed(4)).cuda()
    res = {}
    for engine in ("exact", "tf32"):
        m = _pivot_d32(n_items, n_users, 11)
        m.ce_engine = engine
        m.noise.push("eps", eps)
        loss, rec, kld = get_gen_loss(batch, m, None, 0.01, n_neg=n_items)
        loss.backward()
        res[engine] = (float(loss), {k: N(p.grad) for k, p in m.named_parameters() if p.grad is not None})
    (le, ge), (lt, gt) = res["exact"], res["tf32"]
    assert abs(lt - le) <= 1e-3 * abs(le)
    assert ge.keys() == gt.keys() and len(ge) > 0
    for k in ge:
        assert np.abs(gt[k] - ge[k]).max() <= 1e-2 * max(np.abs(ge[k]).max(), 1e-12), k


def test_pivotcvae_d32_graphed_train_step_tf32():
    """A GraphedTrainStep at D = 32 with the tf32 CE captures (its eager warm-up builds the transposed table image
    outside the capture) and replays; the replayed loss matches an eager step on the same batch and the same Philox
    rows, with the tf32 engine (1e-3 relative) and with the exact one (1e-3 relative)."""
    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.train_generative import get_gen_loss
    n_items, n_users, B = 3001, 50, 64
    m = _pivot_d32(n_items, n_users, 12)
    m.ce_engine = "tf32"
    opt = torch.optim.Adam(m.parameters(), lr=1e-4, capturable=True)
    step = GraphedTrainStep(m, opt, B, 0.01, n_items)
    batch = _batch(np.random.default_rng(5), n_items, n_users, B)
    counter = m.noise.device_counter.clone()
    eager = {}
    for engine in ("tf32", "exact"):
        m.ce_engine = engine
        m.noise.device_counter.copy_(counter)      # the eager step draws the Philox rows the replay will draw
        loss, _, _ = get_gen_loss(batch, m, None, 0.01, n_neg=n_items)
        eager[engine] = float(loss)
    m.ce_engine = "tf32"
    m.noise.device_counter.copy_(counter)
    opt.zero_grad(set_to_none=True)
    loss, rec, kld = step(batch)
    torch.cuda.synchronize()
    lg = float(loss)
    assert np.isfinite(lg)
    assert abs(lg - eager["tf32"]) <= 1e-3 * abs(eager["tf32"])
    assert abs(lg - eager["exact"]) <= 1e-3 * abs(eager["exact"])
    # a second replay runs on the updated parameters
    loss2, _, _ = step(batch)
    torch.cuda.synchronize()
    assert np.isfinite(float(loss2))


def test_ce_tf32_unsupported_dim_names_supported_dims(ops):
    """D = 4 has no tensor-core engine: the tf32 request is an error naming the dims that have one."""
    from pivotcvae_b200 import _lib as L
    rng = np.random.default_rng(4)
    W = _unit_rows(rng, 1000, 4)
    Q = rng.standard_normal((64, 4)).astype(np.float32)
    tg = rng.integers(0, 1000, 64)
    with pytest.raises(L.PcvError, match="8, 16, 32, 64 and 128"):
        ops.ce_fwd_bwd(ops.Table(T(W)), T(Q), T(tg), 1.0, engine="tf32")


def test_ce_tf32_two_dims_one_device(ops):
    """D = 16 and then D = 128 in one process on one device: each instantiation sets its own shared-memory
    attribute before its first launch."""
    for D in (16, 128):
        rng = np.random.default_rng(D)
        n_items, M = 7001, 257
        W = _unit_rows(rng, n_items, D)
        Q = (rng.standard_normal((M, D)) * np.sqrt(8.0 / D)).astype(np.float32)
        tg = rng.integers(0, n_items, M)
        tab = ops.Table(T(W))
        loss, lse, dq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="tf32")
        el, _, edq = ops.ce_fwd_bwd(tab, T(Q), T(tg), 1.0, engine="exact")
        np.testing.assert_allclose(N(loss), N(el), rtol=1e-3, atol=1e-3)
        np.testing.assert_allclose(N(dq), N(edq), rtol=1e-2, atol=1e-3)
