"""-m gpu: the select, top-k, sampler and cross-entropy kernels at the edges of float32 (non-finite, zero, tiny and huge
query rows and table rows), against the CPU oracle bit for bit and against float64 restatements.

The non-finite contract is the one include/pcv_b200.h states and tests/test_float_edges_host.py pins on the oracle:
a NaN score never wins (it counts as -inf), and a row with no score above -inf returns its first index with value
-inf.  Every returned index is copied to the host and range-checked before anything indexes with it."""
import numpy as np
import pytest
import torch

import oracle
from gpu_util import N, T

pytestmark = pytest.mark.gpu

BIG = 1.0e38   # a finite table entry large enough that q . w overflows to +-inf


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _unit(rng, n, d):
    W = rng.standard_normal((n, d)).astype(np.float32)
    return W / np.linalg.norm(W, axis=1, keepdims=True)


def _engines(D):
    return ["simt", "tcgen05", "tcgen05_f16", "auto"] if D == 8 else ["simt", "tcgen05", "auto"]


def _f16_image(W):
    """pcv_table_create builds the f16 image of a D = 8 table iff 0 < max|w| < 1e4 (NaN rows do not count)."""
    ss = np.einsum("ij,ij->i", W.astype(np.float64), W.astype(np.float64))
    ss = ss[~np.isnan(ss)]
    m = np.sqrt(ss.max()) if ss.size else 0.0
    return W.shape[1] == 8 and 0.0 < m < 1.0e4


def _checked(idx, lo, hi):
    """Host copy of returned indices, range-checked before any use."""
    i = N(idx)
    assert i.dtype == np.int64
    bad = (i < lo) | (i >= hi)
    assert not bad.any(), "index outside [%d, %d): rows %s -> %s" % (lo, hi, np.nonzero(bad)[0][:8], i[bad][:8])
    return i


def _select(ops, tab, W, Q, engine, lo=0):
    idx, val = ops.score_select(tab, T(Q), "greedy", engine=engine)
    i = _checked(idx, lo, lo + W.shape[0])
    return i, N(val)


def _assert_select(ops, tab, W, Q, engine, what, lo=0):
    gi, gv = _select(ops, tab, W, Q, engine, lo)
    oi, ov = oracle.score_select(W, Q)
    oi = oi + lo
    bad = np.nonzero((gi != oi) | ~((gv == ov) | (np.isnan(gv) & np.isnan(ov))))[0]
    assert bad.size == 0, "%s [%s]: rows %s: got %s %s, oracle %s %s" % (
        what, engine, bad[:6], gi[bad][:6], gv[bad][:6], oi[bad][:6], ov[bad][:6])


def _edge_queries(rng, D, M=40):
    Q = (rng.standard_normal((M, D)) * rng.uniform(0.1, 3.0, (M, 1))).astype(np.float32)
    Q[1] = 0.0
    Q[2] = np.nan
    Q[3, D // 2] = np.nan
    Q[4, 0] = np.inf
    Q[5, D - 1] = -np.inf
    Q[6, 0], Q[6, 1] = np.inf, -np.inf
    Q[7] = np.inf
    Q[8] = -np.inf
    return Q


# ------------------------------------------------------------------ select: query rows
@pytest.mark.parametrize("D", [8, 16, 64, 128])
@pytest.mark.parametrize("n_items", [3000, 65536])
def test_select_edge_query_rows(ops, D, n_items):
    """Zero, all-NaN, one-NaN and +-inf query rows: every engine equals the oracle (index and value) and stays in the
    catalog.  Before the sentinel fix an all-NaN row came back as index 2^31 - 1."""
    rng = np.random.default_rng(D * 1000 + n_items)
    W = _unit(rng, n_items, D)
    Q = _edge_queries(rng, D)
    tab = ops.Table(T(W))
    for eng in _engines(D):
        _assert_select(ops, tab, W, Q, eng, "edge query rows")


def test_select_edge_query_rows_1m(ops):
    rng = np.random.default_rng(11)
    W = _unit(rng, 1 << 20, 8)
    Q = _edge_queries(rng, 8, 24)
    tab = ops.Table(T(W))
    for eng in _engines(8):
        _assert_select(ops, tab, W, Q, eng, "edge query rows, 1M items")


# ------------------------------------------------------------------ select: norm sweep
NORMS = [1e-30, 1e-25, 1e-22, 1e-15, 1.0, 1e15, 1e25, 1e30]


@pytest.mark.parametrize("D", [8, 16, 64, 128])
def test_select_query_norm_sweep(ops, D):
    """|q| from 1e-30 to 1e30 on a table of near-ties (every row within ~3 % of one direction), where the tf32 / f16
    approximate order differs from the fp32 order: the filters' bands must follow |q| all the way (at 1e30, |q|^2
    overflows while every score stays finite; below ~1e-19 it underflows)."""
    rng = np.random.default_rng(500 + D)
    n = 65536
    u = rng.standard_normal(D).astype(np.float32)
    u /= np.linalg.norm(u)
    W = u[None, :] + 0.03 * rng.standard_normal((n, D)).astype(np.float32)
    W = (W / np.linalg.norm(W, axis=1, keepdims=True)).astype(np.float32)
    base = u[None, :] + 0.03 * rng.standard_normal((64, D)).astype(np.float32)
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    tab = ops.Table(T(W))
    for s in NORMS:
        Q = (base * np.float32(s)).astype(np.float32)
        assert np.all(np.isfinite(Q)) and np.all(np.abs(Q).max(axis=1) > 0)
        for eng in _engines(D):
            _assert_select(ops, tab, W, Q, eng, "|q| = %g" % s)


@pytest.mark.parametrize("D", [8, 16])
def test_select_tiny_q_random_table(ops, D):
    """Tiny |q| on a random unit table, where items anti-aligned with q exist.  Between ~4e-23 and 5e-22, |q|^2 is a
    subnormal that has lost most of its bits: an f16 scale taken from it can push |q'| max|w| past 1, and the approximate
    score 1 + s' of an anti-aligned item below 0, whose f16 sign bit wins the filter's unsigned chunk maxima."""
    rng = np.random.default_rng(600 + D)
    n, M = 65536, 1024
    W = _unit(rng, n, D)
    base = _unit(rng, M, D)
    tab = ops.Table(T(W))
    for s in (5e-23, 1e-22, 2e-22, 3e-22, 1e-20, 1e-17):
        Q = (base * np.float32(s)).astype(np.float32)
        for eng in _engines(D):
            _assert_select(ops, tab, W, Q, eng, "random table, |q| = %g" % s)


# ------------------------------------------------------------------ select: table rows
EDGE_ROWS = ["nan_row", "nan_component", "zero_row", "norm_5e3", "norm_2e4", "norm_1e6", "overflow_row", "inf_row"]


def _edge_row(kind, D, rng):
    w = rng.standard_normal(D).astype(np.float32)
    w /= np.linalg.norm(w)
    if kind == "nan_row":
        return np.full(D, np.nan, np.float32)
    if kind == "nan_component":
        w[D // 2 - 1] = np.nan
        return w
    if kind == "zero_row":
        return np.zeros(D, np.float32)
    if kind.startswith("norm_"):
        return (w * np.float32(float(kind[5:]))).astype(np.float32)
    if kind == "overflow_row":
        return np.full(D, BIG, np.float32)
    if kind == "inf_row":
        return np.full(D, np.inf, np.float32)
    raise ValueError(kind)


def _edge_table(rng, n, D, kind, pos):
    W = _unit(rng, n, D)
    j = {"first": 3, "middle": n // 2 + 17, "last": n - 2}[pos]
    W[j] = _edge_row(kind, D, rng)
    return W, j


def _table_queries(rng, D, M=48):
    Q = (rng.standard_normal((M, D)) * rng.uniform(0.1, 3.0, (M, 1))).astype(np.float32)
    Q[: M // 4] = np.abs(Q[: M // 4])          # aligned with the overflow / inf rows: q . w = +inf
    Q[M // 4] = 0.0
    return Q


@pytest.mark.parametrize("D", [8, 16, 64, 128])
@pytest.mark.parametrize("chunk_tiles", [0, 3])
def test_select_edge_table_rows(ops, D, chunk_tiles, monkeypatch):
    """One NaN row, a row with one NaN component, a zero row, rows of norm 5e3, 2e4 and 1e6 (both sides of the f16
    filter's range (0, 1e4)), a finite row whose scores overflow to +-inf and an inf row, each in the first, a middle and the last
    column chunk (PCV_TC_CHUNK_TILES forces the chunked partition): every engine equals the oracle."""
    if chunk_tiles:
        monkeypatch.setenv("PCV_TC_CHUNK_TILES", str(chunk_tiles))
    rng = np.random.default_rng(900 + D + chunk_tiles)
    n = 3000
    for kind in EDGE_ROWS:
        for pos in ("first", "middle", "last"):
            W, _ = _edge_table(rng, n, D, kind, pos)
            Q = _table_queries(rng, D)
            tab = ops.Table(T(W))
            for eng in _engines(D):
                if eng == "tcgen05_f16" and not _f16_image(W):
                    with pytest.raises(Exception):
                        ops.score_select(tab, T(Q), "greedy", engine=eng)
                    continue
                _assert_select(ops, tab, W, Q, eng, "%s at %s" % (kind, pos))


@pytest.mark.parametrize("D", [8, 64])
def test_select_edge_table_rows_after_refresh(ops, D):
    """The fine_tune path: a handle created from a clean table (D = 8: with an f16 image), then the table is edited in
    place and Table.refresh() re-derives the images.  Same cases as above, same oracle."""
    rng = np.random.default_rng(1300 + D)
    n = 3000
    for kind in EDGE_ROWS:
        for pos in ("first", "middle", "last"):
            W, _ = _edge_table(rng, n, D, kind, pos)
            clean = _unit(rng, n, D)
            Wt = T(clean)
            tab = ops.Table(Wt)
            Wt.copy_(T(W))
            tab.refresh()
            Q = _table_queries(rng, D)
            for eng in _engines(D):
                _assert_select(ops, tab, W, Q, eng, "refreshed, %s at %s" % (kind, pos))


# ------------------------------------------------------------------ select: row shards
@pytest.mark.parametrize("D", [8, 32])
def test_select_row_shards_non_finite(ops, D):
    """Vocab-parallel: every shard's indices lie in its own rows, and the pcv_vp_pack_keys max-merge equals the whole
    table, including rows whose scores are NaN on every shard (NaN query) or on one shard (NaN table rows)."""
    rng = np.random.default_rng(1700 + D)
    n = 9000
    W = _unit(rng, n, D)
    W[3000:3100] = np.nan                 # a block of NaN rows inside shard 1
    W[6000:9000, 0] = np.nan              # shard 2: every score NaN
    Q = _edge_queries(rng, D)
    bounds = [0, 3000, 6000, 9000]
    full_i, full_v = oracle.score_select(W, Q)
    for eng in ("simt", "tcgen05", "auto"):
        keys = []
        for a, b in zip(bounds[:-1], bounds[1:]):
            shard = ops.Table(T(W[a:b]), row_offset=a)
            idx, val = ops.score_select(shard, T(Q), "greedy", engine=eng)
            i = _checked(idx, a, b)
            oi, ov = oracle.score_select(W[a:b], Q)
            assert np.array_equal(i, oi + a) and np.array_equal(N(val), ov), (eng, a)
            keys.append(ops.vp_pack_keys(val, idx))
        mi, mv = ops.vp_unpack_keys(torch.stack(keys).max(dim=0).values)
        assert np.array_equal(_checked(mi, 0, n), full_i) and np.array_equal(N(mv), full_v), eng


# ------------------------------------------------------------------ exprace
def test_exprace_non_finite(ops):
    """The SIMT exponential race (key = -E (1 + exp(-s))) where every key of a row overflows to -inf, with noise
    entries equal to 0, scores of -inf, and NaN queries: the oracle's bits, indices inside the catalog."""
    rng = np.random.default_rng(23)
    n, D, M = 5000, 8, 32
    u = np.ones(D, np.float32) / np.sqrt(D)
    W = (u[None, :] + 0.1 * rng.standard_normal((n, D))).astype(np.float32)
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    Q = (rng.standard_normal((M, D)) * 2.0).astype(np.float32)
    Q[0:8] = -1000.0 * u                           # s ~ -1000: exp(-s) clamps to e^88, E (1 + e^88) overflows
    noise = rng.exponential(1.0, (M, n)).astype(np.float32)
    noise[0:4] = 3.0 + noise[0:4]                  # rows 0..3: every key is -inf
    noise[4, 100] = 0.0                            # row 4: one zero noise entry wins (key -0)
    noise[5, [7, 4000]] = 0.0                      # row 5: two zero entries, lowest index
    noise[6] = 0.0                                 # row 6: all zero
    Q[8, 0] = -np.inf                              # row 8: s = -inf for items with w_0 > 0 ...
    noise[8, :50] = 0.0                            # ... together with E = 0
    Q[9] = np.nan
    Q[10, 3] = np.nan
    Q[11] = 0.0
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "exprace", noise=T(noise), engine="simt")
    i = _checked(idx, 0, n)
    oi, ov = oracle.score_select(W, Q, "exprace", noise)
    assert np.array_equal(i, oi)
    assert np.array_equal(N(val), ov)
    assert np.all(i[0:4] == 0) and np.all(ov[0:4] == -np.inf)
    assert i[4] == 100 and i[5] == 7


# ------------------------------------------------------------------ top-k and no-repeat
def _topk_table(rng, n, D):
    W = _unit(rng, n, D)
    W[10:14] = np.nan                               # NaN scores
    W[20:26] = 0.0
    W[20:26, 0] = -np.inf                           # q_0 > 0: -inf;  q_0 < 0: +inf
    return W


@pytest.mark.parametrize("n", [40, 3000])
def test_topk_non_finite(ops, n):
    """NaN and -inf entries inside the top-k window: only scores above -inf are listed (NaN counts as -inf), the rest
    of the window is -1 / -inf, as past the end of a short catalog."""
    rng = np.random.default_rng(31 + n)
    D, k = 8, 16
    W = _topk_table(rng, n, D)
    Q = (rng.standard_normal((24, D)) * 2.0).astype(np.float32)
    Q[:8, 0] = np.abs(Q[:8, 0]) + 20.0              # -inf on items 20..25, large scores elsewhere
    Q[8:12, 0] = -np.abs(Q[8:12, 0]) - 0.5          # +inf on items 20..25: six ties at +inf
    Q[12] = np.nan
    Q[13, 2] = np.nan
    Q[14] = 0.0
    tab = ops.Table(T(W))
    idx, val = ops.score_topk(tab, T(Q), k)
    gi = N(idx)
    assert np.all((gi == -1) | ((gi >= 0) & (gi < n)))
    oi, ov = oracle.score_topk(W, Q, k)
    assert np.array_equal(gi, oi)
    assert np.array_equal(N(val), ov)
    assert np.all(gi[12] == -1) and np.all(gi[8, :6] == np.arange(20, 26))


@pytest.mark.parametrize("engine", ["simt", "auto"])
def test_no_repeat_non_finite(ops, engine):
    """No-repeat slates with NaN / -inf scores, and slates in which two slots have no orderable score at all."""
    rng = np.random.default_rng(41)
    n, D, L, B = 3000, 8, 5, 24
    W = _topk_table(rng, n, D)
    Q = (rng.standard_normal((B * L, D)) * 2.0).astype(np.float32)
    Q[0:L] = Q[0] + 0.001 * Q[0:L]                  # slate 0: near-identical slots -> duplicates to resolve
    Q[1 * L + 1] = np.nan                           # slate 1: two slots with no orderable score
    Q[1 * L + 3, 4] = np.nan
    Q[2 * L:3 * L] = Q[2 * L]                       # slate 2: identical slots, one NaN
    Q[2 * L + 2] = np.nan
    Q[3 * L:4 * L, 0] = -np.abs(Q[3 * L:4 * L, 0]) - 0.5   # slate 3: every slot has six +inf ties
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine=engine, no_repeat=L)
    gi = _checked(idx, 0, n)
    oi, ov = oracle.slate_no_repeat(W, Q, L)
    assert np.array_equal(gi, oi)
    assert np.array_equal(N(val), ov)
    assert gi[1 * L + 1] == 0 and gi[1 * L + 3] == 0 and ov[1 * L + 1] == -np.inf
    assert np.array_equal(np.sort(gi[3 * L:4 * L]), np.arange(20, 25))


# ------------------------------------------------------------------ sampler
def test_sigmoid_categorical_non_finite(ops):
    """pcv_sigmoid_categorical on NaN, zero, huge and tiny query rows: the oracle's draws bit for bit, in [0, N)."""
    rng = np.random.default_rng(53)
    n, D, M = 4000, 8, 64
    W = _unit(rng, n, D)
    Q = (rng.standard_normal((M, D)) * 2.0).astype(np.float32)
    Q[0] = np.nan
    Q[1, 5] = np.nan
    Q[2] = 0.0
    Q[3:8] *= np.float32(1e30)
    Q[8:12] *= np.float32(1e-30)
    Q[12:16] *= np.float32(1e15)
    tab = ops.Table(T(W))
    idx = ops.sigmoid_categorical(tab, T(Q), seed=1234, offset=7)
    gi = _checked(idx, 0, n)
    oi, _ = oracle.sigmoid_categorical(W, Q, 1234, 7)
    assert np.array_equal(gi, oi)


# ------------------------------------------------------------------ cross-entropy against float64
U = 2.0 ** -24


def _tf32(a):
    """The tf32 engine's operands: fp32 with the low 13 mantissa bits dropped (kind::tf32 truncates)."""
    return (np.ascontiguousarray(a, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def _wmax(W):
    return float(np.sqrt(np.nanmax(np.einsum("ij,ij->i", W.astype(np.float64), W.astype(np.float64)))))


def _ce64(W, Q, tg, keep=None, Wt=None):
    """float64 restatement of the masked CE (train_generative.py:36-59): masked-out logits are 0 and stay in lse.
    Wt: the table the target row of dq is read from (default W).  -> (loss, lse, dq, p)."""
    W64, Q64 = W.astype(np.float64), Q.astype(np.float64)
    y = Q64 @ W64.T
    M = Q.shape[0]
    if keep is not None:
        keep = keep.copy()
        keep[np.arange(M), tg] = True
        y = np.where(keep, y, 0.0)
    m = y.max(axis=1, keepdims=True)
    e = np.exp(y - m)
    lse = m[:, 0] + np.log(e.sum(axis=1))
    p = e / e.sum(axis=1, keepdims=True)
    if keep is not None:
        p = np.where(keep, p, 0.0)
    dq = p @ W64 - (W if Wt is None else Wt).astype(np.float64)[tg]
    return lse - y[np.arange(M), tg], lse, dq, p


def _ce64_tf32(W, Q, tg):
    """The tf32 engine restated in float64: logits of the truncated operands for lse and the soft-max, while the target
    logit (loss = lse - y_t) and the target row of dq are the exact fp32 ones, as ce_finalize_kernel re-derives them."""
    _, lse, dq, p = _ce64(_tf32(W), _tf32(Q), tg, Wt=W)
    yt = np.einsum("id,id->i", Q.astype(np.float64), W.astype(np.float64)[tg])
    return lse - yt, lse, dq, p


def _ce_tol(W, Q, kind, n_terms=None):
    """Per-row bounds on |engine - float64 restatement|, u = 2^-24.

    kind "exact" (against the restatement on the fp32 operands): a logit is a D-term fp32 FMA chain, within
    delta = gamma_D |q| max|w| of the exact one, gamma_D = D u / (1 - D u).
    kind "tf32" (against _ce64_tf32, the restatement on the tf32-truncated operands): the products of two 11-bit mantissas
    are exact in fp32, so only the fp32 accumulation of D of them remains (gamma_D |q| max|w| again, as
    sum_k |q_k w_k| <= |q| |w|); the exponent argument y log2(e) - c is rounded in fp32 (|y|, |c| <= 1.01 |q| max|w|:
    4 u (|q| max|w| + 1)), and ex2.approx is good to 2^-21 relative, one more logit shift of that size.
    Then lse and the target logit move by at most delta each; the fp32 sum of the n exponentials adds at most
    (n + 16) u to log L, and rounding a value of size |lse| a few ulps (8 u |lse|).  dq = sum p w - w_t: a shift of
    every logit by at most delta moves each p by a factor within exp(+-2 delta), so |dq| moves by at most
    (exp(2 delta) - 1) max|w|, and the fp32 accumulation over n items adds n u max|w|.  The tf32 engine's gradient MMA
    truncates P to tf32 (2^-10 relative per term) and may subtract the truncated target row (2^-10 |w_t|): 2^-9 max|w|
    more."""
    D = W.shape[1]
    n = W.shape[0] if n_terms is None else n_terms
    wmax = _wmax(W)
    qw = np.linalg.norm(Q.astype(np.float64), axis=1) * wmax
    delta = D * U / (1 - D * U) * qw
    if kind == "tf32":
        delta = delta + 4 * U * (qw + 1) + 2.0 ** -21
    loss_tol = 2 * delta + (n + 16) * U + 8 * U * (qw + np.log(n))
    dq_tol = (np.expm1(2 * delta) + n * U + (2.0 ** -9 if kind == "tf32" else 0.0)) * wmax + 1e-6
    return loss_tol, dq_tol


def _ce_queries(rng, W, M, qnorm):
    D = W.shape[1]
    Q = rng.standard_normal((M, D))
    Q[: M // 2] += 3.0 * W[rng.integers(0, W.shape[0], M // 2)]   # peaked soft-max: dq = acc / L - w_t cancels
    Q = Q / np.linalg.norm(Q, axis=1, keepdims=True) * qnorm
    return Q.astype(np.float32)


def _assert_ce(got, want, W, Q, kind, rows=None, what="", n_terms=None):
    loss, lse, dq = (N(x) for x in got[:3])
    wl, wlse, wdq = want[:3]
    lt, dt = _ce_tol(W, Q, kind, n_terms)
    r = np.arange(Q.shape[0]) if rows is None else rows
    for name, g, w, t in (("loss", loss, wl, lt), ("lse", lse, wlse, lt)):
        err = np.abs(g[r] - w[r])
        assert np.all(err <= t[r]), "%s %s: max err %g (bound %g)" % (what, name, err.max(), t[r][np.argmax(err - t[r])])
    err = np.abs(dq[r] - wdq[r]).max(axis=1)
    assert np.all(err <= dt[r]), "%s dq: max err %g (bound %g)" % (what, err.max(), dt[r][np.argmax(err - dt[r])])


def _assert_grad(what, dW, want, S):
    """|dW - float64| <= 2 S elementwise (the magnitude sum of test_gpu_table_grad.py's error model)."""
    err = np.abs(N(dW).astype(np.float64) - want)
    bound = 2 * S + 1e-30
    bad = ~(err <= bound)
    assert not bad.any(), "%s: %d elements over the bound, worst err %g (bound there %g)" % (
        what, int(bad.sum()), float(err[bad].max()), float(bound[bad][np.argmax(err[bad])]))


def _tgrad64(W, Q, tg, rs, lse, keep=None, n_terms=None):
    """float64 d(sum_i rs_i CE_i)/dW of the masked CE, and the bound's magnitude sum S.  A term rs_i (p_ij - [t_i = j])
    q_i of dW[j] has p_ij right to a relative expm1(2 delta_i) (the logit error of _ce_tol, kind exact) plus
    |lse_i - lse64_i| (the kernel uses its forward's fp32 lse) plus ~2 ulp of __expf (2e-5 covers it); the fp32 sum of
    at most n_terms terms per element adds n_terms u of their magnitudes."""
    M, D = Q.shape
    _, lse64, _, p = _ce64(W, Q, tg, keep)
    delta = D * U / (1 - D * U) * np.linalg.norm(Q.astype(np.float64), axis=1) * _wmax(W)
    rel = np.expm1(2 * delta) + np.abs(N(lse).astype(np.float64) - lse64) + 2e-5 + (M if n_terms is None else n_terms) * U
    g = p.copy()
    g[np.arange(M), tg] -= 1.0
    mag = p.copy()
    mag[np.arange(M), tg] += 1.0
    Q64 = Q.astype(np.float64)
    return (g * rs[:, None]).T @ Q64, (mag * (np.abs(rs) * rel)[:, None]).T @ np.abs(Q64)


@pytest.mark.parametrize("D", [8, 32, 128])
@pytest.mark.parametrize("qnorm", [30.0, 100.0])
@pytest.mark.parametrize("unit", [True, False])
def test_ce_large_q_float64(ops, D, qnorm, unit):
    """The exact engine (dense and bitmask) and the tf32 engine at |q| = 30 and 100, unit-norm and unnormalised
    tables, against float64 within the derived bounds; the tf32 engine against the restatement on its truncated
    operands, so its bound stays that of an fp32 computation."""
    rng = np.random.default_rng(int(qnorm) + D + 7 * unit)
    n, M = 5000, 256
    W = _unit(rng, n, D)
    if not unit:
        W = (W * rng.uniform(0.2, 3.0, (n, 1))).astype(np.float32)
    Q = _ce_queries(rng, W, M, qnorm)
    tg = rng.integers(0, n, M)
    tab = ops.Table(T(W))
    _assert_ce(ops.ce_fwd_bwd(tab, T(Q), T(tg), engine="exact"), _ce64(W, Q, tg), W, Q, "exact", what="exact dense")
    got = ops.ce_fwd_bwd(tab, T(Q), T(tg), engine="tf32")
    # rows failing the reference-exponent test (lb < ub - 140, ce_ref_kernel) are redone in exact fp32; rows within 1 of
    # that threshold may go either way and are held to the bound of whichever path they took
    ub = np.linalg.norm(Q.astype(np.float64), axis=1) * _wmax(W) * 1.01
    y = Q.astype(np.float64) @ W[:32].astype(np.float64).T
    lb = np.maximum(y.max(axis=1), np.einsum("id,id->i", Q.astype(np.float64), W.astype(np.float64)[tg])) - 0.01 * ub
    margin = lb - (ub - 140.0)
    flagged, tc_rows = np.nonzero(margin < -1.0)[0], np.nonzero(margin > 1.0)[0]
    _assert_ce(got, _ce64_tf32(W, Q, tg), W, Q, "tf32", rows=tc_rows, what="tf32 dense")
    _assert_ce(got, _ce64(W, Q, tg), W, Q, "exact", rows=flagged, what="tf32 dense, flagged rows")
    for r in np.nonzero(np.abs(margin) <= 1.0)[0]:
        try:
            _assert_ce(got, _ce64_tf32(W, Q, tg), W, Q, "tf32", rows=[r], what="tf32 dense, threshold row")
        except AssertionError:
            _assert_ce(got, _ce64(W, Q, tg), W, Q, "exact", rows=[r], what="tf32 dense, threshold row")
    keep = rng.random((M, n)) < 0.3
    Qm = Q.copy()
    # rows whose kept logits (the target aside) are all below -5: the masked-out zeros carry lse
    keep[: M // 4] = (rng.random((M // 4, n)) < 0.05) & (Qm[: M // 4].astype(np.float64) @ W.T.astype(np.float64) < -5.0)
    bits = oracle.pack_bitmask(keep)
    _assert_ce(ops.ce_fwd_bwd(tab, T(Qm), T(tg), bitmask=T(bits.view(np.int32))), _ce64(W, Qm, tg, keep), W, Qm, "exact",
               what="exact bitmask")


@pytest.mark.parametrize("D", [8, 64])
def test_ce_tf32_flagged_rows_large_q_float64(ops, D):
    """|q| = 100 rows whose first 32 items point away from q fail the tf32 engine's reference-exponent test
    (lb < ub - 140): they are redone in exact fp32 and meet the exact engine's float64 bound; the others the tf32 one."""
    rng = np.random.default_rng(61 + D)
    n, M = 5000, 128
    u0 = rng.standard_normal(D).astype(np.float32)
    u0 /= np.linalg.norm(u0)
    W = _unit(rng, n, D)
    head = -u0[None, :] + 0.1 * rng.standard_normal((32, D)).astype(np.float32)
    W[:32] = head / np.linalg.norm(head, axis=1, keepdims=True)
    Q = _ce_queries(rng, W, M, 100.0)
    bad = np.arange(0, M, 9)
    for r in bad:
        v = u0 + 0.05 * rng.standard_normal(D).astype(np.float32)
        Q[r] = 100.0 * v / np.linalg.norm(v)
    ub = np.linalg.norm(Q[bad], axis=1) * 1.01
    assert np.all((Q[bad] @ W[:32].T).max(axis=1) < ub - 140.0)
    tg = rng.integers(32, n, M)
    tg[bad] = 5                                   # a far-off target: lb = max(target, first 32 items) stays low
    tab = ops.Table(T(W))
    got = ops.ce_fwd_bwd(tab, T(Q), T(tg), engine="tf32")
    _assert_ce(got, _ce64(W, Q, tg), W, Q, "exact", rows=bad, what="tf32 flagged rows")
    _assert_ce(got, _ce64_tf32(W, Q, tg), W, Q, "tf32", rows=np.setdiff1d(np.arange(M), bad),
               what="tf32 other rows")


@pytest.mark.parametrize("D", [8, 64])
@pytest.mark.parametrize("qnorm", [30.0, 100.0])
@pytest.mark.parametrize("keep_prob", [1e-4, 0.5])
def test_ce_philox_large_q_float64(ops, D, qnorm, keep_prob):
    """The Philox mask mode (the gap-process mask oracle.bernoulli_bitmask restates) at large |q|: loss, lse, dq and
    the table gradient against float64.  At keep_prob 1e-4 a row keeps its target and a stray column or none: the
    masked-out zeros carry lse."""
    rng = np.random.default_rng(int(qnorm) * 3 + D + int(keep_prob * 10))
    n, M = 5000, 128
    W = _unit(rng, n, D)
    Q = _ce_queries(rng, W, M, qnorm)
    tg = rng.integers(0, n, M)
    rs = rng.standard_normal(M)
    tab = ops.Table(T(W))
    seed, off = 77 + D, 13
    bits = oracle.bernoulli_bitmask(seed, off, M, n, keep_prob)
    keep = np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(bool)
    got = ops.ce_fwd_bwd(tab, T(Q), T(tg), keep_prob, seed=seed, offset=off)
    _assert_ce(got, _ce64(W, Q, tg, keep), W, Q, "exact", what="philox %g" % keep_prob)
    dW = ops.ce_table_grad(tab, T(Q), T(tg), got[1], T(rs.astype(np.float32)), keep_prob, seed=seed, offset=off)
    want, S = _tgrad64(W, Q, tg, rs.astype(np.float32).astype(np.float64), got[1], keep)
    _assert_grad("philox %g table grad" % keep_prob, dW, want, S)


@pytest.mark.parametrize("D", [8, 64])
@pytest.mark.parametrize("qnorm", [30.0, 100.0])
def test_ce_table_grad_large_q_float64(ops, D, qnorm):
    """ce_table_grad at large |q|: the exact engine dense and with a bitmask, and the tf32 engine (error model of
    test_gpu_table_grad.py's tf32 test: tf32 logits, the tf32 forward's lse, the gradient MMA's truncation)."""
    rng = np.random.default_rng(int(qnorm) * 5 + D)
    n, M = 5000, 130
    W = _unit(rng, n, D)
    Q = _ce_queries(rng, W, M, qnorm)
    tg = rng.integers(0, n, M)
    tg[: M // 3] = tg[0]                                   # one item is the target of a third of the rows
    rs = rng.standard_normal(M).astype(np.float32)
    rs[::7] = 0.0
    rs64 = rs.astype(np.float64)
    tab = ops.Table(T(W))
    _, lse, _ = ops.ce_fwd_bwd(tab, T(Q), T(tg), want_dq=False)
    want, S = _tgrad64(W, Q, tg, rs64, lse)
    _assert_grad("exact dense", ops.ce_table_grad(tab, T(Q), T(tg), lse, T(rs)), want, S)
    keep = rng.random((M, n)) < 0.1
    bm = T(oracle.pack_bitmask(keep).view(np.int32))
    _, lse, _ = ops.ce_fwd_bwd(tab, T(Q), T(tg), 0.1, bitmask=bm, want_dq=False)
    want, S = _tgrad64(W, Q, tg, rs64, lse, keep)
    _assert_grad("exact bitmask", ops.ce_table_grad(tab, T(Q), T(tg), lse, T(rs), 0.1, bitmask=bm), want, S)
    _, lse, _ = ops.ce_fwd_bwd(tab, T(Q), T(tg), want_dq=False, engine="tf32")
    dW = ops.ce_table_grad(tab, T(Q), T(tg), lse, T(rs), engine="tf32")
    _, lse64, _, p = _ce64(W, Q, tg)
    qn = np.linalg.norm(Q.astype(np.float64), axis=1)
    rel = np.expm1(2.0 ** -9 * qn) + np.abs(N(lse).astype(np.float64) - lse64) + 2.0 ** -9 + 2e-5 + 2 * M * U
    p[np.arange(M), tg] += 1.0
    _assert_grad("tf32", dW, _tgrad64(W, Q, tg, rs64, lse)[0],
                 (p * (np.abs(rs64) * rel)[:, None]).T @ np.abs(Q.astype(np.float64)))


@pytest.mark.parametrize("D", [8, 64])
@pytest.mark.parametrize("qnorm", [30.0, 100.0])
def test_cand_ce_large_q_float64(ops, D, qnorm):
    """Candidate mode with 1000 candidates per row and the target at a column >= 32: loss, lse, dq and the table
    gradient (duplicate candidates included) against float64."""
    rng = np.random.default_rng(int(qnorm) * 7 + D)
    n, M, nC = 5000, 64, 1000
    W = _unit(rng, n, D)
    Q = _ce_queries(rng, W, M, qnorm)
    cand = rng.integers(0, n, (M, nC))
    cand[:, 40] = cand[:, 0]                               # duplicates within a row
    tpos = rng.integers(32, nC, M)
    tpos[:4] = 40                                          # the target is a duplicated column
    for i in range(M // 2):                                # peaked rows: the target is the item q points at
        cand[i, tpos[i]] = int(np.argmax(W @ Q[i]))
    rs = rng.standard_normal(M).astype(np.float32)
    tab = ops.Table(T(W))
    loss, lse, dq, _ = ops.cand_ce_fwd_bwd(tab, T(Q), T(cand), T(tpos))
    Wc = W.astype(np.float64)[cand]                                      # [M, nC, D]
    X = np.einsum("icd,id->ic", Wc, Q.astype(np.float64))
    mx = X.max(axis=1, keepdims=True)
    lse64 = mx[:, 0] + np.log(np.exp(X - mx).sum(axis=1))
    P = np.exp(X - lse64[:, None])
    want = (lse64 - X[np.arange(M), tpos], lse64, np.einsum("ic,icd->id", P, Wc) - Wc[np.arange(M), tpos])
    _assert_ce((loss, lse, dq), want, W, Q, "exact", what="candidates", n_terms=nC)
    dW = ops.cand_ce_table_grad(tab, T(Q), T(cand), T(tpos), lse, T(rs))
    delta = D * U / (1 - D * U) * np.linalg.norm(Q.astype(np.float64), axis=1) * _wmax(W)
    rel = np.expm1(2 * delta) + np.abs(N(lse).astype(np.float64) - lse64) + 2e-5 + M * nC * U
    G = P.copy()
    G[np.arange(M), tpos] -= 1.0
    Mag = P.copy()
    Mag[np.arange(M), tpos] += 1.0
    Q64 = Q.astype(np.float64)
    want_dW = np.zeros((n, D))
    S = np.zeros((n, D))
    np.add.at(want_dW, cand.reshape(-1), ((G * rs[:, None])[:, :, None] * Q64[:, None, :]).reshape(-1, D))
    np.add.at(S, cand.reshape(-1), ((Mag * (np.abs(rs) * rel)[:, None])[:, :, None] * np.abs(Q64)[:, None, :]).reshape(-1, D))
    _assert_grad("candidate table grad", dW, want_dW, S)


@pytest.mark.parametrize("D", [8, 64])
@pytest.mark.parametrize("qnorm", [30.0, 100.0])
def test_ce_vocab_parallel_large_q_float64(ops, D, qnorm):
    """ce_partials over three row shards + ce_vp_merge, and ce_shard_table_grad on each shard, at large |q| against
    float64: the merge of the shards' (m, l, acc) records must not lose what one shard's rescaling keeps."""
    rng = np.random.default_rng(int(qnorm) * 11 + D)
    n, M = 5000, 96
    W = _unit(rng, n, D)
    Q = _ce_queries(rng, W, M, qnorm)
    tg = rng.integers(0, n, M)
    rs = rng.standard_normal(M).astype(np.float32)
    bounds = [0, 1664, 3328, n]                           # shard offsets: multiples of 128
    shards = [ops.Table(T(W[a:b]), row_offset=a) for a, b in zip(bounds[:-1], bounds[1:])]
    recs = torch.stack([ops.ce_partials(s, T(Q), T(tg)) for s in shards])
    loss, lse, dq = ops.ce_vp_merge(recs, T(W), T(Q), T(tg))
    _assert_ce((loss, lse, dq), _ce64(W, Q, tg), W, Q, "exact", what="vp merge")
    want, S = _tgrad64(W, Q, tg, rs.astype(np.float64), lse)
    for s, a, b in zip(shards, bounds[:-1], bounds[1:]):
        dW = ops.ce_shard_table_grad(s, T(Q), T(tg), lse, T(rs))
        _assert_grad("shard [%d, %d) table grad" % (a, b), dW, want[a:b], S[a:b])


@pytest.mark.parametrize("engine", ["exact", "tf32"])
@pytest.mark.parametrize("D", [8, 64])
def test_ce_nan_row_is_isolated(ops, engine, D):
    """A NaN query row gives NaN loss, lse and dq in that row; every other row is bitwise what it is without it (the
    tf32 engine shares a 128-row tile between them)."""
    rng = np.random.default_rng(71 + D)
    n, M = 3000, 200
    W = _unit(rng, n, D)
    Q = _ce_queries(rng, W, M, 30.0)
    tg = rng.integers(0, n, M)
    tab = ops.Table(T(W))
    ref = [N(x) for x in ops.ce_fwd_bwd(tab, T(Q), T(tg), engine=engine)]
    Qn = Q.copy()
    Qn[5] = np.nan
    Qn[130, 1] = np.nan
    got = [N(x) for x in ops.ce_fwd_bwd(tab, T(Qn), T(tg), engine=engine)]
    other = np.setdiff1d(np.arange(M), [5, 130])
    for g, r in zip(got, ref):
        assert np.all(np.isnan(g[[5, 130]]))
        assert np.array_equal(g[other], r[other])


def test_engines_share_one_workspace(ops):
    """The SIMT engine's partial winners must not land in the head of the workspace that the tcgen05 engine needs zero
    on entry (overflow counter, per-row overflow winners): any order of engines on one table, one M."""
    rng = np.random.default_rng(83)
    n, M = 3000, 512
    W = _unit(rng, n, 8)
    W[100:140] = W[7]                       # exact ties: overflow lists in use
    Q = (rng.standard_normal((M, 8)) * 2.0).astype(np.float32)
    Q[:64] = 1.5 * W[7]
    tab = ops.Table(T(W))
    oi, ov = oracle.score_select(W, Q)
    for eng in ("simt", "tcgen05", "simt", "tcgen05_f16", "simt", "auto", "simt", "tcgen05"):
        gi, gv = _select(ops, tab, W, Q, eng)
        assert np.array_equal(gi, oi) and np.array_equal(gv, ov), eng
