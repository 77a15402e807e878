"""-m gpu: the tcgen05/TMEM/TMA score+select engine (tf32 filter + exact fp32 refine)
must return the same bits as the exact SIMT engine and the CPU oracle."""
import numpy as np
import pytest
import torch

import oracle
from gpu_util import N, T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


@pytest.fixture(params=["tcgen05", "tcgen05_f16"])
def tc_engine(request):
    """D = 8 runs on both tensor-core filters: tf32 operands / fp32 accumulators, and f16 operands / f16 accumulators
    (packed TMEM reads, 16-bit packed maxima); the exact refine makes their results identical."""
    return request.param


def _unit(rng, n, d=8):
    W = rng.standard_normal((n, d)).astype(np.float32)
    return W / np.linalg.norm(W, axis=1, keepdims=True)


@pytest.mark.parametrize("n_items,M", [(256, 128), (300, 1), (2048, 128), (2049, 130), (4095, 77), (50000, 1024),
                                       (65536, 300), (100003, 515), (3707, 320)])
def test_tc_matches_oracle(ops, n_items, M, tc_engine):
    rng = np.random.default_rng(n_items * 7 + M)
    W = _unit(rng, n_items)
    Q = (rng.standard_normal((M, 8)) * rng.uniform(0.05, 3.0, (M, 1))).astype(np.float32)
    if n_items > 600:   # exact ties: duplicated rows in different tiles / splits / column halves
        W[n_items - 1] = W[5]
        W[n_items // 2 + 3] = W[5]
        W[300] = W[5]
        Q[0] = 1.7 * W[5]
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine=tc_engine)
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi)
    assert np.array_equal(N(val), ov)       # the refine is the exact fp32 FMA chain: bitwise
    if n_items > 600:
        assert N(idx)[0] == 5
    si, sv = ops.score_select(tab, T(Q), "greedy", engine="simt")
    assert torch.equal(idx, si) and torch.equal(val, sv)


def test_tc_golden_dims8(ops, golden, tc_engine):
    fx = golden("dims")
    tab = ops.Table(T(fx["d8/W"]))
    idx, val = ops.score_select(tab, T(fx["d8/Q"]), "greedy", engine=tc_engine)
    assert np.array_equal(N(idx), fx["d8/idx"]) and np.array_equal(N(val), fx["d8/val"])   # == torch.mm + torch.max


@pytest.mark.parametrize("D", [16, 32, 64, 128])
def test_tc_golden_other_dims(ops, golden, D):
    """--dim is free in the reference (train_generative.py:302): the tcgen05 filter walks D in k-atoms of 8."""
    fx = golden("dims")
    W, Q = fx["d%d/W" % D], fx["d%d/Q" % D]
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine="tcgen05")
    assert np.array_equal(N(idx), fx["d%d/idx" % D])       # the reference's torch.mm + torch.max indices
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(val), ov)


@pytest.mark.parametrize("n_items,M,D", [(256, 128, 16), (2049, 130, 16), (50000, 1024, 16), (4095, 77, 32), (65536, 300, 32),
                                         (100003, 515, 64), (3707, 320, 64), (300, 1, 128), (40001, 700, 128), (9000, 129, 128)])
def test_tc_other_dims_match_oracle(ops, n_items, M, D):
    rng = np.random.default_rng(n_items * 7 + M + D)
    W = _unit(rng, n_items, D)
    Q = (rng.standard_normal((M, D)) * rng.uniform(0.05, 3.0, (M, 1))).astype(np.float32)
    if n_items > 600:   # exact ties in different tiles / column slices, a tie block that overflows the lists
        W[n_items - 1] = W[5]
        W[n_items // 2 + 3] = W[5]
        W[300] = W[5]
        Q[0] = 1.7 * W[5]
        W[400:400 + 150] = W[400]
        Q[1 % M] = 2.0 * W[400]
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine="tcgen05")
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi)
    assert np.array_equal(N(val), ov)
    si, sv = ops.score_select(tab, T(Q), "greedy", engine="simt")
    assert torch.equal(idx, si) and torch.equal(val, sv)
    ai, av = ops.score_select(tab, T(Q), "greedy", engine="auto")
    assert torch.equal(idx, ai) and torch.equal(val, av)


def test_tc_all_equal_and_heavy_ties(ops, tc_engine):
    """Every item inside the band: lists collapse continuously; the first index must still win."""
    W = np.tile(np.array([[0.5, 0.5, 0.5, 0.5, 0, 0, 0, 0]], dtype=np.float32), (5000, 1))
    Q = np.ones((130, 8), dtype=np.float32)
    idx, _ = ops.score_select(ops.Table(T(W)), T(Q), "greedy", engine=tc_engine)
    assert np.array_equal(N(idx), np.zeros(130, dtype=np.int64))
    rng = np.random.default_rng(0)
    W2 = _unit(rng, 6000)
    W2[1000:1400] = W2[999]          # 401 exact duplicates of the best row for Q2[0]
    Q2 = rng.standard_normal((64, 8)).astype(np.float32)
    Q2[0] = W2[999]
    idx2, val2 = ops.score_select(ops.Table(T(W2)), T(Q2), "greedy", engine=tc_engine)
    oi, ov = oracle.score_select(W2, Q2)
    assert np.array_equal(N(idx2), oi) and np.array_equal(N(val2), ov) and N(idx2)[0] == 999


def test_tc_near_ties_inside_tf32_error(ops, tc_engine):
    """Items whose exact scores differ by less than the tf32 error: the filter may misorder them,
    the refine must not."""
    rng = np.random.default_rng(42)
    W = _unit(rng, 8192)
    q = _unit(rng, 1)[0]
    # rows that score within ~1e-6 of each other around the maximum
    base = q / np.linalg.norm(q)
    for j, d in zip([17, 4000, 8000, 6001], [3e-7, 1e-7, 2e-7, 0.0]):
        pert = base + d * rng.standard_normal(8)
        W[j] = (pert / np.linalg.norm(pert)).astype(np.float32)
    Q = np.repeat(q[None], 128, 0).astype(np.float32) * np.linspace(0.1, 4, 128, dtype=np.float32)[:, None]
    idx, val = ops.score_select(ops.Table(T(W)), T(Q), "greedy", engine=tc_engine)
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(val), ov)


def test_tc_unnormalised_table_and_zero_query(ops, tc_engine):
    rng = np.random.default_rng(9)
    W = (rng.standard_normal((7000, 8)) * rng.uniform(0.1, 20, (7000, 1))).astype(np.float32)
    Q = rng.standard_normal((200, 8)).astype(np.float32) * 5
    Q[3] = 0       # all scores equal (0): index 0 wins
    idx, val = ops.score_select(ops.Table(T(W)), T(Q), "greedy", engine=tc_engine)
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(val), ov) and N(idx)[3] == 0


def test_tc_full_size_properties_packed_key_merge(ops, tc_engine):
    """BASELINE C4 size (1M items, 20480 rows): shard-merge invariance, planted maxima, and the
    winning value re-derived from the returned index (no oracle run at this size)."""
    g = torch.Generator(device="cuda").manual_seed(1)
    n_items, M = 1_000_000, 20480
    W = torch.nn.functional.normalize(torch.randn(n_items, 8, generator=g, device="cuda"), dim=1)
    Q = torch.randn(M, 8, generator=g, device="cuda")
    plant = torch.randint(0, n_items, (64,), generator=g, device="cuda")
    Q[:64] = 2.5 * W[plant]                      # the planted row is the unique maximiser (cos = 1)
    full = ops.Table(W)
    idx, val = ops.score_select(full, Q, "greedy", engine=tc_engine)
    assert torch.equal(W[idx[:64]], W[plant])
    # value == exact chain of the returned index, and no random probe beats it
    probe = torch.randint(0, n_items, (M, 64), generator=g, device="cuda")
    ps = (W[probe] * Q[:, None, :]).sum(-1)
    assert bool((ps.max(1).values <= val + 1e-5).all())
    G = 4
    per = n_items // G
    keys = []
    for s in range(G):
        t = ops.Table(W[s * per:(s + 1) * per], row_offset=s * per)
        i, v = ops.score_select(t, Q, "greedy", engine=tc_engine)
        keys.append(ops.vp_pack_keys(v, i))
    mi, mv = ops.vp_unpack_keys(torch.stack(keys).max(0).values)     # the all-reduce(MAX) merge, on one device
    assert torch.equal(mi, idx) and torch.equal(mv, val)
    si, sv = ops.score_select(full, Q[:2048], "greedy", engine="simt")
    assert torch.equal(si, idx[:2048]) and torch.equal(sv, val[:2048])


def test_tc_row_groups_and_max_size(ops, tc_engine):
    """M large enough that the workspace budget forces several row groups (C5-style: 10 M items)."""
    g = torch.Generator(device="cuda").manual_seed(5)
    n_items, M = 10_000_000, 16384
    W = torch.nn.functional.normalize(torch.randn(n_items, 8, generator=g, device="cuda"), dim=1)
    Q = torch.randn(M, 8, generator=g, device="cuda")
    plant = torch.randint(0, n_items, (M,), generator=g, device="cuda")
    Q[::7] = 1.5 * W[plant[::7]]
    tab = ops.Table(W)
    assert tab.workspace("select", M).numel() <= (200 << 20)
    idx, val = ops.score_select(tab, Q, "greedy", engine=tc_engine)
    assert torch.equal(W[idx[::7]], W[plant[::7]])
    exact = (W[idx] * Q).sum(-1)
    assert bool(((exact - val).abs() <= 1e-5).all())
    si, sv = ops.score_select(tab, Q[:512], "greedy", engine="simt")
    assert torch.equal(si, idx[:512]) and torch.equal(sv, val[:512])


@pytest.mark.parametrize("n_items,M,chunk_tiles", [(50000, 700, 16), (100003, 515, 64), (9000, 300, 3), (65536, 1500, 100)])
def test_tc_column_chunks(ops, monkeypatch, n_items, M, chunk_tiles, tc_engine):
    """Catalogs beyond the L2 are walked in column chunks (32 MB each in production); PCV_TC_CHUNK_TILES forces the
    chunked partition on small catalogs: same bits as the oracle, ties across chunks -> lowest index, heavy ties
    (flagged streams, overflow lists) inside a chunk."""
    monkeypatch.setenv("PCV_TC_CHUNK_TILES", str(chunk_tiles))
    rng = np.random.default_rng(n_items + chunk_tiles)
    W = _unit(rng, n_items)
    Q = (rng.standard_normal((M, 8)) * rng.uniform(0.05, 3.0, (M, 1))).astype(np.float32)
    W[n_items - 1] = W[5]                       # duplicates in the first, a middle and the last chunk
    W[n_items // 2 + 3] = W[5]
    W[chunk_tiles * 256 + 7] = W[5]
    Q[0] = 1.7 * W[5]
    W[n_items // 3: n_items // 3 + 700] = W[n_items // 3]      # 700-way tie block inside one chunk
    Q[1] = 2.0 * W[n_items // 3]
    tab = ops.Table(T(W))
    idx, val = ops.score_select(tab, T(Q), "greedy", engine=tc_engine)
    oi, ov = oracle.score_select(W, Q)
    assert np.array_equal(N(idx), oi) and np.array_equal(N(val), ov)
    assert N(idx)[0] == 5 and N(idx)[1] == n_items // 3
    monkeypatch.delenv("PCV_TC_CHUNK_TILES")
    idx1, val1 = ops.score_select(ops.Table(T(W)), T(Q), "greedy", engine=tc_engine)     # one chunk: same answer
    assert torch.equal(idx, idx1) and torch.equal(val, val1)


def test_f16_filter_hands_over_no_more_than_the_tf32_filter(ops):
    """Regression guard for the f16 filter's band.  Its band is a constant of the scaled domain, so relative to |q| it
    is 1 / (|q'| max|w|) times wider: with a power-of-two scale (|q'| max|w| anywhere in [0.5, 1)) streams at 10 M
    items overflowed their four hand-over slots, were flagged and re-scanned exactly by the refine kernel — still
    bit-exact, but the call took 1.4x (16384 rows) to 2.6x (65536 rows) the tf32 filter's time instead of 0.84x.
    Same results, and the f16 call must not be slower than the tf32 one by more than a generous margin."""
    g = torch.Generator(device="cuda").manual_seed(11)
    n_items, M = 10_000_000, 16384
    W = torch.nn.functional.normalize(torch.randn(n_items, 8, generator=g, device="cuda"), dim=1)
    Q = torch.randn(M, 8, generator=g, device="cuda") * torch.empty(M, 1, device="cuda").uniform_(0.3, 3.0, generator=g)
    tab = ops.Table(W)

    def run(engine):
        out = ops.score_select(tab, Q, "greedy", engine=engine)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.score_select(tab, Q, "greedy", engine=engine)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return out, sorted(ts)[2]

    (ti, tv), t_tf32 = run("tcgen05")
    (hi, hv), t_f16 = run("tcgen05_f16")
    assert torch.equal(ti, hi) and torch.equal(tv, hv)
    print("10 M x %d: tf32 filter %.2f ms, f16 filter %.2f ms" % (M, t_tf32, t_f16))
    assert t_f16 < 1.25 * t_tf32

