"""-m gpu: pcv_table_refresh, the in-place refresh of an item-table handle, and the fine_tune steps built on it.

1. After W changes in place (random perturbation, one row grown so that max|w| grows, the table shrunk), a refreshed
   handle gives BIT FOR BIT what a handle freshly created on the same W gives, at every entry point: select under every
   engine, exprace, top-k, no-repeat, the rejection sampler, the CE forward (exact and tf32), the CE table gradient
   (exact, tf32, candidate mode) and the logits.  Once before the tf32 CE's transposed image exists, twice after.
2. The f16 filter of a handle refreshed out of the f16 range (max|w| >= 1e4) stays exact; back in range, too.
3. The refresh is capturable (no sync, no allocation) and ordered on its stream.
4. Eager fine_tune: item_table() keeps ONE handle across Adam steps, equal to a fresh one, and a steady-state step
   neither synchronises the device nor allocates device memory through the runtime.
5. GraphedTrainStep(train_tables=True) on ListCVAE: the replayed loss equals the eager loss on the parameters the
   previous replay left, both tables move, and recommend() afterwards is the oracle's arg-max on the updated table.

Bitwise checks need no tolerance: both handles run the same kernels on the same bytes.  The one tolerance (5.) is
derived where it is used.
"""
import gc

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
from gpu_util import N

pytestmark = pytest.mark.gpu

DIMS = (4, 8, 16, 32, 64, 128)
TC_DIMS = (8, 16, 32, 64, 128)
U = 2.0 ** -24


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    return o


def _outputs(ops, tab, Q, tg, extra):
    """Every entry point that reads the handle -> {name: tensor}.  extra: fixed noise / candidate inputs."""
    D = tab.dim
    out = {}
    engines = ["auto", "simt"] + (["tcgen05"] if D in TC_DIMS else [])
    if D == 8:
        engines.append("tcgen05_f16")
    for e in engines:
        out["select_" + e], out["select_val_" + e] = ops.score_select(tab, Q, engine=e)
    out["exprace"], out["exprace_key"] = ops.score_select(tab, Q, "exprace", noise=extra["noise"])
    out["topk"], out["topk_val"] = ops.score_topk(tab, Q, 5)
    out["no_repeat"], out["no_repeat_val"] = ops.score_select(tab, Q, engine="auto", no_repeat=5)
    out["sampler"], out["sampler_iters"] = ops.sigmoid_categorical(tab, Q, seed=7, offset=11, want_iters=True)
    out["logits"] = ops.score_logits(tab, Q)
    rs = extra["row_scale"]
    for eng in ["exact"] + (["tf32"] if D in TC_DIMS else []):
        loss, lse, dq = ops.ce_fwd_bwd(tab, Q, tg, engine=eng)
        out["ce_loss_" + eng], out["ce_lse_" + eng], out["ce_dq_" + eng] = loss, lse, dq
        out["ce_dW_" + eng] = ops.ce_table_grad(tab, Q, tg, lse, rs, engine=eng)
    cand, tpos = extra["cand"], extra["tpos"]
    Qc = Q[: cand.shape[0]].contiguous()
    loss, lse, dq, p = ops.cand_ce_fwd_bwd(tab, Qc, cand, tpos, want_logits=True)
    out.update(cand_loss=loss, cand_lse=lse, cand_dq=dq, cand_p=p)
    # every item is a candidate of at most one (row, column): each dW row gets at most one atomic add, so the result
    # does not depend on the order of the float atomics
    out["cand_dW"] = ops.cand_ce_table_grad(tab, Qc, cand, tpos, lse, rs[: cand.shape[0]].contiguous())
    return out


def _assert_same(got, want, what):
    torch.cuda.synchronize()
    for k in want:
        a, b = got[k], want[k]
        assert a.shape == b.shape and torch.equal(a, b), "%s: %s differs from a fresh handle (%d elements)" % (
            what, k, int((a != b).sum()))


def _problem(D, seed, n=3001, M=640):
    g = torch.Generator(device="cuda").manual_seed(seed)
    W = F.normalize(torch.randn(n, D, device="cuda", generator=g), dim=1)
    Q = torch.randn(M, D, device="cuda", generator=g) * 2
    tg = torch.randint(0, n, (M,), device="cuda", generator=g)
    perm = torch.randperm(n, device="cuda", generator=g)
    n_cand = 40
    cand = perm[: 64 * n_cand].view(64, n_cand).contiguous()
    extra = {"noise": torch.empty(M, n, device="cuda").exponential_(generator=g),
             "row_scale": torch.randn(M, device="cuda", generator=g),
             "cand": cand, "tpos": torch.randint(0, n_cand, (64,), device="cuda", generator=g)}
    return W, Q, tg, extra, g


@pytest.mark.parametrize("D", DIMS)
def test_refresh_equals_create(ops, D):
    W, Q, tg, extra, g = _problem(D, 100 + D)
    tab = ops.Table(W)
    ops.score_select(tab, Q)        # the handle is in use before W changes
    m0 = float(W.norm(dim=1).max())
    # (a) random perturbation, refreshed while the transposed CE image does not exist yet (it stays lazy)
    W.add_(0.1 * torch.randn(W.shape, device="cuda", generator=g))
    tab.refresh()
    _assert_same(_outputs(ops, tab, Q, tg, extra), _outputs(ops, ops.Table(W), Q, tg, extra), "perturbed")
    # (b) max|w| grows: one row scaled by 1.5 (the transposed image exists now: the tf32 CE of (a) built it)
    j = int(W.norm(dim=1).argmax())
    W[j].mul_(1.5)
    tab.refresh()
    assert float(W.norm(dim=1).max()) > 1.4 * m0
    _assert_same(_outputs(ops, tab, Q, tg, extra), _outputs(ops, ops.Table(W), Q, tg, extra), "max|w| grown")
    # (c) max|w| shrinks
    W.mul_(0.25)
    tab.refresh()
    _assert_same(_outputs(ops, tab, Q, tg, extra), _outputs(ops, ops.Table(W), Q, tg, extra), "max|w| shrunk")


def test_refresh_out_of_f16_range(ops):
    """max|w| >= 1e4 after a refresh: the f16 filter (whose image the handle keeps) must stay exact."""
    W, Q, _, _, _ = _problem(8, 7, n=20000, M=2048)
    tab = ops.Table(W)
    ref = lambda: oracle.score_select(N(W), N(Q))[0]
    assert np.array_equal(N(ops.score_select(tab, Q, engine="tcgen05_f16")[0]), ref())
    for scale in (3.0e4, 1.0 / 3.0e4):
        W.mul_(scale)
        tab.refresh()
        want = ref()
        for e in ("tcgen05_f16", "auto", "tcgen05"):
            assert np.array_equal(N(ops.score_select(tab, Q, engine=e)[0]), want), (scale, e)


@pytest.mark.parametrize("D", (8, 32))
def test_refresh_captured(ops, D):
    """refresh() inside torch.cuda.graph: capture fails on any sync or allocation; replays follow W."""
    W, Q, tg, extra, g = _problem(D, 200 + D)
    tab = ops.Table(W)
    run = lambda: (ops.score_select(tab, Q, engine="tcgen05")[0], ops.sigmoid_categorical(tab, Q, seed=3),
                   ops.ce_fwd_bwd(tab, Q, tg, engine="tf32"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):       # warm-up: workspaces, the transposed image, kernel attributes
        run()
        tab.refresh()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        tab.refresh()
        sel, smp, (loss, lse, dq) = run()
    for k in range(2):
        W.copy_(F.normalize(torch.randn(W.shape, device="cuda", generator=g), dim=1) * (1.0 + k))
        graph.replay()
        fresh = ops.Table(W)
        want_sel = ops.score_select(fresh, Q, engine="tcgen05")[0]
        want_smp = ops.sigmoid_categorical(fresh, Q, seed=3)
        wl, wlse, wdq = ops.ce_fwd_bwd(fresh, Q, tg, engine="tf32")
        torch.cuda.synchronize()
        assert torch.equal(sel, want_sel) and torch.equal(smp, want_smp)
        assert torch.equal(loss, wl) and torch.equal(lse, wlse) and torch.equal(dq, wdq)


def test_refresh_stream_order(ops):
    """Update, refresh and score on one side stream with no host sync in between."""
    W, Q, _, _, g = _problem(8, 300, n=50000, M=1024)
    tab = ops.Table(W)
    new = F.normalize(torch.randn(W.shape, device="cuda", generator=g), dim=1) * 3.0
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        W.copy_(new)
        tab.refresh()
        got = {e: ops.score_select(tab, Q, engine=e)[0] for e in ("tcgen05_f16", "tcgen05")}
        smp = ops.sigmoid_categorical(tab, Q, seed=5)
    torch.cuda.synchronize()
    want = oracle.score_select(N(new), N(Q))[0]
    for e, v in got.items():
        assert np.array_equal(N(v), want), e
    assert np.array_equal(N(smp), oracle.sigmoid_categorical(N(new), N(Q), 5)[0])


class _Emb:
    def __init__(self, w):
        self.weight = w


def _list_model(D, n_items, n_users, seed, engine):
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    L, Z, H, PH = 5, 16, 64, 32
    g = torch.Generator(device="cuda").manual_seed(seed)
    doc = _Emb(torch.randn(n_items, D, device="cuda", generator=g))
    usr = _Emb(torch.randn(n_users, D, device="cuda", generator=g))
    torch.manual_seed(seed)
    m = UserListCVAEWithPrior(doc, usr, L, D, Z, L + 1, [L * D + L + 1 + D, H, H], [Z + L + 1 + D, H, H, L * D],
                              [L + 1 + D, PH, PH], False, "cuda:0", fine_tune=True)
    m.ce_engine = engine
    return m


def _batch(seed, n_items, n_users, B, L=5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return {"slates": torch.randint(0, n_items, (B, L), device="cuda", generator=g),
            "users": torch.randint(0, n_users, (B, 1), device="cuda", generator=g),
            "responses": (torch.rand(B, L, device="cuda", generator=g) < 0.3).float()}


def test_eager_fine_tune_keeps_one_handle(ops):
    from torch.profiler import ProfilerActivity, profile

    from pivotcvae_b200.train_generative import get_gen_loss
    n_items, n_users, B = 3001, 40, 64
    m = _list_model(8, n_items, n_users, 5, "tf32")
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2)
    batch = _batch(6, n_items, n_users, B)

    def step():
        opt.zero_grad()
        loss, _, _ = get_gen_loss(batch, m, None, 0.01, n_neg=n_items)
        loss.backward()
        opt.step()
        return m.item_table()

    t0 = m.item_table()
    g = torch.Generator(device="cuda").manual_seed(9)
    Q = torch.randn(512, 8, device="cuda", generator=g)
    tg = torch.randint(0, n_items, (512,), device="cuda", generator=g)
    for _ in range(3):
        assert step() is t0
        fresh = ops.Table(m.docEmbed.weight.detach())
        for e in ("tcgen05_f16", "tcgen05"):
            assert torch.equal(ops.score_select(t0, Q, engine=e)[0], ops.score_select(fresh, Q, engine=e)[0])
        assert torch.equal(ops.sigmoid_categorical(t0, Q, seed=1), ops.sigmoid_categorical(fresh, Q, seed=1))
        for a, b in zip(ops.ce_fwd_bwd(t0, Q, tg, engine="tf32"), ops.ce_fwd_bwd(fresh, Q, tg, engine="tf32")):
            assert torch.equal(a, b)
    del fresh
    gc.collect()
    torch.cuda.synchronize()
    # the profiler synchronises the device itself when it stops: only the runtime calls made inside the step's own
    # window count (a stream sync closes that window, so the step's kernels are in the trace)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        with torch.profiler.record_function("fine_tune_step"):
            step()
            torch.cuda.current_stream().synchronize()
    events = prof.events()
    names = [e.name for e in events]
    assert any("table_refresh_kernel" in n for n in names), "the step did not refresh"
    win = next(e for e in events if e.name == "fine_tune_step")
    inside = [e.name for e in events if win.time_range.start <= e.time_range.start <= win.time_range.end]
    assert any(n.startswith("cudaLaunchKernel") for n in inside), "the step window holds no runtime calls"
    for bad in ("cudaDeviceSynchronize", "cudaMalloc", "cudaFree"):
        hits = [n for n in inside if n == bad]
        assert not hits, "%s inside a steady-state fine_tune step (%d calls)" % (bad, len(hits))


@pytest.mark.parametrize("engine", ("exact", "tf32"))
@pytest.mark.parametrize("D", (8, 32))
def test_graphed_fine_tune(ops, D, engine):
    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.train_generative import get_gen_loss
    n_items, n_users, B, L = 3001, 40, 64, 5
    m = _list_model(D, n_items, n_users, 10 + D, engine)
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2, capturable=True)
    step = GraphedTrainStep(m, opt, B, 0.01, n_items, train_tables=True)
    d0, u0 = m.docEmbed.weight.detach().clone(), m.userEmbed.weight.detach().clone()
    batch = _batch(11, n_items, n_users, B)
    step(batch)
    for _ in range(3):
        counter = m.noise.device_counter.clone()
        kept, m._table = m._table, None                 # the eager reference scores against a FRESH handle
        with torch.no_grad():
            eager, _, _ = get_gen_loss(batch, m, None, 0.01, n_neg=n_items)
        eager = float(eager)
        m._table = kept
        m.noise.device_counter.copy_(counter)      # the replay draws the Philox rows the eager call drew
        loss = float(step(batch)[0])
        # Both sides run the same kernels on the same parameters and Philox rows; only sums whose order may differ
        # between them (float atomics, torch's reductions) can move the result.  The loss is a sum of non-negative
        # terms (CE rows, KL), so reordering its at most M = B * L = 320 fp32 additions moves it by at most
        # 2 * 320 * u of its value (Higham's bound for recursive summation): 4e-5 relative.  A replay that read a
        # stale handle scores against the table before the last Adam step (lr 1e-2 on every touched entry).
        assert abs(loss - eager) <= 2 * 320 * U * abs(eager), (loss, eager)
    rows = batch["slates"].unique()
    assert not torch.equal(m.docEmbed.weight[rows], d0[rows])
    assert not torch.equal(m.userEmbed.weight, u0)
    # recommend() on the handle the last replay refreshed (item_table() must not refresh it again)
    l0 = ops.launch_count()
    tab = m.item_table()
    assert tab is step._table and ops.launch_count() == l0
    g = torch.Generator(device="cuda").manual_seed(12)
    ctx = torch.zeros(B, L, device="cuda")
    ctx[:, :2] = 1
    users = torch.randint(0, n_users, (B,), device="cuda", generator=g)
    eps = torch.randn(B, m.latent_size, device="cuda", generator=g)
    m.noise.push("eps", eps)
    with torch.no_grad():
        items, _ = m.recommend(ctx, users, return_item=True)
        m.noise.push("eps", eps)
        rx, _ = m.recommend(ctx, users, return_item=False)
    want, _ = oracle.score_select(N(m.docEmbed.weight), N(rx).reshape(-1, D))
    assert np.array_equal(N(items), want)


@pytest.mark.parametrize("D", TC_DIMS)
def test_tf32_ce_reproducible(ops, D):
    """The tf32 CE forward adds the column slices' partial sums in a fixed order: two calls on one handle (and calls on
    two handles of the same table) agree bit for bit, which the refresh checks above rely on."""
    W, Q, tg, _, _ = _problem(D, 400 + D, n=20000, M=2048)
    t1, t2 = ops.Table(W), ops.Table(W)
    ref = ops.ce_fwd_bwd(t1, Q, tg, engine="tf32")
    for tab in (t1, t2, t1):
        for a, b in zip(ops.ce_fwd_bwd(tab, Q, tg, engine="tf32"), ref):
            assert torch.equal(a, b)
