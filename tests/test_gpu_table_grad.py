"""-m gpu: the embedding tables under fine_tune=True.

1. pcv_ce_table_grad (every mask path) and pcv_cand_ce_table_grad against float64 autograd of the materialised loss;
2. UserListCVAEWithPrior(fine_tune=True): get_gen_loss + backward in every training mode against the golden fixtures
   (MLP gradients) and a float64 restatement of the reference's ListCVAE loss with the tables as leaves (table
   gradients);
3. a few Adam steps, then recommend() against the CPU oracle on the updated table; the guards.

Error model shared by the bounds below (u = 2^-24).  One term of dW[j] is g_i (p_ij - [t_i = j]) q_i: the kernel's
logit x_ij is a D-long fp32 FMA chain (error <= D u |q_i| |w_j|, <= 1e-5 absolute for the unit-norm tables and |q| <= 6
used here), __expf adds ~2 ulp, and the forward's lse is fp32 (a few ulp of |lse| <= 15): p_ij is right to a relative
2e-5 at worst.  The fp32 sum over the M rows adds at most M u relative to S_jk = sum_i |g_i| m_ij (p_ij + [t_i = j])
|q_ik|, the sum of the terms' magnitudes.  So |dW - dW64| <= (2e-5 + M u) S elementwise; every check below uses it with
a 2x margin (the float64 reference is exact to ~1e-15 relative by comparison).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
from gpu_util import N, T, load_sd

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    return o


def _check(name, got, want, bound):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)
    assert not bool(bad.any()), "%s: %d elements over the bound, worst err %g (bound there %g)" % (
        name, int(bad.sum()), float(err[bad].max()), float(bound.expand_as(err)[bad][err[bad].argmax()]))


def _unpack(bits, n):
    """(M, ceil(N/32)) uint32 -> (M, N) bool: bit j % 32 of word j // 32."""
    b = np.unpackbits(np.ascontiguousarray(bits).view(np.uint8), axis=1, bitorder="little")
    return torch.from_numpy(b[:, :n].astype(bool)).cuda()


def _problem(n_items, M, D, seed, rep_targets=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    W = F.normalize(torch.randn(n_items, D, device="cuda", generator=g), dim=1)
    Q = torch.randn(M, D, device="cuda", generator=g) * 2
    tg = torch.randint(0, n_items, (M,), device="cuda", generator=g)
    if rep_targets:
        tg[: M // 2] = tg[0]                       # one item is the target of half the rows
    rs = torch.randn(M, device="cuda", generator=g)
    rs[::5] = 0.0                                  # zero and negative row scales
    return W, Q, tg, rs


def _ref(W, Q, tg, rs, keep=None):
    """float64 autograd of sum_i rs_i CE_i over the materialised masked logits (masked-out logits are 0) -> (dW, S)
    with S the magnitude sum of the error model (module docstring)."""
    M, n = Q.shape[0], W.shape[0]
    W64 = W.double().requires_grad_()
    Q64 = Q.double()
    m = torch.ones(M, n, dtype=torch.bool, device=W.device) if keep is None else keep.clone()
    m[torch.arange(M), tg] = True                  # the target is always kept
    X = (Q64 @ W64.t()) * m
    loss = torch.logsumexp(X, 1) - X[torch.arange(M), tg]
    (loss * rs.double()).sum().backward()
    with torch.no_grad():
        p = torch.exp(X - torch.logsumexp(X, 1, keepdim=True)) * m
        p[torch.arange(M), tg] += 1.0
        S = (p * rs.double().abs()[:, None]).t() @ Q64.abs()
    return W64.grad, S


def _bound(S, M):
    return 2 * (2e-5 + M * U) * S + 1e-30


@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
@pytest.mark.parametrize("n_items,M", [(1, 5), (127, 33), (1025, 70), (100003, 45)])
def test_table_grad_dense_exact(ops, D, n_items, M):
    W, Q, tg, rs = _problem(n_items, M, D, 1000 * D + n_items + M, rep_targets=(n_items > 1))
    tab = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, 1.0, want_dq=False)
    dW = ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0)
    want, S = _ref(W, Q, tg, rs)
    _check("dense D=%d" % D, dW, want, _bound(S, M))
    assert torch.equal(dW, ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0))     # reproducible bit for bit


@pytest.mark.parametrize("D", [8, 32, 128])
def test_table_grad_dense_row_split(ops, D):
    """A small catalog over many rows: the rows are cut into splits and the fixed-order reduce adds them."""
    W, Q, tg, rs = _problem(300, 4000, D, 7 + D)
    tab = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, 1.0, want_dq=False)
    dW = ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0)
    want, S = _ref(W, Q, tg, rs)
    _check("split D=%d" % D, dW, want, _bound(S, 4000))
    assert torch.equal(dW, ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0))


@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
@pytest.mark.parametrize("n_items,M", [(127, 33), (5000, 61)])
def test_table_grad_bitmask(ops, D, n_items, M):
    W, Q, tg, rs = _problem(n_items, M, D, 3 * D + n_items, rep_targets=True)
    rng = np.random.default_rng(D + n_items)
    keep = rng.random((M, n_items)) < 0.1
    keep[:3] = False                               # rows where only the target is kept
    bits = oracle.pack_bitmask(keep)
    bm = T(bits.view(np.int32))
    tab = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, 0.1, bitmask=bm, want_dq=False)
    dW = ops.ce_table_grad(tab, Q, tg, lse, rs, 0.1, bitmask=bm)
    want, S = _ref(W, Q, tg, rs, torch.from_numpy(keep).cuda())
    _check("bitmask D=%d" % D, dW, want, _bound(S, M))
    assert torch.equal(dW, ops.ce_table_grad(tab, Q, tg, lse, rs, 0.1, bitmask=bm))


@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
@pytest.mark.parametrize("n_items,M,keep", [(3000, 50, 0.07), (40000, 64, 0.025), (1025, 37, 0.5)])
def test_table_grad_philox(ops, D, n_items, M, keep):
    """The backward regenerates the forward's gap-process mask; oracle.bernoulli_bitmask restates it bit for bit
    (test_gpu_kernels.py pins it against the forward).  Float atomics: the bound of the module docstring holds for any
    summation order."""
    W, Q, tg, rs = _problem(n_items, M, D, 11 * D + n_items, rep_targets=True)
    tab = ops.Table(W)
    seed, off = 42 + D, 9
    _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, keep, seed=seed, offset=off, want_dq=False)
    dW = ops.ce_table_grad(tab, Q, tg, lse, rs, keep, seed=seed, offset=off)
    bits = oracle.bernoulli_bitmask(seed, off, M, n_items, keep)
    want, S = _ref(W, Q, tg, rs, _unpack(bits, n_items))
    _check("philox D=%d" % D, dW, want, _bound(S, M))
    # the device-side offset counter of CUDA-graph replays is added to `offset`, as in the forward
    cnt = torch.full((1,), 5, dtype=torch.int64, device="cuda")
    _, lse2, _ = ops.ce_fwd_bwd(tab, Q, tg, keep, seed=seed, offset=off - 5, offset_dev=cnt, want_dq=False)
    dW2 = ops.ce_table_grad(tab, Q, tg, lse2, rs, keep, seed=seed, offset=off - 5, offset_dev=cnt)
    _check("philox offset_dev D=%d" % D, dW2, want, _bound(S, M))


@pytest.mark.parametrize("D", [8, 16, 32, 64, 128])
@pytest.mark.parametrize("n_items,M", [(1025, 130), (20000, 96)])
def test_table_grad_tf32_engine(ops, D, n_items, M):
    """engine tf32: the tensor-core sweep (tcgen05, dW resident in TMEM).  Per term g_i (p_ij - [t_i = j]) q_ik:
      - the tf32 logit is within 2^-9 |q_i| |w_j| = 2^-9 |q_i| of the exact one (both operands truncated to 10 mantissa
        bits, 2^-10 relative each), so p_ij is off by a relative expm1(2^-9 |q_i|) at most;
      - lse_i is the tf32 forward's: p_ij is off by a further relative |lse_tf32 - lse64|_i (measured per row);
      - the gradient MMA truncates P^T and Q to tf32 again: 2^-9 relative per term;
      - the fp32 accumulation in tensor memory over M rows: 2 M u relative to the magnitude sum (truncating adds).
    Summed with the magnitudes (p_ij + [t_i = j]) |g_i| |q_ik| of the terms, with a 2x margin."""
    W, Q, tg, rs = _problem(n_items, M, D, 5 * D + n_items, rep_targets=True)
    tab = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, 1.0, want_dq=False, engine="tf32")
    dW = ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0, engine="tf32")
    want, _ = _ref(W, Q, tg, rs)
    with torch.no_grad():
        X = Q.double() @ W.double().t()
        lse64 = torch.logsumexp(X, 1)
        p = torch.exp(X - lse64[:, None])
        p[torch.arange(M), tg] += 1.0
        rel = (torch.expm1(2.0 ** -9 * Q.double().norm(dim=1)) + (lse.double() - lse64).abs() + 2.0 ** -9 + 2e-5 + 2 * M * U)
        S = (p * (rs.double().abs() * rel)[:, None]).t() @ Q.double().abs()
    _check("tf32 D=%d" % D, dW, want, 2 * S + 1e-30)
    assert torch.equal(dW, ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0, engine="tf32"))     # reproducible bit for bit
    # and it is the tensor-core result, not the exact pass: the two differ beyond the exact pass's own bound somewhere
    exact = ops.ce_table_grad(tab, Q, tg, lse, rs, 1.0)
    assert not torch.equal(dW, exact)


def test_table_grad_argument_errors(ops):
    import ctypes

    from pivotcvae_b200 import _lib as L
    lib = L.load()
    W, Q, tg, rs = _problem(500, 16, 8, 3)
    tab = ops.Table(W)
    _, lse, _ = ops.ce_fwd_bwd(tab, Q, tg, 1.0, want_dq=False)
    dW = torch.empty_like(W)
    mask = L.CeMask(1.0)
    ws = tab.workspace("ce_tgrad", 16)
    p = ops._ptr
    args = [tab.handle, p(Q), p(tg), 16, ctypes.byref(mask), p(lse), p(rs), p(dW), p(ws), ws.numel(), None]
    assert lib.pcv_ce_table_grad(*args) == 0
    for k in (0, 1, 2, 5, 6, 7):                                     # NULL pointers
        a = list(args)
        a[k] = None
        assert lib.pcv_ce_table_grad(*a) == -1, k
    need = ctypes.c_size_t()
    assert lib.pcv_ce_table_grad_workspace_bytes(tab.handle, 16, ctypes.byref(mask), ctypes.byref(need)) == 0
    a = list(args)
    a[9] = 0                                                          # too small a workspace
    assert lib.pcv_ce_table_grad(*a) == -4
    assert b"workspace" in lib.pcv_last_error()
    with pytest.raises(L.PcvError, match="row_offset"):               # a vocab-parallel shard
        shard = ops.Table(W[128:], row_offset=128)
        ops.ce_table_grad(shard, Q, tg - 128, lse, rs, 1.0)
    W4, Q4, tg4, rs4 = _problem(500, 16, 4, 4)
    tab4 = ops.Table(W4)
    with pytest.raises(L.PcvError, match="tf32"):                    # no tf32 engine at D = 4
        ops.ce_table_grad(tab4, Q4, tg4, torch.zeros(16, device="cuda"), rs4, 1.0, engine="tf32")
    for fn in (lambda: lib.pcv_cand_ce_table_grad(None, p(Q), p(tg), p(tg), 16, 4, p(lse), p(rs), p(dW), None),
               lambda: lib.pcv_cand_ce_table_grad(tab.handle, p(Q), p(tg), p(tg), 16, 0, p(lse), p(rs), p(dW), None)):
        assert fn() == -1


@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
def test_cand_table_grad(ops, D):
    """Against the float64 gather-bmm-CE autograd (train_generative.py:52-56), duplicate candidates included."""
    n_items, M, nC = 3000, 70, 100
    W, Q, _, rs = _problem(n_items, M, D, 17 * D)
    g = torch.Generator(device="cuda").manual_seed(D)
    cand = torch.randint(0, n_items, (M, nC), device="cuda", generator=g)
    cand[:, 1] = cand[:, 0]                                     # duplicates within a row
    cand[:, 2] = cand[:, 0]
    tpos = torch.randint(0, nC, (M,), device="cuda", generator=g)
    tpos[:5] = 1                                                # the target is one of the duplicated columns
    tab = ops.Table(W)
    _, lse, _, _ = ops.cand_ce_fwd_bwd(tab, Q, cand, tpos, want_dq=False)
    dW = ops.cand_ce_table_grad(tab, Q, cand, tpos, lse, rs)
    W64 = W.double().requires_grad_()
    X = torch.bmm(W64[cand], Q.double()[:, :, None]).squeeze(2)
    (F.cross_entropy(X, tpos, reduction="none") * rs.double()).sum().backward()
    with torch.no_grad():
        P = torch.softmax(X, 1)
        P[torch.arange(M), tpos] += 1.0
        S = torch.zeros_like(W64).index_add_(0, cand.reshape(-1),
                                             ((P * rs.double().abs()[:, None])[:, :, None] * Q.double().abs()[:, None, :])
                                             .reshape(-1, D))
    # per element the same error model as the catalog CE, with nC in place of M (the terms of one row land on its
    # candidates' rows; atomics add them in any order)
    _check("cand D=%d" % D, dW, W64.grad, 2 * (2e-5 + (M * nC) * U) * S + 1e-30)


# ============================================================ model level
class _Emb:
    def __init__(self, w):
        self.weight = torch.from_numpy(np.ascontiguousarray(w))


def _build_list(fx, fine_tune=True):
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    cfg, sd = fx.cfg, fx.sub("sd/")
    L, D, Z, H, PH = cfg["L"], cfg["D"], cfg["Z"], cfg["hidden"], cfg["phidden"]
    ud = 0 if cfg["no_user"] else D
    m = UserListCVAEWithPrior(_Emb(sd["docEmbed.weight"]), None if cfg["no_user"] else _Emb(sd["userEmbed.weight"]),
                              L, D, Z, L + 1, [L * D + L + 1 + ud, H, H], [Z + L + 1 + ud, H, H, L * D],
                              [L + 1 + ud, PH, PH], bool(cfg["no_user"]), "cuda:0", fine_tune=fine_tune)
    return load_sd(m, sd)


def _ref_list_loss(m, slates, users, resp, eps, beta, keep=None, cand=None, tpos=None):
    """float64 restatement of the reference's ListCVAE training loss (listcvae.py:90-168, train_generative.py:44-65)
    with every parameter AND both tables as leaves -> (loss, {name: grad})."""
    P = {k: v.detach().double().requires_grad_() for k, v in m.named_parameters()}
    P["docEmbed.weight"] = m.docEmbed.weight.detach().double().requires_grad_()
    if not m.noUser:
        P["userEmbed.weight"] = m.userEmbed.weight.detach().double().requires_grad_()
    B, Ls = slates.shape
    D = m.feature_size
    lin = lambda name, x: x @ P[name + ".weight"].t() + P[name + ".bias"]
    act = lambda x: F.leaky_relu(x, 0.01)
    cond = F.one_hot(resp.sum(1).long(), Ls + 1).double()
    user = [] if m.noUser else [P["userEmbed.weight"][users.reshape(-1)]]
    h = torch.cat([P["docEmbed.weight"][slates].reshape(B, Ls * D), cond] + user, 1)
    for i in range(len(m.encMLP)):
        h = act(lin("enc_%d" % (i + 1), h))
    mu, lv = lin("encmu", h), lin("enclogvar", h)
    z = eps.double() * torch.exp(0.5 * lv) + mu
    h = torch.cat([z, cond] + user, 1)
    n = len(m.decMLP)
    for i in range(n):
        h = lin("dec_%d" % (i + 1), h)
        h = act(h) if i < n - 1 else h
    rx = h.reshape(B * Ls, D)
    h = torch.cat([cond] + user, 1)
    for i in range(len(m.priorMLP)):
        h = act(lin("prior_%d" % (i + 1), h))
    pmu, plv = lin("priorMu", h), lin("priorLogvar", h)
    t = slates.reshape(-1)
    if cand is not None:
        X = torch.bmm(P["docEmbed.weight"][cand], rx[:, :, None]).squeeze(2)
        rec = F.cross_entropy(X, tpos)
    else:
        X = rx @ P["docEmbed.weight"].t()
        if keep is not None:
            mk = keep.clone()
            mk[torch.arange(B * Ls), t] = True
            X = X * mk
        rec = F.cross_entropy(X, t)
    kld = -0.5 * torch.sum(1 + lv - plv - (torch.exp(lv) + (mu - pmu) ** 2) / torch.exp(plv))
    loss = rec + beta * kld
    loss.backward()
    return loss.detach(), {k: v.grad for k, v in P.items()}


# MLP gradients and the loss: the tolerances of test_gpu_models.py test_list_gen_loss_and_grads (fp32 kernels vs the
# reference's fp32 torch run).  Table gradients against float64: the docEmbed gradient sums the CE's table term (error
# model of the module docstring, <= 2e-5 + M u ~ 3e-5 relative of its magnitude at M = 240 rows) and the encoder's
# gather term (one 3xTF32 input-gradient GEMM chain per row, ~2e-5 relative, test_gpu_backward.py); the userEmbed
# gradient is three gather terms.  rtol 2e-3 with an absolute floor of 1e-4 of the gradient's largest entry covers
# both with margin and still catches a dropped term (each term is O(1) of the gradient).
def _check_tables(m, ref, rtol=2e-3, floor=1e-4):
    names = ["docEmbed.weight"] + ([] if m.noUser else ["userEmbed.weight"])
    for k in names:
        got = dict(m.named_parameters())[k].grad
        assert got is not None, k
        w = ref[k]
        _check(k, got, w, rtol * w.abs() + floor * w.abs().max())


def _batch(fx):
    return {"slates": fx["in/slates"], "users": fx["in/users"].reshape(-1, 1), "responses": fx["in/resp"]}


@pytest.mark.parametrize("name", ["list_small", "list_small_user"])
@pytest.mark.parametrize("ntag", ["mask", "full"])
def test_fine_tune_gen_loss_fixture_modes(golden, name, ntag):
    """The fixtures' own modes (injected eps and bitmask): loss and MLP gradients as the frozen model's, tables vs
    float64."""
    from pivotcvae_b200.train_generative import get_gen_loss
    fx = golden(name)
    m = _build_list(fx)
    t2 = "loss_%s/" % ntag
    m.noise.push("eps", T(fx[t2 + "eps"]))
    bits = fx[t2 + "bitmask"]
    n_neg = int(fx[t2 + "n_neg"])
    m.noise.push("mask", T(bits.view(np.int32)))
    loss, rec, kld = get_gen_loss(_batch(fx), m, None, 0.01, n_neg=n_neg)
    np.testing.assert_allclose([loss.item(), rec.item(), kld.item()], fx[t2 + "loss"], rtol=1e-4)
    loss.backward()
    for pname, prm in m.named_parameters():
        g = fx.sub(t2 + "grad/").get(pname)
        if g is not None:
            np.testing.assert_allclose(N(prm.grad), g, rtol=2e-3, atol=2e-6, err_msg=pname)
    keep = _unpack(bits, m.docEmbed.weight.shape[0])
    want, ref = _ref_list_loss(m, T(fx["in/slates"]), T(fx["in/users"]), T(fx["in/resp"]), T(fx[t2 + "eps"]), 0.01,
                               keep=keep)
    assert abs(loss.item() - want.item()) <= 1e-4 * abs(want.item())
    _check_tables(m, ref)


@pytest.mark.parametrize("name", ["list_small", "list_small_user"])
@pytest.mark.parametrize("mode", ["exact", "tf32", "philox", "candidate"])
def test_fine_tune_gen_loss_modes(golden, name, mode):
    """Full catalog on both engines, the Philox mask and candidate mode, all against the float64 restatement."""
    from pivotcvae_b200.train_generative import get_gen_loss
    fx = golden(name)
    m = _build_list(fx)
    eps = T(fx["loss_full/eps"])
    m.noise.push("eps", eps)
    n_items = m.docEmbed.weight.shape[0]
    batch = _batch(fx)
    M = fx["in/slates"].size
    keep = cand = tpos = None
    n_neg = n_items
    if mode == "tf32":
        m.ce_engine = "tf32"
    elif mode == "philox":
        n_neg = 150
        m.noise.reseed(1234)                    # eps is injected: the mask is the only Philox draw (offset 0)
        keep = _unpack(oracle.bernoulli_bitmask(1234, 0, M, n_items, n_neg / n_items), n_items)
    elif mode == "candidate":
        g = torch.Generator(device="cuda").manual_seed(5)
        cand = torch.randint(0, n_items, (M, 40), device="cuda", generator=g)
        tpos = torch.randint(0, 40, (M,), device="cuda", generator=g)
        cand[:, 1] = cand[:, 0]                                    # duplicate candidates
        cand[torch.arange(M), tpos] = T(fx["in/slates"]).reshape(-1)
        m.candidateFlag = True
        batch = dict(batch, sample_candidates=cand, sample_targets=tpos)
    loss, rec, kld = get_gen_loss(batch, m, None, 0.01, n_neg=n_neg)
    loss.backward()
    want, ref = _ref_list_loss(m, T(fx["in/slates"]), T(fx["in/users"]), T(fx["in/resp"]), eps, 0.01, keep=keep,
                               cand=cand, tpos=tpos)
    # tf32: logits and dq on the tensor cores, loss ~1e-4 / dq ~1e-3 relative (include/pcv_b200.h); the table gradient
    # inherits the forward's lse error and the MLP gradients the dq error, so that mode gets 10x the bounds
    loose = 10.0 if mode == "tf32" else 1.0
    assert abs(loss.item() - want.item()) <= 1e-4 * loose * abs(want.item())
    for pname, prm in m.named_parameters():
        if pname in ref and pname not in ("docEmbed.weight", "userEmbed.weight"):
            w = ref[pname]
            _check(pname, prm.grad, w, 2e-3 * loose * w.abs() + 1e-4 * loose * w.abs().max())
    _check_tables(m, ref, 2e-3 * loose, 1e-4 * loose)


@pytest.mark.parametrize("name", ["list_small", "list_small_user"])
@pytest.mark.parametrize("cand_mode", [False, True])
def test_fine_tune_forward_p_path(golden, name, cand_mode):
    """forward()'s materialised `p` (LogitsFn / CandidateLogitsFn): the same table gradient through torch's CE."""
    fx = golden(name)
    m = _build_list(fx)
    s, r = T(fx["in/slates"]), T(fx["in/resp"])
    u = None if m.noUser else T(fx["in/users"])
    eps = T(fx["loss_full/eps"])
    m.noise.push("eps", eps)
    M, n_items = s.numel(), m.docEmbed.weight.shape[0]
    cand = tpos = None
    if cand_mode:
        g = torch.Generator(device="cuda").manual_seed(9)
        cand = torch.randint(0, n_items, (M, 30), device="cuda", generator=g)
        tpos = torch.randint(0, 30, (M,), device="cuda", generator=g)
        cand[:, 2] = cand[:, 3]
        m.candidateFlag = True
    p, rx, z, emb, mu, lv = m.forward(s, r, cand.reshape(s.shape[0], s.shape[1], -1) if cand_mode else None, u)
    pmu, plv = m.get_prior(r, u)
    rec = F.cross_entropy(p, tpos if cand_mode else s.reshape(-1))
    kld = -0.5 * torch.sum(1 + lv - plv - (torch.exp(lv) + (mu - pmu) ** 2) / torch.exp(plv))
    (rec + 0.01 * kld).backward()
    _, ref = _ref_list_loss(m, s, T(fx["in/users"]), r, eps, 0.01, cand=cand, tpos=tpos)
    _check_tables(m, ref)


@pytest.mark.parametrize("name", ["list_small", "list_small_user"])
def test_fine_tune_philox_with_device_counter(golden, name):
    """With a device-side Philox counter installed (as after building a CUDA-graph generator on the model),
    get_gen_loss advances it (flush_eager) between the CE forward and loss.backward(); the table gradient must still
    use the mask the forward drew, at the counter value the forward read."""
    from pivotcvae_b200.train_generative import get_gen_loss
    fx = golden(name)
    m = _build_list(fx)
    eps = T(fx["loss_full/eps"])
    n_items = m.docEmbed.weight.shape[0]
    M = fx["in/slates"].size
    m.noise.reseed(1234)
    m.noise.counter = 7
    m.noise.begin_graph(torch.device("cuda:0"))         # device counter = 7, host-side offsets restart at 0
    m.noise.push("eps", eps)
    loss, _, _ = get_gen_loss(_batch(fx), m, None, 0.01, n_neg=150)
    assert int(m.noise.device_counter.item()) == 7 + M   # advanced before the backward below
    loss.backward()
    keep = _unpack(oracle.bernoulli_bitmask(1234, 7, M, n_items, 150 / n_items), n_items)
    _, ref = _ref_list_loss(m, T(fx["in/slates"]), T(fx["in/users"]), T(fx["in/resp"]), eps, 0.01, keep=keep)
    _check_tables(m, ref)


def test_fine_tune_adam_then_recommend(golden):
    """Adam steps change both tables; recommend() then scores against the UPDATED table (the handle is re-created
    when the weight's version changes): slates bitwise equal to the CPU oracle's arg-max on the new table."""
    from pivotcvae_b200.train_generative import get_gen_loss
    fx = golden("list_small_user")
    m = _build_list(fx)
    d0, u0 = m.docEmbed.weight.detach().clone(), m.userEmbed.weight.detach().clone()
    opt = torch.optim.Adam(m.parameters(), lr=1e-2)
    m.noise.reseed(77)
    for _ in range(3):
        opt.zero_grad()
        loss, _, _ = get_gen_loss(_batch(fx), m, None, 0.01, n_neg=200)
        loss.backward()
        opt.step()
    rows = T(fx["in/slates"]).unique()
    assert not torch.equal(m.docEmbed.weight[rows], d0[rows])
    assert not torch.equal(m.userEmbed.weight, u0)
    ctx, users = T(fx["rec_k1/ctx"]), T(fx["in/users"])
    eps = T(fx["rec_k1/eps"])
    m.noise.push("eps", eps)
    items, _ = m.recommend(ctx, users, return_item=True)
    m.noise.push("eps", eps)
    rx, _ = m.recommend(ctx, users, return_item=False)
    W = N(m.docEmbed.weight)
    want, _ = oracle.score_select(W, N(rx).reshape(-1, m.feature_size))
    assert np.array_equal(N(items), want)


def test_fine_tune_guards(golden):
    """CUDA-graph capture and vocab-parallel refuse trainable tables; the PivotCVAE family keeps them frozen."""
    from pivotcvae_b200 import _lib as L
    from pivotcvae_b200.graphs import GraphedTrainStep
    from pivotcvae_b200.models.pivotcvae import PIVOTCVAE_MODELS
    from pivotcvae_b200.train_generative import get_gen_loss
    fx = golden("list_small_user")
    m = _build_list(fx)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
    with pytest.raises(L.PcvError, match="fine_tune"):
        GraphedTrainStep(m, opt, 4, 0.01, 100)
    with pytest.raises(L.PcvError, match="fine_tune"):
        m.enable_vocab_parallel()
    m.docEmbed.weight.requires_grad_(False)
    m.userEmbed.weight.requires_grad_(False)
    assert m.trainable_tables() == []
    # PivotCVAE family: the flag is accepted and ignored (the reference's subclasses pass False, SURVEY F8)
    fp = golden("pivot_small")
    cfg, sd = fp.cfg, fp.sub("sd/")
    pm = PIVOTCVAE_MODELS["pivotcvae_gt_pi"](_Emb(sd["docEmbed.weight"]), _Emb(sd["userEmbed.weight"]), cfg["L"], cfg["D"],
                                             cfg["Z"], cfg["L"] + 1, list(fp["cfg/enc"]), list(fp["cfg/psm"]),
                                             list(fp["cfg/scm"]), list(fp["cfg/prior"]), bool(cfg["no_user"]), "cuda:0",
                                             fine_tune=True)
    load_sd(pm, sd)
    assert not pm.docEmbed.weight.requires_grad and not pm.userEmbed.weight.requires_grad
    t2 = "loss_gt_full/"
    pm.noise.push("eps", T(fp[t2 + "eps"]))
    pm.noise.push("mask", T(fp[t2 + "bitmask"].view(np.int32)))
    batch = {"slates": fp["in/slates"], "users": fp["in/users"].reshape(-1, 1), "responses": fp["in/resp"]}
    loss, _, _ = get_gen_loss(batch, pm, None, 0.01, n_neg=int(fp[t2 + "n_neg"]))
    loss.backward()
    assert pm.docEmbed.weight.grad is None and pm.userEmbed.weight.grad is None
