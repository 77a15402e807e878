"""-m gpu: the backward half of every training step against float64 references.

Covers the tcgen05 GEMM epilogues, split-K slices, the deterministic weight-gradient reduce and the batched transpose
(csrc/gemm_tc.cu), FusedMLPFn.backward over the block kinds the models build (autograd.py), the pre-training kernels
(csrc/pretrain.cu), the KL kernel at training sizes, 1024-wide response MLPs, and full PivotCVAE / ListCVAE gradients
at the C3 training batch.

Where a result is exact (copies, residuals, activation-derivative masks, a fixed-order float32 sum) it is compared
bitwise.  Every other bound is derived in a comment next to it; u = 2^-24 is the float32 unit roundoff.  The worst
error / bound ratio of each tolerance check is printed at the end of the module (run with -s to see it).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
ACT_NONE, ACT_LEAKY, ACT_RELU = 0, 1, 2
SLOPE = {ACT_LEAKY: 0.01, ACT_RELU: 0.0}
SENT = 7.0                      # sentinel: what a kernel must leave alone still reads 7.0 afterwards

_WORST = {}


def _check(name, err, bound):
    """assert err <= bound elementwise; remember the worst err / bound of the check for the module's summary."""
    err = torch.as_tensor(err, dtype=torch.float64)
    bound = torch.as_tensor(bound, dtype=torch.float64, device=err.device).expand_as(err)
    bad = ~(err <= bound)
    assert not bool(bad.any()), "%s: %d elements over the bound, worst err %g (bound %g)" % (
        name, int(bad.sum()), float(err[bad].max()) if bool(torch.isfinite(err[bad]).any()) else float("nan"),
        float(bound[bad].flatten()[0]))
    nz = bound > 0
    r = float((err[nz] / bound[nz]).max()) if bool(nz.any()) else 0.0
    _WORST[name] = max(_WORST.get(name, 0.0), r)


@pytest.fixture(scope="module", autouse=True)
def _margins():
    yield
    if _WORST:
        print("\nworst error / bound per check (test_gpu_backward.py):")
        for k in sorted(_WORST):
            print("  %-40s %.3g" % (k, _WORST[k]))


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _lo(x):
    """tf32 residual x - trunc10(x): exact in float32 (the kernels' tf32_lo)."""
    return x - (x.view(torch.int32) & -8192).view(torch.float32)


def _pad4(n):
    return (n + 3) // 4 * 4


def _mat(g, r, c):
    """[r, c] operand in a buffer with a padded (multiple of 4) leading dimension, padding zero."""
    buf = torch.zeros(r, _pad4(c), device="cuda")
    buf[:, :c] = torch.randn(r, c, generator=g, device="cuda")
    return buf


def _buf(rows, ld):
    """output buffer with one spare row below the output, every float a sentinel."""
    return torch.full((rows + 1, ld), SENT, device="cuda")


def _untouched(buf, rows, cols):
    """nothing written right of `cols` in the first `rows` rows, nor in the spare row."""
    return bool((buf[:rows, cols:] == SENT).all()) and bool((buf[rows:] == SENT).all())


# ================================================================== 1. GEMM epilogue matrix
GEMM_SHAPES = [   # M, N, K, ldc, ldct
    (17, 40, 54, 43, 21),       # M < 32: one partial sub-tile; ldc, ldct % 4 != 0: every store scalar
    (300, 129, 33, 131, 301),   # M % 32, M % 128, N % 32, K % 32 != 0
    (129, 200, 96, 200, 132),   # aligned strides: full 32 x 32 sub-tiles take the 128-bit stores, the tails the scalar ones
]
OUTPUTS = [("C",), ("C", "C_lo"), ("Ct", "Ct_lo"), ("C", "C_lo", "Ct", "Ct_lo")]


def _act64(x, act):
    if act == ACT_LEAKY:
        return torch.where(x > 0, x, 0.01 * x)
    if act == ACT_RELU:
        return x.clamp_min(0.0)
    return x


@pytest.mark.parametrize("shape", GEMM_SHAPES)
@pytest.mark.parametrize("split3", [False, True])
def test_gemm_epilogue_matrix(ops, shape, split3):
    """Every epilogue (act x act' x bias x output set) of ops.gemm_tn.  The plain result C0 of each (bias, act) is
    checked against float64; every other output of the same product must then be C0 exactly: C0 * act'(saved)
    (a float32 product with 1, 0.01f or 0), its tf32 residual, its transpose and the transposed residual."""
    M, N, K, ldc, ldct = shape
    g = torch.Generator(device="cuda").manual_seed(M * 1000 + N)
    A, Bm = _mat(g, M, K), _mat(g, N, K)
    res = dict(A_lo=_lo(A), B_lo=_lo(Bm)) if split3 else {}
    bias = torch.randn(N, generator=g, device="cuda")
    sbuf = torch.randn(M, N + 5, generator=g, device="cuda")
    sbuf[:, ::7] = 0.0                 # saved == 0 is not > 0: the negative-side derivative applies
    saved = sbuf[:, :N]                # ld_dact = N + 5
    A64, B64 = A[:, :K].double(), Bm[:, :K].double()
    lin = A64 @ B64.t()
    mag = A64.abs() @ B64.abs().t()
    # 3xTF32: fp32-grade; one pass: 2 * 2^-10 operand truncation (test_gpu_gemm.py).  bias is added once in fp32 and
    # both activations are 1-Lipschitz, so |bias| joins the scale and the bound carries through act().
    tol = 3e-6 if split3 else 2.5e-3
    tag = "gemm 3xTF32" if split3 else "gemm one pass"

    def run(outs, **epi):
        bufs = {k: _buf(M, ldc) if k in ("C", "C_lo") else _buf(N, ldct) for k in outs}
        views = {k: (b[:M] if k in ("C", "C_lo") else b[:N]) for k, b in bufs.items()}
        ops.gemm_tn(A, Bm, M, N, K, **res, **views, **epi)
        return bufs

    for use_bias in (False, True):
        bkw = dict(bias=bias) if use_bias else {}
        for act in (ACT_NONE, ACT_LEAKY, ACT_RELU):
            C0 = run(("C",), act=act, **bkw)["C"][:M, :N].clone()
            want = _act64(lin + (bias.double() if use_bias else 0.0), act)
            scale = mag + (bias.double().abs() if use_bias else 0.0)
            _check(tag, (C0.double() - want).abs(), tol * scale)
            for dact in (None, ACT_LEAKY, ACT_RELU):
                if dact is None:
                    expect, dkw = C0, {}
                else:
                    expect = C0 * torch.where(saved > 0, 1.0, SLOPE[dact])      # float32 factors 1, 0.01f, 0
                    dkw = dict(dact_src=saved, dact=dact)
                for outs in OUTPUTS:
                    b = run(outs, act=act, **bkw, **dkw)
                    what = "act %d dact %s bias %d outputs %s" % (act, dact, use_bias, "+".join(outs))
                    if "C" in outs:
                        assert torch.equal(b["C"][:M, :N], expect), what
                        assert _untouched(b["C"], M, N), what
                    if "C_lo" in outs:
                        assert torch.equal(b["C_lo"][:M, :N], _lo(expect)), what
                        assert _untouched(b["C_lo"], M, N), what
                    if "Ct" in outs:
                        assert torch.equal(b["Ct"][:N, :M], expect.t()), what
                        assert _untouched(b["Ct"], N, M), what
                    if "Ct_lo" in outs:
                        assert torch.equal(b["Ct_lo"][:N, :M], _lo(expect).t()), what
                        assert _untouched(b["Ct_lo"], N, M), what


# ================================================================== 2. split-K, reduce, transpose
@pytest.mark.parametrize("n_out,n_in,Bsz,splits", [
    (40, 54, 64, 5),          # 2 K blocks over 5 slices: slices 2..4 are empty
    (256, 1024, 5000, 32),    # 157 K blocks: 31 slices of 5, the last of 2
    (30, 33, 9473, 32),       # 297 K blocks: slices of 10, slice 29 ragged, slices 30 and 31 empty
])
def test_split_k_slices_and_reduce(ops, n_out, n_in, Bsz, splits):
    """dW = G^T X as the MLP backward runs it: every split-K slice against float64, empty slices exact zeros,
    wgrad_reduce's dW bitwise equal to the float32 sum of the slices in slice order, db within its rounding bound."""
    g = torch.Generator(device="cuda").manual_seed(n_out * 7 + splits)
    G = torch.randn(Bsz, n_out, generator=g, device="cuda")
    X = torch.randn(Bsz, n_in, generator=g, device="cuda")
    ldb = _pad4(Bsz)
    Gt, Gtlo = torch.zeros(n_out, ldb, device="cuda"), torch.zeros(n_out, ldb, device="cuda")
    Xt, Xtlo = torch.zeros(n_in, ldb, device="cuda"), torch.zeros(n_in, ldb, device="cuda")
    ops.transpose_batch([dict(src=G, rows=Bsz, cols=n_out, dst=Gt, dst_lo=Gtlo),
                         dict(src=X, rows=Bsz, cols=n_in, dst=Xt, dst_lo=Xtlo)])
    part = torch.full((splits, n_out, _pad4(n_in)), SENT, device="cuda")
    ops.gemm_tn(Gt, Xt, n_out, n_in, Bsz, A_lo=Gtlo, B_lo=Xtlo, C=part, split_k=splits)
    per = -(-(-(-Bsz // 32)) // splits) * 32            # K rows per slice
    G64, X64 = G.double(), X.double()
    empty = 0
    for z in range(splits):
        k0, k1 = min(Bsz, z * per), min(Bsz, (z + 1) * per)
        sl = part[z, :, :n_in]
        if k0 >= k1:
            assert torch.equal(sl, torch.zeros_like(sl)), "empty split-K slice %d is not zero" % z
            empty += 1
            continue
        ref = G64[k0:k1].t() @ X64[k0:k1]
        mag = G64[k0:k1].abs().t() @ X64[k0:k1].abs()
        _check("split-K slice 3xTF32", (sl.double() - ref).abs(), 3e-6 * mag)
    assert empty == {5: 3, 32: 0 if Bsz == 5000 else 2}[splits]
    assert bool((part[:, :, n_in:] == SENT).all())
    dW = torch.empty(n_out, n_in, device="cuda")
    db = torch.empty(n_out, device="cuda")
    ops.wgrad_reduce(part, n_out, n_in, dW, Gt=Gt, B=Bsz, db=db)
    acc = part[0, :, :n_in].clone()
    for z in range(1, splits):
        acc = acc + part[z, :, :n_in]
    assert torch.equal(dW, acc), "wgrad_reduce is not the slice-order float32 sum"
    # db[o]: each of 256 threads adds ceil(B / 256) terms in sequence, then 5 butterfly levels and 8 warp partials:
    # at most ceil(B / 256) + 13 roundings, each <= u of the running |sum| <= sum |G|
    bound = (-(-Bsz // 256) + 13) * U * G64.abs().sum(0)
    _check("wgrad_reduce db", (db.double() - G64.sum(0)).abs(), bound)


TR_SHAPES = [(1, 1), (33, 70), (129, 31), (300, 257), (5, 1000), (64, 96)]


def _tr_jobs(g, shapes):
    jobs = []
    for r, c in shapes:
        src = torch.randn(r, c + 3, generator=g, device="cuda")          # ld_src = c + 3: a strided source
        jobs.append(dict(src=src, rows=r, cols=c, dst=_buf(c, r + 5), dst_lo=_buf(c, r + 5),
                         src_lo=torch.full((r, c + 3), SENT, device="cuda")))
    return jobs


def _tr_verify(jobs):
    for j in jobs:
        r, c, s = j["rows"], j["cols"], j["src"][:, :j["cols"]]
        assert torch.equal(j["dst"][:c, :r], s.t()), (r, c)
        assert torch.equal(j["dst_lo"][:c, :r], _lo(s).t()), (r, c)
        assert torch.equal(j["src_lo"][:, :c], _lo(s)), (r, c)
        assert bool((j["src_lo"][:, c:] == SENT).all()), (r, c)
        assert _untouched(j["dst"], c, r) and _untouched(j["dst_lo"], c, r), (r, c)


def test_transpose_batch_ragged(ops):
    g = torch.Generator(device="cuda").manual_seed(3)
    jobs = _tr_jobs(g, TR_SHAPES)
    ops.transpose_batch(jobs)
    _tr_verify(jobs)


@pytest.mark.parametrize("n_jobs", [13, 17, 25])
def test_transpose_batch_chunks_beyond_12_jobs(ops, n_jobs):
    """ops.transpose_batch splits the jobs into launches of at most 12 (an 8-layer block needs 17)."""
    g = torch.Generator(device="cuda").manual_seed(n_jobs)
    jobs = _tr_jobs(g, [TR_SHAPES[i % len(TR_SHAPES)] for i in range(n_jobs)])
    ops.transpose_batch(jobs)
    _tr_verify(jobs)


def test_transpose_batch_entry_point_rejects_13_jobs(ops):
    from pivotcvae_b200 import _lib as L
    g = torch.Generator(device="cuda").manual_seed(13)
    jobs = _tr_jobs(g, [(40, 24)] * 13)
    arr = (L.TransposeJob * 13)()
    for a, j in zip(arr, jobs):
        a.src, a.ld_src, a.rows, a.cols = j["src"].data_ptr(), j["src"].stride(0), j["rows"], j["cols"]
        a.dst, a.ld_dst, a.dst_lo, a.src_lo = j["dst"].data_ptr(), j["dst"].stride(0), None, None
    with pytest.raises(L.PcvError, match="1..12 jobs"):
        L.check(L.load().pcv_transpose_batch(arr, 13, ops._stream()), "pcv_transpose_batch")
    torch.cuda.synchronize()
    assert all(bool((j["dst"] == SENT).all()) for j in jobs)


# ================================================================== 3. FusedMLPFn backward over the block kinds
LS, DIM, Z = 5, 8, 16
N_DOC, N_USR = 500, 300


def _block_kinds(d):
    """name -> block description, built over the batch inputs d (segments as the models build them)."""
    oh = ("onehot", d["r"])
    gdoc = ("gather", d["doc"], d["s"])
    gusr = ("gather", d["usr"], d["u"].reshape(-1, 1))
    return {
        "dense": dict(segs=[("dense", 0)], dense=[(54, True)], hidden=[256, 256], n_out=32),
        # encoder heads on ids only: no dense input, so the backward stops before the layer-0 input gradient;
        # d_out + d_z through the fused reparam_bwd
        "enc_heads": dict(segs=[gdoc, oh, gusr], dense=[], hidden=[256, 256], n_out=2 * Z, latent=True, use=("out", "z")),
        "prior_dz_only": dict(segs=[oh, gusr], dense=[], hidden=[128, 128], n_out=2 * Z, latent=True, use=("z",)),
        "heads_dout_only": dict(segs=[("dense", 0), oh, gusr], dense=[(16, True)], hidden=[64], n_out=2 * Z,
                                latent=True, use=("out",)),
        # heads written at column 5 of a wider output: the unfused latent path
        "latent_col0": dict(segs=[("dense", 0), oh], dense=[(16, True)], hidden=[64], n_out=2 * Z, latent=True,
                            use=("out", "z"), out_col0=5, out_ld=5 + 2 * Z + 3),
        # the SCM: pivot row copied into columns 0..D-1, the MLP output behind it
        "scm": dict(segs=[("dense", 0), oh, ("gather", d["doc"], d["s"][:, :1]), gusr], dense=[(Z, True)],
                    hidden=[256, 256], n_out=(LS - 1) * DIM, out_ld=LS * DIM, out_col0=DIM, copy_seg=2),
        # one-hot and gather segments before and between dense inputs; n_out % 4 != 0
        "seg_off": dict(segs=[oh, ("dense", 0), ("gather", d["doc"], d["s"][:, :2]), ("dense", 1)],
                        dense=[(10, True), (7, True)], hidden=[64], n_out=30),
        "seg_off_frozen": dict(segs=[oh, ("dense", 0), ("gather", d["doc"], d["s"][:, :2]), ("dense", 1)],
                               dense=[(10, False), (7, True)], hidden=[64], n_out=30),
        "frozen_dense": dict(segs=[("dense", 0)], dense=[(20, False)], hidden=[64], n_out=8),
        # 8 layers: 2 * 8 + 1 = 17 transpose jobs, two launches; ReLU chain
        "relu8": dict(segs=[("dense", 0)], dense=[(33, True)], hidden=[64, 48, 64, 40, 64, 36, 64], n_out=30,
                      act=ACT_RELU),
    }


def _x0_64(segs, dense64, B):
    parts = []
    for s in segs:
        if s[0] == "dense":
            parts.append(dense64[s[1]])
        elif s[0] == "onehot":
            parts.append(F.one_hot(s[1].sum(1).long(), s[1].shape[1] + 1).double())
        else:
            parts.append(s[1].double()[s[2].reshape(B, -1)].reshape(B, -1))
    return torch.cat(parts, 1)


def _chain64(x, Ws, bs, acts, masks_from):
    """Linear/activation chain in float64.  The activation derivative is taken where the forward under test decided
    it (the saved float32 outputs): a pre-activation within float32 rounding of 0 may land on either side, and the
    backward must follow the forward it differentiates."""
    h = x
    for l, (W, b, a) in enumerate(zip(Ws, bs, acts)):
        h = h @ W.t() + b
        if a != ACT_NONE:
            one = torch.ones((), dtype=torch.float64, device=h.device)
            h = h * torch.where(masks_from[l] > 0, one, one * SLOPE[a])
    return h


KINDS = ["dense", "enc_heads", "prior_dz_only", "heads_dout_only", "latent_col0", "scm", "seg_off", "seg_off_frozen",
         "frozen_dense", "relu8"]


@pytest.mark.parametrize("B", [1, 31, 129, 4096, 9473])
@pytest.mark.parametrize("kind", KINDS)
def test_fused_mlp_backward_block_kinds(ops, kind, B):
    """FusedMLPFn.backward under tc3 and tc against float64 autograd of the same chain: every parameter gradient,
    every dense-input gradient, None for inputs that need none.  B = 9473 runs the streaming forward at CT = 4."""
    from pivotcvae_b200 import autograd as ag
    g = torch.Generator(device="cuda").manual_seed(B * 31 + KINDS.index(kind))
    rnd = lambda *s: torch.randn(*s, generator=g, device="cuda")
    d = dict(r=(torch.rand(B, LS, generator=g, device="cuda") < 0.5).float(),
             s=torch.randint(0, N_DOC, (B, LS), generator=g, device="cuda"),
             u=torch.randint(0, N_USR, (B,), generator=g, device="cuda"),
             doc=rnd(N_DOC, DIM), usr=rnd(N_USR, DIM))
    k = _block_kinds(d)[kind]
    latent = k.get("latent", False)
    act = k.get("act", ACT_LEAKY)
    c0, n_out = k.get("out_col0", 0), k["n_out"]
    out_ld = k.get("out_ld", c0 + n_out)
    dense = [rnd(B, w) for w, _ in k["dense"]]
    n_in0 = sum(dense[s[1]].shape[1] if s[0] == "dense" else
                (s[1].shape[1] + 1 if s[0] == "onehot" else s[1].shape[1] * s[2].reshape(B, -1).shape[1])
                for s in k["segs"])
    dims = [n_in0] + k["hidden"] + [n_out]
    Ws = [rnd(dims[i + 1], dims[i]) / dims[i] ** 0.5 for i in range(len(dims) - 1)]
    bs = [0.1 * rnd(dims[i + 1]) for i in range(len(dims) - 1)]
    acts = [act] * (len(dims) - 2) + [ACT_NONE]
    eps = rnd(B, Z) if latent else None
    use = k.get("use", ("out",))
    d_out = rnd(B, out_ld) if "out" in use else None       # columns outside the block's own must be ignored
    d_z = rnd(B, Z) if "z" in use else None

    spec = ag.MlpSpec(k["segs"], acts, latent=Z if latent else 0, eps=eps, out_ld=out_ld if out_ld != n_out else None,
                      out_col0=c0, copy_seg=k.get("copy_seg", -1), save=True)
    dense_in = [t.clone().requires_grad_(need) for t, (_, need) in zip(dense, k["dense"])]
    params = [t.clone().requires_grad_(True) for pair in zip(Ws, bs) for t in pair]
    res = ag.FusedMLPFn.apply(spec, B, len(dense_in), *dense_in, *params)
    out = res[0] if latent else res
    node = out.grad_fn
    sv = node.saved_tensors
    nl = node.n_layers
    x0_k, acts_k, out_k = sv[0], sv[1:nl], sv[nl]

    dense64 = [t.double().requires_grad_(need) for t, (_, need) in zip(dense, k["dense"])]
    x64 = _x0_64(k["segs"], dense64, B)
    assert torch.equal(x0_k, x64.float()), "saved x0 is not the concatenated segments"
    W64 = [W.double().requires_grad_(True) for W in Ws]
    b64 = [b.double().requires_grad_(True) for b in bs]
    h = _chain64(x64, W64, b64, acts, list(acts_k) + [out_k[:, c0:c0 + n_out]])
    loss = 0.0
    if d_out is not None:
        loss = loss + (h * d_out[:, c0:c0 + n_out].double()).sum()
    if d_z is not None:
        z = eps.double() * torch.exp(0.5 * h[:, Z:]) + h[:, :Z]
        loss = loss + (z * d_z.double()).sum()
    loss.backward()
    want = [t.grad for t in dense64] + [t.grad for pair in zip(W64, b64) for t in pair]

    # tc3: fp32-grade products, 2e-5; tc: one tf32 pass, 5e-3 (test_gpu_gemm.py test_mlp_backward_engines_agree, a
    # 3-layer chain).  The gradient of layer l passes through nl - 1 - l input-gradient GEMMs and one weight-gradient
    # GEMM, each adding its own relative error, so the bounds of the 3-layer chain scale with nl / 3 for deeper ones.
    depth = max(1.0, nl / 3)
    try:
        for engine, tol in (("tc3", 2e-5 * depth), ("tc", 5e-3 * depth)):
            ag.MLP_BWD_ENGINE = engine
            got = ag.FusedMLPFn.backward(node, d_out, d_z)
            assert got[:3] == (None, None, None)
            got_dense, got_wb = got[3:3 + len(dense)], got[3 + len(dense):]
            for gd, (_, need) in zip(got_dense, k["dense"]):
                assert (gd is None) == (not need), "dense-input gradient presence"
            for i, (a, w) in enumerate(zip(list(got_dense) + list(got_wb), want)):
                if w is None:
                    continue
                assert a.shape == w.shape, (i, a.shape, w.shape)
                _check("FusedMLPFn grad " + engine, (a.double() - w).abs().max(), tol * w.abs().max())
    finally:
        ag.MLP_BWD_ENGINE = "tc3"


# ================================================================== 4. pre-training kernels and KL
@pytest.mark.parametrize("Ls,D", [(5, 8), (3, 20), (3, 32), (2, 128)])
@pytest.mark.parametrize("no_user", [False, True])
def test_gather_norm_fwd_bwd(ops, Ls, D, no_user):
    """x0 = [normalize(concat doc[slates]) | normalize(usr[users])] and its backward scattered into the tables, with
    ids repeated thousands of times (within a slate too), all-zero slates and users (norm clamped at 1e-12)."""
    g = torch.Generator(device="cuda").manual_seed(Ls * 1000 + D + no_user)
    B, n_doc, n_usr = 3000, 40, 20
    doc = torch.randn(n_doc, D, generator=g, device="cuda")
    usr = torch.randn(n_usr, D, generator=g, device="cuda")
    doc[0], usr[0] = 0.0, 0.0
    slates = torch.randint(1, 7, (B, Ls), generator=g, device="cuda")           # heavy repeats
    slates[1::3] = torch.randint(1, n_doc, (len(range(1, B, 3)), Ls), generator=g, device="cuda")
    slates[::50] = 0                                                             # zero rows: norm 0
    users = torch.randint(1, 4, (B,), generator=g, device="cuda")
    users[::40] = 0
    Gup = torch.randn(B, (Ls + (0 if no_user else 1)) * D, generator=g, device="cuda")
    x0, inv = ops.gather_norm_fwd(doc, None if no_user else usr, slates, users)
    d_doc, d_usr = ops.gather_norm_bwd(Gup, x0, inv, slates, users, tuple(doc.shape), None if no_user else tuple(usr.shape))
    assert (d_usr is None) == no_user

    doc64 = doc.double().requires_grad_(True)
    usr64 = usr.double().requires_grad_(True)
    segs = [(doc64[slates].reshape(B, Ls * D), slates.reshape(-1), Ls * D, "doc")]
    if not no_user:
        segs.append((usr64[users], users, D, "usr"))
    parts = [F.normalize(raw, dim=1, eps=1e-12) for raw, _, _, _ in segs]
    x64 = torch.cat(parts, 1)
    (x64 * Gup.double()).sum().backward()

    off = 0
    for (raw, ids, n, name), xh in zip(segs, parts):
        xk = x0[:, off:off + n].double()
        # forward: sum of squares by fmaf, ceil(n / 32) per lane then 5 butterfly levels, all terms >= 0: relative
        # error <= (ceil(n/32) + 5) u; sqrt halves it and adds u, the reciprocal and the product u each
        ex = ((-(-n // 32) + 5) / 2 + 3) * U
        _check("gather_norm_fwd", (xk - xh.detach()).abs(), ex * xh.detach().abs())
        zero = (slates == 0).all(1) if name == "doc" else users == 0
        assert bool((x0[zero, off:off + n] == 0).all()), "all-zero rows must normalise to 0"
        # backward per element: d = (g - x dot) inv, dot = sum_k x_k g_k by fmaf (ceil(n/32) + 5 roundings of at most
        # S = sum_k |x_k g_k|), x and inv carry the forward's relative error ex, three more roundings; so
        # |err| <= (2 (ceil(n/32) + 5) + 2 ex / u + 3) u A,  A = inv (|g| + |x| S).  R atomicAdds into one table
        # entry in any order add <= R u sum |d| <= R u sum A.
        gk = Gup[:, off:off + n].double()
        S = (xh.detach().abs() * gk.abs()).sum(1, keepdim=True)
        inv64 = 1.0 / raw.detach().norm(dim=1, keepdim=True).clamp_min(1e-12)
        A = inv64 * (gk.abs() + xh.detach().abs() * S)
        A_tab = torch.zeros((n_doc if name == "doc" else n_usr), D, dtype=torch.float64, device="cuda")
        A_tab.index_add_(0, ids, A.reshape(-1, D))
        R = int(torch.bincount(ids).max())
        K = 2 * (-(-n // 32) + 5) + 2 * ex / U + 3 + R
        got, ref = (d_doc, doc64.grad) if name == "doc" else (d_usr, usr64.grad)
        _check("gather_norm_bwd", (got.double() - ref).abs(), K * U * A_tab)
        off += n


def _bce_ref(p, t):
    """float64 reference of nn.BCELoss()(sigmoid(p), t) as float32 torch computes it: s rounded to float32 (expf
    overflows to inf below p = -88.72, so s = 0 there, and s = 1 exactly for p >= 17.4), the -100 log clamp of
    BCELoss, the gradient from torch autograd of BCELoss times the sigmoid backward s (1 - s).
    -> (loss, dp, loss bound, dp bound)."""
    p64 = p.double()
    e32 = torch.exp(-p64).float().double()
    s = (1.0 / (1.0 + e32)).float().double()
    t64 = t.double()
    sl = s.clone().requires_grad_(True)
    loss = F.binary_cross_entropy(sl, t64)
    loss.backward()
    dp = sl.grad * s * (1.0 - s)
    n = p.numel()
    # kernel s = 1 / (1 + expf(-p)): expf <= 2 ulp, the add and the divide 1 ulp more, the reference's own rounding
    # of s half an ulp: |s_k - s| <= 4 ulp <= eps_s s with eps_s = 2^-21.  Where s is 0 or 1 both sides are exact.
    eps_s = 2.0 ** -21
    sat = (s == 0) | (s == 1)
    term = -(t64 * torch.log(s).clamp_min(-100) + (1 - t64) * torch.log1p(-s).clamp_min(-100))
    # d log(s) = eps_s, d log(1 - s) = eps_s s / (1 - s); logf 1 ulp and the two products and the sum: 4u |term|
    ratio = torch.where(sat, torch.zeros_like(s), s / (1 - s).clamp_min(1e-300))
    e = torch.where(sat, torch.zeros_like(s), eps_s * (t64 + (1 - t64) * ratio)) + 4 * U * term.abs()
    # one block of 1024 threads: ceil(n / 1024) sequential adds per thread, 5 butterfly levels, 32 warp partials;
    # then * (1 / n) rounded twice
    red = (-(-n // 1024) + 37) * U * term.abs().sum()
    loss_bound = (e.sum() + red) / n + 2 * U * abs(loss.item())
    # dp = (s - t) * [v / max(v, 1e-12)] / n, v = s (1 - s): the bracket is exactly 1 for v >= 1e-12 and continuous
    # with relative error <= eps_s + 4u below; (s - t) moves by eps_s s + u |s - t|; 1/n and the products 3u
    dp_bound = eps_s * (s + 3 * (s - t64).abs()) / n + 4 * U * dp.abs()
    dp_bound = torch.where(sat, 4 * U * dp.abs(), dp_bound)
    return loss.item(), dp, loss_bound, dp_bound


def _bce_inputs(g, n, soft):
    """|p| up to 120 in three regions: |p| <= 8; 20 <= |p| <= 80; 95 <= |p| <= 120.  Left out are 8 < p < 20,
    where 1 - s is a few float32 ulps of 1 and log(1 - s) is decided by the last bit of s (any two float32
    implementations, torch's included, differ there by O(1) per element), and -95 < p < -80, whose s is near
    the float32 denormal / expf-overflow boundary."""
    reg = torch.randint(0, 3, (n,), generator=g, device="cuda")
    u01 = torch.rand(n, generator=g, device="cuda")
    mag = torch.where(reg == 0, 8 * u01, torch.where(reg == 1, 20 + 60 * u01, 95 + 25 * u01))
    sign = torch.where(torch.rand(n, generator=g, device="cuda") < 0.5, -1.0, 1.0)
    p = mag * sign
    p[0] = -120.0                      # s = 0: log(s) clamps at -100
    if n > 1:
        p[1] = 120.0                   # s = 1: log(1 - s) clamps at -100
    t = torch.rand(n, generator=g, device="cuda")
    if not soft:
        t = (t < 0.5).float()
    return p, t


@pytest.mark.parametrize("n", [1, 1023, 1025, 5_000_000])
@pytest.mark.parametrize("soft", [False, True])
def test_bce_sigmoid(ops, n, soft):
    g = torch.Generator(device="cuda").manual_seed(n + soft)
    p, t = _bce_inputs(g, n, soft)
    loss, dp = ops.bce_sigmoid(p, t)
    ref, dp_ref, lb, db = _bce_ref(p, t)
    _check("bce_sigmoid loss", abs(float(loss) - ref), lb)
    _check("bce_sigmoid dpred", (dp.double() - dp_ref).abs(), db)


@pytest.mark.parametrize("B,Zl", [(1, 16), (300, 5), (4097, 16)])
@pytest.mark.parametrize("which", ["both", "d_out", "d_z"])
def test_reparam_bwd(ops, B, Zl, which):
    """gradient w.r.t. [mu | logvar] with z = eps exp(0.5 logvar) + mu folded in; d_out a strided view."""
    g = torch.Generator(device="cuda").manual_seed(B + Zl)
    out_buf = 2 * torch.randn(B, 2 * Zl + 7, generator=g, device="cuda")
    out = out_buf[:, :2 * Zl]
    dbuf = torch.randn(B, 2 * Zl + 9, generator=g, device="cuda")
    d_out = dbuf[:, 3:3 + 2 * Zl] if which in ("both", "d_out") else None
    d_z = torch.randn(B, Zl, generator=g, device="cuda") if which in ("both", "d_z") else None
    eps = torch.randn(B, Zl, generator=g, device="cuda")
    got = ops.reparam_bwd(d_out, d_z, eps, out, Zl)
    o64 = out.double().requires_grad_(True)
    loss = 0.0
    if d_out is not None:
        loss = loss + (o64 * d_out.double()).sum()
    if d_z is not None:
        z = eps.double() * torch.exp(0.5 * o64[:, Zl:]) + o64[:, :Zl]
        loss = loss + (z * d_z.double()).sum()
    loss.backward()
    ref = o64.grad
    if d_z is None:
        assert torch.equal(got, d_out)
        return
    # mu half: one float32 add (or a copy): correctly rounded, so bitwise the float32 sum
    assert torch.equal(got[:, :Zl], d_z if d_out is None else d_out[:, :Zl] + d_z)
    # logvar half: d_z eps (0.5 expf(0.5 lv)): expf 2 ulp = 4u, two products 2u; then the add u |result|
    term = (d_z.double() * eps.double() * 0.5 * torch.exp(0.5 * out[:, Zl:].double())).abs()
    _check("reparam_bwd", (got[:, Zl:].double() - ref[:, Zl:]).abs(), 8 * U * term + U * ref[:, Zl:].abs())


@pytest.mark.parametrize("rows", [4096, 65536])
def test_kl_fwd_bwd_training_sizes(ops, rows):
    """KL (one CTA, fixed reduction order) at the C3 batch and 16x it, against float64 autograd."""
    g = torch.Generator(device="cuda").manual_seed(rows)
    mu, lv, pmu, plv = (0.7 * torch.randn(rows, 16, generator=g, device="cuda") for _ in range(4))
    out, grads = ops.kl_fwd_bwd(mu, lv, pmu, plv)
    a64 = [x.double().requires_grad_(True) for x in (mu, lv, pmu, plv)]
    m, v, pm, pv = a64
    kl = -0.5 * (1 + v - pv - (torch.exp(v) + (m - pm) ** 2) / torch.exp(pv)).sum()
    kl.backward()
    with torch.no_grad():
        ev, ipv = torch.exp(v), torch.exp(-pv)
        ratio = (ev + (m - pm) ** 2) * ipv
        T = 1 + v.abs() + pv.abs() + ratio
    n = mu.numel()
    # per term: two expf (4u each) and four roundings in ratio, three in 1 + v - pv - ratio: <= 15u T; the sum:
    # ceil(n / 1024) sequential adds per thread and two 5-level butterflies
    _check("kl value", abs(float(out) - kl.item()),0.5 * (15 + -(-n // 1024) + 10) * U * float(T.sum()))
    # dmu, dpmu = +-(mu - pmu) e^-pv: 4u + 2u; dlv = -0.5 (1 - ev ipv): 8u ev ipv + 2u; dplv = -0.5 (ratio - 1): 13u ratio + u
    bounds = [8 * U * m.grad.abs(), 5 * U * (1 + ev * ipv), 8 * U * pm.grad.abs(), 7 * U * (ratio + 1)]
    for name, gk, x, b in zip(("dmu", "dlogvar", "dpmu", "dplogvar"), grads, a64, bounds):
        _check("kl " + name, (gk.double() - x.grad).abs(), b)


# ================================================================== 5. 1024-wide response MLP
def _resp_env(seed, n_items, n_users, width):
    from pivotcvae_b200.env.response_model import UserResponseModel_MLP
    torch.manual_seed(seed)
    env = UserResponseModel_MLP(n_items - 1, n_users - 1, DIM, LS, [(LS + 1) * DIM, width, width, LS], "cuda:0", False)
    return env.to("cuda:0")


def _sd(m):
    return {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}


def _N(t):
    return t.detach().cpu().numpy()


def _resp_batch(rng, B, n_items, n_users):
    return rng.integers(0, n_items, (B, LS)), rng.integers(0, n_users, B)


def test_resp_mlp_1024_forward(ops):
    """ld = 1024: inference at B = 1, 777 (streaming CT 1), 5000, 20000 (CT 2: CT 4 would need 361 472 B of shared
    memory) bitwise equal to the oracle, under the "exact", "auto" and "tc" policies (the tc engine must leave
    1024-wide blocks to the exact engines); the training forward with saved outputs at B = 20000 (CT 2) bitwise
    equal to the oracle's chain over the saved x0, every saved activation included."""
    import oracle
    n_items, n_users = 3000, 500
    env = _resp_env(11, n_items, n_users, 1024)
    esd = _sd(env)
    rng = np.random.default_rng(5)
    for B in (1, 777, 5000, 20000):
        slates, users = _resp_batch(rng, B, n_items, n_users)
        want = oracle.resp_mlp(esd, slates, users, False)
        st, ut = torch.from_numpy(slates).cuda(), torch.from_numpy(users).cuda()
        for policy in ("exact", "auto", "tc"):
            with torch.no_grad(), ops.mlp_engine(policy):
                got = env(st, ut)
            assert np.array_equal(_N(got), want), (B, policy)
    env.differentiable = True
    pred = env(st, ut)                                       # B = 20000, grad mode: GatherNormFn + FusedMLPFn(save)
    sv = pred.grad_fn.saved_tensors
    h = _N(sv[0])
    for i in (1, 2):
        h = oracle.linear(h, esd["mlp_%d.weight" % i], esd["mlp_%d.bias" % i], oracle.ACT_RELU)
        assert np.array_equal(_N(sv[i]), h), "saved activation %d" % i
    h = oracle.linear(h, esd["mlp_3.weight"], esd["mlp_3.bias"], oracle.ACT_NONE)
    assert np.array_equal(_N(pred), h) and np.array_equal(_N(sv[3]), h)


def _clean_rows(env, slates, users, need):
    """First `need` rows whose every hidden pre-activation lies farther from 0 than the float32 forward's error bound,
    so the float32 forward and the float64 oracle take the same ReLU branch everywhere.  (A row with a pre-activation
    inside the bound may differ by a whole term of a weight-gradient row between two correct implementations.)
    Bound per layer: (K + 3) u (sum_k |a_k w_k| + |b|) + sum_k e_k |w_k|, e the error of the layer's input; x0 starts
    at 16u |x0| (the gather-normalise forward's bound for L D = 40, D = 8 is 6.5u)."""
    with torch.no_grad():
        doc, usr = env.docEmbed.weight.double(), env.userEmbed.weight.double()
        x = torch.cat([F.normalize(doc[slates].reshape(len(slates), -1), dim=1, eps=1e-12),
                       F.normalize(usr[users], dim=1, eps=1e-12)], 1)
        e = 16 * U * x.abs()
        ok = torch.ones(len(slates), dtype=torch.bool, device=x.device)
        for m in env.mlp[:-1]:
            W, b = m.weight.double(), m.bias.double()
            pre = x @ W.t() + b
            e = (W.shape[1] + 3) * U * (x.abs() @ W.abs().t() + b.abs()) + e @ W.abs().t()
            ok &= (pre.abs() > e).all(1)
            x = pre.clamp_min(0)
    idx = torch.nonzero(ok).flatten()[:need]
    assert len(idx) == need, "only %d rows clear of the float32 bound" % len(idx)
    return idx


def test_resp_1024_train_step_vs_oracle(ops):
    """One response_loss step with backward (gather-normalise, 48-1024-1024-5 MLP, BCE) at B = 512 against
    oracle.resp_train_step (float64), every parameter gradient, embedding tables included."""
    import oracle
    from pivotcvae_b200.pretrain_env import response_loss
    n_items, n_users, B = 3000, 500, 512
    env = _resp_env(12, n_items, n_users, 1024)
    env.differentiable = True
    g = torch.Generator(device="cuda").manual_seed(12)
    slates = torch.randint(0, n_items, (8 * B, LS), generator=g, device="cuda")   # about a quarter of rows are clear
    users = torch.randint(0, n_users, (8 * B,), generator=g, device="cuda")
    keep = _clean_rows(env, slates, users, B)
    slates, users = slates[keep], users[keep]
    resp = (torch.rand(B, LS, generator=g, device="cuda") < 0.3).float()
    loss = response_loss(env, {"slates": _N(slates), "users": _N(users), "responses": _N(resp)})   # a loader's batch
    loss.backward()
    esd = _sd(env)
    ref_loss, ref_pred, ref_grads = oracle.resp_train_step(esd, _N(slates), _N(users), _N(resp), False)
    # loss: the kernel's BCE rounding on its own pred (the bce bound) plus the float32 forward's error on pred,
    # |d loss / d pred| = |s - t| / n times its bound (the _clean_rows propagation carried to the last layer)
    with torch.no_grad():
        pred_k = env(slates, users)
    _, _, lb, _ = _bce_ref(pred_k.reshape(-1), resp.reshape(-1))
    with torch.no_grad():
        doc, usr = env.docEmbed.weight.double(), env.userEmbed.weight.double()
        x = torch.cat([F.normalize(doc[slates].reshape(B, -1), dim=1, eps=1e-12), F.normalize(usr[users], dim=1, eps=1e-12)], 1)
        e = 16 * U * x.abs()
        for m in env.mlp:
            W, b = m.weight.double(), m.bias.double()
            pre = x @ W.t() + b
            e = (W.shape[1] + 3) * U * (x.abs() @ W.abs().t() + b.abs()) + e @ W.abs().t()
            x = pre.clamp_min(0) if m is not env.mlp[-1] else pre
        s = torch.sigmoid(torch.from_numpy(ref_pred).cuda())
        fwd = float(((s - resp.double()).abs() * e).sum()) / resp.numel()
    _check("resp step loss", abs(loss.item() - ref_loss), lb + fwd)
    for name, prm in env.named_parameters():
        ref = ref_grads[name]
        # tc3 MLP-gradient bound (test_gpu_gemm.py): fp32-grade products
        _check("resp step grad tc3", np.abs(_N(prm.grad).astype(np.float64) - ref).max(), 2e-5 * np.abs(ref).max())


# ================================================================== 6. gradients at the C3 batch
def _fused_nodes(t):
    """FusedMLPFn nodes of the autograd graph behind t, keyed by the first-layer weight's data pointer."""
    found, seen, stack = {}, set(), [t.grad_fn]
    while stack:
        n = stack.pop()
        if n is None or n in seen:
            continue
        seen.add(n)
        if type(n).__name__ == "FusedMLPFnBackward":
            nl = n.n_layers
            sv = n.saved_tensors
            found[sv[nl + 1].data_ptr()] = list(sv[1:nl]) + [sv[nl]]
        stack.extend(f for f, _ in n.next_functions)
    return found


def _masks(nodes, first_layer):
    """saved post-activation outputs of the hidden layers of the block whose first layer is `first_layer`"""
    return nodes[first_layer.weight.data_ptr()]


@pytest.mark.parametrize("model_kind", ["pivot", "list"])
def test_c3_batch_gradients(ops, model_kind):
    """get_gen_loss + backward at the C3 training batch (B = 4096, 20 480 CE rows, full 20 000-item soft-max, pushed
    eps) against a float64 torch restatement of oracle.gen_loss: encoder -> reparam -> prior -> KL -> SCM or decoder
    -> full-catalog CE.  The LeakyReLU derivatives follow the forward's saved outputs (see _chain64)."""
    from pivotcvae_b200.models.listcvae import UserListCVAEWithPrior
    from pivotcvae_b200.models.pivotcvae import PIVOTCVAE_MODELS
    from pivotcvae_b200.train_generative import get_gen_loss
    n_items, n_users, B, beta = 20000, 2000, 4096, 0.001
    torch.manual_seed(33)
    emb = torch.nn.Embedding(n_items, DIM)
    uemb = torch.nn.Embedding(n_users, DIM)
    if model_kind == "pivot":
        m = PIVOTCVAE_MODELS["pivotcvae_gt_pi"](emb, uemb, LS, DIM, Z, LS + 1, [54, 256, 256], [30, 256, 256, DIM],
                                               [38, 256, 256, (LS - 1) * DIM], [14, 128, 128], False, "cuda:0")
    else:
        m = UserListCVAEWithPrior(emb, uemb, LS, DIM, Z, LS + 1, [54, 256, 256], [30, 256, 256, LS * DIM],
                                  [14, 128, 128], False, "cuda:0")
    g = torch.Generator(device="cuda").manual_seed(34)
    slates = torch.randint(0, n_items, (B, LS), generator=g, device="cuda")
    users = torch.randint(0, n_users, (B,), generator=g, device="cuda")
    resp = (torch.rand(B, LS, generator=g, device="cuda") < 0.4).float()
    eps = torch.randn(B, Z, generator=g, device="cuda")
    m.noise.push("eps", eps)
    loss, rec, kld = get_gen_loss({"slates": slates, "users": users, "responses": resp}, m, None, beta, n_neg=n_items)
    nodes = _fused_nodes(loss)
    loss.backward()

    P = {k: v.detach().double().requires_grad_(True) for k, v in m.named_parameters() if v.requires_grad}
    doc, usr = m.docEmbed.weight.double(), m.userEmbed.weight.double()
    cond = F.one_hot(resp.sum(1).long(), LS + 1).double()
    ue = usr[users]

    def mlp(x, prefix, n, heads, last_act, masks):
        Ws = [P["%s_%d.weight" % (prefix, i + 1)] for i in range(n)]
        bs = [P["%s_%d.bias" % (prefix, i + 1)] for i in range(n)]
        acts = [ACT_LEAKY] * n
        if heads:
            Ws.append(torch.cat([P[heads[0] + ".weight"], P[heads[1] + ".weight"]], 0))
            bs.append(torch.cat([P[heads[0] + ".bias"], P[heads[1] + ".bias"]], 0))
            acts.append(ACT_NONE)
        else:
            acts[-1] = last_act
        return _chain64(x, Ws, bs, acts, masks)

    enc = mlp(torch.cat([doc[slates].reshape(B, -1), cond, ue], 1), "enc", 2, ("encmu", "enclogvar"), None,
              _masks(nodes, m.encMLP[0]))
    mu, lv = enc[:, :Z], enc[:, Z:]
    z = eps.double() * torch.exp(0.5 * lv) + mu
    pr = mlp(torch.cat([cond, ue], 1), "prior", 2, ("priorMu", "priorLogvar"), None, _masks(nodes, m.priorMLP[0]))
    pmu, plv = pr[:, :Z], pr[:, Z:]
    if model_kind == "pivot":
        piv = doc[slates[:, 0]]
        sc = mlp(torch.cat([z, cond, piv, ue], 1), "scm", 3, None, ACT_NONE, _masks(nodes, m.scmMLP[0]))
        rx = torch.cat([piv, sc], 1)
    else:
        rx = mlp(torch.cat([z, cond, ue], 1), "dec", 3, None, ACT_NONE, _masks(nodes, m.decMLP[0]))
    q = rx.reshape(B * LS, DIM)
    logits = q @ doc.t()
    rec64 = (torch.logsumexp(logits, 1) - logits.gather(1, slates.reshape(-1, 1)).squeeze(1)).mean()
    del logits
    kld64 = -0.5 * (1 + lv - plv - (torch.exp(lv) + (mu - pmu) ** 2) / torch.exp(plv)).sum()
    loss64 = rec64 + beta * kld64
    loss64.backward()
    # the C3 bounds of test_big_parity.py test_gpu_loss_and_grads_c3: loss 1e-4 relative, every gradient 2e-3 of its
    # largest element (fp32 full-catalog soft-max and 3xTF32 backward GEMMs)
    for name, got, ref in (("loss", loss, loss64), ("rec", rec, rec64), ("kld", kld, kld64)):
        _check("C3 %s" % name, abs(float(got) - float(ref)), 1e-4 * abs(float(ref)))
    for name, prm in m.named_parameters():
        if name not in P:
            assert prm.grad is None, name
            continue
        ref = P[name].grad
        if ref is None:
            assert prm.grad is None, name            # the PSM is never differentiated
            continue
        _check("C3 %s grad" % model_kind, (prm.grad.double() - ref).abs().max(), 2e-3 * ref.abs().max())
