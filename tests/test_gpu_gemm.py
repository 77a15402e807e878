"""-m gpu: the tcgen05 TN GEMM of the MLP blocks (csrc/gemm_tc.cu) against float64 matmul: tf32 single pass
(reduced-precision tolerance), 3xTF32 (fp32-grade), ragged shapes, every epilogue, split-K + reduce."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from pivotcvae_b200 import ops as o
    o.device_ok()
    return o


def _lo(x):
    return x - (x.view(torch.int32) & -8192).view(torch.float32)


def _mat(g, r, c):
    """[r, c] view with a padded (multiple of 4) leading dimension, like the buffers of the training path."""
    buf = torch.zeros(r, (c + 3) // 4 * 4, device="cuda")
    buf[:, :c] = torch.randn(r, c, generator=g, device="cuda")
    return buf


@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (256, 128, 64), (4096, 256, 256), (1000, 40, 54), (77, 300, 14),
                                   (129, 129, 33), (5, 8, 256), (2048, 32, 38)])
@pytest.mark.parametrize("split3", [False, True])
def test_gemm_matches_float64(ops, M, N, K, split3):
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A, B = _mat(g, M, K), _mat(g, N, K)
    C = torch.full((M, (N + 3) // 4 * 4), 7.0, device="cuda")
    kw = dict(A_lo=_lo(A), B_lo=_lo(B)) if split3 else {}
    ops.gemm_tn(A, B, M, N, K, C=C, **kw)
    want = A[:, :K].double() @ B[:, :K].double().t()
    scale = (A[:, :K].double().abs() @ B[:, :K].double().abs().t()).clamp_min(1e-30)
    err = ((C[:, :N].double() - want).abs() / scale).max().item()
    assert err < (3e-6 if split3 else 2.5e-3), err          # 3xTF32: fp32-grade; one pass: 2 * 2^-10 operand truncation
    if N < C.shape[1]:
        assert bool((C[:, N:] == 7.0).all())                # nothing written beyond N


def test_gemm_epilogues(ops):
    g = torch.Generator(device="cuda").manual_seed(1)
    M, N, K = 700, 200, 96
    A, B = _mat(g, M, K), _mat(g, N, K)
    bias = torch.randn(N, generator=g, device="cuda")
    saved = torch.randn(M, N, generator=g, device="cuda")
    C, Clo = torch.zeros(M, N, device="cuda"), torch.zeros(M, N, device="cuda")
    Ct, Ctlo = torch.zeros(N, M, device="cuda"), torch.zeros(N, M, device="cuda")
    ops.gemm_tn(A, B, M, N, K, A_lo=_lo(A), B_lo=_lo(B), C=C, C_lo=Clo, Ct=Ct, Ct_lo=Ctlo, bias=bias, act=1, dact_src=saved, dact=2)
    y = torch.nn.functional.leaky_relu(A.double() @ B.double().t() + bias.double(), 0.01) * (saved > 0).double()
    scale = A.double().abs() @ B.double().abs().t() + bias.double().abs()
    assert ((C.double() - y).abs() / scale).max().item() < 3e-6
    assert torch.equal(Ct, C.t()) and torch.equal(Clo, _lo(C)) and torch.equal(Ctlo, _lo(C).t())


@pytest.mark.parametrize("n_out,n_in,Bsz,splits", [(256, 54, 4096, 16), (32, 256, 1000, 7), (8, 30, 333, 4)])
def test_wgrad_split_k_and_reduce(ops, n_out, n_in, Bsz, splits):
    """dW = G^T X and db = column sums of G, the way the backward of a Linear layer uses the pieces."""
    g = torch.Generator(device="cuda").manual_seed(n_out)
    G, X = torch.randn(Bsz, n_out, generator=g, device="cuda"), torch.randn(Bsz, n_in, generator=g, device="cuda")
    ldb = (Bsz + 3) // 4 * 4
    Gt, Gtlo = torch.zeros(n_out, ldb, device="cuda"), torch.zeros(n_out, ldb, device="cuda")
    Xt, Xtlo = torch.zeros(n_in, ldb, device="cuda"), torch.zeros(n_in, ldb, device="cuda")
    ops.transpose_batch([dict(src=G, rows=Bsz, cols=n_out, dst=Gt, dst_lo=Gtlo), dict(src=X, rows=Bsz, cols=n_in, dst=Xt, dst_lo=Xtlo)])
    assert torch.equal(Gt[:, :Bsz], G.t()) and torch.equal(Xtlo[:, :Bsz], _lo(X).t())
    part = torch.empty(splits, n_out, (n_in + 3) // 4 * 4, device="cuda")
    ops.gemm_tn(Gt, Xt, n_out, n_in, Bsz, A_lo=Gtlo, B_lo=Xtlo, C=part, split_k=splits)
    dW, db = torch.empty(n_out, n_in, device="cuda"), torch.empty(n_out, device="cuda")
    ops.wgrad_reduce(part, n_out, n_in, dW, Gt=Gt, B=Bsz, db=db)
    want = G.double().t() @ X.double()
    assert torch.allclose(dW.double(), want, rtol=1e-4, atol=1e-3 * want.abs().max().item() * 1e-2)
    assert torch.allclose(db.double(), G.double().sum(0), rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("B", [64, 1000, 4096])
def test_mlp_backward_engines_agree(ops, B):
    """FusedMLPFn.backward on the library's tcgen05 GEMMs (3xTF32 and one tf32 pass) vs plain torch autograd of the
    same Linear/LeakyReLU chain (float64)."""
    from pivotcvae_b200 import _lib as L
    from pivotcvae_b200 import autograd as ag
    g = torch.Generator(device="cuda").manual_seed(B)
    dims = [54, 256, 256, 32]
    x = torch.randn(B, dims[0], generator=g, device="cuda")
    up = torch.randn(B, dims[-1], generator=g, device="cuda")
    Ws = [(torch.randn(dims[i + 1], dims[i], generator=g, device="cuda") / dims[i] ** 0.5) for i in range(3)]
    bs = [0.1 * torch.randn(dims[i + 1], generator=g, device="cuda") for i in range(3)]
    acts = [L.ACT_LEAKY, L.ACT_LEAKY, L.ACT_NONE]

    def run(engine):
        ag.MLP_BWD_ENGINE = engine
        xs = x.clone().requires_grad_(True)
        ps = [t.clone().requires_grad_(True) for pair in zip(Ws, bs) for t in pair]
        spec = ag.MlpSpec([("dense", 0)], acts, save=True)
        out = ag.FusedMLPFn.apply(spec, B, 1, xs, *ps)
        (out * up).sum().backward()
        return [xs.grad] + [p.grad for p in ps]

    try:
        got3, got1 = run("tc3"), run("tc")
        with pytest.raises(ValueError):
            run("torch")
    finally:
        ag.MLP_BWD_ENGINE = "tc3"
    xd = x.double().requires_grad_(True)
    pd = [t.double().requires_grad_(True) for pair in zip(Ws, bs) for t in pair]
    h = xd
    for i in range(3):
        h = h @ pd[2 * i].t() + pd[2 * i + 1]
        if i < 2:
            h = torch.nn.functional.leaky_relu(h, 0.01)
    (h * up.double()).sum().backward()
    want = [xd.grad] + [p.grad for p in pd]
    for a3, a1, w in zip(got3, got1, want):
        sc = w.abs().max().item()
        assert (a3.double() - w).abs().max().item() <= 2e-5 * sc           # fp32-grade
        assert (a1.double() - w).abs().max().item() <= 5e-3 * sc           # one tf32 pass: reduced precision
