"""-m gpu: SURVEY 8f N4 — one response-model pre-training step (pretrain_env.py:76-88) and the biased-MF top-k
recommendation (models/deterministic.py:97-124) against the reference's own outputs (tests/golden/n4.npz)."""
import numpy as np
import pytest
import torch

from gpu_util import N, T, load_sd

pytestmark = pytest.mark.gpu


class _E:
    def __init__(self, w):
        self.weight = torch.from_numpy(np.ascontiguousarray(w))


@pytest.mark.parametrize("tag,no_user", [("mlp_user", False), ("mlp_nouser", True)])
@pytest.mark.parametrize("engine", ["tc3"])
def test_response_pretrain_step(golden, tag, no_user, engine):
    from pivotcvae_b200 import autograd as ag
    from pivotcvae_b200.env.response_model import UserResponseModel_MLP
    from pivotcvae_b200.pretrain_env import response_loss
    fx = golden("n4")
    n_items, n_users, Ls, D, B = [int(v) for v in fx["cfg"]]
    m = UserResponseModel_MLP(n_items - 1, n_users - 1, D, Ls, [(Ls if no_user else Ls + 1) * D, 64, 32, Ls], "cuda:0", no_user).to("cuda:0")
    load_sd(m, fx.sub(tag + "/sd/"))
    m.differentiable = True
    batch = {"slates": fx[tag + "/slates"], "users": fx[tag + "/users"], "responses": fx[tag + "/resp"]}
    ag.MLP_BWD_ENGINE = engine
    try:
        loss = response_loss(m, batch)
        loss.backward()
    finally:
        ag.MLP_BWD_ENGINE = "tc3"
    assert abs(float(loss) - float(fx[tag + "/loss"])) <= 1e-5 * abs(float(fx[tag + "/loss"]))
    with torch.no_grad():
        pred = m(T(fx[tag + "/slates"]), T(fx[tag + "/users"]))        # inference path: the fused block
    np.testing.assert_allclose(N(pred), fx[tag + "/pred"], rtol=1e-4, atol=1e-5)
    ref = fx.sub(tag + "/grad/")
    for name, p in m.named_parameters():
        assert p.grad is not None, name
        np.testing.assert_allclose(N(p.grad), ref[name], rtol=2e-3, atol=2e-6, err_msg=name)


def test_train_response_model_loop(tmp_path):
    """The drop-in training loop runs end to end and the loss goes down (pretrain_env.py:25-139)."""
    from pivotcvae_b200.pretrain_env import train_response_model

    class DS(torch.utils.data.Dataset):
        noUser = False

        def __init__(self, n, seed):
            rng = np.random.default_rng(seed)
            self.s = rng.integers(0, 200, (n, 5))
            self.u = rng.integers(0, 30, (n, 1))
            self.r = ((self.s % 3 == 0) ^ (self.u % 2 == 0)).astype(float)     # learnable from the ids
            self.max_iid, self.max_uid = 199, 29

        def __len__(self):
            return len(self.s)

        def __getitem__(self, i):
            return {"slates": self.s[i], "users": self.u[i], "responses": self.r[i]}

    class Log:
        def log(self, s):
            pass

    torch.manual_seed(0)
    tr, va = train_response_model(DS(2048, 1), DS(256, 2), 8, 5, [48, 64, 5], 256, 6, 1e-2, 1e-6, "cuda:0",
                                  str(tmp_path / "resp.pkl"), Log())
    assert tr[-1] < tr[0] - 0.02 and (tmp_path / "resp.pkl").exists()


def test_mf_forward_and_topk_recommend(golden):
    from pivotcvae_b200.models.deterministic import MF
    fx = golden("n4")
    n_items, n_users, Ls, D, _ = [int(v) for v in fx["cfg"]]
    mf = MF(_E(fx["mf/doc"]), _E(fx["mf/usr"]), Ls, D, "cuda:0")
    with torch.no_grad():
        mf.userBias.weight.copy_(T(fx["mf/user_bias"]))
        mf.docBias.weight.copy_(T(fx["mf/doc_bias"]))
        pred = mf.forward(T(fx["mf/slates"]), None, u=T(fx["mf/users"]))
        items, _ = mf.recommend(None, u=T(fx["mf/users"]), return_item=True)
        rx, _ = mf.recommend(None, u=T(fx["mf/users"]))
    np.testing.assert_allclose(N(pred), fx["mf/pred"], rtol=1e-5, atol=1e-6)
    got, want = N(items), fx["mf/items"]
    p_all = fx["mf/p_all"]
    # torch.topk order == ours unless two scores are closer than the fp32 rounding of the two summation orders
    same = (got == want)
    for i, j in zip(*np.nonzero(~same)):
        assert abs(p_all[i, got[i, j]] - p_all[i, want[i, j]]) <= 2e-6, (i, j)
    assert same.mean() > 0.99 and rx.shape == (len(want), Ls * D)
