"""Parity at the BASELINE.json config sizes against the UNMODIFIED reference (fixtures big_c2/c3/c4.npz,
made by tests/golden/make_golden_big.py): C2 = 50 000 items / L=10 / nouser / B=256, C3 = 100 000 items /
B=256 training loss + gradients, C4 = 1 000 000 items / B=64.

Tables, MLP weights, the Exp(1) race noise and the Bernoulli mask are regenerated from seeds
(tests/golden/synth.py) and pinned by the checksums in the fixture; eps and every reference output are stored.

Slate parity is audited, not just asserted: the MLP blocks here are a sequential-k FMA chain, within ~1e-6 of
torch's addmm but not bit-identical to it, so a query row can differ from the reference's by |dq| ~ 1e-6 and an
arg-max whose reference top-1/top-2 gap is below 2*|dq| may legitimately flip (table rows have unit norm, so a
logit moves by at most |dq|).  Every mismatch must be such a near-tie; anything else fails.  The counts go to the
JSON file named by $PCV_PARITY_REPORT when it is set (profiles/*_parity_big.json, quoted in DESIGN.md).

CPU legs (-m "not gpu") run the same audit on the oracle; GPU legs (-m gpu) on the drop-in classes through the C ABI.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import synth  # noqa: E402

import oracle  # noqa: E402

REPORT = os.environ.get("PCV_PARITY_REPORT")

_fx_cache, _w_cache = {}, {}


def big(name):
    if name not in _fx_cache:
        _fx_cache[name] = dict(np.load(os.path.join(HERE, "golden", "big_%s.npz" % name)))
    return _fx_cache[name]


def weights(workload, kind, fx, prefix=""):
    key = (workload, kind)
    if key not in _w_cache:
        w, sd, env_sd = synth.weights(workload, kind)
        for k, v in synth.weights_checksums(sd, env_sd).items():
            assert int(fx[prefix + k]) == int(v), "regenerated synthetic weights differ from the fixture's (%s)" % k
        _w_cache[key] = (w, sd, env_sd)
    return _w_cache[key]


def report(key, entry):
    if not REPORT:
        return
    os.makedirs(os.path.dirname(os.path.abspath(REPORT)), exist_ok=True)
    data = {}
    if os.path.exists(REPORT):
        try:
            data = json.load(open(REPORT))
        except Exception:
            data = {}
    data[key] = entry
    json.dump(data, open(REPORT, "w"), indent=1, sort_keys=True)


def audit_slates(tag_name, fx, tag, w, got_items, got_rx, got_pivot=None, got_pivot_out=None, sampled=False):
    """Compare slates with the reference's; every mismatch must be a near-tie (see module docstring)."""
    L, D = w["L"], w["D"]
    B = got_items.size // L
    ref_items = fx[tag + "items"].reshape(B, L)
    got_items = got_items.reshape(B, L)
    dq = np.linalg.norm((got_rx.reshape(B, L, D).astype(np.float64) - fx[tag + "rx"].reshape(B, L, D)), axis=2)
    gap = (fx[tag + "slot_top2"][:, 0].astype(np.float64) - fx[tag + "slot_top2"][:, 1]).reshape(B, L)
    pivot_flips = np.zeros(B, dtype=bool)
    if got_pivot is not None:
        pivot_flips = got_pivot.reshape(-1) != fx[tag + "pivot_idx"]
        if pivot_flips.any():
            dpo = np.linalg.norm(got_pivot_out.astype(np.float64) - fx[tag + "pivot_out"], axis=1)
            if sampled:
                k2 = fx[tag + "pivot_key_top2"].astype(np.float64)
                rel = (k2[:, 0] - k2[:, 1]) / k2[:, 0]
                # key = sigmoid(s)/sum/E: a logit change of |dq| moves it by at most |dq| relative (sigmoid' <= sigmoid)
                bad = pivot_flips & (rel > 2 * dpo + 1e-6)
            else:
                pg = fx[tag + "pivot_top2"][:, 0].astype(np.float64) - fx[tag + "pivot_top2"][:, 1]
                bad = pivot_flips & (pg > 2 * dpo)
            assert not bad.any(), "%s: pivot differs from the reference's on rows %s and it is not a near-tie" % (tag_name, np.nonzero(bad)[0])
    same_pivot = ~pivot_flips
    mism = (got_items != ref_items) & same_pivot[:, None]
    bad = mism & (gap > 2 * dq)
    entry = {"rows": int(B * L), "slates": int(B), "pivot_flips": int(pivot_flips.sum()),
             "slot_mismatches": int(mism.sum()), "unexplained": int(bad.sum()),
             "max_dq": float(dq[same_pivot].max()) if same_pivot.any() else 0.0, "min_ref_gap": float(gap.min())}
    report(tag_name, entry)
    assert not bad.any(), "%s: %d slots differ from the reference with a top1-top2 gap above the rounding difference: %s" % (
        tag_name, bad.sum(), entry)
    return entry


# ----------------------------------------------------------------------------------------------
# CPU: the oracle against the reference at the BASELINE sizes
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,tag", [("c2", "greedy_k3/"), ("c2", "greedy_k10/"), ("c4", "greedy_k2/")])
def test_oracle_greedy_slates_at_baseline_sizes(name, tag):
    fx = big(name)
    w, sd, _ = weights(name, "pivot", fx)
    B = int(fx["B"])
    oracle.set_threads(min(8, os.cpu_count() or 1))
    try:
        ref = oracle.pivot_recommend(sd, synth.contexts(B, w["L"], int(fx[tag + "k"])), fx["users"], fx[tag + "eps"], w["no_user"], "max")
    finally:
        oracle.set_threads(1)
    e = audit_slates("oracle/%s/%s" % (name, tag[:-1]), fx, tag, w, ref["items"], ref["rx"], ref["pivot"], ref["pivot_out"])
    np.testing.assert_allclose(ref["z_mu"], fx[tag + "z_mu"], rtol=2e-5, atol=2e-6)
    assert e["unexplained"] == 0


def test_oracle_sampled_and_list_slates_c2():
    fx = big("c2")
    w, sd, _ = weights("c2", "pivot", fx)
    B, tag = int(fx["B"]), "sampled_k2/"
    race = synth.race_noise(int(fx[tag + "race_seed"]), B, w["n_items"])
    assert synth.checksum(race) == int(fx[tag + "race_sum"])
    oracle.set_threads(min(8, os.cpu_count() or 1))
    try:
        ref = oracle.pivot_recommend(sd, synth.contexts(B, w["L"], int(fx[tag + "k"])), fx["users"], fx[tag + "eps"], True, "sample", race)
        audit_slates("oracle/c2/sampled_k2", fx, tag, w, ref["items"], ref["rx"], ref["pivot"], ref["pivot_out"], sampled=True)
        wl, sdl, _ = weights("c2", "list", fx, "list/")
        lfx = {k[5:]: v for k, v in fx.items() if k.startswith("list/")}
        tag = "list_k4/"
        ref = oracle.list_recommend(sdl, synth.contexts(B, wl["L"], int(lfx[tag + "k"])), fx["users"], lfx[tag + "eps"], True)
        audit_slates("oracle/c2/list_k4", lfx, tag, wl, ref["items"], ref["rx"])
    finally:
        oracle.set_threads(1)


@pytest.mark.parametrize("tag", ["nneg1000/", "full/"])
def test_oracle_loss_c3(tag):
    fx = big("c3")
    w, sd, _ = weights("c3", "pivot", fx)
    M, N = int(fx["B"]) * w["L"], w["n_items"]
    bitmask = None
    if tag == "nneg1000/":
        bitmask = synth.pack_bitmask(synth.bernoulli_mask(int(fx[tag + "mask_seed"]), M, N, int(fx[tag + "n_neg"]) / N))
        assert synth.checksum(bitmask) == int(fx[tag + "mask_sum"])
    oracle.set_threads(min(8, os.cpu_count() or 1))
    try:
        got = oracle.gen_loss(sd, fx["slates"], fx["responses"], fx["users"].reshape(-1), fx[tag + "eps"], False, 0.001, bitmask)
    finally:
        oracle.set_threads(1)
    np.testing.assert_allclose(got, fx[tag + "loss"], rtol=1e-4)     # north_star: losses within 1e-4 relative


# ----------------------------------------------------------------------------------------------
# GPU: the drop-in classes through the C ABI against the reference at the BASELINE sizes
# ----------------------------------------------------------------------------------------------
def _gpu_model(workload, kind, fx, key="pivotcvae_gt_pi", prefix=""):
    import bench
    w, sd, env_sd = weights(workload, kind, fx, prefix)
    m, env = bench.build_gpu(w, sd, env_sd, "list" if kind == "list" else ("sampled" if key.endswith("_spi") else "greedy"), "cuda:0")
    return w, sd, env_sd, m, env


def _pivot_pieces(m, ctx, users):
    """recommend()'s own sequence (models/pivotcvae.py), exposing the intermediates the audit needs."""
    with torch.no_grad():
        r, u, _ = m._inputs(ctx, users)
        out, z, pivot_out = m._prior_chain(r, u, m.psmMLP)
        pidx = m._pick_index(pivot_out, None)
        rx = m._scm(z, ("onehot", r), pidx, None if m.noUser else m._user_seg(u), [])
        items = m.get_recommended_item(rx)
    return items, out[:, :m.latent_size], rx, pidx, pivot_out


@pytest.mark.gpu
@pytest.mark.parametrize("name,tag", [("c2", "greedy_k3/"), ("c2", "greedy_k10/"), ("c4", "greedy_k2/")])
@pytest.mark.parametrize("engine", ["auto", "simt"])
def test_gpu_greedy_slates_at_baseline_sizes(name, tag, engine):
    from gpu_util import N, T
    fx = big(name)
    w, sd, env_sd, m, env = _gpu_model(name, "pivot", fx)
    m.select_engine = engine
    B = int(fx["B"])
    ctx = T(synth.contexts(B, w["L"], int(fx[tag + "k"])))
    users = None if w["no_user"] else T(fx["users"])
    m.noise.push("eps", T(fx[tag + "eps"]))
    items, z_mu = m.recommend(ctx, users, return_item=True)          # the public call
    m.noise.push("eps", T(fx[tag + "eps"]))
    items2, z_mu2, rx, pidx, pivot_out = _pivot_pieces(m, ctx, users)
    assert torch.equal(items, items2)
    e = audit_slates("gpu-%s/%s/%s" % (engine, name, tag[:-1]), fx, tag, w, N(items), N(rx), N(pidx), N(pivot_out))
    np.testing.assert_allclose(N(z_mu), fx[tag + "z_mu"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(N(rx).reshape(-1), fx[tag + "rx"].reshape(-1), rtol=1e-4, atol=1e-5)
    # and the CUDA path is bit-identical to the oracle on the same inputs
    oracle.set_threads(min(8, os.cpu_count() or 1))
    try:
        ref = oracle.pivot_recommend(sd, N(ctx), fx["users"], fx[tag + "eps"], w["no_user"], "max")
    finally:
        oracle.set_threads(1)
    assert np.array_equal(N(items), ref["items"])
    if name == "c2" and tag == "greedy_k3/":
        resp = env(items.view(B, -1), T(fx["users"]))
        if e["pivot_flips"] == 0 and e["slot_mismatches"] == 0:
            np.testing.assert_allclose(N(resp), fx[tag + "resp"], rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("name,tag", [("c2", "greedy_k3/"), ("c2", "greedy_k10/"), ("c4", "greedy_k2/")])
def test_gpu_tc_mlp_engine_slates_at_baseline_sizes(name, tag):
    """The tcgen05 engine of the MLP blocks (mlp_engine="tc": 3xTF32, fp32-grade but not bit-identical to the FMA
    chain) against the UNMODIFIED reference at the BASELINE sizes: every slot audited, a mismatch is accepted only if
    the reference's own top1-top2 gap is below the measured |dq| |w| (audit_slates), z_mu / rx within 1e-4."""
    from gpu_util import N, T
    from pivotcvae_b200 import ops
    fx = big(name)
    w, sd, env_sd, m, env = _gpu_model(name, "pivot", fx)
    m.mlp_engine = env.mlp_engine = "tc"
    B = int(fx["B"])
    ctx = T(synth.contexts(B, w["L"], int(fx[tag + "k"])))
    users = None if w["no_user"] else T(fx["users"])
    m.noise.push("eps", T(fx[tag + "eps"]))
    items, z_mu = m.recommend(ctx, users, return_item=True)          # the public call
    with ops.mlp_engine("tc"):
        m.noise.push("eps", T(fx[tag + "eps"]))
        items2, z_mu2, rx, pidx, pivot_out = _pivot_pieces(m, ctx, users)
    assert torch.equal(items, items2)
    m.mlp_engine = None
    m.noise.push("eps", T(fx[tag + "eps"]))
    rx_exact, _ = m.recommend(ctx, users, return_item=False)
    assert not torch.equal(rx.view(-1), rx_exact.reshape(-1))        # the tc engine really ran
    e = audit_slates("gpu-mlp-tc/%s/%s" % (name, tag[:-1]), fx, tag, w, N(items), N(rx), N(pidx), N(pivot_out))
    assert e["unexplained"] == 0
    np.testing.assert_allclose(N(z_mu), fx[tag + "z_mu"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(N(rx).reshape(-1), fx[tag + "rx"].reshape(-1), rtol=1e-4, atol=1e-5)
    if name == "c2" and tag == "greedy_k3/":
        resp = env(items.view(B, -1), T(fx["users"]))
        if e["pivot_flips"] == 0 and e["slot_mismatches"] == 0:
            np.testing.assert_allclose(N(resp), fx[tag + "resp"], rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_gpu_tc_mlp_engine_list_slates_c2():
    from gpu_util import N, T
    fx = big("c2")
    w, sd, env_sd, m, env = _gpu_model("c2", "list", fx, prefix="list/")
    m.mlp_engine = "tc"
    lfx = {k[5:]: v for k, v in fx.items() if k.startswith("list/")}
    B, tag = int(fx["B"]), "list_k4/"
    ctx = T(synth.contexts(B, w["L"], int(lfx[tag + "k"])))
    m.noise.push("eps", T(lfx[tag + "eps"]))
    items, z_mu = m.recommend(ctx, None, return_item=True)
    m.noise.push("eps", T(lfx[tag + "eps"]))
    rx, _ = m.recommend(ctx, None, return_item=False)
    e = audit_slates("gpu-mlp-tc/c2/list_k4", lfx, tag, w, N(items), N(rx))
    assert e["unexplained"] == 0
    np.testing.assert_allclose(N(z_mu), lfx[tag + "z_mu"], rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_gpu_sampled_slates_c2_identical_rng():
    from gpu_util import N, T
    fx = big("c2")
    w, sd, env_sd, m, env = _gpu_model("c2", "pivot", fx, "pivotcvae_gt_spi")
    B, tag = int(fx["B"]), "sampled_k2/"
    race = synth.race_noise(int(fx[tag + "race_seed"]), B, w["n_items"])
    assert synth.checksum(race) == int(fx[tag + "race_sum"])
    ctx = T(synth.contexts(B, w["L"], int(fx[tag + "k"])))
    m.noise.push("eps", T(fx[tag + "eps"]))
    m.noise.push("race", T(race))
    items, _ = m.recommend(ctx, None, return_item=True)
    m.noise.push("eps", T(fx[tag + "eps"]))
    m.noise.push("race", T(race))
    items2, _, rx, pidx, pivot_out = _pivot_pieces(m, ctx, None)
    assert torch.equal(items, items2)
    audit_slates("gpu/c2/sampled_k2", fx, tag, w, N(items), N(rx), N(pidx), N(pivot_out), sampled=True)


@pytest.mark.gpu
def test_gpu_list_slates_c2():
    from gpu_util import N, T
    fx = big("c2")
    w, sd, env_sd, m, env = _gpu_model("c2", "list", fx, prefix="list/")
    lfx = {k[5:]: v for k, v in fx.items() if k.startswith("list/")}
    B, tag = int(fx["B"]), "list_k4/"
    ctx = T(synth.contexts(B, w["L"], int(lfx[tag + "k"])))
    m.noise.push("eps", T(lfx[tag + "eps"]))
    items, z_mu = m.recommend(ctx, None, return_item=True)
    m.noise.push("eps", T(lfx[tag + "eps"]))
    rx, _ = m.recommend(ctx, None, return_item=False)
    audit_slates("gpu/c2/list_k4", lfx, tag, w, N(items), N(rx))
    np.testing.assert_allclose(N(z_mu), lfx[tag + "z_mu"], rtol=2e-5, atol=2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["nneg1000/", "full/"])
def test_gpu_loss_and_grads_c3(tag):
    """get_gen_loss + backward at 100 000 items, B=256 (train_generative.py:44-65, 133): loss within 1e-4 relative,
    every parameter gradient within 2e-3 of torch autograd on the reference."""
    from gpu_util import N, T
    from pivotcvae_b200.train_generative import get_gen_loss
    fx = big("c3")
    w, sd, env_sd, m, env = _gpu_model("c3", "pivot", fx)
    M, Nn = int(fx["B"]) * w["L"], w["n_items"]
    n_neg = int(fx[tag + "n_neg"])
    m.noise.push("eps", T(fx[tag + "eps"]))
    if tag == "nneg1000/":
        bitmask = synth.pack_bitmask(synth.bernoulli_mask(int(fx[tag + "mask_seed"]), M, Nn, n_neg / Nn))
        assert synth.checksum(bitmask) == int(fx[tag + "mask_sum"])
        m.noise.push("mask", T(bitmask.view(np.int32)))
    batch = {"slates": fx["slates"], "users": fx["users"], "responses": fx["responses"]}
    loss, rec, kld = get_gen_loss(batch, m, None, 0.001, n_neg=n_neg)
    got = [loss.item(), rec.item(), kld.item()]
    np.testing.assert_allclose(got, fx[tag + "loss"], rtol=1e-4)
    loss.backward()
    worst = 0.0
    grads = {k[len(tag) + 5:]: v for k, v in fx.items() if k.startswith(tag + "grad/")}
    assert grads
    for pname, prm in m.named_parameters():
        if pname in grads:
            g = N(prm.grad)
            scale = np.abs(grads[pname]).max() + 1e-30
            worst = max(worst, float(np.abs(g - grads[pname]).max() / scale))
            np.testing.assert_allclose(g, grads[pname], rtol=2e-3, atol=2e-3 * scale, err_msg=pname)
        else:
            assert prm.grad is None, pname
    report("gpu/c3/loss_" + tag[:-1], {"loss": got, "reference": [float(v) for v in fx[tag + "loss"]],
                                       "rel_err": float(abs(got[0] - fx[tag + "loss"][0]) / fx[tag + "loss"][0]),
                                       "worst_grad_err_over_max": worst})
