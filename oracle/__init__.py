"""CPU oracle for the PivotCVAE hot path — TEST INFRASTRUCTURE ONLY.

ctypes wrapper over oracle/pcv_oracle.c plus numpy compositions that restate the
reference's call stacks (SURVEY §3).  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference leg may import this package; nothing
under pivotcvae_b200/ does.  Parity pinning: tests/test_oracle_golden.py checks
every function here against fixtures produced by the reference's own classes
(tests/golden/make_golden.py).

Weight dictionaries (`sd`) use the reference's state_dict names
(models/pivotcvae.py:112-152): enc_i.weight, encmu.weight, psm_i.weight, ...
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpcv_oracle.so")

ACT_NONE, ACT_LEAKY, ACT_RELU = 0, 1, 2


def build(force=False):
    src = os.path.join(_HERE, "pcv_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-B", "-C", _HERE], check=True, stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.orc_kl.restype = ctypes.c_double
        _lib.orc_get_threads.restype = ctypes.c_int
    return _lib


def set_threads(n):
    lib().orc_set_threads(ctypes.c_int(int(n)))


def get_threads():
    return lib().orc_get_threads()


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


I64 = ctypes.c_int64
I32 = ctypes.c_int
U64 = ctypes.c_uint64


# ----------------------------------------------------------------------------
# primitives
# ----------------------------------------------------------------------------
def expf(x):
    x = _f32(x)
    y = np.empty_like(x)
    lib().orc_expf(_p(x), I64(x.size), _p(y))
    return y


def philox4x32_10(ctr, key):
    c = np.ascontiguousarray(ctr, dtype=np.uint32)
    k = np.ascontiguousarray(key, dtype=np.uint32)
    o = np.empty(4, dtype=np.uint32)
    lib().orc_philox4x32_10(_p(c), _p(k), _p(o))
    return o


def bernoulli_bitmask(seed, offset, M, N, keep_prob):
    bits = np.empty((M, (N + 31) // 32), dtype=np.uint32)
    lib().orc_bernoulli_bitmask(U64(seed), U64(offset), I64(M), I64(N), ctypes.c_double(keep_prob), _p(bits))
    return bits


def pack_bitmask(mask):
    """(M, N) {0,1} -> (M, ceil(N/32)) uint32, bit j%32 of word j//32."""
    mask = np.asarray(mask) != 0
    M, N = mask.shape
    words = (N + 31) // 32
    pad = np.zeros((M, words * 32), dtype=bool)
    pad[:, :N] = mask
    b = pad.reshape(M, words, 32).astype(np.uint64)
    return (b << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32)


def normalize_rows(W):
    W = _f32(W)
    out = np.empty_like(W)
    lib().orc_normalize_rows(_p(W), I64(W.shape[0]), I32(W.shape[1]), _p(out))
    return out


def condition(r):
    r = _f32(r)
    B, L = r.shape
    c = np.empty((B, L + 1), dtype=np.float32)
    lib().orc_condition(_p(r), I64(B), I32(L), _p(c))
    return c


def linear(x, W, b, act=ACT_NONE):
    x, W, b = _f32(x), _f32(W), _f32(b)
    B, K = x.shape
    N = W.shape[0]
    assert W.shape[1] == K and b.shape[0] == N
    y = np.empty((B, N), dtype=np.float32)
    lib().orc_linear(_p(x), I64(B), I32(K), _p(W), _p(b), I32(N), I32(act), _p(y))
    return y


def reparam(mu, logvar, eps):
    mu, logvar, eps = _f32(mu), _f32(logvar), _f32(eps)
    z = np.empty_like(mu)
    lib().orc_reparam(_p(mu), _p(logvar), _p(eps), I64(mu.size), _p(z))
    return z


def score_select(W, Q, mode="greedy", noise=None):
    """argmax_j <q_i, w_j> (greedy) or the sigmoid exponential race. -> (idx int64[M], val f32[M]).  Greedy: a NaN
    score never wins (it counts as -inf); a row with no score above -inf returns index 0 and value -inf."""
    W, Q = _f32(W), _f32(Q)
    N, D = W.shape
    M = Q.shape[0]
    idx = np.empty(M, dtype=np.int64)
    val = np.empty(M, dtype=np.float32)
    m = 0
    if mode != "greedy":
        m = 1
        noise = _f32(noise)
        assert noise.shape == (M, N)
    lib().orc_score_select(_p(W), I64(N), I32(D), _p(Q), I64(M), I32(m), _p(noise), _p(idx), _p(val))
    return idx, val


def sigmoid_categorical(W, Q, seed, offset=0):
    """Throughput-mode draw from Categorical(sigmoid(Q W^T)) (pivotcvae.py:349-351): the rejection sampler of
    csrc/sampler.cu restated -> (idx int64[M], proposals used int32[M], -1 = inverse-CDF fallback)."""
    W, Q = _f32(W), _f32(Q)
    M = Q.shape[0]
    idx = np.empty(M, dtype=np.int64)
    iters = np.empty(M, dtype=np.int32)
    lib().orc_sigmoid_categorical(_p(W), I64(W.shape[0]), I32(W.shape[1]), _p(Q), I64(M), U64(seed), U64(offset), _p(idx), _p(iters))
    return idx, iters


def score_logits(W, Q):
    W, Q = _f32(W), _f32(Q)
    out = np.empty((Q.shape[0], W.shape[0]), dtype=np.float32)
    lib().orc_score_logits(_p(W), I64(W.shape[0]), I32(W.shape[1]), _p(Q), I64(Q.shape[0]), _p(out))
    return out


def score_topk(W, Q, k):
    """torch.topk of every score row, restated: score descending, equal scores by ascending index (the order a
    first-index arg-max repeated k times gives).  Non-finite rule (include/pcv_b200.h): a NaN score counts as -inf, and
    only scores above -inf are listed; the slots after them hold index -1 and value -inf, as past the end of a short
    catalog.  -> (idx int64[M, k], val f32[M, k])."""
    p = score_logits(W, Q)
    key = np.where(np.isnan(p), -np.inf, p).astype(np.float64)
    order = np.lexsort((np.broadcast_to(np.arange(p.shape[1]), p.shape), -key), axis=1)[:, :k]
    val = np.take_along_axis(key, order, 1).astype(np.float32)
    idx = np.where(val > -np.inf, order, -1).astype(np.int64)
    return idx, val


def slate_no_repeat(W, Q, L):
    """Opt-in no-repeat selection (NOT reference behaviour, SURVEY F1): rows of Q are the L slots of M/L slates;
    slot l takes arg-max_j <q, w_j> (ties -> lowest j) over the items slots 0..l-1 of its slate have taken, among the
    scores above -inf (a NaN score counts as -inf).  A slot with no such item keeps its plain arg-max
    (score_select's result), which may repeat an earlier slot's item; it does not count as taken."""
    p = score_logits(W, Q)
    p = np.where(np.isnan(p), np.float32(-np.inf), p)
    M = p.shape[0]
    items = np.empty(M, dtype=np.int64)
    vals = np.empty(M, dtype=np.float32)
    for b in range(M // L):
        taken = []
        for l in range(L):
            row = p[b * L + l]
            free = row.copy()
            free[taken] = -np.inf
            if free.max() > -np.inf:
                j = int(np.argmax(free))          # numpy arg-max returns the first maximal index
                taken.append(j)
            else:
                j = int(np.argmax(row))           # all -inf: index 0, as score_select
            items[b * L + l], vals[b * L + l] = j, row[j]
    return items, vals


def ce(W, Q, targets, bitmask=None):
    """-> (loss_rows[M], lse[M], dq[M, D]); bitmask None = full-catalog soft-max."""
    W, Q, targets = _f32(W), _f32(Q), _i64(targets).reshape(-1)
    N, D = W.shape
    M = Q.shape[0]
    if bitmask is not None:
        bitmask = np.ascontiguousarray(bitmask, dtype=np.uint32)
        assert bitmask.shape == (M, (N + 31) // 32)
    loss = np.empty(M, dtype=np.float32)
    lse = np.empty(M, dtype=np.float32)
    dq = np.empty((M, D), dtype=np.float32)
    lib().orc_ce(_p(W), I64(N), I32(D), _p(Q), _p(targets), I64(M), _p(bitmask), _p(loss), _p(lse), _p(dq))
    return loss, lse, dq


def cand_ce(W, Q, candidates, target_pos):
    """-> (loss_rows[M], dq[M, D], p[M, nC]) for the sampled soft-max mode."""
    W, Q = _f32(W), _f32(Q)
    M, D = Q.shape
    cand = _i64(candidates).reshape(M, -1)
    tpos = _i64(target_pos).reshape(-1)
    nC = cand.shape[1]
    loss = np.empty(M, dtype=np.float32)
    dq = np.empty((M, D), dtype=np.float32)
    p = np.empty((M, nC), dtype=np.float32)
    lib().orc_cand_ce(_p(W), I32(D), _p(Q), _p(cand), _p(tpos), I64(M), I32(nC), _p(loss), _p(dq), _p(p))
    return loss, dq, p


def kl(mu, lv, pmu, plv, grads=False):
    mu, lv, pmu, plv = _f32(mu), _f32(lv), _f32(pmu), _f32(plv)
    if grads:
        g = [np.empty_like(mu) for _ in range(4)]
        v = lib().orc_kl(_p(mu), _p(lv), _p(pmu), _p(plv), I64(mu.size), *[_p(a) for a in g])
        return v, g
    return lib().orc_kl(_p(mu), _p(lv), _p(pmu), _p(plv), I64(mu.size), None, None, None, None)


def urm(variant, doc, usr, item_bias, user_bias, slates, users, pos_bias=None, pos_dep=None, mr_factor=0.0):
    doc, usr = _f32(doc), _f32(usr)
    ib, ub = _f32(item_bias).reshape(-1), _f32(user_bias).reshape(-1)
    slates, users = _i64(slates), _i64(users).reshape(-1)
    B, L = slates.shape
    D = doc.shape[1]
    pb = _f32(pos_bias) if pos_bias is not None else None
    pd = _f32(pos_dep).reshape(-1) if pos_dep is not None else None
    out = np.empty((B, L), dtype=np.float32)
    lib().orc_urm(I32(variant), _p(doc), _p(usr), _p(ib), _p(ub), _p(pb), _p(pd), ctypes.c_float(mr_factor),
                  I32(L), I32(D), _p(slates), _p(users), I64(B), _p(out))
    return out


def resp_input(doc, usr, slates, users, no_user):
    doc = _f32(doc)
    slates = _i64(slates)
    B, L = slates.shape
    D = doc.shape[1]
    usr_a = _f32(usr) if not no_user else None
    users_a = _i64(users).reshape(-1) if not no_user else None
    x = np.empty((B, L * D + (0 if no_user else D)), dtype=np.float32)
    lib().orc_resp_input(_p(doc), _p(usr_a), I32(L), I32(D), _p(slates), _p(users_a), I64(B), I32(int(no_user)), _p(x))
    return x


# ----------------------------------------------------------------------------
# compositions (the reference's call stacks, SURVEY §3)
# ----------------------------------------------------------------------------
def _count_layers(sd, prefix):
    n = 0
    while "%s_%d.weight" % (prefix, n + 1) in sd:
        n += 1
    return n


def mlp(x, sd, prefix, last_act, hidden_act=ACT_LEAKY):
    """prefix_1 .. prefix_n; hidden layers use hidden_act, the last one last_act."""
    n = _count_layers(sd, prefix)
    for i in range(1, n + 1):
        act = hidden_act if i < n else last_act
        x = linear(x, sd["%s_%d.weight" % (prefix, i)], sd["%s_%d.bias" % (prefix, i)], act)
    return x


def prior(sd, r, u, no_user):
    """get_prior: pivotcvae.py:229-240 / listcvae.py:121-132."""
    c = condition(r)
    x = c if no_user else np.concatenate([c, _f32(sd["userEmbed.weight"])[_i64(u).reshape(-1)]], 1)
    h = mlp(x, sd, "prior", ACT_LEAKY)
    return linear(h, sd["priorMu.weight"], sd["priorMu.bias"]), linear(h, sd["priorLogvar.weight"], sd["priorLogvar.bias"])


def encode(sd, s, r, u, no_user):
    """forward()'s encoder half: pivotcvae.py:250-259, 159-174."""
    W = _f32(sd["docEmbed.weight"])
    s = _i64(s)
    emb = W[s.reshape(-1)].reshape(s.shape[0], -1)
    c = condition(r)
    parts = [emb, c]
    if not no_user:
        parts.append(_f32(sd["userEmbed.weight"])[_i64(u).reshape(-1)])
    h = mlp(np.concatenate(parts, 1), sd, "enc", ACT_LEAKY)
    mu = linear(h, sd["encmu.weight"], sd["encmu.bias"])
    lv = linear(h, sd["enclogvar.weight"], sd["enclogvar.bias"])
    return mu, lv, emb


def pick_pivot(sd, pivot_out, how, true_pivot=None, noise=None):
    """pivotcvae.py:186-195 and the variant overrides. how in {'gt','max','sample','sample_gt'}."""
    W = _f32(sd["docEmbed.weight"])
    if how == "gt":
        return _i64(true_pivot)
    if how == "max":
        return score_select(W, pivot_out, "greedy")[0]
    if how == "sample":
        return score_select(W, pivot_out, "exprace", noise)[0]
    if how == "sample_gt":
        return score_select(W, W[_i64(true_pivot)], "exprace", noise)[0]
    raise ValueError(how)


def pivot_decode(sd, z, c, uemb, how, true_pivot=None, noise=None):
    """decode: pivotcvae.py:197-227 -> (rx[B,L,D], pivot_idx, pivot_out)."""
    W = _f32(sd["docEmbed.weight"])
    parts = [z, c] + ([uemb] if uemb is not None else [])
    pivot_out = mlp(np.concatenate(parts, 1), sd, "psm", ACT_NONE)
    p = pick_pivot(sd, pivot_out, how, true_pivot, noise)
    pe = W[p]
    parts = [z, c, pe] + ([uemb] if uemb is not None else [])
    out = mlp(np.concatenate(parts, 1), sd, "scm", ACT_NONE)
    B, D = pe.shape
    rx = np.concatenate([pe.reshape(B, 1, D), out.reshape(B, -1, D)], 1)
    return rx, p, pivot_out


def pivot_recommend(sd, r, u, eps, no_user, infer="max", noise=None):
    """recommend(return_item=True): pivotcvae.py:278-296 -> dict."""
    mu, lv = prior(sd, r, u, no_user)
    z = reparam(mu, lv, eps)
    c = condition(r)
    uemb = None if no_user else _f32(sd["userEmbed.weight"])[_i64(u).reshape(-1)]
    rx, p, pivot_out = pivot_decode(sd, z, c, uemb, infer, noise=noise)
    D = rx.shape[2]
    items, vals = score_select(_f32(sd["docEmbed.weight"]), rx.reshape(-1, D), "greedy")
    return dict(items=items, z_mu=mu, z_logvar=lv, z=z, rx=rx, pivot=p, pivot_out=pivot_out, vals=vals)


def list_decode(sd, z, c, uemb):
    parts = [z, c] + ([uemb] if uemb is not None else [])
    return mlp(np.concatenate(parts, 1), sd, "dec", ACT_NONE)


def list_recommend(sd, r, u, eps, no_user):
    """listcvae.py:170-188."""
    mu, lv = prior(sd, r, u, no_user)
    z = reparam(mu, lv, eps)
    c = condition(r)
    uemb = None if no_user else _f32(sd["userEmbed.weight"])[_i64(u).reshape(-1)]
    rx = list_decode(sd, z, c, uemb)
    W = _f32(sd["docEmbed.weight"])
    items, vals = score_select(W, rx.reshape(-1, W.shape[1]), "greedy")
    return dict(items=items, z_mu=mu, z_logvar=lv, z=z, rx=rx, vals=vals)


def pivot_forward(sd, s, r, u, eps, no_user, train="gt", noise=None):
    """forward(): pivotcvae.py:242-276 (full-catalog branch), without materialising p."""
    mu, lv, emb = encode(sd, s, r, u, no_user)
    z = reparam(mu, lv, eps)
    c = condition(r)
    uemb = None if no_user else _f32(sd["userEmbed.weight"])[_i64(u).reshape(-1)]
    rx, p, pivot_out = pivot_decode(sd, z, c, uemb, train, true_pivot=_i64(s)[:, 0], noise=noise)
    return dict(rx=rx, z=z, emb=emb, z_mu=mu, z_logvar=lv, pivot=p)


def list_forward(sd, s, r, u, eps, no_user):
    mu, lv, emb = encode(sd, s, r, u, no_user)
    z = reparam(mu, lv, eps)
    c = condition(r)
    uemb = None if no_user else _f32(sd["userEmbed.weight"])[_i64(u).reshape(-1)]
    rx = list_decode(sd, z, c, uemb)
    return dict(rx=rx, z=z, emb=emb, z_mu=mu, z_logvar=lv)


def gen_loss(sd, s, r, u, eps, no_user, beta, bitmask=None, model="pivot", train="gt", noise=None):
    """get_gen_loss, mask-train branch: train_generative.py:44-65 -> (loss, recLoss, KLD)."""
    pmu, plv = prior(sd, r, u, no_user)
    f = pivot_forward(sd, s, r, u, eps, no_user, train, noise) if model == "pivot" else list_forward(sd, s, r, u, eps, no_user)
    W = _f32(sd["docEmbed.weight"])
    q = f["rx"].reshape(-1, W.shape[1])
    loss_rows, _, _ = ce(W, q, _i64(s).reshape(-1), bitmask)
    rec = float(np.mean(loss_rows.astype(np.float64)))
    kld = kl(f["z_mu"], f["z_logvar"], pmu, plv)
    return rec + beta * kld, rec, kld


def gen_loss_candidates(sd, s, r, u, eps, no_user, beta, candidates, target_pos, model="pivot"):
    """get_gen_loss, candidate branch (train_generative.py:52-56) -> (loss, recLoss, KLD)."""
    pmu, plv = prior(sd, r, u, no_user)
    f = pivot_forward(sd, s, r, u, eps, no_user, "gt") if model == "pivot" else list_forward(sd, s, r, u, eps, no_user)
    W = _f32(sd["docEmbed.weight"])
    q = f["rx"].reshape(-1, W.shape[1])
    loss_rows, _, _ = cand_ce(W, q, candidates, target_pos)
    rec = float(np.mean(loss_rows.astype(np.float64)))
    kld = kl(f["z_mu"], f["z_logvar"], pmu, plv)
    return rec + beta * kld, rec, kld


def resp_mlp(sd, slates, users, no_user):
    """UserResponseModel_MLP.forward: env/response_model.py:76-87 (plain ReLU)."""
    x = resp_input(sd["docEmbed.weight"], None if no_user else sd["userEmbed.weight"], slates, users, no_user)
    return mlp(x, sd, "mlp", ACT_NONE, hidden_act=ACT_RELU)


def ils(table, slates):
    """analysis.py:13-30 get_ILS -> f32[B]."""
    table, slates = _f32(table), _i64(slates)
    B, L = slates.shape
    out = np.empty(B, dtype=np.float32)
    lib().orc_ils(_p(table), I32(table.shape[1]), _p(slates), I64(B), I32(L), _p(out))
    return out


def coverage(slates, N):
    """analysis.py:5-11 get_coverage."""
    return len(np.unique(np.asarray(slates))) * 1.0 / N


# ---------------------------------------------------------------------------
# SURVEY 8f N4: response-model pre-training step (pretrain_env.py:76-88) and the biased MF (deterministic.py:97-124)
# ---------------------------------------------------------------------------
def resp_train_step(sd, slates, users, resp, no_user):
    """forward (env/response_model.py:76-87) -> BCELoss(sigmoid(pred), resp) -> gradients of every parameter incl. the
    embedding tables.  numpy float64 restatement (small cases only).  -> (loss, pred, {name: grad})."""
    doc = sd["docEmbed.weight"].astype(np.float64)
    B, Ls = slates.shape
    D = doc.shape[1]
    raw = doc[slates].reshape(B, Ls * D)
    nrm = np.maximum(np.linalg.norm(raw, axis=1, keepdims=True), 1e-12)
    parts, raws, norms = [raw / nrm], [raw], [nrm]
    if not no_user:
        usr = sd["userEmbed.weight"].astype(np.float64)
        ur = usr[users.reshape(-1)]
        un = np.maximum(np.linalg.norm(ur, axis=1, keepdims=True), 1e-12)
        parts.append(ur / un)
        raws.append(ur)
        norms.append(un)
    x0 = np.concatenate(parts, 1)
    n_layers = _count_layers(sd, "mlp")
    acts, h = [x0], x0
    for i in range(1, n_layers + 1):
        h = h @ sd["mlp_%d.weight" % i].astype(np.float64).T + sd["mlp_%d.bias" % i].astype(np.float64)
        if i < n_layers:
            h = np.maximum(h, 0.0)
        acts.append(h)
    pred = h
    s = 1.0 / (1.0 + np.exp(-pred))
    t = resp.astype(np.float64)
    loss = float(np.mean(-(t * np.maximum(np.log(s), -100) + (1 - t) * np.maximum(np.log(1 - s), -100))))
    g = (s - t) / pred.size
    grads = {}
    for i in range(n_layers, 0, -1):
        if i < n_layers:
            g = g * (acts[i] > 0)
        grads["mlp_%d.weight" % i] = g.T @ acts[i - 1]
        grads["mlp_%d.bias" % i] = g.sum(0)
        g = g @ sd["mlp_%d.weight" % i].astype(np.float64)
    def unnorm(gx, xhat, nrm):  # noqa: E306
        return (gx - xhat * (xhat * gx).sum(1, keepdims=True)) / nrm
    gd = unnorm(g[:, :Ls * D], parts[0], norms[0]).reshape(B, Ls, D)
    d_doc = np.zeros_like(doc)
    np.add.at(d_doc, slates, gd)
    grads["docEmbed.weight"] = d_doc
    if not no_user:
        gu = unnorm(g[:, Ls * D:], parts[1], norms[1])
        d_usr = np.zeros_like(sd["userEmbed.weight"].astype(np.float64))
        np.add.at(d_usr, users.reshape(-1), gu)
        grads["userEmbed.weight"] = d_usr
    return loss, pred, grads


def mf_scores(doc, usr, doc_bias, user_bias, users):
    """p[i, j] = <normalize(usr)[u_i], normalize(doc)[j]> + b_u + b_j (deterministic.py:36-47, 97-112), float64."""
    d = doc.astype(np.float64)
    u = usr.astype(np.float64)
    d = d / np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-12)
    u = u / np.maximum(np.linalg.norm(u, axis=1, keepdims=True), 1e-12)
    return u[users] @ d.T + user_bias.astype(np.float64)[users].reshape(-1, 1) + doc_bias.astype(np.float64).reshape(1, -1)
