"""autograd glue around the fused CUDA blocks.

Forward passes are single calls into libpcv_b200.so.  Backward of the catalog
cross-entropy is free (the forward kernel already produced d loss/d q).  Backward
of the MLP blocks runs on the library's own tensor-core GEMMs (csrc/gemm_tc.cu):
per layer one split-K weight-gradient GEMM (+ a deterministic reduce that also
emits the bias gradient) and one input-gradient GEMM whose epilogue applies the
activation derivative and writes the transposed copy the next weight-gradient
GEMM consumes.  MLP_BWD_ENGINE = "tc3" (3xTF32: fp32-grade products, default)
or "tc" (one tf32 pass: the reduced-precision training config).  The PSM block
never needs a backward (SURVEY F6).
"""
import torch

from . import _lib as L
from . import ops


class MlpSpec:
    """Static description of one fused block.

    segs: list of ('dense', k) | ('onehot', r) | ('gather', table, idx[, normalize]);
          ('dense', k) refers to the k-th differentiable dense input of the call.
    acts: activation id per layer.
    """

    def __init__(self, segs, acts, latent=0, eps=None, seed=0, offset=0, out_ld=None, out_col0=0, copy_seg=-1,
                 save=True, offset_dev=None):
        self.segs, self.acts = segs, list(acts)
        self.save = save
        self.latent, self.eps, self.seed, self.offset = latent, eps, seed, offset
        self.offset_dev = offset_dev
        self.out_ld, self.out_col0, self.copy_seg = out_ld, out_col0, copy_seg

    def build_segments(self, dense):
        out = []
        for s in self.segs:
            if s[0] == "dense":
                out.append(ops.Dense(dense[s[1]]))
            elif s[0] == "onehot":
                out.append(ops.OneHot(s[1]))
            else:
                out.append(ops.Gather(s[1], s[2], normalize=(len(s) > 3 and s[3])))
        return out


MLP_BWD_ENGINE = "tc3"


_SM_COUNT = {}


def _sm_count(device):
    n = _SM_COUNT.get(device)
    if n is None:
        n = _SM_COUNT[device] = torch.cuda.get_device_properties(device).multi_processor_count
    return n


def _padded(rows, cols, like):
    """[rows, cols] view of a fresh buffer whose leading dimension is a multiple of 4 floats (TMA operand rule)."""
    return torch.empty(rows, ops.pad4(cols), dtype=torch.float32, device=like.device)


def _mlp_backward_tc(g, x0, acts, Ws, act_ids, need_input_grad, split3):
    """Backward of Linear/activation chain on the tcgen05 GEMMs.  g: [B, n_out_last] gradient w.r.t. the last layer's
    PRE-activation output (callers fold a last-layer activation in beforehand).  Returns (grads_wb, g_in | None)."""
    nl = len(Ws)
    B = g.shape[0]
    Bp = ops.pad4(B)
    inputs = [x0] + list(acts)                       # input of layer l (post-activation output of layer l - 1)
    # ---- one batched launch: K-major (transposed) copies of every saved input, of the top gradient and of the weights
    jobs, XT, XTlo, WT, WTlo = [], [], [], [None] * nl, [None] * nl
    for l in range(nl):
        n_in = Ws[l].shape[1]
        xt = torch.empty(n_in, Bp, dtype=torch.float32, device=g.device)
        xl = torch.empty_like(xt) if split3 else None
        jobs.append(dict(src=inputs[l], rows=B, cols=n_in, dst=xt, dst_lo=xl))
        XT.append(xt)
        XTlo.append(xl)
        if l > 0 or need_input_grad:
            n_out = Ws[l].shape[0]
            wt = _padded(n_in, n_out, g)
            wl = torch.empty_like(wt) if split3 else None
            jobs.append(dict(src=Ws[l], rows=n_out, cols=n_in, dst=wt, dst_lo=wl))
            WT[l], WTlo[l] = wt, wl
    n_top = Ws[-1].shape[0]
    if n_top % 4 == 0 and g.is_contiguous() and g.data_ptr() % 16 == 0:
        gp = g                                       # already a legal TMA operand
    else:
        gp = _padded(B, n_top, g)
        gp[:, :n_top].copy_(g)
    gt = torch.empty(n_top, Bp, dtype=torch.float32, device=g.device)
    gp_lo = torch.empty_like(gp) if split3 else None
    gt_lo = torch.empty_like(gt) if split3 else None
    jobs.append(dict(src=gp, rows=B, cols=n_top, dst=gt, dst_lo=gt_lo, src_lo=gp_lo))
    ops.transpose_batch(jobs)
    grads_wb = [None] * (2 * nl)
    g_in = None
    for l in range(nl - 1, -1, -1):
        n_out, n_in = Ws[l].shape
        tiles = -(-n_out // 128) * -(-n_in // 128)
        splits = max(1, min(-(-B // 128), _sm_count(g.device) // tiles, 32))     # ~one CTA per SM, >= 128 batch rows per slice
        part = torch.empty(splits, n_out, ops.pad4(n_in), dtype=torch.float32, device=g.device)
        ops.gemm_tn(gt, XT[l], n_out, n_in, B, A_lo=gt_lo, B_lo=XTlo[l], C=part, split_k=splits)
        dW = torch.empty(n_out, n_in, dtype=torch.float32, device=g.device)
        db = torch.empty(n_out, dtype=torch.float32, device=g.device)
        ops.wgrad_reduce(part, n_out, n_in, dW, Gt=gt, B=B, db=db)
        grads_wb[2 * l], grads_wb[2 * l + 1] = dW, db
        if l == 0 and not need_input_grad:
            break
        nxt = _padded(B, n_in, g)
        nxt_lo = torch.empty_like(nxt) if split3 else None
        nxt_t = torch.empty(n_in, Bp, dtype=torch.float32, device=g.device) if l > 0 else None
        nxt_t_lo = torch.empty_like(nxt_t) if (split3 and l > 0) else None
        ops.gemm_tn(gp, WT[l], B, n_in, n_out, A_lo=gp_lo, B_lo=WTlo[l], C=nxt, C_lo=nxt_lo if l > 0 else None, Ct=nxt_t,
                    Ct_lo=nxt_t_lo, dact_src=acts[l - 1] if l > 0 else None, dact=act_ids[l - 1] if l > 0 else 0)
        if l == 0:
            g_in = nxt
        gp, gp_lo, gt, gt_lo = nxt, nxt_lo, nxt_t, nxt_t_lo
    return grads_wb, g_in


def _act_grad(g, a_out, act):
    """d/d(pre-activation) from the saved post-activation output (same sign for both activations): one kernel."""
    if act == L.ACT_LEAKY:
        return torch.ops.aten.leaky_relu_backward(g, a_out, 0.01, True)
    if act == L.ACT_RELU:
        return torch.ops.aten.threshold_backward(g, a_out, 0.0)
    return g


class FusedMLPFn(torch.autograd.Function):
    """apply(spec, B, n_dense, *dense_inputs, W0, b0, W1, b1, ...) -> out[, z]"""

    @staticmethod
    def forward(ctx, spec, B, n_dense, *tensors):
        ctx.set_materialize_grads(False)      # an unused output (out or z) arrives as None, not as a zero-filled tensor
        dense = tensors[:n_dense]
        wb = tensors[n_dense:]
        layers = [(wb[2 * i], wb[2 * i + 1], spec.acts[i]) for i in range(len(wb) // 2)]
        need = spec.save and any(t.requires_grad for t in tensors)
        segments = spec.build_segments(dense)
        res = ops.mlp_forward(segments, layers, B, out_ld=spec.out_ld, out_col0=spec.out_col0,
                              copy_seg=spec.copy_seg, save=need, latent=spec.latent, eps=spec.eps,
                              seed=spec.seed, offset=spec.offset, offset_dev=spec.offset_dev)
        ctx.spec, ctx.n_dense, ctx.n_layers = spec, n_dense, len(layers)
        ctx.n_out = layers[-1][0].shape[0]
        if need:
            offs, o = [], 0
            for s in segments:
                offs.append(o)
                o += s.width
            ctx.seg_off = offs
            ctx.seg_width = [s.width for s in segments]
            saved = [res["x0"]] + res["acts"] + [res["out"]] + [w for (w, _, _) in layers]
            if spec.latent:
                saved.append(res["eps"])
            ctx.save_for_backward(*saved)
        if spec.latent:
            return res["out"], res["z"]
        return res["out"]

    @staticmethod
    def backward(ctx, d_out, d_z=None):
        spec, nl = ctx.spec, ctx.n_layers
        saved = ctx.saved_tensors
        x0, acts, out = saved[0], saved[1:nl], saved[nl]
        Ws = saved[nl + 1:nl + 1 + nl]
        c0 = spec.out_col0
        g = None
        if MLP_BWD_ENGINE not in ("tc3", "tc"):
            raise ValueError("MLP_BWD_ENGINE must be 'tc3' or 'tc'")
        if spec.latent and (d_z is not None) and c0 == 0 and ctx.n_out == 2 * spec.latent:
            # [mu | logvar] block: the reparameterisation's backward and the sum with d_out in ONE kernel
            do = d_out if (d_out is None or d_out.stride(1) == 1) else d_out.contiguous()
            g = ops.reparam_bwd(do, d_z, saved[-1], out, spec.latent)
        else:
            if d_out is not None:
                g = d_out[:, c0:c0 + ctx.n_out]
            if spec.latent:
                Z = spec.latent
                if d_z is not None:
                    eps = saved[-1]
                    std = torch.exp(0.5 * out[:, c0 + Z:c0 + 2 * Z])
                    gz = torch.cat([d_z, d_z * eps * 0.5 * std], 1)
                    g = gz if g is None else g + gz
        if g is None:
            return (None,) * (3 + ctx.n_dense + 2 * nl)
        g = g.contiguous()
        g = _act_grad(g, out[:, c0:c0 + ctx.n_out], spec.acts[nl - 1])      # identity for every block of the path
        need_in = any(s[0] == "dense" and ctx.needs_input_grad[3 + s[1]] for s in spec.segs)
        grads_wb, g = _mlp_backward_tc(g, x0, acts, Ws, spec.acts, need_in, MLP_BWD_ENGINE == "tc3")
        d_dense = [None] * ctx.n_dense
        for si, s in enumerate(spec.segs):
            if s[0] == "dense" and ctx.needs_input_grad[3 + s[1]]:
                o = ctx.seg_off[si]
                d_dense[s[1]] = g[:, o:o + ctx.seg_width[si]]
        return (None, None, None, *d_dense, *grads_wb)


class CatalogCEFn(torch.autograd.Function):
    """mean_i [ logsumexp_j(mask * <q_i, w_j>) - <q_i, w_{t_i}> ] over the whole catalog
    (train_generative.py:36-42, 59) without materialising logits."""

    @staticmethod
    def forward(ctx, q, table, targets, keep_prob, bitmask, seed, offset, offset_dev=None, engine="exact"):
        ctx.set_materialize_grads(False)
        loss_rows, lse, dq = ops.ce_fwd_bwd(table, q, targets, keep_prob, bitmask, seed, offset,
                                            want_dq=q.requires_grad, offset_dev=offset_dev, engine=engine)
        ctx.M = q.shape[0]
        if dq is not None:
            ctx.save_for_backward(dq)
        ctx.mark_non_differentiable(lse)
        return loss_rows.mean(), loss_rows, lse

    @staticmethod
    def backward(ctx, g_mean, g_rows, _g_lse):
        (dq,) = ctx.saved_tensors
        d = dq * (g_mean / ctx.M) if g_mean is not None else None
        if g_rows is not None:
            d = dq * g_rows.unsqueeze(1) if d is None else d + dq * g_rows.unsqueeze(1)
        return d, None, None, None, None, None, None, None, None


class VocabParallelCEFn(torch.autograd.Function):
    """The same mean CE with the catalog sharded over the ranks of `group` (SURVEY §8e): local partial records over
    this rank's row shard, ONE all-gather of [M, 2 + D] floats, merge.  Every rank gets the full loss and the full
    d loss / d q, so the replicated MLPs see identical gradients without any further collective."""

    @staticmethod
    def forward(ctx, q, shard, full_weight, targets, group, engine="exact"):
        import torch.distributed as dist
        ctx.set_materialize_grads(False)
        rec = ops.ce_partials(shard, q, targets, engine=engine)
        world = dist.get_world_size(group)
        recs = torch.empty(world * rec.shape[0], rec.shape[1], dtype=rec.dtype, device=rec.device)
        dist.all_gather_into_tensor(recs, rec, group=group)
        recs = recs.view(world, rec.shape[0], rec.shape[1])
        loss_rows, lse, dq = ops.ce_vp_merge(recs, full_weight, q, targets, want_dq=q.requires_grad)
        ctx.M = q.shape[0]
        if dq is not None:
            ctx.save_for_backward(dq)
        ctx.mark_non_differentiable(lse)
        return loss_rows.mean(), loss_rows, lse

    @staticmethod
    def backward(ctx, g_mean, g_rows, _g_lse):
        (dq,) = ctx.saved_tensors
        d = dq * (g_mean / ctx.M) if g_mean is not None else None
        if g_rows is not None:
            d = dq * g_rows.unsqueeze(1) if d is None else d + dq * g_rows.unsqueeze(1)
        return d, None, None, None, None, None


class GatherNormFn(torch.autograd.Function):
    """x0 = [normalize(concat doc[slates]) | normalize(usr[users])] with trainable tables (the response model's
    prologue, env/response_model.py:76-83, as pretrain_env.py trains it)."""

    @staticmethod
    def forward(ctx, doc, usr, slates, users):
        x0, inv = ops.gather_norm_fwd(doc, usr, slates, users)
        ctx.save_for_backward(x0, inv, slates, users if usr is not None else slates)
        ctx.doc_shape, ctx.usr_shape = tuple(doc.shape), (tuple(usr.shape) if usr is not None else None)
        return x0

    @staticmethod
    def backward(ctx, g):
        x0, inv, slates, users = ctx.saved_tensors
        d_doc, d_usr = ops.gather_norm_bwd(g.contiguous(), x0, inv, slates, users, ctx.doc_shape, ctx.usr_shape)
        return d_doc, d_usr, None, None


class BCESigmoidFn(torch.autograd.Function):
    """nn.BCELoss()(sigmoid(pred), target) in one kernel (pretrain_env.py:57-58, 84)."""

    @staticmethod
    def forward(ctx, pred, target):
        loss, dp = ops.bce_sigmoid(pred, target, want_grad=pred.requires_grad)
        ctx.shape = pred.shape
        if dp is not None:
            ctx.save_for_backward(dp)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dp,) = ctx.saved_tensors
        return (dp * g).view(ctx.shape), None


class KLFn(torch.autograd.Function):
    """-0.5 * sum(1 + lv - plv - (exp(lv) + (mu-pmu)^2)/exp(plv))  (train_generative.py:61)."""

    @staticmethod
    def forward(ctx, mu, lv, pmu, plv):
        out, g = ops.kl_fwd_bwd(mu, lv, pmu, plv, grads=True)
        ctx.save_for_backward(*g)
        return out

    @staticmethod
    def backward(ctx, go):
        return tuple(torch._foreach_mul(list(ctx.saved_tensors), go))      # one multi-tensor launch for the four gradients


class LogitsFn(torch.autograd.Function):
    """p = q @ W^T materialised, for forward()'s API parity (pivotcvae.py:274)."""

    @staticmethod
    def forward(ctx, q, table):
        ctx.table = table
        return ops.score_logits(table, q)

    @staticmethod
    def backward(ctx, dp):
        return dp.mm(ctx.table.weight), None


class CandidateCEFn(torch.autograd.Function):
    """mean CE over per-row candidate lists (train_generative.py:52-56)."""

    @staticmethod
    def forward(ctx, q, table, candidates, target_pos):
        loss_rows, lse, dq, _ = ops.cand_ce_fwd_bwd(table, q, candidates, target_pos, want_dq=q.requires_grad)
        ctx.M = q.shape[0]
        if dq is not None:
            ctx.save_for_backward(dq)
        return loss_rows.mean()

    @staticmethod
    def backward(ctx, g):
        (dq,) = ctx.saved_tensors
        return dq * (g / ctx.M), None, None, None


class CandidateLogitsFn(torch.autograd.Function):
    """p[i, c] = <W[cand[i, c]], q_i> materialised (forward()'s candidate branch, pivotcvae.py:265-271)."""

    @staticmethod
    def forward(ctx, q, table, candidates):
        M = q.shape[0]
        tp = torch.zeros(M, dtype=torch.int64, device=q.device)
        _, _, _, p = ops.cand_ce_fwd_bwd(table, q, candidates, tp, want_dq=False, want_logits=True)
        ctx.table, ctx.cand = table, candidates
        return p

    @staticmethod
    def backward(ctx, dp):
        w = ctx.table.weight[ctx.cand.reshape(dp.shape[0], -1)]          # (M, nC, D) plain gather
        return torch.bmm(dp.unsqueeze(1), w).squeeze(1), None, None
