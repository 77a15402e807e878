"""PivotCVAE family — drop-in for the reference's models/pivotcvae.py:33-461.

Eight registry entries = 4 training-time pivot choices x 2 inference-time ones
(pivotcvae.py:10-30).  Here they are one class parameterised by two strategy
strings; the reference's class names are kept so pickles and imports resolve.

  training : 'gt'  ground-truth pivot      'max' arg-max of the PSM output
             'sample' Categorical(sigmoid(PSM . table))   'sample_gt' same around the GT row
  inference: 'max' | 'sample'
"""
import torch

from .. import _lib as L
from .cvae import BaseCVAE


class UserPivotCVAE(BaseCVAE):
    train_pick = "gt"
    infer_pick = "max"

    def __init__(self, embeddings, u_embeddings, slate_size, feature_size, latent_size, condition_size,
                 encoder_struct, psm_struct, scm_struct, prior_struct, no_user, device, fine_tune=False):
        super().__init__(embeddings, u_embeddings, slate_size, latent_size, no_user, device, False)
        ud = 0 if no_user else feature_size
        # shape contracts of pivotcvae.py:58-71
        assert encoder_struct[0] == slate_size * feature_size + condition_size + ud
        assert psm_struct[0] == latent_size + condition_size + ud
        assert psm_struct[-1] == feature_size
        assert scm_struct[0] == latent_size + condition_size + feature_size + ud
        assert scm_struct[-1] == (slate_size - 1) * feature_size
        assert prior_struct[0] == condition_size + ud
        assert condition_size == slate_size + 1, "the condition is one-hot(#clicks) of width slate_size+1 (cvae.py:90)"
        self.feature_size = feature_size
        self.condition_size = condition_size
        self.encoderStruct, self.psmStruct = encoder_struct, psm_struct
        self.scmStruct, self.priorStruct = scm_struct, prior_struct
        self.encMLP = self._build_mlp("enc", encoder_struct)
        self.encmu = torch.nn.Linear(encoder_struct[-1], latent_size)
        self.enclogvar = torch.nn.Linear(encoder_struct[-1], latent_size)
        self.psmMLP = self._build_mlp("psm", psm_struct)
        self.scmMLP = self._build_mlp("scm", scm_struct)
        self.priorMLP = self._build_mlp("prior", prior_struct)
        self.priorMu = torch.nn.Linear(prior_struct[-1], latent_size)
        self.priorLogvar = torch.nn.Linear(prior_struct[-1], latent_size)
        self.to(self.device)

    # ------------------------------------------------------------------ pivot
    def _pick_index(self, pivot_output, true_pivot):
        """-> int64 (B,) item ids (pivotcvae.py:186-195 and the variant overrides)."""
        training = true_pivot is not None and len(true_pivot) > 0
        how = self.train_pick if training else self.infer_pick
        if how == "gt":
            return true_pivot.to(self._dev(), torch.int64).reshape(-1)
        if how == "max":
            q = pivot_output
        elif how == "sample":
            q = pivot_output
        else:  # 'sample_gt': scores are taken around the ground-truth pivot's own row
            q = self.docEmbed.weight[true_pivot.to(self._dev(), torch.int64).reshape(-1)]
        q = q.detach()
        if how == "max":
            return self._select(q, "greedy")
        noise = self.noise.pop("race")
        if noise is not None:
            noise = noise.to(self._dev())
            if self._vp is not None:      # external noise is [B, N]: every shard reads its own columns
                noise = noise[:, self._vp[1]:self._vp[2]].contiguous()
            return self._select(q, "exprace", noise=noise)
        # throughput mode: the same Categorical(sigmoid(scores)) drawn exactly in O(1) per row (csrc/sampler.cu);
        # needs the whole catalog, which every vocab-parallel rank keeps anyway -> no collective
        from .. import ops
        return ops.sigmoid_categorical(self.full_table(), q, **self._stream_args(q.shape[0]))

    def pick_pivot(self, pivot_output, true_pivot=[]):
        return self.docEmbed.weight[self._pick_index(pivot_output, true_pivot)]

    # ------------------------------------------------------------------ decoder
    def _psm(self, z, cond_seg, user_seg, dense):
        """[z, c, u] -> psm_i (LeakyReLU except last) -> pivot_output (B, D); never differentiated (SURVEY F6)."""
        with torch.no_grad():
            d = [z.detach()] + [t.detach() for t in dense]
            segs = [("dense", 0), cond_seg] + ([user_seg] if user_seg is not None else [])
            layers = self._stack(self.psmMLP, L.ACT_LEAKY, L.ACT_NONE)
            return self._run_block(segs, layers, z.shape[0], dense=tuple(d))

    def _scm(self, z, cond_seg, pivot_idx, user_seg, dense):
        """[z, c, pivot, u] -> scm_i -> rx (B, L*D) with the pivot's row in slot 0 (pivotcvae.py:214-224)."""
        D, Ls = self.feature_size, self.slate_size
        segs = [("dense", 0), cond_seg, ("gather", self.docEmbed.weight, pivot_idx.reshape(-1, 1))]
        if user_seg is not None:
            segs.append(user_seg)
        layers = self._stack(self.scmMLP, L.ACT_LEAKY, L.ACT_NONE)
        return self._run_block(segs, layers, z.shape[0], dense=(z,) + tuple(dense), out_ld=Ls * D, out_col0=D,
                               copy_seg=2)

    def _decode(self, z, cond_seg, user_seg, dense, true_pivot):
        pivot_output = self._psm(z, cond_seg, user_seg, dense)
        p = self._pick_index(pivot_output, true_pivot)
        return self._scm(z, cond_seg, p, user_seg, dense)

    def decode(self, z, c, u_emb=None, true_pivot=[]):
        """P(x|z) on already-built tensors (pivotcvae.py:197-227) -> rx (B, L, D)."""
        dense = [c] + ([] if self.noUser else [u_emb])
        user_seg = None if self.noUser else ("dense", 2)
        rx = self._decode(z, ("dense", 1), user_seg, dense, true_pivot)
        return rx.view(z.shape[0], self.slate_size, self.feature_size)

    # ------------------------------------------------------------------ public paths
    def forward_latent(self, s, r, u=None):
        """forward() without the (B*L, N) logits: what the fused training loss consumes."""
        r, u, s = self._inputs(r, u, s)
        out, z = self._encode_ids(s, r, u, reparam=True)
        Z = self.latent_size
        user_seg = None if self.noUser else self._user_seg(u)
        rx = self._decode(z, ("onehot", r), user_seg, [], s[:, 0])
        return rx, z, out[:, :Z], out[:, Z:], s

    def forward(self, s, r, candidates=None, u=None):
        """-> (p, rx, z, emb, z_mu, z_logvar) as pivotcvae.py:242-276."""
        rx, z, mu, lv, s = self.forward_latent(s, r, u)
        B = s.shape[0]
        emb = self.docEmbed.weight[s.reshape(-1)].view(B, -1)  # returned for API parity only
        p = self._logits(rx.view(-1, self.feature_size), candidates)
        return p, rx.view(B, self.slate_size, self.feature_size), z, emb, mu, lv

    def _generate(self, r, u):
        """prior -> z -> PSM in one launch, pivot pick, SCM -> (prior [mu | logvar], rx (B, L*D))."""
        out, z, pivot_output = self._prior_chain(r, u, self.psmMLP)
        user_seg = None if self.noUser else self._user_seg(u)
        return out, self._scm(z, ("onehot", r), self._pick_index(pivot_output, None), user_seg, [])

    def recommend(self, r, u=None, return_item=False, random_pivot=False):
        """prior -> z -> pivot -> slate completion -> arg-max items, or rx as (B, L, D) (pivotcvae.py:278-296)."""
        res, z_mu = super().recommend(r, u, return_item)
        return (res if return_item else res.view(res.shape[0], self.slate_size, self.feature_size)), z_mu

    def log(self, logger):
        for k, v in (("feature size", self.feature_size), ("slate size", self.slate_size),
                     ("z size", self.latent_size), ("condition size", self.condition_size),
                     ("user is ignored", self.noUser), ("encoder struct", self.encoderStruct),
                     ("psm struct", self.psmStruct), ("scm struct", self.scmStruct),
                     ("prior struct", self.priorStruct), ("device", self.device),
                     ("pivot (train/infer)", "%s/%s" % (self.train_pick, self.infer_pick))):
            logger.log("\t%s: %s" % (k, v))


def _variant(name, train_pick, infer_pick):
    return type(name, (UserPivotCVAE,), {"train_pick": train_pick, "infer_pick": infer_pick,
                                         "__module__": __name__, "__qualname__": name})


UserPivotCVAE2 = _variant("UserPivotCVAE2", "max", "max")
UserPivotCVAE_PrePermute = _variant("UserPivotCVAE_PrePermute", "sample", "max")
UserPivotCVAE_PrePermute2 = _variant("UserPivotCVAE_PrePermute2", "sample_gt", "max")
UserPivotCVAE_PrePermute3 = _variant("UserPivotCVAE_PrePermute3", "gt", "sample")
UserPivotCVAE_PrePermute4 = _variant("UserPivotCVAE_PrePermute4", "max", "sample")
UserPivotCVAE_PrePermute5 = _variant("UserPivotCVAE_PrePermute5", "sample", "sample")
UserPivotCVAE_PrePermute6 = _variant("UserPivotCVAE_PrePermute6", "sample_gt", "sample")

PIVOTCVAE_MODELS = {
    "pivotcvae_gt_pi": UserPivotCVAE, "pivotcvae_pt_pi": UserPivotCVAE2,
    "pivotcvae_spt_pi": UserPivotCVAE_PrePermute, "pivotcvae_sgt_pi": UserPivotCVAE_PrePermute2,
    "pivotcvae_gt_spi": UserPivotCVAE_PrePermute3, "pivotcvae_pt_spi": UserPivotCVAE_PrePermute4,
    "pivotcvae_spt_spi": UserPivotCVAE_PrePermute5, "pivotcvae_sgt_spi": UserPivotCVAE_PrePermute6,
}
