"""ListCVAE with a learned prior — drop-in for the reference's models/listcvae.py:8-199.

Same as PivotCVAE minus the pivot: one decoder MLP emits all L*D slate features.
"""
import torch

from .. import _lib as L
from .cvae import BaseCVAE


class UserListCVAEWithPrior(BaseCVAE):
    def __init__(self, embeddings, u_embeddings, slate_size, feature_size, latent_size, condition_size,
                 encoder_struct, decoder_struct, prior_struct, no_user, device, fine_tune=False):
        super().__init__(embeddings, u_embeddings, slate_size, latent_size, no_user, device, fine_tune)
        ud = 0 if no_user else feature_size
        # shape contracts of listcvae.py:35-44
        assert encoder_struct[0] == slate_size * feature_size + condition_size + ud
        assert decoder_struct[0] == latent_size + condition_size + ud
        assert decoder_struct[-1] == slate_size * feature_size
        assert prior_struct[0] == condition_size + ud
        assert condition_size == slate_size + 1
        self.feature_size = feature_size
        self.condition_size = condition_size
        self.encoderStruct, self.decoderStruct, self.priorStruct = encoder_struct, decoder_struct, prior_struct
        self.encMLP = self._build_mlp("enc", encoder_struct)
        self.encmu = torch.nn.Linear(encoder_struct[-1], latent_size)
        self.enclogvar = torch.nn.Linear(encoder_struct[-1], latent_size)
        self.decMLP = self._build_mlp("dec", decoder_struct)
        self.priorMLP = self._build_mlp("prior", prior_struct)
        self.priorMu = torch.nn.Linear(prior_struct[-1], latent_size)
        self.priorLogvar = torch.nn.Linear(prior_struct[-1], latent_size)
        self.to(self.device)

    def _decode(self, z, cond_seg, user_seg, dense):
        """[z, c, u] -> dec_i (LeakyReLU except last) -> (B, L*D)  (listcvae.py:106-119)."""
        segs = [("dense", 0), cond_seg] + ([user_seg] if user_seg is not None else [])
        layers = self._stack(self.decMLP, L.ACT_LEAKY, L.ACT_NONE)
        return self._run_block(segs, layers, z.shape[0], dense=(z,) + tuple(dense))

    def decode(self, z, c, u_emb=None):
        dense = [c] + ([] if self.noUser else [u_emb])
        return self._decode(z, ("dense", 1), None if self.noUser else ("dense", 2), dense)

    def forward_latent(self, s, r, u=None):
        r, u, s = self._inputs(r, u, s)
        out, z = self._encode_ids(s, r, u, reparam=True)
        Z = self.latent_size
        rx = self._decode(z, ("onehot", r), None if self.noUser else self._user_seg(u), [])
        return rx, z, out[:, :Z], out[:, Z:], s

    def forward(self, s, r, candidates=None, u=None):
        """-> (p, rx, z, emb, z_mu, z_logvar) as listcvae.py:134-168 (rx stays (B, L*D) there)."""
        rx, z, mu, lv, s = self.forward_latent(s, r, u)
        emb = self.docEmbed.weight[s.reshape(-1)].view(s.shape[0], -1)  # returned for API parity only
        p = self._logits(rx.view(-1, self.feature_size), candidates)
        return p, rx, z, emb, mu, lv

    def _generate(self, r, u):
        """prior -> z -> decoder in one launch -> (prior [mu | logvar], rx (B, L*D)); recommend() is listcvae.py:170-188."""
        out, _, rx = self._prior_chain(r, u, self.decMLP)
        return out, rx

    def log(self, logger):
        for k, v in (("feature size", self.feature_size), ("slate size", self.slate_size),
                     ("z size", self.latent_size), ("condition size", self.condition_size),
                     ("user is ignored", self.noUser), ("encoder struct", self.encoderStruct),
                     ("decoder struct", self.decoderStruct), ("prior struct", self.priorStruct),
                     ("device", self.device)):
            logger.log("\t%s: %s" % (k, v))
