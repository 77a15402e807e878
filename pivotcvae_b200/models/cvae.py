"""BaseCVAE — drop-in for the reference's models/cvae.py:7-118, running on libpcv_b200.

Same constructor, attributes (docEmbed, userEmbed, slate_size, latent_size,
noUser, device, candidateFlag) and methods (reparametrize, get_condition,
get_recommended_item, sample_encoding); the arithmetic is the sm_100a kernels.
"""
import torch
from torch import nn

from .. import _lib as L
from .. import ops
from ..autograd import FusedMLPFn, MlpSpec
from ..noise import NoiseSource


def with_mlp_engine(fn):
    """Run a method under the object's `mlp_engine` ("exact" / "tc"; None = the process default ops.MLP_ENGINE)."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        eng = getattr(self, "mlp_engine", None)
        if eng is None:
            return fn(self, *a, **k)
        with ops.mlp_engine(eng):
            return fn(self, *a, **k)
    return wrapper


def _require_cuda(device):
    dev = torch.device(device)
    if dev.type != "cuda":
        raise L.PcvError("pivotcvae_b200 models run on a B200 only (device=%r); there is no CPU path" % (device,))
    return dev


class BaseCVAE(nn.Module):
    # inference engine of the fused MLP blocks in recommend(): None = ops.MLP_ENGINE (default "exact": the FFMA engines,
    # bit-identical to the CPU oracle); "tc" = tcgen05 3xTF32 (csrc/mlp_tc.cu), fp32-grade, several times faster
    mlp_engine = None

    def __init__(self, embeddings, u_embeddings, slate_size, latent_size, no_user, device, fine_tune=False):
        super().__init__()
        self.candidateFlag = False
        self.slate_size = slate_size
        self.latent_size = latent_size
        self.noUser = no_user
        self.device = device
        dev = _require_cuda(device)
        # row-L2-normalised copies of the pretrained tables (cvae.py:27-41); fine_tune=True trains both with the rest of
        # the model (the CE's table gradient is pcv_ce_table_grad, the MLP gathers scatter theirs)
        with torch.no_grad():
            src = embeddings.weight.detach().to(dev, torch.float32)
            self.docEmbed = nn.Embedding(src.shape[0], src.shape[1], device=dev)
            self.docEmbed.weight.data.copy_(ops.normalize_rows(src))
            self.docEmbed.weight.requires_grad = fine_tune
            if not no_user:
                usrc = u_embeddings.weight.detach().to(dev, torch.float32)
                self.userEmbed = nn.Embedding(usrc.shape[0], usrc.shape[1], device=dev)
                self.userEmbed.weight.data.copy_(ops.normalize_rows(usrc))
                self.userEmbed.weight.requires_grad = fine_tune
        self.noise = NoiseSource()
        self.select_engine = "auto"
        self.ce_engine = "exact"   # "tf32": full-catalog CE logits and gradient on the tensor cores, D = 8..128 (reduced-precision tolerance)
        # Opt-in extension, OFF by default because the reference has no such logic (SURVEY F1: cvae.py:97-101 picks
        # every slot independently, duplicates allowed).  True: a slot never repeats an item an earlier slot of
        # the same slate took (sequential arg-max without replacement; include/pcv_b200.h pcv_slate_no_repeat).
        self.no_repeat = False
        self._table = None
        self._full = None    # full-catalog handle while vocab-parallel (the sampler draws over every row)
        self._vp = None      # vocab-parallel state: (group, lo, hi) once enable_vocab_parallel() is called
        self._vp_train = False   # enable_vocab_parallel(train_tables=True): the tables train on the sharded catalog
        self._vp_hooks = []      # their row-exchange hooks (removable handles)

    # ---- extension state is rebuilt lazily (whole-model pickling, train_generative.py:199)
    def __getstate__(self):
        st = self.__dict__.copy()
        st["_table"] = None
        st["_full"] = None
        st["_vp"] = None
        st["_vp_train"] = False
        st["_vp_hooks"] = []
        st.pop("_rows", None)
        st.pop("_head_cache", None)
        return st

    # ---- vocab-parallel scoring (SURVEY §8e): every rank keeps the full fp32 table (<= 320 MB) for the
    # gathers, but scores only its own 128-aligned row shard; one all-gather of (val, idx) per scoring step
    def enable_vocab_parallel(self, group=None, shard_rows=True, train_tables=False):
        """Score against this rank's row shard of the catalog only.  shard_rows (default): in recommend() the MLP
        blocks run on this rank's 1/world slice of the batch instead of redundantly on all of it, and the
        queries are all-gathered before every sharded scoring step (a few hundred KB over NVLink).

        train_tables: required when the tables are trainable (fine_tune=True).  The catalog cross-entropy's table
        gradient is then computed for this rank's rows only, and after every backward a hook on each trainable table
        all-gathers each rank's own rows of its .grad (parallel.exchange_owned_rows: N * D * 4 bytes per table), so
        that every rank holds the same full gradient and the replicated tables take identical optimizer steps."""
        import torch.distributed as dist
        from ..parallel import exchange_owned_rows, shard_bounds
        tabs = self.trainable_tables()
        if tabs and not train_tables:
            raise L.PcvError("enable_vocab_parallel: the embedding tables are trainable (fine_tune=True); pass "
                             "train_tables=True to train them on the sharded catalog")
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        lo, hi = shard_bounds(self.docEmbed.weight.shape[0], world, rank)
        self._vp = (group, lo, hi)
        self._vp_rows = bool(shard_rows)
        self._vp_train = bool(train_tables)
        self._table = None
        for h in getattr(self, "_vp_hooks", ()):     # a second call replaces the hooks of the first
            h.remove()
        self._vp_hooks = []
        if train_tables:
            for w in tabs:
                self._vp_hooks.append(w.register_post_accumulate_grad_hook(
                    lambda p: exchange_owned_rows(p.grad, group)))

    def trainable_tables(self):
        """The embedding tables that require grad (fine_tune=True)."""
        tabs = [self.docEmbed.weight] + ([] if self.noUser else [self.userEmbed.weight])
        return [w for w in tabs if w.requires_grad]

    def _vp_row_slice(self, B):
        """(world, first row, rows per rank) when recommend() may shard its MLP rows over the vocab-parallel group:
        throughput mode only (queued parity-mode noise tensors address the whole batch) and an evenly split batch."""
        if self._vp is None or not getattr(self, "_vp_rows", False):
            return None
        if any(self.noise._queue[k] for k in ("eps", "race")):
            return None
        import torch.distributed as dist
        world, rank = dist.get_world_size(self._vp[0]), dist.get_rank(self._vp[0])
        if world == 1 or B % world:
            return None
        return world, rank * (B // world), B // world

    def _stream_args(self, rows):
        """Philox rows of one op.  While the MLP rows are sharded, every rank reserves the rows of the WHOLE batch and
        draws those of its own slice, so the noise is exactly that of the unsharded run."""
        sl = getattr(self, "_rows", None)
        if sl is None:
            return self.noise.stream_args(rows)
        kw = self.noise.stream_args(sl[1])
        kw["offset"] += sl[0]
        return kw

    def _select(self, q, mode="greedy", **kw):
        """score+select over the (possibly sharded) catalog -> global item ids int64 (rows,).  While recommend() shards
        the MLP rows (self._rows), each rank's rows are scored against the whole catalog, which every rank keeps anyway
        (<= 320 MB), so the pick needs no exchange."""
        engine = self.select_engine if mode == "greedy" else "auto"
        if self._vp is None or getattr(self, "_rows", None) is not None:
            return ops.score_select(self.full_table(), q, mode, engine=engine, want_val=False, **kw)[0]
        from ..parallel import VocabParallelSelector
        local = lambda x: ops.score_select(self.item_table(), x, mode, engine=engine, **kw)
        return VocabParallelSelector(local, self._vp[0])(q)[0]

    def _apply(self, fn, *a, **k):
        self._table = None
        self._full = None
        return super()._apply(fn, *a, **k)

    def full_table(self):
        """Handle over the WHOLE catalog (== item_table() unless vocab-parallel)."""
        if self._vp is None:
            return self.item_table()
        w = self.docEmbed.weight
        t = getattr(self, "_full", None)
        if t is None or t.weight.data_ptr() != w.data_ptr() or t.weight.shape != w.shape:
            t = ops.Table(w.detach())
            t.version = w._version
            self._full = t
        elif t.version != w._version:   # updated in place (an optimizer step): refresh the handle on the stream
            t.refresh()
            t.version = w._version
        return t

    def item_table(self):
        w = self.docEmbed.weight
        t = self._table
        if self._vp is not None:
            _, lo, hi = self._vp
            if (t is None or t.row_offset != lo or t.n_rows != hi - lo or t.weight.data_ptr() != w[lo:hi].data_ptr()
                    or t.dim != w.shape[1]):
                t = ops.Table(w.detach()[lo:hi], row_offset=lo)
                t.version = w._version
                self._table = t
            elif t.version != w._version:
                t.refresh()
                t.version = w._version
            return t
        if t is None or t.weight.data_ptr() != w.data_ptr() or t.weight.shape != w.shape:
            t = ops.Table(w.detach())
            t.version = w._version
            self._table = t
        elif t.version != w._version:   # updated in place (an optimizer step): refresh the handle on the stream
            t.refresh()
            t.version = w._version
        return t

    # ---- helpers shared by the subclasses
    @staticmethod
    def _stack(mods, hidden_act, last_act):
        """[(W, b, act)] for a list of nn.Linear."""
        n = len(mods)
        return [(m.weight, m.bias, hidden_act if i < n - 1 else last_act) for i, m in enumerate(mods)]

    def _heads(self, mu_lin, lv_lin):
        """The two latent heads as ONE linear layer emitting [mu | logvar].  Under no_grad the
        concatenation is cached until one of the four parameters changes (in-place updates bump
        `_version`); with autograd on it is rebuilt so the gradient splits back onto the heads."""
        if torch.is_grad_enabled():
            return torch.cat([mu_lin.weight, lv_lin.weight], 0), torch.cat([mu_lin.bias, lv_lin.bias], 0)
        key = (id(mu_lin), mu_lin.weight.data_ptr(), lv_lin.weight.data_ptr(), mu_lin.weight._version,
               lv_lin.weight._version, mu_lin.bias._version, lv_lin.bias._version)
        cache = self.__dict__.setdefault("_head_cache", {})
        hit = cache.get(id(mu_lin))
        if hit is None or hit[0] != key:
            hit = (key, torch.cat([mu_lin.weight, lv_lin.weight], 0).detach(),
                   torch.cat([mu_lin.bias, lv_lin.bias], 0).detach())
            cache[id(mu_lin)] = hit
        return hit[1], hit[2]

    def _run_block(self, segs, layers, B, dense=(), **kw):
        """One fused MLP block; differentiable when grad mode is on."""
        spec = MlpSpec(segs, [a for (_, _, a) in layers], save=torch.is_grad_enabled(), train_tables=True, **kw)
        flat = []
        for (W, b, _) in layers:
            flat += [W, b]
        tables = [segs[i][1] for i in spec.train_segs]          # fine_tune: gather tables that get a gradient
        return FusedMLPFn.apply(spec, B, len(dense), *dense, *flat, *tables)

    def _user_seg(self, u):
        return ("gather", self.userEmbed.weight, u.reshape(-1, 1))

    def _eps_args(self, B):
        eps = self.noise.pop("eps")
        if eps is not None:
            return dict(eps=eps.to(self.docEmbed.weight.device))
        return self._stream_args(B)

    # ---- reference API
    def reparametrize(self, mu, logvar):
        """z = eps * exp(0.5*logvar) + mu (cvae.py:79-83); eps from the model's NoiseSource.
        Runs the kernel's reparameterisation epilogue behind an identity layer."""
        B, Z = mu.shape
        x = torch.cat([mu, logvar], 1)
        eye = torch.eye(2 * Z, device=x.device)
        _, z = self._run_block([("dense", 0)], [(eye, torch.zeros(2 * Z, device=x.device), L.ACT_NONE)], B,
                               dense=(x,), latent=Z, **self._eps_args(B))
        return z

    def get_condition(self, r):
        """one-hot of the number of clicks (cvae.py:85-92)."""
        r = r.to(self.docEmbed.weight.device, torch.float32)
        B, Ls = r.shape
        eye = torch.eye(Ls + 1, device=r.device)
        res = ops.mlp_forward([ops.OneHot(r)], [(eye, torch.zeros(Ls + 1, device=r.device), L.ACT_NONE)], B)
        return res["out"]

    def get_recommended_item(self, embeddings):
        """arg-max item per row over the whole catalog (cvae.py:97-101) -> int64 (rows,)."""
        q = embeddings.reshape(-1, self.feature_size)
        q = q.detach()
        if getattr(self, "no_repeat", False):
            if q.shape[0] % self.slate_size:
                raise L.PcvError("no_repeat: rows must be whole slates (multiple of slate_size)")
            if self._vp is None:
                return ops.score_select(self.item_table(), q, "greedy", engine=self.select_engine, want_val=False,
                                        no_repeat=self.slate_size)[0]
            # vocab-parallel: sharded top-1, then this shard's top-L lists of the duplicate-holding slates, one
            # all-gather of them and the same merge on every rank
            from ..parallel import no_repeat_exchange
            table, Ls = self.item_table(), self.slate_size
            items = self._select(q, "greedy")
            return no_repeat_exchange(lambda it: ops.slate_no_repeat_partials(table, q, it, Ls), items, Ls, self._vp[0])
        return self._select(q, "greedy")

    @with_mlp_engine
    def recommend(self, r, u=None, return_item=False):
        """prior -> z -> decoder (_generate) -> per-slot arg-max items, or the flat (B, L*D) slate features; and z_mu.
        Vocab-parallel with shard_rows, this rank runs _generate on its B/world rows and ONE all-gather carries
        [rx | z_mu] of every rank; the per-slot scoring then is the catalog-sharded select of _select()."""
        with torch.no_grad():
            r, u, _ = self._inputs(r, u)
            B = r.shape[0]
            sl = self._vp_row_slice(B)
            if sl is not None:
                _, r0, per = sl
                r, u = r[r0:r0 + per], None if u is None else u[r0:r0 + per]
                self._rows = (r0, B)
            try:
                out, rx = self._generate(r, u)
            finally:
                self._rows = None
            z_mu = out[:, :self.latent_size]
            if sl is not None:
                from ..parallel import all_gather_rows
                both = all_gather_rows(torch.cat([rx, z_mu], 1), self._vp[0])       # [B, L * D + Z]
                rx, z_mu = both[:, :rx.shape[1]].contiguous(), both[:, rx.shape[1]:]
            res = self.get_recommended_item(rx) if return_item else rx
            self.noise.flush_eager()
            return res, z_mu

    def sample_encoding(self, s, r, u=None):
        """encoder only (cvae.py:103-115) -> (z_mu, z_logvar)."""
        out = self._encode_ids(s, r, u)
        Z = self.latent_size
        return out[:, :Z], out[:, Z:]

    # ---- fused blocks shared by PivotCVAE and ListCVAE ----------------------
    def _dev(self):
        return self.docEmbed.weight.device

    def _inputs(self, r=None, u=None, s=None):
        dev = self._dev()
        if r is not None:
            r = r.to(dev, torch.float32)
        if u is not None:
            u = u.to(dev, torch.int64).reshape(-1)
        if s is not None:
            s = s.to(dev, torch.int64)
        return r, u, s

    def _build_mlp(self, prefix, struct):
        """nn.Linear chain registered as <prefix>_1.. (same names/init as the reference,
        pivotcvae.py:108-113) so reference state_dicts load."""
        mods = []
        for i in range(len(struct) - 1):
            m = nn.Linear(struct[i], struct[i + 1])
            nn.init.kaiming_uniform_(m.weight)
            self.add_module("%s_%d" % (prefix, i + 1), m)
            mods.append(m)
        return mods

    def _prior_block(self, r, u, reparam):
        """[onehot(r), user] -> prior_i (LeakyReLU each) -> [mu | logvar] (+ z).
        pivotcvae.py:229-240 / 279-290, listcvae.py:121-132 / 171-182."""
        segs = [("onehot", r)] + ([] if self.noUser else [self._user_seg(u)])
        layers = self._stack(self.priorMLP, L.ACT_LEAKY, L.ACT_LEAKY)
        hw, hb = self._heads(self.priorMu, self.priorLogvar)
        layers.append((hw, hb, L.ACT_NONE))
        B = r.shape[0]
        if reparam:
            return self._run_block(segs, layers, B, latent=self.latent_size, **self._eps_args(B))
        return self._run_block(segs, layers, B), None

    def _prior_chain(self, r, u, next_mods, last_act=L.ACT_NONE):
        """Inference only: prior block (+ reparameterisation) and the block that consumes z
        ([z, onehot(r), user] -> next_mods) in ONE kernel launch.  -> (mu|logvar, z, next block's output)"""
        B = r.shape[0]
        cond = ops.OneHot(r)
        user = [] if self.noUser else [ops.Gather(self.userEmbed.weight.detach(), u.reshape(-1, 1))]
        layers = [(w.detach(), b.detach(), a) for (w, b, a) in self._stack(self.priorMLP, L.ACT_LEAKY, L.ACT_LEAKY)]
        hw, hb = self._heads(self.priorMu, self.priorLogvar)
        layers.append((hw.detach(), hb.detach(), L.ACT_NONE))
        first = ([cond] + user, layers, dict(latent=self.latent_size, **self._eps_args(B)))
        nxt = [(w.detach(), b.detach(), a) for (w, b, a) in self._stack(next_mods, L.ACT_LEAKY, last_act)]

        def second(res):
            return [ops.Dense(res["z"]), cond] + user, nxt, {}

        ra, rb = ops.mlp_forward_chain(first, second, B)
        return ra["out"], ra["z"], rb["out"]

    def _encode_ids(self, s, r, u, reparam=False):
        """[docEmbed(s), onehot(r), user] -> enc_i (LeakyReLU each) -> [mu | logvar] (+ z).
        pivotcvae.py:250-260, 159-174."""
        r, u, s = self._inputs(r, u, s)
        segs = [("gather", self.docEmbed.weight, s), ("onehot", r)] + ([] if self.noUser else [self._user_seg(u)])
        layers = self._stack(self.encMLP, L.ACT_LEAKY, L.ACT_LEAKY)
        hw, hb = self._heads(self.encmu, self.enclogvar)
        layers.append((hw, hb, L.ACT_NONE))
        B = s.shape[0]
        if reparam:
            return self._run_block(segs, layers, B, latent=self.latent_size, **self._eps_args(B))
        return self._run_block(segs, layers, B)

    def encode(self, emb, c, u_emb=None):
        """Q(z|s) on already-gathered tensors (pivotcvae.py:159-174) -> (z_mu, z_logvar)."""
        dense = [emb, c] + ([] if self.noUser else [u_emb])
        segs = [("dense", i) for i in range(len(dense))]
        layers = self._stack(self.encMLP, L.ACT_LEAKY, L.ACT_LEAKY)
        hw, hb = self._heads(self.encmu, self.enclogvar)
        layers.append((hw, hb, L.ACT_NONE))
        out = self._run_block(segs, layers, emb.shape[0], dense=tuple(dense))
        Z = self.latent_size
        return out[:, :Z], out[:, Z:]

    def get_prior(self, r, u=None):
        r, u, _ = self._inputs(r, u)
        out, _ = self._prior_block(r, u, reparam=False)
        Z = self.latent_size
        return out[:, :Z], out[:, Z:]

    def _logits(self, rx_flat, candidates=None):
        """forward()'s `p`: scores against the whole table, or (candidateFlag) against the per-slot
        candidate lists (B, L, nC) as pivotcvae.py:265-271 does with gather + bmm."""
        from ..autograd import CandidateLogitsFn, LogitsFn
        if self.candidateFlag:
            cand = candidates.to(self._dev(), torch.int64).reshape(rx_flat.shape[0], -1)
            return CandidateLogitsFn.apply(rx_flat, self.item_table(), cand, self.docEmbed.weight)
        return LogitsFn.apply(rx_flat, self.item_table(), self.docEmbed.weight)
