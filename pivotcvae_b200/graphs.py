"""CUDA-graph capture of the slate-generation step (launch-bound inner loop -> one graph launch).

GraphedSlateGenerator captures `model.recommend(ctx, users, return_item=True)` followed by the
response model's score of the generated slates into ONE CUDA graph over static buffers.  Random
draws stay fresh on every replay: the Philox row counter lives in device memory
(pcv_*.offset_dev) and the last node of the graph advances it (pcv_counter_add).

The graph reads the MLP weights through the pre-tiled copies of the packed engine (ops.packed_weight)
and the concatenated latent heads, i.e. it SNAPSHOTS the weights at capture time: build a new
generator after the model has been trained further.
"""
import torch

from . import ops


class GraphedSlateGenerator:
    def __init__(self, model, env, batch, warmup=3):
        dev = model.docEmbed.weight.device
        self.model, self.env, self.batch = model, env, batch
        L = model.slate_size
        self.ctx = torch.zeros(batch, L, device=dev)
        self.users = torch.zeros(batch, dtype=torch.int64, device=dev)
        self.no_user = model.noUser
        model.noise.begin_graph(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):     # builds the table handle, workspaces, smem attributes
                self._step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        l0 = ops.launch_count()
        with torch.cuda.graph(self.graph):
            self.items, self.z_mu, self.resp = self._step()
        self.launches_per_step = ops.launch_count() - l0
        model.item_table().pin_workspaces()     # their pointers are baked into the graph
        if getattr(model, "_vp", None) is not None:
            model.full_table().pin_workspaces()  # vocab-parallel: the row-parallel pivot pick scores the whole catalog
        ops.pin_packed()

    def _step(self):
        items, z_mu = self.model.recommend(self.ctx, None if self.no_user else self.users, return_item=True)
        sl = self.model._vp_row_slice(self.batch)
        if sl is not None:      # vocab-parallel: the response model scores this rank's slates only, one all-gather
            from .parallel import all_gather_rows
            _, r0, per = sl
            resp = all_gather_rows(self.env(items.view(self.batch, -1)[r0:r0 + per], self.users[r0:r0 + per]),
                                   self.model._vp[0])
        else:
            resp = self.env(items.view(self.batch, -1), self.users)
        self.model.noise.end_graph_step()
        return items, z_mu, resp

    def load_inputs(self, ctx, users=None):
        self.ctx.copy_(ctx, non_blocking=True)
        if users is not None:
            self.users.copy_(users, non_blocking=True)

    def replay(self):
        self.graph.replay()
        return self.items, self.resp

    def __call__(self, ctx, users=None):
        """-> (items int64[B*L], resp f32[B, L]) in static buffers (overwritten by the next call)."""
        self.load_inputs(ctx, users)
        return self.replay()


class GraphedTrainStep:
    """One training step (get_gen_loss -> backward -> Adam.step, train_generative.py:124-134)
    captured as ONE CUDA graph over static batch buffers.  The optimizer must be built with
    capturable=True.  Philox masks / eps stay fresh per replay (device-side counter).

    train_tables=True captures a fine_tune step too (trainable docEmbed / userEmbed): the step ends by refreshing the
    item-table handle in place (pcv_table_refresh) after the optimizer has updated docEmbed, so the next replay's
    cross-entropy reads packed images and a max|w| that match the table.  userEmbed has no handle: only the fused MLP
    gathers read it."""

    def __init__(self, model, optimizer, batch, beta, n_neg, warmup=3, train_tables=False):
        from . import _lib
        from .train_generative import get_gen_loss
        trainable = any(getattr(model, k).weight.requires_grad for k in ("docEmbed", "userEmbed") if hasattr(model, k))
        if trainable and not train_tables:
            raise _lib.PcvError("GraphedTrainStep: the embedding tables are trainable (fine_tune=True); pass "
                                "train_tables=True to capture a step that refreshes the item-table handle after every "
                                "optimizer step, or train with fine_tune eagerly.")
        dev = model.docEmbed.weight.device
        L = model.slate_size
        self.model, self.opt = model, optimizer
        self.static = {"slates": torch.zeros(batch, L, dtype=torch.int64, device=dev),
                       "users": torch.zeros(batch, 1, dtype=torch.int64, device=dev),
                       "responses": torch.zeros(batch, L, device=dev)}

        # the one handle every replay reads (and refreshes); kept alive with the graph that baked its pointers in
        self._table = model.item_table() if trainable else None

        def step():
            optimizer.zero_grad(set_to_none=True)
            loss, rec, kld = get_gen_loss(self.static, model, None, beta, n_neg=n_neg)
            loss.backward()
            optimizer.step()
            if self._table is not None:     # docEmbed moved in place: bring the handle along, once per step
                self._table.refresh()
                self._mark_current()
            model.noise.end_graph_step()
            return loss.detach(), rec.detach(), kld.detach()

        self._step = step
        self._params = [p for p in model.parameters() if p.requires_grad]
        # the warm-up runs real Adam updates on the (all-zero) static batch: snapshot the parameters and the
        # optimizer state first and put them back IN PLACE afterwards (pointers must not move before capture)
        with torch.no_grad():
            snap_p = [p.detach().clone() for p in self._params]
            snap_s = [{k: v.clone() for k, v in optimizer.state.get(p, {}).items() if torch.is_tensor(v)}
                      for p in self._params]
        model.noise.begin_graph(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                step()
            with torch.no_grad():
                for p, sp, ss in zip(self._params, snap_p, snap_s):
                    p.copy_(sp)
                    for k, v in optimizer.state.get(p, {}).items():
                        if torch.is_tensor(v):
                            v.copy_(ss[k]) if k in ss else v.zero_()   # state created by the warm-up starts at zero
            if self._table is not None:     # the restore changed docEmbed in place: the first replay reads the handle
                self._table.refresh()
                self._mark_current()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        l0 = ops.launch_count()
        with torch.cuda.graph(self.graph):
            self.loss, self.rec, self.kld = step()
        self.launches_per_step = ops.launch_count() - l0
        model.item_table().pin_workspaces()
        ops.pin_packed()

    def _mark_current(self):
        """The handle matches docEmbed as it is now: item_table() must not refresh it again."""
        self._table.version = self.model.docEmbed.weight._version

    def __call__(self, batch):
        if self._table is not None and self._table is not self.model.item_table():
            raise RuntimeError("GraphedTrainStep: docEmbed was re-allocated or reshaped since the capture; build a new step")
        for k, v in self.static.items():
            v.copy_(batch[k].reshape(v.shape), non_blocking=True)
        self.graph.replay()
        # the replayed optimizer step changed the parameters behind autograd's back: advance their version
        # counters so every cache keyed on them (packed weights, concatenated heads) refreshes on next use
        for p in self._params:
            torch.autograd.graph.increment_version(p)
        if self._table is not None:     # ... except the item-table handle: the replay's last node refreshed it
            self._mark_current()
        return self.loss, self.rec, self.kld
