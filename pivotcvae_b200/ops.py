"""Torch-facing wrappers of the C ABI: tensors in, tensors out, current CUDA stream.

torch is plumbing here (device memory, streams, autograd bookkeeping); all the
arithmetic of the hot path happens in libpcv_b200.so.  Every function raises if
handed a non-CUDA tensor — there is no fallback.
"""
import collections
import ctypes

import torch

from . import _lib as L


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class KernelTimer:
    """CUDA-event timing of individual library calls on the launching stream
    (bench.py's roofline leg).  Usage: with ops.KernelTimer() as kt: ...; kt.summary()."""

    active = None

    def __init__(self):
        self.events = []

    def __enter__(self):
        KernelTimer.active = self
        return self

    def __exit__(self, *exc):
        KernelTimer.active = None

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.events:
            tot, n = out.get(name, (0.0, 0))
            out[name] = (tot + a.elapsed_time(b), n + 1)
        return {k: {"ms_total": v[0], "calls": v[1], "ms_avg": v[0] / v[1]} for k, v in out.items()}


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        kt = KernelTimer.active
        if kt is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        kt = KernelTimer.active
        if kt is not None:
            self.b.record()
            kt.events.append((self.name, self.a, self.b))


def _req(t, dtype, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise L.PcvError("%s must be a CUDA tensor (libpcv_b200 has no CPU path)" % name)
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def _f32(t, name="tensor"):
    return _req(t, torch.float32, name)


def _i64(t, name="index tensor"):
    return _req(t, torch.int64, name)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def launch_count():
    return int(L.load().pcv_launch_count())


def device_ok(device=None):
    dev = torch.cuda.current_device() if device is None else torch.device(device).index or 0
    L.check(L.load().pcv_device_ok(dev), "pcv_device_ok")
    return True


# ----------------------------------------------------------------------------
# item table handle
# ----------------------------------------------------------------------------
class Table:
    """Borrowed view of the item table (cvae.py:30-32) + cached workspaces.  The handle derives packed images and
    max|w| from the weight's values: after an in-place update call refresh(); re-create it when the weight moves."""

    def __init__(self, weight, row_offset=0):
        self.weight = _f32(weight, "item table")
        if self.weight.dim() != 2:
            raise L.PcvError("item table must be 2-D")
        self.n_rows, self.dim = self.weight.shape
        self.row_offset = int(row_offset)
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.weight.device):
            L.check(L.load().pcv_table_create(_ptr(self.weight), self.n_rows, self.dim, self.row_offset,
                                              ctypes.byref(self._h)), "pcv_table_create")
        self._ws = collections.OrderedDict()
        self.version = None     # set by the owner: version counter of the weight the handle snapshotted

    def __del__(self):
        try:
            if self._h:
                L.load().pcv_table_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def refresh(self):
        """Bring the handle up to date with an in-place update of the weight (same storage and shape), on the current
        stream: no allocation and no host sync, so a CUDA graph may capture it.  The object, its workspaces and their
        pins stay."""
        with torch.cuda.device(self.weight.device):
            L.check(L.load().pcv_table_refresh(self._h, _stream()), "pcv_table_refresh")

    def workspace(self, kind, M):
        key = (kind, int(M))
        ws = self._ws.get(key)
        if ws is not None:
            self._ws.move_to_end(key)
        if ws is None:
            n = ctypes.c_size_t()
            lib = L.load()
            fns = {"select": [lib.pcv_score_select_workspace_bytes], "ce": [lib.pcv_ce_workspace_bytes],
                   "topk": [lib.pcv_score_topk_workspace_bytes],
                   # table gradient: the dense-mask query, the largest of the mask modes (row-split partials >= gap table)
                   "ce_tgrad": [lambda h, m, out: lib.pcv_ce_table_grad_workspace_bytes(h, m, ctypes.byref(L.CeMask(1.0)), out)],
                   # no-repeat select: the top-1 workspace followed by the top-k one (include/pcv_b200.h)
                   "select_nr": [lib.pcv_score_select_workspace_bytes, lib.pcv_score_topk_workspace_bytes]}[kind]
            total = 0
            for fn in fns:
                L.check(fn(self._h, int(M), ctypes.byref(n)), "workspace query")
                total += int(n.value)
            n = ctypes.c_size_t(total)
            ws = torch.zeros(max(int(n.value), 256), dtype=torch.uint8, device=self.weight.device)  # zero-filled once (ABI contract)
            # least-recently-used eviction, one entry at a time; a workspace whose pointer a live CUDA graph
            # baked in is pinned by that graph object (pin_workspaces) and is never dropped
            while len(self._ws) >= self.WS_MAX:
                victim = next((k for k in self._ws if k not in self._pinned), None)
                if victim is None:
                    break
                del self._ws[victim]
            self._ws[key] = ws
        return ws

    WS_MAX = 16
    _pinned = frozenset()

    def pin_workspaces(self):
        """Called by the Graphed* objects after capture: every workspace allocated so far stays alive
        (and is never evicted) for the lifetime of this table handle."""
        self._pinned = frozenset(self._pinned | set(self._ws))


def normalize_rows(W):
    W = _f32(W, "W")
    out = torch.empty_like(W)
    with torch.cuda.device(W.device):
        L.check(L.load().pcv_normalize_rows(_ptr(W), W.shape[0], W.shape[1], _ptr(out), _stream()), "pcv_normalize_rows")
    return out


# ----------------------------------------------------------------------------
# score + select
# ----------------------------------------------------------------------------
def counter_add(counter, inc):
    """counter (int64[1] CUDA tensor) += inc on the current stream (Philox row counter of graph replays)."""
    with torch.cuda.device(counter.device):
        L.check(L.load().pcv_counter_add(_ptr(counter), int(inc), _stream()), "pcv_counter_add")


def score_select(table, Q, mode="greedy", noise=None, engine="auto", want_val=True, no_repeat=0):
    """-> (idx int64[M], val f32[M]).  mode 'greedy' | 'exprace' (needs noise: [M, n_rows] Exp(1) draws).  no_repeat=L
    (opt-in, NOT reference behaviour): rows are the L slots of M/L slates; a slot never repeats an item an earlier slot
    of its slate took."""
    Q = _f32(Q, "Q")
    M, D = Q.shape
    if D != table.dim:
        raise L.PcvError("Q has dim %d, table has dim %d" % (D, table.dim))
    opts = L.SelectOpts()
    opts.mode = L.SELECT_GREEDY if mode == "greedy" else L.SELECT_EXPRACE
    opts.engine = {"auto": L.ENGINE_AUTO, "simt": L.ENGINE_SIMT, "tcgen05": L.ENGINE_TCGEN05,
                   "tcgen05_f16": L.ENGINE_TCGEN05_F16}[engine]
    if noise is not None:
        noise = _f32(noise, "noise")
        if tuple(noise.shape) != (M, table.n_rows):
            raise L.PcvError("noise must be [M, n_rows]")
    opts.noise = noise.data_ptr() if noise is not None else None
    opts.no_repeat = int(no_repeat)
    idx = torch.empty(M, dtype=torch.int64, device=Q.device)
    val = torch.empty(M, dtype=torch.float32, device=Q.device) if want_val else None
    ws = table.workspace("select_nr" if no_repeat else "select", M)
    with torch.cuda.device(Q.device), _timed("score_select_%s_M%d" % (mode, M)):
        L.check(L.load().pcv_score_select(table.handle, _ptr(Q), M, ctypes.byref(opts), _ptr(idx), _ptr(val),
                                          _ptr(ws), ws.numel(), _stream()), "pcv_score_select")
    return idx, val


def score_topk(table, Q, k):
    """Exact top-k over the catalog -> (idx int64[M, k], val f32[M, k]), score descending, ties by ascending index."""
    Q = _f32(Q, "Q")
    M, D = Q.shape
    if D != table.dim:
        raise L.PcvError("Q has dim %d, table has dim %d" % (D, table.dim))
    idx = torch.empty(M, k, dtype=torch.int64, device=Q.device)
    val = torch.empty(M, k, dtype=torch.float32, device=Q.device)
    ws = table.workspace("topk", M)
    with torch.cuda.device(Q.device), _timed("score_topk_M%d" % M):
        L.check(L.load().pcv_score_topk(table.handle, _ptr(Q), M, int(k), _ptr(idx), _ptr(val), _ptr(ws), ws.numel(),
                                        _stream()), "pcv_score_topk")
    return idx, val


def slate_no_repeat(table, Q, items, slate_size, vals=None):
    """In place: re-select the slates of `items` ([B*L] top-1 picks for the slot queries Q [B*L, D]) that contain a
    duplicate, sequentially without replacement (opt-in extension; include/pcv_b200.h)."""
    Q, items = _f32(Q, "Q"), _i64(items, "items")
    M, D = Q.shape
    if M % slate_size or items.numel() != M:
        raise L.PcvError("items / Q rows must be B * slate_size")
    ws = table.workspace("topk", M)
    with torch.cuda.device(Q.device), _timed("slate_no_repeat_M%d" % M):
        L.check(L.load().pcv_slate_no_repeat(table.handle, _ptr(Q), M // slate_size, int(slate_size), _ptr(items),
                                             _ptr(vals), _ptr(ws), ws.numel(), _stream()), "pcv_slate_no_repeat")
    return items


def slate_no_repeat_partials(table, Q, items, slate_size):
    """Shard half of the no-repeat selection on a vocab-parallel catalog: for the slates of `items` ([B*L] GLOBAL top-1
    picks) that hold a duplicate, this shard's top-L of each row -> int64 [B*L, L] keys (include/pcv_b200.h)."""
    Q, items = _f32(Q, "Q"), _i64(items, "items")
    M, D = Q.shape
    if D != table.dim:
        raise L.PcvError("Q has dim %d, table has dim %d" % (D, table.dim))
    if M % slate_size or items.numel() != M:
        raise L.PcvError("items / Q rows must be B * slate_size")
    keys = torch.empty(M, slate_size, dtype=torch.int64, device=Q.device)
    ws = table.workspace("topk", M)
    with torch.cuda.device(Q.device), _timed("slate_no_repeat_partials_M%d" % M):
        L.check(L.load().pcv_slate_no_repeat_partials(table.handle, _ptr(Q), M // slate_size, int(slate_size), _ptr(items),
                                                      _ptr(keys), _ptr(ws), ws.numel(), _stream()),
                "pcv_slate_no_repeat_partials")
    return keys


def slate_no_repeat_merge(keys, items, slate_size, vals=None):
    """In place: re-select the duplicate-holding slates of `items` from keys [G, B*L, L], the partials of the G shards
    in shard order; the result equals slate_no_repeat on the whole catalog."""
    keys = _i64(keys, "keys")
    if not items.is_cuda or items.dtype != torch.int64 or not items.is_contiguous():
        raise L.PcvError("items must be a contiguous int64 CUDA tensor (it is updated in place)")
    if vals is not None and (not vals.is_cuda or vals.dtype != torch.float32 or not vals.is_contiguous()
                             or vals.numel() != items.numel()):
        raise L.PcvError("vals must be a contiguous float32 CUDA tensor like items (it is updated in place)")
    M = items.numel()
    if keys.dim() != 3 or tuple(keys.shape[1:]) != (M, slate_size) or M % slate_size:
        raise L.PcvError("keys must be [G, B * slate_size, slate_size]")
    with torch.cuda.device(items.device), _timed("slate_no_repeat_merge_M%d" % M):
        L.check(L.load().pcv_slate_no_repeat_merge(_ptr(keys), keys.shape[0], M // slate_size, int(slate_size),
                                                   _ptr(items), _ptr(vals), _stream()), "pcv_slate_no_repeat_merge")
    return items


def sigmoid_categorical(table, Q, seed=0, offset=0, offset_dev=None, want_iters=False):
    """idx[i] ~ Categorical(sigmoid(Q[i] . W^T)) over the whole catalog, exact rejection sampler (csrc/sampler.cu)."""
    Q = _f32(Q, "Q")
    M, D = Q.shape
    if D != table.dim:
        raise L.PcvError("Q has dim %d, table has dim %d" % (D, table.dim))
    idx = torch.empty(M, dtype=torch.int64, device=Q.device)
    iters = torch.empty(M, dtype=torch.int32, device=Q.device) if want_iters else None
    with torch.cuda.device(Q.device), _timed("sigmoid_categorical_M%d" % M):
        L.check(L.load().pcv_sigmoid_categorical(table.handle, _ptr(Q), M, int(seed), int(offset), _ptr(offset_dev),
                                                 _ptr(idx), _ptr(iters), _stream()), "pcv_sigmoid_categorical")
    return (idx, iters) if want_iters else idx


def score_logits(table, Q):
    Q = _f32(Q, "Q")
    out = torch.empty(Q.shape[0], table.n_rows, dtype=torch.float32, device=Q.device)
    with torch.cuda.device(Q.device):
        L.check(L.load().pcv_score_logits(table.handle, _ptr(Q), Q.shape[0], _ptr(out), _stream()), "pcv_score_logits")
    return out


def vp_pack_keys(vals, idx):
    """(val f32[M], global idx int64[M]) -> int64[M] keys whose signed MAX over shards is the winner."""
    vals, idx = _f32(vals, "vals"), _i64(idx, "idx")
    keys = torch.empty(vals.shape[0], dtype=torch.int64, device=vals.device)
    with torch.cuda.device(vals.device):
        L.check(L.load().pcv_vp_pack_keys(_ptr(vals), _ptr(idx), vals.shape[0], _ptr(keys), _stream()), "pcv_vp_pack_keys")
    return keys


def vp_unpack_keys(keys):
    keys = _i64(keys, "keys")
    M = keys.shape[0]
    oi = torch.empty(M, dtype=torch.int64, device=keys.device)
    ov = torch.empty(M, dtype=torch.float32, device=keys.device)
    with torch.cuda.device(keys.device):
        L.check(L.load().pcv_vp_unpack_keys(_ptr(keys), M, _ptr(oi), _ptr(ov), _stream()), "pcv_vp_unpack_keys")
    return oi, ov


# ----------------------------------------------------------------------------
# fused MLP block
# ----------------------------------------------------------------------------
class Dense:
    def __init__(self, t):
        self.t = _f32(t, "dense segment")
        self.width = self.t.shape[1]

    def fill(self, seg, keep):
        seg.kind, seg.ptr, seg.idx = L.SEG_DENSE, self.t.data_ptr(), None
        seg.width, seg.count, seg.norm = self.width, 1, L.NORM_NONE
        keep.append(self.t)


class OneHot:
    """one-hot(sum_l r[b, l]) of width L+1 (cvae.py:85-92)."""

    def __init__(self, r):
        self.r = _f32(r, "responses")
        self.width = self.r.shape[1] + 1

    def fill(self, seg, keep):
        seg.kind, seg.ptr, seg.idx = L.SEG_ONEHOT, self.r.data_ptr(), None
        seg.width, seg.count, seg.norm = self.width, self.r.shape[1], L.NORM_NONE
        keep.append(self.r)


class Gather:
    """rows table[idx[b, :]] concatenated (nn.Embedding lookups, pivotcvae.py:253)."""

    def __init__(self, table, idx, normalize=False):
        self.table = _f32(table, "gather table")
        idx = _i64(idx, "gather index")
        self.idx = idx.reshape(idx.shape[0], -1)
        self.count = self.idx.shape[1]
        self.width = self.count * self.table.shape[1]
        self.normalize = normalize

    def fill(self, seg, keep):
        seg.kind, seg.ptr, seg.idx = L.SEG_GATHER, self.table.data_ptr(), self.idx.data_ptr()
        seg.width, seg.count = self.table.shape[1], self.count
        seg.norm = L.NORM_SEGMENT if self.normalize else L.NORM_NONE
        keep.extend([self.table, self.idx])


# ---- packed weights of the TMA MLP engine (inference): one pre-tiled copy per weight tensor, rebuilt
# IN PLACE when the tensor's version counter moves (so CUDA graphs that captured the pointer stay valid
# after `repack_stale()`).  An entry pins the weight's storage, so a data_ptr can not be recycled by
# another tensor while it is cached.
_PACKED = collections.OrderedDict()   # (data_ptr, kind) -> [version, shape, storage, packed, weight, kind]
_PACKED_MAX = 512
_PACKED_PINNED = set()                # keys a live CUDA graph reads through: never evicted


def pin_packed():
    """Called by the Graphed* objects after capture: the packed copies that exist now were baked into a
    graph as raw pointers, so they are exempt from the cache's eviction."""
    _PACKED_PINNED.update(_PACKED.keys())


def _pack_into(W, packed, kind):
    with torch.cuda.device(W.device):
        if kind == "tc":
            L.check(L.load().pcv_mlp_tc_pack(_ptr(W), W.shape[1], W.shape[0], _ptr(packed), _stream()), "pcv_mlp_tc_pack")
        else:
            L.check(L.load().pcv_mlp_pack(_ptr(W), W.shape[1], W.shape[0], _ptr(packed), _stream()), "pcv_mlp_pack")


def packed_weight(W, kind="ffma"):
    """Pre-tiled copy of an nn.Linear weight (cached per tensor + version): kind "ffma" = pcv_linear.Wp (the
    packed-weight cluster engine), kind "tc" = pcv_linear.Wt (tf32 hi | lo images of the tensor-core engine)."""
    key = (W.data_ptr(), kind)
    hit = _PACKED.get(key)
    if hit is not None and hit[1] == tuple(W.shape):
        if hit[0] != W._version:
            _pack_into(W, hit[3], kind)
            hit[0] = W._version
        _PACKED.move_to_end(key)
        return hit[3]
    lib = L.load()
    nbytes = (lib.pcv_mlp_tc_packed_bytes if kind == "tc" else lib.pcv_mlp_packed_bytes)(W.shape[1], W.shape[0])
    packed = torch.empty(nbytes // 4, dtype=torch.float32, device=W.device)
    _pack_into(W, packed, kind)
    if not torch.cuda.is_current_stream_capturing():   # graph-pool memory must not outlive its graph in the cache
        _PACKED[key] = [W._version, tuple(W.shape), W.untyped_storage(), packed, W, kind]
        while len(_PACKED) > _PACKED_MAX:
            victim = next((k for k in _PACKED if k not in _PACKED_PINNED), None)
            if victim is None:
                break
            del _PACKED[victim]
    return packed


def repack_stale():
    """Re-tile (in place) every cached weight whose tensor changed since it was packed; call it after
    updating weights that a captured CUDA graph reads through the packed copies."""
    for hit in _PACKED.values():
        if hit[0] != hit[4]._version:
            _pack_into(hit[4], hit[3], hit[5])
            hit[0] = hit[4]._version


# Inference engine of the fused MLP blocks: "exact" = the FFMA engines (sequential-k FMA chain, bit-identical to the
# CPU oracle); "tc" = the tcgen05 3xTF32 engine (csrc/mlp_tc.cu: fp32-grade, ~1e-6 of torch's addmm) wherever every
# block of a launch fits it, the exact engines elsewhere; "auto" = "tc" for large batches, "exact" below.  The library
# decides which kernel runs (pcv_mlp_plan, include/pcv_b200.h).
MLP_ENGINE = "exact"
_MLP_POLICY = {"exact": L.MLP_EXACT, "tc": L.MLP_TC, "auto": L.MLP_AUTO}


class mlp_engine:
    """Context manager: `with ops.mlp_engine("tc"): ...`"""

    def __init__(self, name):
        if name not in _MLP_POLICY:
            raise ValueError("mlp engine must be 'exact', 'tc' or 'auto'")
        self.name = name

    def __enter__(self):
        global MLP_ENGINE
        self.prev, MLP_ENGINE = MLP_ENGINE, self.name

    def __exit__(self, *exc):
        global MLP_ENGINE
        MLP_ENGINE = self.prev


def _mlp_desc(segments, layers, B, *, out=None, out_ld=None, out_col0=0, copy_seg=-1, save=False,
              latent=0, eps=None, seed=0, offset=0, offset_dev=None):
    """Build a pcv_mlp_desc without weight images (+ its output tensors); returns ((desc, keep-alive list, the layers'
    fp32 weights), results, device)."""
    if len(segments) > L.PCV_MAX_SEGMENTS or len(layers) > L.PCV_MAX_LAYERS:
        raise L.PcvError("too many segments / layers for one fused block")
    d = L.MlpDesc()
    keep = []
    d.n_segments = len(segments)
    for i, s in enumerate(segments):
        s.fill(d.seg[i], keep)
    n_in0 = sum(s.width for s in segments)
    d.n_layers = len(layers)
    prev = n_in0
    dev = None
    Ws = []
    for i, (W, b, act) in enumerate(layers):
        W, b = _f32(W, "weight"), _f32(b, "bias")
        dev = W.device
        d.layer[i].W, d.layer[i].b = W.data_ptr(), b.data_ptr()
        d.layer[i].n_in, d.layer[i].n_out, d.layer[i].act = W.shape[1], W.shape[0], act
        keep.extend([W, b])
        Ws.append(W)
        prev = W.shape[0]
    n_out = prev
    if out is None:
        out_ld = out_col0 + n_out if out_ld is None else out_ld
        out = torch.empty(B, out_ld, dtype=torch.float32, device=dev)
    d.out, d.out_ld, d.out_col0, d.copy_seg = out.data_ptr(), int(out_ld), int(out_col0), int(copy_seg)
    res = {"out": out}
    if save:
        x0 = torch.empty(B, n_in0, dtype=torch.float32, device=dev)
        d.x0 = x0.data_ptr()
        acts = []
        for i, (W, _, _) in enumerate(layers[:-1]):
            a = torch.empty(B, W.shape[0], dtype=torch.float32, device=dev)
            d.acts[i] = a.data_ptr()
            acts.append(a)
        res["x0"], res["acts"] = x0, acts
    d.latent = int(latent)
    if latent:
        z = torch.empty(B, latent, dtype=torch.float32, device=dev)
        d.z = z.data_ptr()
        res["z"] = z
        if eps is not None:
            eps = _f32(eps, "eps")
            d.eps = eps.data_ptr()
            keep.append(eps)
            res["eps"] = eps
        else:
            eo = torch.empty(B, latent, dtype=torch.float32, device=dev)
            d.eps_out = eo.data_ptr()
            res["eps"] = eo
        d.seed, d.offset = int(seed), int(offset)
        d.offset_dev = offset_dev.data_ptr() if offset_dev is not None else None
    return (d, keep, Ws), res, dev


def _mlp_launch(blocks, B, dev):
    """One launch of one or two blocks from _mlp_desc under MLP_ENGINE: the library plans which kernel runs them, every
    layer gets the weight image that kernel reads, then the same call launches it."""
    lib, engine = L.load(), _MLP_POLICY[MLP_ENGINE]
    descs = [ctypes.byref(d) for d, _, _ in blocks]
    with torch.cuda.device(dev):
        kernel = ctypes.c_int()
        L.check(lib.pcv_mlp_plan(descs[0], descs[1] if len(descs) > 1 else None, int(B), engine, ctypes.byref(kernel)),
                "pcv_mlp_plan")
        if kernel.value != L.MLP_KERNEL_STREAM:
            field, kind = ("Wt", "tc") if kernel.value == L.MLP_KERNEL_TC else ("Wp", "ffma")
            for d, keep, Ws in blocks:
                for i, W in enumerate(Ws):
                    keep.append(packed_weight(W, kind))
                    setattr(d.layer[i], field, keep[-1].data_ptr())
        name = "pcv_mlp_fwd" if len(descs) == 1 else "pcv_mlp_fwd2"
        with _timed(name[4:]):
            L.check(getattr(lib, name)(*descs, int(B), engine, _stream()), name)


def mlp_forward(segments, layers, B, **kw):
    """Run one fused MLP block.

    segments: list of Dense/OneHot/Gather; layers: list of (W[n_out,n_in], b[n_out], act).
    Returns dict(out=..., z=..., eps=..., x0=..., acts=[...]) (entries present when requested).
    """
    block, res, dev = _mlp_desc(segments, layers, B, **kw)
    _mlp_launch([block], B, dev)
    return res


def mlp_forward_chain(first, second_builder, B):
    """Two chained blocks in one launch.  first = (segments, layers, kwargs); second_builder(res_first)
    -> (segments, layers, kwargs) may reference the first block's output tensors (e.g. its z)."""
    block_a, ra, dev = _mlp_desc(first[0], first[1], B, **first[2])
    segs_b, layers_b, kw_b = second_builder(ra)
    block_b, rb, _ = _mlp_desc(segs_b, layers_b, B, **kw_b)
    _mlp_launch([block_a, block_b], B, dev)
    return ra, rb


# ----------------------------------------------------------------------------
# tensor-core GEMMs of the MLP blocks (csrc/gemm_tc.cu)
# ----------------------------------------------------------------------------
def pad4(n):
    return (int(n) + 3) // 4 * 4


def gemm_tn(A, B, M, N, K, *, A_lo=None, B_lo=None, C=None, C_lo=None, Ct=None, Ct_lo=None, bias=None, act=0,
            dact_src=None, dact=0, split_k=1):
    """C[M, N] = A[M, K] . B[N, K]^T on the tensor cores (tf32; 3xTF32 when the residual operands are given).
    A / B are 2-D fp32 CUDA tensors whose row stride is a multiple of 4 floats (they may be wider than K: padded
    leading dimension).  Outputs are written into the given buffers (row strides taken from them); with split_k > 1
    C is [split_k, M, ldc] raw partial sums."""
    d = L.GemmDesc()
    d.A, d.lda, d.B, d.ldb = A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0)
    d.A_lo = A_lo.data_ptr() if A_lo is not None else None
    d.B_lo = B_lo.data_ptr() if B_lo is not None else None
    d.M, d.N, d.K, d.split_k = int(M), int(N), int(K), int(split_k)
    if C is not None:
        d.C, d.ldc = C.data_ptr(), C.stride(-2)
        d.c_split_stride = C.stride(0) if split_k > 1 else 0
    d.C_lo = C_lo.data_ptr() if C_lo is not None else None
    if Ct is not None:
        d.Ct, d.ldct = Ct.data_ptr(), Ct.stride(0)
    d.Ct_lo = Ct_lo.data_ptr() if Ct_lo is not None else None
    d.bias = bias.data_ptr() if bias is not None else None
    d.act = int(act)
    if dact_src is not None:
        d.dact_src, d.ld_dact, d.dact = dact_src.data_ptr(), dact_src.stride(0), int(dact)
    with torch.cuda.device(A.device), _timed("gemm_tn"):
        L.check(L.load().pcv_gemm_tn(ctypes.byref(d), _stream()), "pcv_gemm_tn")


def transpose_batch(jobs):
    """jobs: list of dict(src=[rows, >=cols] tensor, rows, cols, dst=[cols, >=rows] tensor, dst_lo=None, src_lo=None)."""
    for i in range(0, len(jobs), 12):
        chunk = jobs[i:i + 12]
        arr = (L.TransposeJob * len(chunk))()
        for a, j in zip(arr, chunk):
            a.src, a.ld_src, a.rows, a.cols = j["src"].data_ptr(), j["src"].stride(0), int(j["rows"]), int(j["cols"])
            a.dst, a.ld_dst = j["dst"].data_ptr(), j["dst"].stride(0)
            a.dst_lo = j["dst_lo"].data_ptr() if j.get("dst_lo") is not None else None
            a.src_lo = j["src_lo"].data_ptr() if j.get("src_lo") is not None else None
        with torch.cuda.device(chunk[0]["src"].device):
            L.check(L.load().pcv_transpose_batch(arr, len(chunk), _stream()), "pcv_transpose_batch")


def wgrad_reduce(part, n_out, n_in, dW, Gt=None, B=0, db=None):
    """dW[n_out, n_in] = sum over the split-K slices of part [S, n_out, ld]; db[n_out] = row sums of Gt [n_out, >=B]."""
    S = part.shape[0]
    with torch.cuda.device(part.device):
        L.check(L.load().pcv_wgrad_reduce(_ptr(part), S, part.stride(0), part.stride(1), int(n_out), int(n_in), _ptr(dW),
                                          dW.stride(0), _ptr(Gt), Gt.stride(0) if Gt is not None else 0, int(B), _ptr(db),
                                          _stream()), "pcv_wgrad_reduce")


# ----------------------------------------------------------------------------
# KL, CE, response models
# ----------------------------------------------------------------------------
def kl_fwd_bwd(mu, logvar, pmu, plogvar, grads=True):
    mu, logvar, pmu, plogvar = (_f32(t) for t in (mu, logvar, pmu, plogvar))
    out = torch.empty((), dtype=torch.float32, device=mu.device)
    g = [torch.empty_like(mu) for _ in range(4)] if grads else [None] * 4
    with torch.cuda.device(mu.device):
        L.check(L.load().pcv_kl_fwd_bwd(_ptr(mu), _ptr(logvar), _ptr(pmu), _ptr(plogvar), mu.numel(), _ptr(out),
                                        _ptr(g[0]), _ptr(g[1]), _ptr(g[2]), _ptr(g[3]), _stream()), "pcv_kl_fwd_bwd")
    return out, g


def _ce_mask(table, M, keep_prob, bitmask, seed, offset, offset_dev, engine):
    mask = L.CeMask()
    mask.keep_prob = float(keep_prob)
    if bitmask is not None:
        if not bitmask.is_cuda:
            raise L.PcvError("bitmask must be a CUDA tensor")
        bitmask = bitmask.contiguous()
        if bitmask.dtype not in (torch.int32, torch.uint32) or tuple(bitmask.shape) != (M, (table.n_rows + 31) // 32):
            raise L.PcvError("bitmask must be int32/uint32 [M, ceil(N/32)]")
        mask.bitmask = bitmask.data_ptr()
    mask.seed, mask.offset = int(seed), int(offset)
    mask.offset_dev = offset_dev.data_ptr() if offset_dev is not None else None
    mask.engine = 1 if engine == "tf32" else 0
    return mask, bitmask


def ce_fwd_bwd(table, Q, targets, keep_prob=1.0, bitmask=None, seed=0, offset=0, want_dq=True, offset_dev=None,
               engine="exact"):
    """-> (loss_rows[M], lse[M], dq[M, D] or None); see include/pcv_b200.h."""
    Q, targets = _f32(Q, "Q"), _i64(targets, "targets").reshape(-1)
    M, D = Q.shape
    mask, bitmask = _ce_mask(table, M, keep_prob, bitmask, seed, offset, offset_dev, engine)
    loss = torch.empty(M, dtype=torch.float32, device=Q.device)
    lse = torch.empty(M, dtype=torch.float32, device=Q.device)
    dq = torch.empty(M, D, dtype=torch.float32, device=Q.device) if want_dq else None
    ws = table.workspace("ce", M)
    with torch.cuda.device(Q.device), _timed("ce_fwd_bwd"):
        L.check(L.load().pcv_ce_fwd_bwd(table.handle, _ptr(Q), _ptr(targets), M, ctypes.byref(mask), _ptr(loss),
                                        _ptr(lse), _ptr(dq), _ptr(ws), ws.numel(), _stream()), "pcv_ce_fwd_bwd")
    return loss, lse, dq


def ce_table_grad(table, Q, targets, lse, row_scale, keep_prob=1.0, bitmask=None, seed=0, offset=0, offset_dev=None,
                  engine="exact"):
    """dW [n_rows, D] = d (sum_i row_scale[i] loss_rows[i]) / d table for the mask of the matching ce_fwd_bwd call;
    see include/pcv_b200.h pcv_ce_table_grad."""
    Q, targets = _f32(Q, "Q"), _i64(targets, "targets").reshape(-1)
    lse, row_scale = _f32(lse, "lse"), _f32(row_scale, "row_scale")
    M = Q.shape[0]
    mask, bitmask = _ce_mask(table, M, keep_prob, bitmask, seed, offset, offset_dev, engine)
    dW = torch.empty(table.n_rows, table.dim, dtype=torch.float32, device=Q.device)
    ws = table.workspace("ce_tgrad", M)
    with torch.cuda.device(Q.device), _timed("ce_table_grad"):
        L.check(L.load().pcv_ce_table_grad(table.handle, _ptr(Q), _ptr(targets), M, ctypes.byref(mask), _ptr(lse),
                                           _ptr(row_scale), _ptr(dW), _ptr(ws), ws.numel(), _stream()), "pcv_ce_table_grad")
    return dW


def cand_ce_table_grad(table, Q, candidates, target_pos, lse, row_scale):
    """dW [n_rows, D] (zero-filled here) += the candidate-mode CE gradient w.r.t. the table rows each row's candidate
    list names; see include/pcv_b200.h pcv_cand_ce_table_grad."""
    Q = _f32(Q, "Q")
    M = Q.shape[0]
    candidates = _i64(candidates, "candidates").reshape(M, -1)
    target_pos = _i64(target_pos, "target_pos").reshape(-1)
    lse, row_scale = _f32(lse, "lse"), _f32(row_scale, "row_scale")
    dW = torch.zeros(table.n_rows, table.dim, dtype=torch.float32, device=Q.device)
    with torch.cuda.device(Q.device), _timed("cand_ce_table_grad"):
        L.check(L.load().pcv_cand_ce_table_grad(table.handle, _ptr(Q), _ptr(candidates), _ptr(target_pos), M,
                                                candidates.shape[1], _ptr(lse), _ptr(row_scale), _ptr(dW), _stream()),
                "pcv_cand_ce_table_grad")
    return dW


def ce_partials(shard, Q, targets, engine="exact"):
    """Vocab-parallel CE, local step: partial records [M, 2 + D] = {m, l, acc[D]} of this rank's row shard
    (full-catalog soft-max); see include/pcv_b200.h pcv_ce_partials."""
    Q, targets = _f32(Q, "Q"), _i64(targets, "targets").reshape(-1)
    M, D = Q.shape
    mask = L.CeMask()
    mask.keep_prob = 1.0
    mask.engine = 1 if engine == "tf32" else 0
    rec = torch.empty(M, 2 + D, dtype=torch.float32, device=Q.device)
    ws = shard.workspace("ce", M)
    with torch.cuda.device(Q.device), _timed("ce_partials"):
        L.check(L.load().pcv_ce_partials(shard.handle, _ptr(Q), _ptr(targets), M, ctypes.byref(mask), _ptr(rec), _ptr(ws),
                                         ws.numel(), _stream()), "pcv_ce_partials")
    return rec


def ce_vp_merge(recs, W_full, Q, targets, want_dq=True):
    """recs [G, M, 2 + D] gathered from the G shards -> (loss_rows[M], lse[M], dq[M, D] | None)."""
    recs, W_full, Q = _f32(recs, "recs"), _f32(W_full, "W_full"), _f32(Q, "Q")
    targets = _i64(targets, "targets").reshape(-1)
    G, M, R = recs.shape
    D = Q.shape[1]
    if R != 2 + D or W_full.shape[1] != D:
        raise L.PcvError("records must be [G, M, 2 + D]")
    loss = torch.empty(M, dtype=torch.float32, device=Q.device)
    lse = torch.empty(M, dtype=torch.float32, device=Q.device)
    dq = torch.empty(M, D, dtype=torch.float32, device=Q.device) if want_dq else None
    with torch.cuda.device(Q.device), _timed("ce_vp_merge"):
        L.check(L.load().pcv_ce_vp_merge(_ptr(recs), G, _ptr(W_full), D, _ptr(Q), _ptr(targets), M, _ptr(loss), _ptr(lse),
                                         _ptr(dq), _stream()), "pcv_ce_vp_merge")
    return loss, lse, dq


def cand_ce_fwd_bwd(table, Q, candidates, target_pos, want_dq=True, want_logits=False):
    """Sampled soft-max CE over per-row candidate lists -> (loss_rows[M], lse[M], dq[M,D]|None, p[M,nC]|None)."""
    Q = _f32(Q, "Q")
    M, D = Q.shape
    candidates = _i64(candidates, "candidates").reshape(M, -1)
    target_pos = _i64(target_pos, "target_pos").reshape(-1)
    nC = candidates.shape[1]
    loss = torch.empty(M, dtype=torch.float32, device=Q.device)
    lse = torch.empty(M, dtype=torch.float32, device=Q.device)
    dq = torch.empty(M, D, dtype=torch.float32, device=Q.device) if want_dq else None
    p = torch.empty(M, nC, dtype=torch.float32, device=Q.device) if want_logits else None
    with torch.cuda.device(Q.device), _timed("cand_ce_fwd_bwd"):
        L.check(L.load().pcv_cand_ce_fwd_bwd(table.handle, _ptr(Q), _ptr(candidates), _ptr(target_pos), M, nC, _ptr(loss),
                                             _ptr(lse), _ptr(dq), _ptr(p), _stream()), "pcv_cand_ce_fwd_bwd")
    return loss, lse, dq, p


def gather_norm_fwd(doc, usr, slates, users):
    """[normalize(concat doc[slates]) | normalize(usr[users])] -> (x0 [B, W], inv_norm [B, 2]); usr None = no user."""
    doc, slates = _f32(doc, "doc table"), _i64(slates, "slates")
    B, Ls = slates.shape
    D = doc.shape[1]
    W = (Ls + (0 if usr is None else 1)) * D
    x0 = torch.empty(B, W, dtype=torch.float32, device=doc.device)
    inv = torch.empty(B, 2, dtype=torch.float32, device=doc.device)
    if usr is not None:
        usr, users = _f32(usr, "user table"), _i64(users, "users").reshape(-1)
    with torch.cuda.device(doc.device):
        L.check(L.load().pcv_gather_norm_fwd(_ptr(doc), _ptr(usr), _ptr(slates), _ptr(users) if usr is not None else None, B, Ls, D,
                                             _ptr(x0), W, _ptr(inv), _stream()), "pcv_gather_norm_fwd")
    return x0, inv


def gather_norm_bwd(g, x0, inv, slates, users, doc_shape, usr_shape):
    """-> (d_doc, d_usr | None): gradient of the gather + normalise prologue scattered into table-shaped tensors."""
    g = _f32(g, "g")
    B, Ls = slates.shape
    D = doc_shape[1]
    d_doc = torch.zeros(doc_shape, dtype=torch.float32, device=g.device)
    d_usr = torch.zeros(usr_shape, dtype=torch.float32, device=g.device) if usr_shape is not None else None
    with torch.cuda.device(g.device):
        L.check(L.load().pcv_gather_norm_bwd(_ptr(g), g.stride(0), _ptr(x0), x0.stride(0), _ptr(inv), _ptr(slates),
                                             _ptr(users) if d_usr is not None else None, B, Ls, D, _ptr(d_doc), _ptr(d_usr),
                                             _stream()), "pcv_gather_norm_bwd")
    return d_doc, d_usr


def reparam_bwd(d_out, d_z, eps, out, Z):
    """Gradient w.r.t. a block's [mu | logvar] output with the reparameterisation's backward folded in (one launch).
    d_out: [B, >= 2Z] view or None, d_z: [B, Z] or None, out: the block's saved output (columns 0..2Z-1)."""
    B = out.shape[0]
    g = torch.empty(B, 2 * Z, dtype=torch.float32, device=out.device)
    if d_z is not None:
        d_z, eps = _f32(d_z, "d_z"), _f32(eps, "eps")
    with torch.cuda.device(out.device):
        L.check(L.load().pcv_reparam_bwd(_ptr(d_out), d_out.stride(0) if d_out is not None else 0, _ptr(d_z), _ptr(eps),
                                         _ptr(out), out.stride(0), B, int(Z), _ptr(g), _stream()), "pcv_reparam_bwd")
    return g


def bce_sigmoid(pred, target, want_grad=True):
    """nn.BCELoss()(sigmoid(pred), target) -> (loss scalar tensor, dpred | None)."""
    pred, target = _f32(pred, "pred").reshape(-1), _f32(target, "target").reshape(-1)
    loss = torch.empty((), dtype=torch.float32, device=pred.device)
    dp = torch.empty_like(pred) if want_grad else None
    with torch.cuda.device(pred.device):
        L.check(L.load().pcv_bce_sigmoid(_ptr(pred), _ptr(target), pred.numel(), _ptr(loss), _ptr(dp), _stream()), "pcv_bce_sigmoid")
    return loss, dp


def urm_forward(variant, doc, usr, item_bias, user_bias, slates, users, pos_bias=None, pos_dep=None, mr_factor=0.0):
    doc, usr = _f32(doc), _f32(usr)
    ib, ub = _f32(item_bias).reshape(-1), _f32(user_bias).reshape(-1)
    slates, users = _i64(slates), _i64(users).reshape(-1)
    B, Ls = slates.shape
    d = L.UrmDesc()
    d.variant = variant
    d.doc_table, d.user_table, d.item_bias, d.user_bias = doc.data_ptr(), usr.data_ptr(), ib.data_ptr(), ub.data_ptr()
    keep = [doc, usr, ib, ub]
    if pos_bias is not None:
        pb, pd = _f32(pos_bias).reshape(-1), _f32(pos_dep).reshape(-1)
        d.pos_bias, d.pos_dep = pb.data_ptr(), pd.data_ptr()
        keep += [pb, pd]
    d.mr_factor, d.L, d.D = float(mr_factor), Ls, doc.shape[1]
    out = torch.empty(B, Ls, dtype=torch.float32, device=doc.device)
    with torch.cuda.device(doc.device):
        L.check(L.load().pcv_urm_fwd(ctypes.byref(d), _ptr(slates), _ptr(users), B, _ptr(out), _stream()), "pcv_urm_fwd")
    return out
