"""CPU tests of pcv_mlp_plan, the library's one choice of the kernel that runs a fused MLP launch (include/pcv_b200.h).
Descriptors are built by hand with fake device pointers: planning reads shapes only and needs no GPU."""
import ctypes

import pytest

from pivotcvae_b200 import _lib as L

FAKE = 1 << 20          # 16-byte aligned stand-in for a device pointer; never dereferenced
TC, CLUSTER, STREAM = L.MLP_KERNEL_TC, L.MLP_KERNEL_CLUSTER, L.MLP_KERNEL_STREAM


def desc(segs, widths, x0=False):
    """segs: ("dense", width) | ("onehot", clicks) each; widths: n_out of each layer."""
    d = L.MlpDesc()
    d.n_segments = len(segs)
    n_in = 0
    for i, (kind, n) in enumerate(segs):
        s = d.seg[i]
        s.ptr = FAKE
        if kind == "dense":
            s.kind, s.width, s.count = L.SEG_DENSE, n, 1
            n_in += n
        else:
            s.kind, s.width, s.count = L.SEG_ONEHOT, n + 1, n
            n_in += n + 1
    d.n_layers = len(widths)
    for i, n_out in enumerate(widths):
        layer = d.layer[i]
        layer.W = layer.b = FAKE
        layer.n_in, layer.n_out = n_in, n_out
        n_in = n_out
    d.out, d.out_ld, d.copy_seg = FAKE, n_in, -1
    if x0:
        d.x0 = FAKE
    return d


def plan(engine, B, a, b=None):
    kernel = ctypes.c_int(-1)
    L.check(L.load().pcv_mlp_plan(ctypes.byref(a), ctypes.byref(b) if b is not None else None, B, engine,
                                  ctypes.byref(kernel)), "pcv_mlp_plan")
    return kernel.value


ENC = [("dense", 43), ("onehot", 5), ("dense", 8)]      # 43 + 6 + 8 = 57 wide


def test_exact_runs_the_cluster_engine():
    assert plan(L.MLP_EXACT, 1000, desc(ENC, [256, 256, 32])) == CLUSTER


@pytest.mark.parametrize("engine", [L.MLP_EXACT, L.MLP_TC, L.MLP_AUTO])
def test_saved_outputs_run_the_streaming_engine(engine):
    assert plan(engine, 4096, desc(ENC, [256, 256, 32], x0=True)) == STREAM


@pytest.mark.parametrize("segs,widths", [([("dense", 64)], [256, 256, 32]),                 # the widest input
                                         ([("onehot", 16), ("dense", 47)], [256, 8]),      # 16 clicks
                                         (ENC, [256, 256, 32])])
def test_tc_runs_a_block_that_fits(segs, widths):
    assert plan(L.MLP_TC, 1000, desc(segs, widths)) == TC


@pytest.mark.parametrize("segs,widths", [([("dense", 65)], [256, 32]),                      # input 65 wide
                                         ([("dense", 54)], [256, 257, 32]),                # a 257-wide layer
                                         ([("onehot", 17), ("dense", 8)], [256, 32]),      # 17 clicks
                                         ([("onehot", 5), ("onehot", 5)], [256, 32])])     # two one-hot segments
def test_tc_leaves_a_block_that_does_not_fit_to_the_cluster_engine(segs, widths):
    assert plan(L.MLP_TC, 1000, desc(segs, widths)) == CLUSTER


def test_a_chain_is_planned_as_one_launch():
    """prior [one-hot, user] -> z, then a block on [z 16 | one-hot 6 | user 64] = 86 wide: the second block does not
    fit the tc engine, so neither block runs on it."""
    prior = desc([("onehot", 5), ("dense", 8)], [128, 128, 32])
    nxt = desc([("dense", 16), ("onehot", 5), ("dense", 64)], [256, 256, 8])
    assert plan(L.MLP_TC, 777, prior) == TC
    assert plan(L.MLP_TC, 777, prior, nxt) == CLUSTER
    assert plan(L.MLP_TC, 777, nxt, prior) == CLUSTER


def test_auto_takes_the_tc_engine_from_2048_rows():
    d = desc(ENC, [256, 256, 32])
    assert plan(L.MLP_AUTO, 2047, d) == CLUSTER
    assert plan(L.MLP_AUTO, 2048, d) == TC


@pytest.mark.parametrize("engine", [L.MLP_EXACT, L.MLP_TC])
def test_activations_too_wide_for_the_cluster_engine_stream(engine):
    assert plan(engine, 1000, desc([("dense", 54)], [1024, 1024, 32])) == STREAM


def test_bad_arguments_are_rejected():
    lib, k = L.load(), ctypes.c_int()
    d = desc(ENC, [256, 32])
    assert lib.pcv_mlp_plan(ctypes.byref(d), None, 1000, 3, ctypes.byref(k)) == -1        # unknown engine
    assert lib.pcv_mlp_plan(ctypes.byref(d), None, 0, L.MLP_EXACT, ctypes.byref(k)) == -1
    assert lib.pcv_mlp_plan(ctypes.byref(d), None, 1000, L.MLP_EXACT, None) == -1


@pytest.mark.parametrize("engine,image", [(L.MLP_EXACT, "Wp"), (L.MLP_TC, "Wt")])
def test_launch_without_the_planned_image_is_an_error(engine, image):
    """The kernel the plan names reads its weight image on every layer; a missing one is an error before any device
    work, never a fall-back to another engine."""
    lib = L.load()
    d = desc(ENC, [256, 256, 32])
    d.layer[0].Wp = d.layer[0].Wt = FAKE
    assert lib.pcv_mlp_fwd(ctypes.byref(d), 1000, engine, None) == -1
    msg = lib.pcv_last_error().decode()
    assert "layer 1" in msg and image in msg, msg
