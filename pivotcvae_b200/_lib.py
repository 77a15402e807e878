"""ctypes binding of libpcv_b200.so (the C ABI declared in include/pcv_b200.h).

There is no CPU or eager-PyTorch fallback: if the shared library is missing the
import fails loudly, and every op raises when its tensors are not on a CUDA
sm_100 device.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpcv_b200.so")

PCV_MAX_SEGMENTS = 6
PCV_MAX_LAYERS = 8
PCV_MAX_WIDTH = 1024

ACT_NONE, ACT_LEAKY, ACT_RELU = 0, 1, 2
SEG_DENSE, SEG_ONEHOT, SEG_GATHER = 0, 1, 2
NORM_NONE, NORM_SEGMENT = 0, 1
SELECT_GREEDY, SELECT_EXPRACE = 0, 1
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05, ENGINE_TCGEN05_F16 = 0, 1, 2, 3
URM, URM_P, URM_P_MR = 0, 1, 2
MLP_EXACT, MLP_TC, MLP_AUTO = 0, 1, 2
MLP_KERNEL_TC, MLP_KERNEL_CLUSTER, MLP_KERNEL_STREAM = 0, 1, 2

c_void_p, c_int, c_int64, c_uint64, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                ctypes.c_uint64, ctypes.c_size_t)


class PcvError(RuntimeError):
    pass


class SelectOpts(ctypes.Structure):
    _fields_ = [("mode", c_int), ("engine", c_int), ("noise", c_void_p), ("no_repeat", c_int)]


class Linear(ctypes.Structure):
    _fields_ = [("W", c_void_p), ("b", c_void_p), ("n_in", c_int), ("n_out", c_int), ("act", c_int),
                ("Wp", c_void_p), ("Wt", c_void_p)]


class Segment(ctypes.Structure):
    _fields_ = [("kind", c_int), ("ptr", c_void_p), ("idx", c_void_p), ("width", c_int),
                ("count", c_int), ("norm", c_int)]


class MlpDesc(ctypes.Structure):
    _fields_ = [("n_segments", c_int), ("seg", Segment * PCV_MAX_SEGMENTS), ("n_layers", c_int),
                ("layer", Linear * PCV_MAX_LAYERS), ("out", c_void_p), ("out_ld", c_int),
                ("out_col0", c_int), ("copy_seg", c_int), ("x0", c_void_p),
                ("acts", c_void_p * PCV_MAX_LAYERS), ("latent", c_int), ("eps", c_void_p),
                ("seed", c_uint64), ("offset", c_uint64), ("z", c_void_p), ("eps_out", c_void_p),
                ("offset_dev", c_void_p)]


class CeMask(ctypes.Structure):
    _fields_ = [("keep_prob", ctypes.c_double), ("bitmask", c_void_p), ("seed", c_uint64),
                ("offset", c_uint64), ("offset_dev", c_void_p), ("engine", c_int)]


class GemmDesc(ctypes.Structure):
    _fields_ = [("A", c_void_p), ("A_lo", c_void_p), ("lda", c_int64), ("B", c_void_p), ("B_lo", c_void_p), ("ldb", c_int64),
                ("M", c_int64), ("N", c_int64), ("K", c_int64), ("split_k", c_int), ("C", c_void_p), ("ldc", c_int64),
                ("c_split_stride", c_int64), ("C_lo", c_void_p), ("Ct", c_void_p), ("Ct_lo", c_void_p), ("ldct", c_int64),
                ("bias", c_void_p), ("act", c_int), ("dact_src", c_void_p), ("ld_dact", c_int64), ("dact", c_int)]


class TransposeJob(ctypes.Structure):
    _fields_ = [("src", c_void_p), ("ld_src", c_int64), ("rows", c_int), ("cols", c_int), ("dst", c_void_p),
                ("ld_dst", c_int64), ("dst_lo", c_void_p), ("src_lo", c_void_p)]


class UrmDesc(ctypes.Structure):
    _fields_ = [("variant", c_int), ("doc_table", c_void_p), ("user_table", c_void_p),
                ("item_bias", c_void_p), ("user_bias", c_void_p), ("pos_bias", c_void_p),
                ("pos_dep", c_void_p), ("mr_factor", ctypes.c_float), ("L", c_int), ("D", c_int)]


EXPORTS = {
    "pcv_abi_version": (c_int, []),
    "pcv_last_error": (ctypes.c_char_p, []),
    "pcv_device_ok": (c_int, [c_int]),
    "pcv_launch_count": (c_int64, []),
    "pcv_counter_add": (c_int, [c_void_p, c_uint64, c_void_p]),
    "pcv_table_create": (c_int, [c_void_p, c_int64, c_int, c_int64, ctypes.POINTER(c_void_p)]),
    "pcv_table_destroy": (None, [c_void_p]),
    "pcv_normalize_rows": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "pcv_score_select_workspace_bytes": (c_int, [c_void_p, c_int64, ctypes.POINTER(c_size_t)]),
    "pcv_score_select": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(SelectOpts), c_void_p,
                                 c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcv_score_logits": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "pcv_score_topk_workspace_bytes": (c_int, [c_void_p, c_int64, ctypes.POINTER(c_size_t)]),
    "pcv_score_topk": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcv_slate_no_repeat": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcv_slate_no_repeat_partials": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                             c_void_p]),
    "pcv_slate_no_repeat_merge": (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "pcv_sigmoid_categorical": (c_int, [c_void_p, c_void_p, c_int64, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pcv_vp_pack_keys": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "pcv_vp_unpack_keys": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "pcv_mlp_plan": (c_int, [ctypes.POINTER(MlpDesc), ctypes.POINTER(MlpDesc), c_int64, c_int, ctypes.POINTER(c_int)]),
    "pcv_mlp_fwd": (c_int, [ctypes.POINTER(MlpDesc), c_int64, c_int, c_void_p]),
    "pcv_mlp_fwd2": (c_int, [ctypes.POINTER(MlpDesc), ctypes.POINTER(MlpDesc), c_int64, c_int, c_void_p]),
    "pcv_gemm_tn": (c_int, [ctypes.POINTER(GemmDesc), c_void_p]),
    "pcv_transpose_batch": (c_int, [ctypes.POINTER(TransposeJob), c_int, c_void_p]),
    "pcv_wgrad_reduce": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64, c_int64,
                                 c_void_p, c_void_p]),
    "pcv_gather_norm_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "pcv_gather_norm_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p]),
    "pcv_reparam_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "pcv_bce_sigmoid": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "pcv_kl_fwd_bwd": (c_int, [c_void_p] * 4 + [c_int64] + [c_void_p] * 5 + [c_void_p]),
    "pcv_ce_workspace_bytes": (c_int, [c_void_p, c_int64, ctypes.POINTER(c_size_t)]),
    "pcv_ce_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, ctypes.POINTER(CeMask), c_void_p,
                               c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcv_ce_partials": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, ctypes.POINTER(CeMask), c_void_p, c_void_p, c_size_t,
                                c_void_p]),
    "pcv_ce_vp_merge": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                c_void_p]),
    "pcv_cand_ce_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p]),
    "pcv_ce_table_grad_workspace_bytes": (c_int, [c_void_p, c_int64, ctypes.POINTER(CeMask), ctypes.POINTER(c_size_t)]),
    "pcv_ce_table_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, ctypes.POINTER(CeMask), c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_size_t, c_void_p]),
    "pcv_cand_ce_table_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "pcv_mlp_packed_bytes": (ctypes.c_size_t, [c_int, c_int]),
    "pcv_mlp_pack": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "pcv_mlp_tc_packed_bytes": (ctypes.c_size_t, [c_int, c_int]),
    "pcv_mlp_tc_pack": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "pcv_slate_metrics": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "pcv_popcount": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "pcv_urm_fwd": (c_int, [ctypes.POINTER(UrmDesc), c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PcvError(
            "libpcv_b200.so is missing at %s: build it with `python -m pivotcvae_b200.build` "
            "(needs nvcc; this package has no CPU / eager fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the ABI drifted from include/pcv_b200.h
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().pcv_last_error().decode("utf-8", "replace")
        raise PcvError("%s failed (%d): %s" % (what or "libpcv_b200 call", rc, msg))
