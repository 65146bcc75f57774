"""ctypes binding of libvo_b200.so (the C ABI declared in include/vo_b200.h).

The library is the product; this file only loads it and spells out the prototypes.  There is
no fallback: if the shared object is missing, or the device is not sm_100, importing / creating
a context raises.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VO_B200_LIB") or os.path.join(_HERE, "libvo_b200.so")   # (override: A/B runs of two builds)

# ---- constants mirrored from include/vo_b200.h ---------------------------------------------
VO_ABI_VERSION = 5
VO_OK, VO_ERR_ARG, VO_ERR_CUDA, VO_ERR_UNSUPPORTED = 0, -1, -2, -3
VO_ST_OK, VO_ST_NO_MODEL, VO_ST_TOO_FEW_POINTS, VO_ST_KP_OUT_OF_IMAGE, VO_ST_BAD_INPUT = 0, 1, 2, 4, 8
VO_NORM_HAMMING, VO_NORM_L2_U8, VO_NORM_HAMMING_TC = 0, 1, 2
VO_METRIC_L2, VO_METRIC_COSINE = 0, 1
(VO_MODE_RATIO, VO_MODE_MUTUAL, VO_MODE_RATIO_MUTUAL, VO_MODE_THRESH_MUTUAL, VO_MODE_THRESH,
 VO_MODE_NN) = range(6)
VO_PREC_TF32X3, VO_PREC_TF32X1, VO_PREC_FP32_SIMT, VO_PREC_F16X1, VO_PREC_F16X3 = 0, 1, 2, 3, 4
VO_PNP_THROUGHPUT, VO_PNP_REFERENCE = 0, 1

c_void_p, c_int, c_float, c_double = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_double
c_u64, c_i64 = ctypes.c_uint64, ctypes.c_int64


class KnnOut(ctypes.Structure):
    _fields_ = [("row_idx", c_void_p), ("row_val", c_void_p), ("col_idx", c_void_p)]


class PipelineArgs(ctypes.Structure):
    _fields_ = [
        ("B", c_int), ("n_stride", c_int), ("m_stride", c_int),
        ("n_ref", c_void_p), ("n_cur", c_void_p),
        ("ref_u8", c_void_p), ("cur_u8", c_void_p),
        ("ref_f32", c_void_p), ("cur_f32", c_void_p),
        ("norm_or_metric", c_int), ("mode", c_int), ("precision", c_int),
        ("match_param", c_double),
        ("ref_kp", c_void_p), ("cur_kp", c_void_p),
        ("kp_stride", c_int),
        ("depth", c_void_p),
        ("H", c_int), ("W", c_int),
        ("K_h", c_void_p),
        ("min_flow_px", c_float), ("z_min", c_float), ("z_max", c_float),
        ("n_hyp", c_int),
        ("seed", c_u64),
        ("pair0", c_i64),
        ("thr_px", c_float),
        ("min_inliers", c_int), ("refine_iters", c_int),
        ("T_rel", c_void_p), ("rt", c_void_p),
        ("n_matches", c_void_p), ("n_corr", c_void_p), ("n_inl", c_void_p), ("status", c_void_p),
        ("depth_kp", c_void_p),
        ("u8_bytes", c_int),
        ("pnp_mode", c_int),
        ("ref_restarts", c_int), ("ref_iters", c_int),
        ("ref_confidence", c_double),
    ]


class SeqConfig(ctypes.Structure):
    _fields_ = [
        ("desc_is_f32", c_int), ("n_cap", c_int), ("kp_stride", c_int), ("H", c_int), ("W", c_int),
        ("K", c_double * 9),
        ("norm_or_metric", c_int), ("mode", c_int), ("precision", c_int),
        ("match_param", c_double),
        ("min_flow_px", c_float), ("z_min", c_float), ("z_max", c_float),
        ("n_hyp", c_int),
        ("seed", c_u64),
        ("thr_px", c_float),
        ("min_inliers", c_int), ("refine_iters", c_int),
        ("max_step_m", c_double),
        ("kf_min_common", c_int), ("kf_min_inliers", c_int),
        ("kf_max_dist", c_double),
        ("bad_pnp_limit", c_int), ("max_frames", c_int),
        ("pnp_mode", c_int),
        ("ref_restarts", c_int), ("ref_iters", c_int),
        ("ref_confidence", c_double),
        ("n_seqs", c_int),
        ("seeds", c_void_p),
    ]


class R2d2Layer(ctypes.Structure):
    _fields_ = [("cin", c_int), ("cout", c_int), ("k", c_int), ("dil", c_int), ("bn", c_int), ("relu", c_int),
                ("pool_after", c_int), ("w", c_void_p), ("bias", c_void_p), ("bn_mean", c_void_p), ("bn_var", c_void_p)]


class R2d2Config(ctypes.Structure):
    _fields_ = [("H", c_int), ("W", c_int), ("n_layers", c_int), ("layers", ctypes.POINTER(R2d2Layer)), ("upsample", c_int),
                ("clf_w", c_void_p), ("clf_b", c_void_p), ("sal_w", c_void_p), ("sal_b", c_void_p), ("bn_eps", c_float),
                ("max_kp", c_int)]


class OrbConfig(ctypes.Structure):
    _fields_ = [("H", c_int), ("W", c_int), ("nfeatures", c_int), ("nlevels", c_int), ("fast_threshold", c_int)]


class SiftConfig(ctypes.Structure):
    _fields_ = [("H", c_int), ("W", c_int), ("max_keypoints", c_int)]


PROTOTYPES = {
    "vo_create": (c_int, [c_int, ctypes.POINTER(c_void_p)]),
    "vo_destroy": (None, [c_void_p]),
    "vo_abi_version": (c_int, []),
    "vo_last_error": (ctypes.c_char_p, []),
    "vo_launch_count": (ctypes.c_longlong, [c_void_p]),
    "vo_workspace_generation": (ctypes.c_ulonglong, [c_void_p]),
    "vo_match_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                            c_int, c_double, c_void_p, c_void_p, c_void_p, ctypes.POINTER(KnnOut), c_void_p]),
    "vo_match_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                             c_int, c_double, c_int, c_void_p, c_void_p, c_void_p, ctypes.POINTER(KnnOut),
                             c_void_p, c_void_p]),
    "vo_backproject_dense": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vo_gather_backproject": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                      c_int, c_void_p, c_int, c_int, c_void_p, c_float, c_float, c_float,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_sample_depth": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p,
                                c_void_p]),
    "vo_hypotheses": (c_int, [c_void_p, c_void_p, c_int, c_int, c_u64, c_i64, c_void_p, c_void_p]),
    "vo_pnp_ransac": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int,
                              c_float, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_void_p]),
    "vo_pnp_ransac_ref": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_float, c_double, c_int, c_int,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_bootstrap": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_u64, c_i64, c_void_p, c_void_p]),
    "vo_pnp_ransac_ref_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_float,
                                        c_double, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p]),
    "vo_pipeline": (c_int, [c_void_p, ctypes.POINTER(PipelineArgs), c_void_p]),
    "vo_seq_create": (c_int, [c_void_p, ctypes.POINTER(SeqConfig), ctypes.POINTER(c_void_p)]),
    "vo_seq_destroy": (None, [c_void_p]),
    "vo_seq_push": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "vo_seq_frames": (c_int, [c_void_p]),
    "vo_seq_read": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vo_seq_push_all": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_seq_frames_at": (c_int, [c_void_p, c_int]),
    "vo_seq_read_at": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vo_seq_graph_captures": (c_int, [c_void_p]),
    "vo_seq_push_all_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_seq_lost_frames_at": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "vo_conv2d": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                          c_void_p, c_void_p]),
    "vo_r2d2_create": (c_int, [c_void_p, ctypes.POINTER(R2d2Config), ctypes.POINTER(c_void_p)]),
    "vo_r2d2_destroy": (None, [c_void_p]),
    "vo_r2d2_out_shape": (c_int, [c_void_p, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "vo_r2d2_extract": (c_int, [c_void_p, c_void_p, c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    "vo_orb_create": (c_int, [c_void_p, ctypes.POINTER(OrbConfig), ctypes.POINTER(c_void_p)]),
    "vo_orb_destroy": (None, [c_void_p]),
    "vo_orb_capacity": (c_int, [c_void_p]),
    "vo_orb_extract": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_orb_extract_batch": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_orb_debug_read": (c_int, [c_void_p, c_int, c_int, c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    "vo_sift_create": (c_int, [c_void_p, ctypes.POINTER(SiftConfig), ctypes.POINTER(c_void_p)]),
    "vo_sift_destroy": (None, [c_void_p]),
    "vo_sift_capacity": (c_int, [c_void_p]),
    "vo_sift_extract": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vo_profile_enable": (c_int, [c_void_p, c_int]),
    "vo_profile_collect": (c_int, [c_void_p, c_void_p, c_void_p]),
}

STAGES = ("fill", "prep", "match", "finalize", "gather", "hyp", "p3p", "score", "refit", "dense")

_lib = None
_lock = threading.Lock()


class VoError(RuntimeError):
    pass


def load():
    """Load libvo_b200.so (once) and attach prototypes.  Raises if it is not built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise VoError(
                    f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(or visual-odometry-pipeline_b200/csrc/build.sh).  There is no CPU fallback.")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in PROTOTYPES.items():
                fn = getattr(lib, name)  # AttributeError here = header/library drift
                fn.restype = res
                fn.argtypes = args
            if lib.vo_abi_version() != VO_ABI_VERSION:
                raise VoError(f"ABI mismatch: library {lib.vo_abi_version()} vs binding {VO_ABI_VERSION}")
            _lib = lib
    return _lib


def check(rc, what):
    if rc != VO_OK:
        msg = load().vo_last_error()
        raise VoError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


class Context:
    """vo_ctx handle for one CUDA device (see include/vo_b200.h: vo_create)."""

    def __init__(self, device=0):
        lib = load()
        h = c_void_p()
        check(lib.vo_create(int(device), ctypes.byref(h)), "vo_create")
        self.handle = h
        self.device = int(device)
        self.lib = lib

    def launch_count(self):
        return int(self.lib.vo_launch_count(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.vo_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
