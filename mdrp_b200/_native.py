"""ctypes binding of librepose_b200.so (include/repose_b200.h).

The library is the product: there is no Python / CPU fallback.  If the shared object is
missing or no CUDA device is present, every entry point raises.
"""
import ctypes as C
import os
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "librepose_b200.so")

CALIB, CALIB_SHIFT, SHARED, VARYING = 0, 1, 2, 3
VARIANTS = {"calib": CALIB, "calib_shift": CALIB_SHIFT, "shared": SHARED, "varying": VARYING}
PAIR_OK, PAIR_DEGENERATE, PAIR_EVENTS_RERUN, PAIR_CONTINUED, PAIR_FAILED = 0, 1, 2, 4, -1   # enum rp_pair_state
LOSS = {"TRIVIAL": 0, "TRUNCATED": 1, "HUBER": 2, "CAUCHY": 3, "TRUNCATED_CAUCHY": 4}

EXPORTS = [
    "rp_create", "rp_destroy", "rp_last_error", "rp_default_options", "rp_launch_count",
    "rp_estimate_batch_host", "rp_estimate_batch_dev", "rp_sample_batch", "rp_sample_batch_prosac", "rp_solve_batch",
    "rp_score_batch", "rp_refine_batch", "rp_measure_pipes", "rp_last_timing", "rp_gather_depths_dev", "rp_tc_count_batch", "rp_pair_status", "rp_gather_depths_batch_dev",
    "rp_estimate_batch_host_f32", "rp_estimate_batch_dev_f32", "rp_gather_depths_dev_f32", "rp_gather_depths_batch_dev_f32",
    "rp_estimate_batch_host_quality", "rp_estimate_batch_dev_quality", "rp_estimate_batch_host_f32_quality",
    "rp_estimate_batch_dev_f32_quality", "rp_order_by_quality",
    "rp_gather_depths_dev_quality", "rp_gather_depths_dev_f32_quality", "rp_gather_depths_batch_dev_quality",
    "rp_gather_depths_batch_dev_f32_quality",
    "rp_refine_pairs_host", "rp_refine_pairs_dev", "rp_refine_pairs_host_f32", "rp_refine_pairs_dev_f32",
    "rp_estimate_batch_host_init", "rp_estimate_batch_dev_init", "rp_estimate_batch_host_f32_init",
    "rp_estimate_batch_dev_f32_init",
]
ORDER_SMEM_CAP = 12288   # RP_ORDER_SMEM_CAP: larger pairs are ordered in global scratch


class NativeError(RuntimeError):
    pass


class Model(C.Structure):
    _fields_ = [("q", C.c_double * 4), ("t", C.c_double * 3), ("scale", C.c_double),
                ("shift1", C.c_double), ("shift2", C.c_double), ("f1", C.c_double), ("f2", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("refinements", C.c_int64), ("iterations", C.c_int64), ("num_inliers", C.c_int64),
                ("inlier_ratio", C.c_double), ("model_score", C.c_double)]


class Options(C.Structure):
    _fields_ = [("max_iterations", C.c_int64), ("min_iterations", C.c_int64),
                ("dyn_num_trials_mult", C.c_double), ("success_prob", C.c_double),
                ("max_reproj_error", C.c_double), ("max_epipolar_error", C.c_double),
                ("seed", C.c_uint64), ("estimate_shift", C.c_int32), ("progressive_sampling", C.c_int32),
                ("weight_sampson", C.c_double), ("bundle_max_iterations", C.c_int64),
                ("loss_type", C.c_int32), ("reserved1", C.c_int32), ("loss_scale", C.c_double),
                ("gradient_tol", C.c_double), ("step_tol", C.c_double), ("initial_lambda", C.c_double),
                ("min_lambda", C.c_double), ("max_lambda", C.c_double), ("max_prosac_iterations", C.c_int64)]


class BundleOptions(C.Structure):
    _fields_ = [("max_iterations", C.c_int64), ("loss_type", C.c_int32), ("reserved", C.c_int32),
                ("loss_scale", C.c_double), ("gradient_tol", C.c_double), ("step_tol", C.c_double),
                ("initial_lambda", C.c_double), ("min_lambda", C.c_double), ("max_lambda", C.c_double)]


class BundleStats(C.Structure):
    _fields_ = [("iterations", C.c_int64), ("initial_cost", C.c_double), ("cost", C.c_double),
                ("lam", C.c_double), ("invalid_steps", C.c_int64), ("step_norm", C.c_double),
                ("grad_norm", C.c_double)]


MODEL_DTYPE = np.dtype([("q", "<f8", 4), ("t", "<f8", 3), ("scale", "<f8"), ("shift1", "<f8"),
                        ("shift2", "<f8"), ("f1", "<f8"), ("f2", "<f8")])
STATS_DTYPE = np.dtype([("refinements", "<i8"), ("iterations", "<i8"), ("num_inliers", "<i8"),
                        ("inlier_ratio", "<f8"), ("model_score", "<f8")])
BSTATS_DTYPE = np.dtype([("iterations", "<i8"), ("initial_cost", "<f8"), ("cost", "<f8"), ("lam", "<f8"),
                         ("invalid_steps", "<i8"), ("step_norm", "<f8"), ("grad_norm", "<f8")])
assert MODEL_DTYPE.itemsize == C.sizeof(Model) == 96
assert STATS_DTYPE.itemsize == C.sizeof(Stats) == 40

_lib = None
DP = C.POINTER(C.c_double)
VP = C.c_void_p


def load():
    """dlopen the CUDA library; raises NativeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise NativeError(f"{SO_PATH} is missing: run `python -m mdrp_b200.build` "
                          "(there is no CPU fallback)")
    L = C.CDLL(SO_PATH)
    L.rp_create.restype = C.c_int
    L.rp_create.argtypes = [C.c_int, C.POINTER(VP)]
    L.rp_destroy.restype = None
    L.rp_destroy.argtypes = [VP]
    L.rp_last_error.restype = C.c_char_p
    L.rp_last_error.argtypes = [VP]
    L.rp_default_options.restype = None
    L.rp_default_options.argtypes = [C.POINTER(Options)]
    L.rp_launch_count.restype = C.c_int64
    L.rp_launch_count.argtypes = [VP]
    est_args = [VP, C.c_int, C.c_int64, VP, VP, VP, VP, VP, VP, C.POINTER(Options), VP, VP, VP]
    L.rp_estimate_batch_host.restype = C.c_int
    L.rp_estimate_batch_host.argtypes = est_args
    L.rp_estimate_batch_dev.restype = C.c_int
    L.rp_estimate_batch_dev.argtypes = est_args + [VP]
    L.rp_estimate_batch_host_f32.restype = C.c_int
    L.rp_estimate_batch_host_f32.argtypes = est_args
    L.rp_estimate_batch_dev_f32.restype = C.c_int
    L.rp_estimate_batch_dev_f32.argtypes = est_args + [VP]
    est_q_args = est_args[:8] + [VP] + est_args[8:]   # quality after d2
    for name in ("rp_estimate_batch_host_quality", "rp_estimate_batch_host_f32_quality"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = est_q_args
    for name in ("rp_estimate_batch_dev_quality", "rp_estimate_batch_dev_f32_quality"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = est_q_args + [VP]
    # rp_estimate_batch_*_init: the quality twin's arguments (quality nullable) with init after opt
    est_init_args = est_q_args[:11] + [VP] + est_q_args[11:]
    for name in ("rp_estimate_batch_host_init", "rp_estimate_batch_host_f32_init"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = est_init_args
    for name in ("rp_estimate_batch_dev_init", "rp_estimate_batch_dev_f32_init"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = est_init_args + [VP]
    # rp_refine_pairs_*: the estimator's arguments up to opt, then init, subset, models, bstats, num_inliers, inliers
    refine_args = est_args[:10] + [VP, VP, VP, VP, VP, VP]
    for name in ("rp_refine_pairs_host", "rp_refine_pairs_host_f32"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = refine_args
    for name in ("rp_refine_pairs_dev", "rp_refine_pairs_dev_f32"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = refine_args + [VP]
    L.rp_order_by_quality.restype = C.c_int
    L.rp_order_by_quality.argtypes = [VP, C.c_int64, VP, VP, VP]
    L.rp_sample_batch.restype = C.c_int
    L.rp_sample_batch.argtypes = [VP, C.c_int64, C.c_uint64, C.c_int64, VP]
    L.rp_sample_batch_prosac.restype = C.c_int
    L.rp_sample_batch_prosac.argtypes = [VP, C.c_int64, C.c_uint64, C.c_int64, C.c_int32, C.c_int64, VP]
    L.rp_solve_batch.restype = C.c_int
    L.rp_solve_batch.argtypes = [VP, C.c_int, C.c_int64, VP, VP, VP, VP, VP, VP]
    L.rp_score_batch.restype = C.c_int
    L.rp_score_batch.argtypes = [VP, C.c_int, C.c_int64, VP, C.c_int64, VP, VP, C.c_double, VP, VP, VP]
    L.rp_tc_count_batch.restype = C.c_int
    L.rp_tc_count_batch.argtypes = [VP, C.c_int, C.c_int64, VP, C.c_int64, VP, VP, C.c_double, VP]
    L.rp_refine_batch.restype = C.c_int
    L.rp_refine_batch.argtypes = [VP, C.c_int, C.c_int64, VP, C.c_int64, VP, VP, VP, VP, VP, C.c_double,
                                  C.c_double, C.POINTER(BundleOptions), VP]
    L.rp_gather_depths_dev.restype = C.c_int
    L.rp_gather_depths_dev.argtypes = [VP, VP, C.c_int, C.c_int, VP, C.c_int, C.c_int, VP, VP, C.c_int64, VP, VP, VP, VP,
                                       C.POINTER(C.c_int64), VP]
    L.rp_gather_depths_batch_dev.restype = C.c_int
    L.rp_gather_depths_batch_dev.argtypes = [VP, C.c_int64, VP, VP, C.c_int, C.c_int, C.c_int, VP, VP, VP, VP, VP, VP, VP, VP, VP, VP]
    for f in (L.rp_gather_depths_dev_f32, L.rp_gather_depths_batch_dev_f32):
        f.restype = C.c_int
    L.rp_gather_depths_dev_f32.argtypes = L.rp_gather_depths_dev.argtypes
    L.rp_gather_depths_batch_dev_f32.argtypes = L.rp_gather_depths_batch_dev.argtypes
    # the _quality gathers: the twin's arguments with quality after kp2 and quality_out after d2
    for twin, kp2, d2 in (("rp_gather_depths_dev", 8, 13), ("rp_gather_depths_batch_dev", 10, 14)):
        t = getattr(L, twin).argtypes
        for name in (twin + "_quality", twin + "_f32_quality"):
            getattr(L, name).restype = C.c_int
            getattr(L, name).argtypes = t[:kp2 + 1] + [VP] + t[kp2 + 1:d2 + 1] + [VP] + t[d2 + 1:]
    L.rp_measure_pipes.restype = C.c_int
    L.rp_measure_pipes.argtypes = [VP, DP, DP]
    L.rp_pair_status.restype = C.c_int
    L.rp_pair_status.argtypes = [VP, C.c_int64, VP]
    L.rp_last_timing.restype = C.c_int
    L.rp_last_timing.argtypes = [VP, DP, C.POINTER(C.c_int64)]
    _lib = L
    return L


def default_options() -> Options:
    o = Options()
    load().rp_default_options(C.byref(o))
    return o


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a):
    return a.ctypes.data if a is not None else None


TIMING_KEYS = ["prepare", "sample", "solve", "score_minimal", "scan", "lo_refine", "lo_score_merge",
               "final_refine", "device_total", "h2d", "d2h", "bound_kernel", "tc_kernel", "widen", "order", "r15"]
COUNTER_KEYS = ["hypotheses", "point_scores", "lm_problems", "lm_iterations", "chunks", "exact_models",
                "bound_evaluated", "head_models", "tc_evaluated", "tc_selected", "lm_flops", "c11", "c12", "c13", "c14", "c15"]


class Context:
    """One rp_ctx = one GPU (workspace + stream)."""

    def __init__(self, device: int = 0):
        self._lib = load()
        h = VP()
        rc = self._lib.rp_create(device, C.byref(h))
        if rc != 0:
            raise NativeError(f"rp_create({device}) failed ({rc}): "
                              f"{self._lib.rp_last_error(None).decode()}")
        self._h = h
        self.device = device
        # One rp_ctx owns one device workspace, its events and work counters, and ctypes releases the GIL
        # during a native call: calls on the SAME context from several Python threads are serialised here
        # (the reference binding is re-entrant; INTEGRATION.md: one rp_ctx per concurrently calling thread).
        self._lock = threading.RLock()

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise NativeError(f"librepose_b200 error {rc}: {self._lib.rp_last_error(self._h).decode()}")

    def _call(self, fn, *args):
        """One native call on this context: serialised per context, error code turned into NativeError."""
        with self._lock:
            self._check(fn(*args))

    @property
    def launch_count(self) -> int:
        return int(self._lib.rp_launch_count(self._h))

    def last_timing(self):
        ms = (C.c_double * 16)()
        cn = (C.c_int64 * 16)()
        self._call(self._lib.rp_last_timing, self._h, ms, cn)
        return dict(zip(TIMING_KEYS, list(ms))), dict(zip(COUNTER_KEYS, list(cn)))

    def pair_status(self, n_pairs):
        """rp_pair_state of every pair of the last estimate call (0 ok, 1 degenerate, bits 2 / 4 re-run, -1 failed)."""
        out = np.zeros(n_pairs, dtype=np.int32)
        self._call(self._lib.rp_pair_status, self._h, n_pairs, _ptr(out))
        return out

    def measure_pipes(self):
        a, b = C.c_double(0), C.c_double(0)
        self._call(self._lib.rp_measure_pipes, self._h, C.byref(a), C.byref(b))
        return a.value, b.value

    # ---- hot path -------------------------------------------------------------------------
    def estimate_batch_host(self, variant, offsets, x1, x2, d1, d2, cams, opt: Options):
        """Packed host arrays in, (models, stats, masks) numpy structured arrays out."""
        return self._estimate_host(self._lib.rp_estimate_batch_host, _f64, variant, offsets, x1, x2, d1, d2, cams, opt)

    def estimate_batch_host_f32(self, variant, offsets, x1, x2, d1, d2, cams, opt: Options):
        """`estimate_batch_host` for float32 points and depths (rp_estimate_batch_host_f32): half the upload, the same
        bytes out as `estimate_batch_host` on the values converted to float64."""
        return self._estimate_host(self._lib.rp_estimate_batch_host_f32, _f32, variant, offsets, x1, x2, d1, d2, cams, opt)

    def estimate_batch_host_quality(self, variant, offsets, x1, x2, d1, d2, cams, opt: Options, quality):
        """`estimate_batch_host` with one match quality per correspondence (rp_estimate_batch_host[_f32]_quality): every
        pair is ordered by decreasing float32 quality on the device (ties: original index), masks come back in the
        caller's order.  float32 points and depths (all four) take the float32 entry point, anything else float64."""
        quality = _f32(quality)
        if all(getattr(a, "dtype", None) == np.float32 for a in (x1, x2, d1, d2)):
            fn, conv = self._lib.rp_estimate_batch_host_f32_quality, _f32
        else:
            fn, conv = self._lib.rp_estimate_batch_host_quality, _f64
        return self._estimate_host(fn, conv, variant, offsets, x1, x2, d1, d2, cams, opt, quality)

    def estimate_batch_host_init(self, variant, offsets, x1, x2, d1, d2, cams, opt: Options, init, quality=None):
        """`estimate_batch_host` from one prior per pair (rp_estimate_batch_host[_f32]_init): `init` (MODEL_DTYPE [P], a
        NaN row leaves its pair without a prior) is scored and locally optimised before RANSAC's first iteration.
        `quality` (optional) as in `estimate_batch_host_quality`; float32 points and depths (all four) take the float32
        entry point, anything else float64."""
        init = np.ascontiguousarray(init, dtype=MODEL_DTYPE).reshape(-1)
        if init.shape != (len(offsets) - 1,):
            raise ValueError("init must hold one model per pair")
        quality = _f32(quality) if quality is not None else None
        if all(getattr(a, "dtype", None) == np.float32 for a in (x1, x2, d1, d2)):
            fn, conv = self._lib.rp_estimate_batch_host_f32_init, _f32
        else:
            fn, conv = self._lib.rp_estimate_batch_host_init, _f64
        return self._estimate_host(fn, conv, variant, offsets, x1, x2, d1, d2, cams, opt, quality, init)

    def _estimate_host(self, fn, conv, variant, offsets, x1, x2, d1, d2, cams, opt, quality=None, init=None):
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_pairs = len(offsets) - 1
        x1, x2, d1, d2 = conv(x1), conv(x2), conv(d1), conv(d2)
        ntot = int(offsets[-1]) if n_pairs >= 0 else 0
        if x1.shape != (ntot, 2) or x2.shape != (ntot, 2) or d1.shape != (ntot,) or d2.shape != (ntot,):
            raise ValueError("x1/x2 must be [N,2] and d1/d2 [N] with N = offsets[-1]")
        if quality is not None and quality.shape != (ntot,):
            raise ValueError("quality must be [N] with N = offsets[-1]")
        cams = _f64(cams) if cams is not None else None
        if cams is not None and cams.shape != (n_pairs, 8):
            raise ValueError("cams must be [n_pairs, 8]")
        models = np.zeros(n_pairs, dtype=MODEL_DTYPE)
        stats = np.zeros(n_pairs, dtype=STATS_DTYPE)
        masks = np.zeros(max(ntot, 1), dtype=np.uint8)
        data = [_ptr(x1), _ptr(x2), _ptr(d1), _ptr(d2)] + ([_ptr(quality)] if quality is not None or init is not None else [])
        prior = [_ptr(init)] if init is not None else []
        self._call(fn,
            self._h, int(variant), n_pairs, _ptr(offsets), *data,
            _ptr(cams), C.byref(opt), *prior, _ptr(models), _ptr(stats), _ptr(masks))
        return models, stats, masks[:ntot]

    def estimate_batch_dev(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options,
                           models_ptr, stats_ptr, masks_ptr, stream=0):
        """Raw device pointers (e.g. torch tensor .data_ptr()); offsets is a host int64 array."""
        self._estimate_dev(self._lib.rp_estimate_batch_dev, variant, offsets, [x1_ptr, x2_ptr, d1_ptr, d2_ptr], cams_ptr, opt,
                           models_ptr, stats_ptr, masks_ptr, stream)

    def estimate_batch_dev_f32(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options,
                               models_ptr, stats_ptr, masks_ptr, stream=0):
        """`estimate_batch_dev` with x1, x2, d1, d2 pointing at float32 device arrays (rp_estimate_batch_dev_f32)."""
        self._estimate_dev(self._lib.rp_estimate_batch_dev_f32, variant, offsets, [x1_ptr, x2_ptr, d1_ptr, d2_ptr], cams_ptr,
                           opt, models_ptr, stats_ptr, masks_ptr, stream)

    def estimate_batch_dev_quality(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options,
                                   models_ptr, stats_ptr, masks_ptr, quality_ptr, stream=0):
        """`estimate_batch_dev` with a float32 device array of match qualities (rp_estimate_batch_dev_quality)."""
        self._estimate_dev(self._lib.rp_estimate_batch_dev_quality, variant, offsets,
                           [x1_ptr, x2_ptr, d1_ptr, d2_ptr, quality_ptr or None], cams_ptr, opt, models_ptr, stats_ptr,
                           masks_ptr, stream)

    def estimate_batch_dev_f32_quality(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options,
                                       models_ptr, stats_ptr, masks_ptr, quality_ptr, stream=0):
        """`estimate_batch_dev_f32` with a float32 device array of match qualities (rp_estimate_batch_dev_f32_quality)."""
        self._estimate_dev(self._lib.rp_estimate_batch_dev_f32_quality, variant, offsets,
                           [x1_ptr, x2_ptr, d1_ptr, d2_ptr, quality_ptr or None], cams_ptr, opt, models_ptr, stats_ptr,
                           masks_ptr, stream)

    def estimate_batch_dev_init(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options, init_ptr,
                                models_ptr, stats_ptr, masks_ptr, quality_ptr=None, stream=0):
        """`estimate_batch_dev` from one prior per pair (rp_estimate_batch_dev_init): `init_ptr` points at [P] rp_model
        in device memory (NaN rows: no prior); `quality_ptr` (optional) at float32 match qualities."""
        self._estimate_dev(self._lib.rp_estimate_batch_dev_init, variant, offsets,
                           [x1_ptr, x2_ptr, d1_ptr, d2_ptr, quality_ptr or None], cams_ptr, opt, models_ptr, stats_ptr,
                           masks_ptr, stream, init_ptr)

    def estimate_batch_dev_f32_init(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options,
                                    init_ptr, models_ptr, stats_ptr, masks_ptr, quality_ptr=None, stream=0):
        """`estimate_batch_dev_init` with x1, x2, d1, d2 pointing at float32 device arrays (rp_estimate_batch_dev_f32_init)."""
        self._estimate_dev(self._lib.rp_estimate_batch_dev_f32_init, variant, offsets,
                           [x1_ptr, x2_ptr, d1_ptr, d2_ptr, quality_ptr or None], cams_ptr, opt, models_ptr, stats_ptr,
                           masks_ptr, stream, init_ptr)

    def _estimate_dev(self, fn, variant, offsets, data, cams_ptr, opt, models_ptr, stats_ptr, masks_ptr, stream,
                      init_ptr=None):
        """`data`: the device pointers between offsets and cams (x1, x2, d1, d2 and, for quality and prior calls,
        quality); `init_ptr`: the priors of the _init calls."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        prior = [init_ptr] if init_ptr is not None else []
        self._call(fn,
            self._h, int(variant), len(offsets) - 1, _ptr(offsets), *data,
            cams_ptr, C.byref(opt), *prior, models_ptr, stats_ptr, masks_ptr, stream or None)

    # ---- refinement of caller-supplied models (rp_refine_pairs_*) --------------------------------
    def refine_pairs_host(self, variant, offsets, x1, x2, d1, d2, cams, opt: Options, init, subset=None):
        """The estimator's final refinement from `init` (MODEL_DTYPE [P]) on each pair's `subset` (uint8 [N], None: every
        correspondence).  Returns (models, bstats, num_inliers int64 [P], inliers uint8 [N]) of the refined models."""
        return self._refine_host(self._lib.rp_refine_pairs_host, _f64, variant, offsets, x1, x2, d1, d2, cams, opt, init,
                                 subset)

    def refine_pairs_host_f32(self, variant, offsets, x1, x2, d1, d2, cams, opt: Options, init, subset=None):
        """`refine_pairs_host` for float32 points and depths (rp_refine_pairs_host_f32): half the upload, the same bytes
        out as `refine_pairs_host` on the values converted to float64."""
        return self._refine_host(self._lib.rp_refine_pairs_host_f32, _f32, variant, offsets, x1, x2, d1, d2, cams, opt,
                                 init, subset)

    def _refine_host(self, fn, conv, variant, offsets, x1, x2, d1, d2, cams, opt, init, subset):
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_pairs = len(offsets) - 1
        x1, x2, d1, d2 = conv(x1), conv(x2), conv(d1), conv(d2)
        ntot = int(offsets[-1]) if n_pairs >= 0 else 0
        if x1.shape != (ntot, 2) or x2.shape != (ntot, 2) or d1.shape != (ntot,) or d2.shape != (ntot,):
            raise ValueError("x1/x2 must be [N,2] and d1/d2 [N] with N = offsets[-1]")
        init = np.ascontiguousarray(init, dtype=MODEL_DTYPE).reshape(-1)
        if init.shape != (n_pairs,):
            raise ValueError("init must hold one model per pair")
        if subset is not None:
            subset = np.ascontiguousarray(subset, dtype=np.uint8).reshape(-1)
            if subset.shape != (ntot,):
                raise ValueError("subset must be [N] with N = offsets[-1]")
        cams = _f64(cams) if cams is not None else None
        if cams is not None and cams.shape != (n_pairs, 8):
            raise ValueError("cams must be [n_pairs, 8]")
        models = np.zeros(n_pairs, dtype=MODEL_DTYPE)
        bstats = np.zeros(n_pairs, dtype=BSTATS_DTYPE)
        num_inliers = np.zeros(n_pairs, dtype=np.int64)
        inliers = np.zeros(max(ntot, 1), dtype=np.uint8)
        self._call(fn, self._h, int(variant), n_pairs, _ptr(offsets), _ptr(x1), _ptr(x2), _ptr(d1), _ptr(d2), _ptr(cams),
                   C.byref(opt), _ptr(init), _ptr(subset), _ptr(models), _ptr(bstats), _ptr(num_inliers), _ptr(inliers))
        return models, bstats, num_inliers, inliers[:ntot]

    def refine_pairs_dev(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options, init_ptr,
                         subset_ptr, models_ptr, bstats_ptr, num_inliers_ptr, inliers_ptr, stream=0):
        """rp_refine_pairs_dev: raw device pointers (subset, bstats, num_inliers, inliers may be None); offsets is a host
        int64 array."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self._call(self._lib.rp_refine_pairs_dev, self._h, int(variant), len(offsets) - 1, _ptr(offsets), x1_ptr, x2_ptr,
                   d1_ptr, d2_ptr, cams_ptr, C.byref(opt), init_ptr, subset_ptr or None, models_ptr, bstats_ptr or None,
                   num_inliers_ptr or None, inliers_ptr or None, stream or None)

    def refine_pairs_dev_f32(self, variant, offsets, x1_ptr, x2_ptr, d1_ptr, d2_ptr, cams_ptr, opt: Options, init_ptr,
                             subset_ptr, models_ptr, bstats_ptr, num_inliers_ptr, inliers_ptr, stream=0):
        """`refine_pairs_dev` with x1, x2, d1, d2 pointing at float32 device arrays (rp_refine_pairs_dev_f32)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self._call(self._lib.rp_refine_pairs_dev_f32, self._h, int(variant), len(offsets) - 1, _ptr(offsets), x1_ptr,
                   x2_ptr, d1_ptr, d2_ptr, cams_ptr, C.byref(opt), init_ptr, subset_ptr or None, models_ptr,
                   bstats_ptr or None, num_inliers_ptr or None, inliers_ptr or None, stream or None)

    # ---- stage entry points -----------------------------------------------------------------
    def order(self, offsets, quality):
        """rp_order_by_quality: per pair, the pair-local indices in (float32 quality descending, index ascending)
        order (NaN as -inf, -0 as +0); int32 [N]."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        quality = _f32(quality)
        n = int(offsets[-1]) if len(offsets) else 0
        if len(offsets) < 1 or quality.shape != (n,):
            raise ValueError("quality must be [N] with N = offsets[-1]")
        perm = np.zeros(n, dtype=np.int32)
        self._call(self._lib.rp_order_by_quality, self._h, len(offsets) - 1, _ptr(offsets), _ptr(quality), _ptr(perm))
        return perm

    def sample(self, n, seed, iters, progressive_sampling=False, max_prosac_iterations=100000):
        out = np.zeros((iters, 3), dtype=np.int32)
        if progressive_sampling:
            self._call(self._lib.rp_sample_batch_prosac, self._h, n, seed, iters, 1, max_prosac_iterations, _ptr(out))
        else:
            self._call(self._lib.rp_sample_batch, self._h, n, seed, iters, _ptr(out))
        return out

    def solve(self, variant, x1h, x2h, d1, d2):
        x1h, x2h, d1, d2 = _f64(x1h), _f64(x2h), _f64(d1), _f64(d2)
        n = x1h.shape[0]
        models = np.zeros((n, 4), dtype=MODEL_DTYPE)
        counts = np.zeros(n, dtype=np.int32)
        self._call(self._lib.rp_solve_batch, self._h, int(variant), n, _ptr(x1h), _ptr(x2h), _ptr(d1),
                                             _ptr(d2), _ptr(models), _ptr(counts))
        return models, counts

    def score(self, variant, models, x1, x2, sq_thr, want_masks=False):
        models = np.ascontiguousarray(models, dtype=MODEL_DTYPE)
        x1, x2 = _f64(x1), _f64(x2)
        n, npts = len(models), len(x1)
        scores = np.zeros(n)
        counts = np.zeros(n, dtype=np.int64)
        masks = np.zeros((n, npts), dtype=np.uint8) if want_masks else None
        self._call(self._lib.rp_score_batch, self._h, int(variant), n, _ptr(models), npts, _ptr(x1), _ptr(x2),
                                             float(sq_thr), _ptr(scores), _ptr(counts), _ptr(masks))
        return (scores, counts, masks) if want_masks else (scores, counts)

    def tc_count(self, variant, models, x1, x2, sq_thr):
        """Certain-outlier counts of the tensor-core tier (rp_tc_count_batch)."""
        models = np.ascontiguousarray(models, dtype=MODEL_DTYPE)
        x1, x2 = _f64(x1), _f64(x2)
        out = np.zeros(len(models), dtype=np.int64)
        self._call(self._lib.rp_tc_count_batch, self._h, int(variant), len(models), _ptr(models), len(x1), _ptr(x1), _ptr(x2),
                   float(sq_thr), _ptr(out))
        return out

    def refine(self, variant, models, x1, x2, d1, d2, scale_reproj, weight_sampson, bopt: BundleOptions,
               mask=None):
        models = np.ascontiguousarray(models, dtype=MODEL_DTYPE).copy()
        x1, x2, d1, d2 = _f64(x1), _f64(x2), _f64(d1), _f64(d2)
        mk = np.ascontiguousarray(mask, dtype=np.uint8) if mask is not None else None
        stats = np.zeros(len(models), dtype=BSTATS_DTYPE)
        self._call(self._lib.rp_refine_batch, self._h, int(variant), len(models), _ptr(models), len(x1), _ptr(x1),
                                              _ptr(x2), _ptr(d1), _ptr(d2), _ptr(mk), float(scale_reproj),
                                              float(weight_sampson), C.byref(bopt), _ptr(stats))
        return models, stats


def bundle_options(max_iterations=100, loss_type="CAUCHY", loss_scale=1.0, gradient_tol=1e-10, step_tol=1e-8,
                   initial_lambda=1e-3, min_lambda=1e-10, max_lambda=1e10) -> BundleOptions:
    lt = LOSS[loss_type] if isinstance(loss_type, str) else int(loss_type)
    return BundleOptions(max_iterations, lt, 0, loss_scale, gradient_tol, step_tol, initial_lambda, min_lambda,
                         max_lambda)
