"""Host-side mirror of the reference's Python surface for the RePoseD hot path.

Same names, argument meaning, return objects and `info` keys as the PoseLib binding the
reference calls (whl:_core.pyi:446-501; call sites /root/reference/make_pair.py:111,
make_video.py:284, README.md:86-96), plus the PoseLib-mdrp fork names the eval drivers use
(/root/reference/eval.py:153, eval_shared_f.py:177, eval_varying_f.py:168) and batched entry
points, which are the unit the GPU actually wants.  All numerics run in librepose_b200.so
(CUDA, sm_100a); there is no CPU fallback.

Error behaviour (SURVEY.md §8b): unknown dict keys are ignored; N < 3 returns the identity
model with iterations = 0, model_score = DBL_MAX and an all-False mask; x1/x2/d1/d2 length
mismatches raise ValueError (the reference silently reads out of bounds there).
"""
import sys
import threading

import numpy as np

from . import _native as nv

DBL_MAX = sys.float_info.max

_CAMERA_MODELS = {"SIMPLE_PINHOLE": 0, "PINHOLE": 1}


class Camera:
    """poselib.Camera for the two models the reference's callers use (whl:_core.pyi:76-123)."""

    def __init__(self, model="SIMPLE_PINHOLE", params=None, width=-1, height=-1):
        if model not in _CAMERA_MODELS:
            raise ValueError(f"camera model {model!r} is outside this build (SIMPLE_PINHOLE / PINHOLE; "
                             "undistort on the host first)")
        self._model = model
        self.model_id = _CAMERA_MODELS[model]
        self.params = [float(p) for p in (params if params is not None else [1.0, 0.0, 0.0])]
        self.width, self.height = int(width), int(height)

    @classmethod
    def from_any(cls, cam):
        if isinstance(cam, Camera):
            return cam
        if isinstance(cam, dict):
            return cls(cam.get("model", "SIMPLE_PINHOLE"), cam.get("params"), cam.get("width", -1),
                       cam.get("height", -1))
        # duck-typed poselib.Camera
        return cls(cam.model_name(), list(cam.params), cam.width, cam.height)

    def model_name(self):
        return self._model

    def focal_x(self):
        return self.params[0]

    def focal_y(self):
        return self.params[0] if self._model == "SIMPLE_PINHOLE" else self.params[1]

    def focal(self):
        return 0.5 * (self.focal_x() + self.focal_y())

    def principal_point(self):
        return np.array(self.params[1:3] if self._model == "SIMPLE_PINHOLE" else self.params[2:4])

    def fxfycxcy(self):
        pp = self.principal_point()
        return [self.focal_x(), self.focal_y(), float(pp[0]), float(pp[1])]

    def unproject(self, x):
        x = np.asarray(x, dtype=np.float64)
        f = np.array([self.focal_x(), self.focal_y()])
        return (x - self.principal_point()) / f

    def project(self, x):
        x = np.asarray(x, dtype=np.float64)
        f = np.array([self.focal_x(), self.focal_y()])
        return x * f + self.principal_point()

    def __repr__(self):
        return f"[{self._model} {self.width} {self.height} {self.params}]"


class CameraPose:
    """poselib.CameraPose: q (w first), t; R/Rt derived (whl:_core.pyi:125-152)."""

    def __init__(self, q=(1.0, 0.0, 0.0, 0.0), t=(0.0, 0.0, 0.0)):
        self.q = np.array(q, dtype=np.float64)
        self.t = np.array(t, dtype=np.float64)

    @property
    def R(self):
        w, x, y, z = self.q
        return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                         [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                         [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])

    @property
    def Rt(self):
        return np.concatenate([self.R, self.t[:, None]], axis=1)

    def center(self):
        return -self.R.T @ self.t

    def __repr__(self):
        return f"[q: {self.q}, t: {self.t}]"


class MonoDepthTwoViewGeometry:
    """X2 = scale (d2+shift2) K2^-1 x2 = R (d1+shift1) K1^-1 x1 + t (whl:_core.pyi:178-204)."""

    def __init__(self, pose=None, scale=1.0, shift1=0.0, shift2=0.0):
        self.pose = pose if pose is not None else CameraPose()
        self.scale, self.shift1, self.shift2 = float(scale), float(shift1), float(shift2)

    def __repr__(self):
        return f"[pose: {self.pose}, scale: {self.scale}, shift1: {self.shift1}, shift2: {self.shift2}]"


class MonoDepthImagePair:
    """geometry + two SIMPLE_PINHOLE cameras [f, 0, 0] (whl:_core.pyi:171-176).  `.pose` aliases
    geometry.pose: the eval drivers of the fork read image_pair.pose (eval_shared_f.py:84)."""

    def __init__(self, geometry=None, camera1=None, camera2=None):
        self.geometry = geometry if geometry is not None else MonoDepthTwoViewGeometry()
        self.camera1 = camera1 if camera1 is not None else Camera()
        self.camera2 = camera2 if camera2 is not None else Camera()

    @property
    def pose(self):
        return self.geometry.pose


# ---- option dicts --------------------------------------------------------------------------------
_RANSAC_KEYS = ("max_iterations", "min_iterations", "dyn_num_trials_mult", "success_prob", "max_reproj_error",
                "max_epipolar_error", "seed")


def make_options(ransac_opt=None, bundle_opt=None, focal_variant=False) -> nv.Options:
    """dict -> rp_options with the binding's defaults (whl:METADATA:71-107); unknown keys ignored."""
    ransac_opt = ransac_opt or {}
    bundle_opt = bundle_opt or {}
    o = nv.default_options()
    for k in _RANSAC_KEYS:
        if k in ransac_opt:
            setattr(o, k, type(getattr(o, k))(ransac_opt[k]))
    # PROSAC (RandomSampler::initialize_prosac so@0x4f8a20): the caller passes correspondences sorted by
    # decreasing quality, exactly as with the reference
    o.progressive_sampling = int(bool(ransac_opt.get("progressive_sampling", False)))
    if "max_prosac_iterations" in ransac_opt:
        o.max_prosac_iterations = int(ransac_opt["max_prosac_iterations"])
    o.estimate_shift = int(bool(ransac_opt.get("monodepth_estimate_shift", False)))
    o.weight_sampson = float(np.float32(ransac_opt.get("monodepth_weight_sampson", 1.0)))
    if "max_iterations" in bundle_opt:
        o.bundle_max_iterations = int(bundle_opt["max_iterations"])
    # the binding matches the loss name case-insensitively and keeps its default (CAUCHY) for a name it
    # does not know (verified on the wheel: 'cauchy' == 'CAUCHY', 'bogus' -> CAUCHY)
    lt = bundle_opt.get("loss_type", "CAUCHY")
    if isinstance(lt, str):
        if lt.upper() == "TRUNCATED_LE_ZACH":
            raise NotImplementedError("TRUNCATED_LE_ZACH loss is outside this build")
        o.loss_type = nv.LOSS.get(lt.upper(), nv.LOSS["CAUCHY"])
    else:
        o.loss_type = int(lt)
    # focal variants honour the user's loss_scale (default 0.5*max_epipolar_error); the calibrated
    # variant overwrites it with half the normalised threshold (SURVEY.md §8b "Errors")
    o.loss_scale = float(bundle_opt.get("loss_scale", 0.5 * o.max_epipolar_error if focal_variant else 1.0))
    for k in ("gradient_tol", "step_tol", "initial_lambda", "min_lambda", "max_lambda"):
        if k in bundle_opt:
            setattr(o, k, float(bundle_opt[k]))
    return o


# ---- context per device ----------------------------------------------------------------------------
_ctx = {}
_ctx_lock = threading.Lock()


def context(device: int = 0) -> nv.Context:
    with _ctx_lock:
        if device not in _ctx:
            _ctx[device] = nv.Context(device)
        return _ctx[device]


def _pack(list_x1, list_x2, list_d1, list_d2):
    n = [len(d) for d in list_d1]
    for a, b, c, d in zip(list_x1, list_x2, list_d1, list_d2):
        a = np.asarray(a)
        if a.ndim != 2 or a.shape[1] != 2 or np.asarray(b).shape != a.shape:
            raise TypeError("points must be [N, 2] arrays")
        if not (len(a) == len(c) == len(d)):
            raise ValueError("points and depths must have the same length")
    offsets = np.zeros(len(n) + 1, dtype=np.int64)
    offsets[1:] = np.cumsum(n)
    cat = lambda xs, shape: (np.concatenate([np.asarray(x, dtype=np.float64).reshape(shape) for x in xs])
                             if len(xs) else np.zeros(shape if shape[0] != -1 else (0,) + shape[1:]))
    x1 = cat(list_x1, (-1, 2))
    x2 = cat(list_x2, (-1, 2))
    d1 = cat(list_d1, (-1,))
    d2 = cat(list_d2, (-1,))
    return offsets, x1, x2, d1, d2


def _all_float32(*lists):
    """True when every point and depth array of the batch is float32 (and there is at least one pair): those batches take
    the float32 entry points, which widen on the device and return the same bytes with half the upload."""
    arrays = [a for xs in lists for a in xs]
    return len(arrays) > 0 and all(getattr(a, "dtype", None) == np.float32 for a in arrays)


def _pack_f32(list_x1, list_x2, list_d1, list_d2):
    """`_pack` for a batch whose arrays are all float32 (`_all_float32`): the same checks and offsets, float32 packed
    arrays, so no FP64 copy of the batch is made on the host."""
    for a, b, c, d in zip(list_x1, list_x2, list_d1, list_d2):
        if a.ndim != 2 or a.shape[1] != 2 or b.shape != a.shape:
            raise TypeError("points must be [N, 2] arrays")
        if not (len(a) == len(c) == len(d)):
            raise ValueError("points and depths must have the same length")
    offsets = np.zeros(len(list_d1) + 1, dtype=np.int64)
    offsets[1:] = np.cumsum([len(d) for d in list_d1])
    cat = lambda xs, shape: np.concatenate([np.asarray(x).reshape(shape) for x in xs])
    return offsets, cat(list_x1, (-1, 2)), cat(list_x2, (-1, 2)), cat(list_d1, (-1,)), cat(list_d2, (-1,))


def _pack_auto(list_x1, list_x2, list_d1, list_d2):
    """`_pack_f32` when every array is float32, else `_pack` (float64)."""
    if _all_float32(list_x1, list_x2, list_d1, list_d2):
        return _pack_f32(list_x1, list_x2, list_d1, list_d2)
    return _pack(list_x1, list_x2, list_d1, list_d2)


def _pack_quality(quality, offsets):
    """One match-quality array per pair -> packed float32 [N].  The values are converted to float32 first, so the order
    the estimator uses is that of the float32 values.  A pair count or length that does not match the points raises
    ValueError."""
    n = np.diff(offsets)
    if len(quality) != len(n):
        raise ValueError(f"quality needs one array per pair ({len(n)}), got {len(quality)}")
    qs = [np.asarray(q, dtype=np.float32).reshape(-1) for q in quality]
    for i, (q, k) in enumerate(zip(qs, n)):
        if len(q) != k:
            raise ValueError(f"quality of pair {i} has {len(q)} values for {k} correspondences")
    return np.concatenate(qs) if qs else np.zeros(0, dtype=np.float32)


def _pack_priors(rows, n_pairs):
    """One rp_model row per pair (None for a pair: no prior) -> MODEL_DTYPE [n_pairs] with NaN rows for the Nones; a
    pair count that does not match the points raises ValueError."""
    if len(rows) != n_pairs:
        raise ValueError(f"initial models need one entry per pair ({n_pairs}), got {len(rows)}")
    out = np.zeros(n_pairs, dtype=nv.MODEL_DTYPE)
    out.view(np.float64).reshape(n_pairs, 12)[:] = np.nan
    for i, r in enumerate(rows):
        if r is not None:
            out[i] = r
    return out


def _estimate_host(ctx, variant, offsets, x1, x2, d1, d2, cams, opt, quality=None, init=None):
    """Packed host arrays through the float32 entry point when they are float32, else the FP64 one; with a packed
    `quality` through the quality entry point of that dtype; with packed priors `init` through the _init entry point."""
    if init is not None:
        return ctx.estimate_batch_host_init(variant, offsets, x1, x2, d1, d2, cams, opt, init, quality)
    if quality is not None:
        return ctx.estimate_batch_host_quality(variant, offsets, x1, x2, d1, d2, cams, opt, quality)
    if x1.dtype == np.float32 and x2.dtype == np.float32 and d1.dtype == np.float32 and d2.dtype == np.float32:
        return ctx.estimate_batch_host_f32(variant, offsets, x1, x2, d1, d2, cams, opt)
    return ctx.estimate_batch_host(variant, offsets, x1, x2, d1, d2, cams, opt)


def _info(stats_row, mask):
    return {"refinements": int(stats_row["refinements"]), "iterations": int(stats_row["iterations"]),
            "num_inliers": int(stats_row["num_inliers"]), "inlier_ratio": float(stats_row["inlier_ratio"]),
            "model_score": float(stats_row["model_score"]), "inliers": [bool(b) for b in mask]}


def _geometry(m):
    return MonoDepthTwoViewGeometry(CameraPose(m["q"], m["t"]), m["scale"], m["shift1"], m["shift2"])


# ---- batched entry points (the unit of GPU work) -----------------------------------------------------
def estimate_monodepth_relative_pose_batch(points2D_1, points2D_2, depth_1, depth_2, cameras1, cameras2,
                                           ransac_opt=None, bundle_opt=None, device=0, quality=None,
                                           initial_geometries=None):
    """Lists (one entry per image pair) in, list of (MonoDepthTwoViewGeometry, info) out.  When every point and depth
    array is float32 the batch goes through the float32 entry point (same results, half the upload).

    `quality` (optional): one array of match qualities per pair (matcher scores, higher is better).  Each pair is then
    ordered by decreasing float32 quality on the device (ties: original index; NaN lowest) before the estimator runs,
    which is the order PROSAC (`progressive_sampling`) expects; the inlier lists come back in the caller's order.

    `initial_geometries` (optional): one MonoDepthTwoViewGeometry per pair (None: no prior for that pair), e.g. a
    tracker's previous pose.  RANSAC scores and locally optimises it before its first iteration, so the result is never
    worse than the locally optimised prior, and then samples as usual, so a wrong prior is recovered from;
    `info["iterations"]` counts only the sampled iterations and `info["refinements"]` includes the prior's LO."""
    offsets, x1, x2, d1, d2 = _pack_auto(points2D_1, points2D_2, depth_1, depth_2)
    q = _pack_quality(quality, offsets) if quality is not None else None
    init = (_pack_priors([None if g is None else _model_row(g) for g in initial_geometries], len(offsets) - 1)
            if initial_geometries is not None else None)
    cams = np.array([Camera.from_any(a).fxfycxcy() + Camera.from_any(b).fxfycxcy()
                     for a, b in zip(cameras1, cameras2)], dtype=np.float64).reshape(-1, 8)
    opt = make_options(ransac_opt, bundle_opt, focal_variant=False)
    variant = nv.CALIB_SHIFT if opt.estimate_shift else nv.CALIB
    models, stats, masks = _estimate_host(context(device), variant, offsets, x1, x2, d1, d2, cams, opt, q, init)
    return [(_geometry(models[i]), _info(stats[i], masks[offsets[i]:offsets[i + 1]])) for i in range(len(models))]


def _focal_batch(variant, points2D_1, points2D_2, depth_1, depth_2, ransac_opt, bundle_opt, device, quality=None,
                 initial_image_pairs=None):
    offsets, x1, x2, d1, d2 = _pack_auto(points2D_1, points2D_2, depth_1, depth_2)
    q = _pack_quality(quality, offsets) if quality is not None else None
    init = (_pack_priors([None if p is None else _model_row(p.geometry, Camera.from_any(p.camera1).focal(),
                                                            Camera.from_any(p.camera2).focal())
                          for p in initial_image_pairs], len(offsets) - 1)
            if initial_image_pairs is not None else None)
    opt = make_options(ransac_opt, bundle_opt, focal_variant=True)
    models, stats, masks = _estimate_host(context(device), variant, offsets, x1, x2, d1, d2, None, opt, q, init)
    out = []
    for i, m in enumerate(models):
        pair = MonoDepthImagePair(_geometry(m), Camera("SIMPLE_PINHOLE", [m["f1"], 0.0, 0.0]),
                                  Camera("SIMPLE_PINHOLE", [m["f2"], 0.0, 0.0]))
        out.append((pair, _info(stats[i], masks[offsets[i]:offsets[i + 1]])))
    return out


def estimate_monodepth_shared_focal_relative_pose_batch(points2D_1, points2D_2, depth_1, depth_2,
                                                        ransac_opt=None, bundle_opt=None, device=0, quality=None,
                                                        initial_image_pairs=None):
    """`quality`: as in estimate_monodepth_relative_pose_batch.  `initial_image_pairs` (optional): one MonoDepthImagePair
    per pair (None: no prior), used as `initial_geometries` there; its cameras' focal lengths are the prior's."""
    return _focal_batch(nv.SHARED, points2D_1, points2D_2, depth_1, depth_2, ransac_opt, bundle_opt, device, quality,
                        initial_image_pairs)


def estimate_monodepth_varying_focal_relative_pose_batch(points2D_1, points2D_2, depth_1, depth_2,
                                                         ransac_opt=None, bundle_opt=None, device=0, quality=None,
                                                         initial_image_pairs=None):
    """`quality`, `initial_image_pairs`: as in estimate_monodepth_shared_focal_relative_pose_batch."""
    return _focal_batch(nv.VARYING, points2D_1, points2D_2, depth_1, depth_2, ransac_opt, bundle_opt, device, quality,
                        initial_image_pairs)


# ---- refinement of caller-supplied models (rp_refine_pairs_host[_f32]) ----------------------------------------
def _model_row(geometry, f1=1.0, f2=1.0):
    """MonoDepthTwoViewGeometry (or a duck-typed one) -> one rp_model: q w-first as the pose stores it, t, scale, shifts,
    and the two focal lengths (1 for the calibrated variants, which do not read them)."""
    m = np.zeros((), dtype=nv.MODEL_DTYPE)
    m["q"] = np.asarray(geometry.pose.q, dtype=np.float64)
    m["t"] = np.asarray(geometry.pose.t, dtype=np.float64)
    m["scale"], m["shift1"], m["shift2"] = geometry.scale, geometry.shift1, geometry.shift2
    m["f1"], m["f2"] = f1, f2
    return m


def _pack_subsets(subsets, offsets):
    """One boolean / 0-1 array per pair (None for a pair: every correspondence) -> packed uint8 [N]; ValueError on a
    pair count or length that does not match the points."""
    n = np.diff(offsets)
    if len(subsets) != len(n):
        raise ValueError(f"subsets needs one entry per pair ({len(n)}), got {len(subsets)}")
    out = []
    for i, (s, k) in enumerate(zip(subsets, n)):
        s = np.ones(k, dtype=np.uint8) if s is None else (np.asarray(s).reshape(-1) != 0).astype(np.uint8)
        if len(s) != k:
            raise ValueError(f"subset of pair {i} has {len(s)} entries for {k} correspondences")
        out.append(s)
    return np.concatenate(out) if out else np.zeros(0, dtype=np.uint8)


def _refine_host(variant, points2D_1, points2D_2, depth_1, depth_2, cams, init, ransac_opt, bundle_opt, subsets, device,
                 focal_variant):
    """Packed refinement of one model per pair: (models, bstats, num_inliers, inliers, offsets)."""
    if not (len(points2D_1) == len(points2D_2) == len(depth_1) == len(depth_2) == len(init)):
        raise ValueError("points, depths and initial models need one entry per pair")
    offsets, x1, x2, d1, d2 = _pack_auto(points2D_1, points2D_2, depth_1, depth_2)
    subset = _pack_subsets(subsets, offsets) if subsets is not None else None
    opt = make_options(ransac_opt, bundle_opt, focal_variant=focal_variant)
    if variant == nv.CALIB and opt.estimate_shift:
        variant = nv.CALIB_SHIFT
    ctx = context(device)
    fn = ctx.refine_pairs_host_f32 if x1.dtype == np.float32 else ctx.refine_pairs_host
    init = np.array(init, dtype=nv.MODEL_DTYPE).reshape(-1)
    return fn(variant, offsets, x1, x2, d1, d2, cams, opt, init, subset) + (offsets,)


def _refine_info(bstats_row, num_inliers, mask):
    n = len(mask)
    return {"iterations": int(bstats_row["iterations"]), "initial_cost": float(bstats_row["initial_cost"]),
            "cost": float(bstats_row["cost"]), "lambda": float(bstats_row["lam"]),
            "invalid_steps": int(bstats_row["invalid_steps"]), "step_norm": float(bstats_row["step_norm"]),
            "grad_norm": float(bstats_row["grad_norm"]), "num_inliers": int(num_inliers),
            "inlier_ratio": float(num_inliers) / n if n else 0.0, "inliers": [bool(b) for b in mask]}


def refine_monodepth_relative_pose_batch(points2D_1, points2D_2, depth_1, depth_2, cameras1, cameras2,
                                         initial_geometries, ransac_opt=None, bundle_opt=None, subsets=None, device=0):
    """The estimator's final refinement (hybrid Sampson + reprojection cost, the bundle options' loss) from caller-supplied
    start geometries, one per pair, instead of RANSAC's models: a tracker's previous poses, another method's poses, or an
    estimate to re-refine with other bundle options.  `subsets` (optional): one boolean array per pair selecting the
    correspondences the refinement uses (None, or a None entry: all of them); a pair with at most 3 selected
    correspondences keeps its start geometry.  Thresholds and `monodepth_estimate_shift` come from `ransac_opt` as for
    the estimator.  Returns a list of (MonoDepthTwoViewGeometry, info): info holds BundleStats (iterations, initial_cost,
    cost, lambda, invalid_steps, step_norm, grad_norm) and num_inliers, inlier_ratio and inliers of the refined model."""
    if not (len(cameras1) == len(cameras2) == len(points2D_1)):
        raise ValueError("cameras1 / cameras2 need one camera per pair")
    cams = np.array([Camera.from_any(a).fxfycxcy() + Camera.from_any(b).fxfycxcy()
                     for a, b in zip(cameras1, cameras2)], dtype=np.float64).reshape(-1, 8)
    init = [_model_row(g) for g in initial_geometries]
    models, bstats, num_inl, inl, offsets = _refine_host(nv.CALIB, points2D_1, points2D_2, depth_1, depth_2, cams, init,
                                                         ransac_opt, bundle_opt, subsets, device, False)
    return [(_geometry(models[i]), _refine_info(bstats[i], num_inl[i], inl[offsets[i]:offsets[i + 1]]))
            for i in range(len(models))]


def _refine_focal_batch(variant, points2D_1, points2D_2, depth_1, depth_2, initial_image_pairs, ransac_opt, bundle_opt,
                        subsets, device):
    init = [_model_row(p.geometry, Camera.from_any(p.camera1).focal(), Camera.from_any(p.camera2).focal())
            for p in initial_image_pairs]
    models, bstats, num_inl, inl, offsets = _refine_host(variant, points2D_1, points2D_2, depth_1, depth_2, None, init,
                                                         ransac_opt, bundle_opt, subsets, device, True)
    out = []
    for i, m in enumerate(models):
        pair = MonoDepthImagePair(_geometry(m), Camera("SIMPLE_PINHOLE", [m["f1"], 0.0, 0.0]),
                                  Camera("SIMPLE_PINHOLE", [m["f2"], 0.0, 0.0]))
        out.append((pair, _refine_info(bstats[i], num_inl[i], inl[offsets[i]:offsets[i + 1]])))
    return out


def refine_monodepth_shared_focal_relative_pose_batch(points2D_1, points2D_2, depth_1, depth_2, initial_image_pairs,
                                                      ransac_opt=None, bundle_opt=None, subsets=None, device=0):
    """`refine_monodepth_relative_pose_batch` for the shared-focal estimator: principal-point-centred points, start
    MonoDepthImagePairs (focal from camera.focal()); returns (MonoDepthImagePair, info) per pair."""
    return _refine_focal_batch(nv.SHARED, points2D_1, points2D_2, depth_1, depth_2, initial_image_pairs, ransac_opt,
                               bundle_opt, subsets, device)


def refine_monodepth_varying_focal_relative_pose_batch(points2D_1, points2D_2, depth_1, depth_2, initial_image_pairs,
                                                       ransac_opt=None, bundle_opt=None, subsets=None, device=0):
    """`refine_monodepth_shared_focal_relative_pose_batch` for the varying-focal estimator."""
    return _refine_focal_batch(nv.VARYING, points2D_1, points2D_2, depth_1, depth_2, initial_image_pairs, ransac_opt,
                               bundle_opt, subsets, device)


def refine_monodepth_relative_pose(points2D_1, points2D_2, depth_1, depth_2, camera1, camera2, initial_geometry,
                                   ransac_opt={}, bundle_opt={}, subset=None):
    """One pair of `refine_monodepth_relative_pose_batch`."""
    return refine_monodepth_relative_pose_batch([points2D_1], [points2D_2], [depth_1], [depth_2], [camera1], [camera2],
                                                [initial_geometry], ransac_opt, bundle_opt,
                                                None if subset is None else [subset])[0]


def refine_monodepth_shared_focal_relative_pose(points2D_1, points2D_2, depth_1, depth_2, initial_image_pair,
                                                ransac_opt={}, bundle_opt={}, subset=None):
    """One pair of `refine_monodepth_shared_focal_relative_pose_batch`."""
    return refine_monodepth_shared_focal_relative_pose_batch([points2D_1], [points2D_2], [depth_1], [depth_2],
                                                             [initial_image_pair], ransac_opt, bundle_opt,
                                                             None if subset is None else [subset])[0]


def refine_monodepth_varying_focal_relative_pose(points2D_1, points2D_2, depth_1, depth_2, initial_image_pair,
                                                 ransac_opt={}, bundle_opt={}, subset=None):
    """One pair of `refine_monodepth_varying_focal_relative_pose_batch`."""
    return refine_monodepth_varying_focal_relative_pose_batch([points2D_1], [points2D_2], [depth_1], [depth_2],
                                                              [initial_image_pair], ransac_opt, bundle_opt,
                                                              None if subset is None else [subset])[0]


# ---- the reference's single-pair surface ---------------------------------------------------------------
def estimate_monodepth_relative_pose(points2D_1, points2D_2, depth_1, depth_2, camera1, camera2,
                                     ransac_opt={}, bundle_opt={}, initial_pose=None):
    """poselib.estimate_monodepth_relative_pose (whl:_core.pyi:446-475).  `initial_pose` is accepted
    and ignored, exactly like the reference (ransac_monodepth_relpose so@0x228c20 resets it)."""
    return estimate_monodepth_relative_pose_batch([points2D_1], [points2D_2], [depth_1], [depth_2], [camera1],
                                                  [camera2], ransac_opt, bundle_opt)[0]


def estimate_monodepth_shared_focal_relative_pose(points2D_1, points2D_2, depth_1, depth_2, ransac_opt={},
                                                  bundle_opt={}, initial_image_pair=None):
    """poselib.estimate_monodepth_shared_focal_relative_pose (whl:_core.pyi:477-488)."""
    return estimate_monodepth_shared_focal_relative_pose_batch([points2D_1], [points2D_2], [depth_1], [depth_2],
                                                               ransac_opt, bundle_opt)[0]


def estimate_monodepth_varying_focal_relative_pose(points2D_1, points2D_2, depth_1, depth_2, ransac_opt={},
                                                   bundle_opt={}, initial_image_pair=None):
    """poselib.estimate_monodepth_varying_focal_relative_pose (whl:_core.pyi:490-501)."""
    return estimate_monodepth_varying_focal_relative_pose_batch([points2D_1], [points2D_2], [depth_1], [depth_2],
                                                                ransac_opt, bundle_opt)[0]


# ---- PoseLib-mdrp fork names used by eval.py / eval_shared_f.py / eval_varying_f.py --------------------
def _fork_ransac(ransac_dict):
    """Experiment flags of eval.py:105-123 -> upstream keys (SURVEY.md §8b fork-API row)."""
    r = dict(ransac_dict)
    r["monodepth_estimate_shift"] = bool(r.get("solver_shift", False)) and bool(r.get("use_ours", False)) \
        and not bool(r.get("use_p3p", False))
    if "weight_sampson" in r:
        r["monodepth_weight_sampson"] = r["weight_sampson"]
    return r


def estimate_relative_pose_w_mono_depth(kp1, kp2, d, camera1, camera2, ransac_dict={}, bundle_dict={}):
    """eval.py:153 — depths arrive as one [N,2] array; returns (CameraPose-like, info)."""
    d = np.asarray(d, dtype=np.float64)
    geom, info = estimate_monodepth_relative_pose(kp1, kp2, d[:, 0], d[:, 1], camera1, camera2,
                                                  _fork_ransac(ransac_dict), bundle_dict)
    return geom.pose, info


def estimate_shared_focal_monodepth_relative_pose(kp1, kp2, d, ransac_dict={}, bundle_dict={}):
    """eval_shared_f.py:177."""
    d = np.asarray(d, dtype=np.float64)
    return estimate_monodepth_shared_focal_relative_pose(kp1, kp2, d[:, 0], d[:, 1], _fork_ransac(ransac_dict),
                                                         bundle_dict)


def estimate_varying_focal_monodepth_relative_pose(kp1, kp2, d, ransac_dict={}, bundle_dict={}):
    """eval_varying_f.py:168."""
    d = np.asarray(d, dtype=np.float64)
    return estimate_monodepth_varying_focal_relative_pose(kp1, kp2, d[:, 0], d[:, 1], _fork_ransac(ransac_dict),
                                                          bundle_dict)


# ---- minimal solvers exposed by the reference (whl:_core.pyi:614, :871, :914) ---------------------------
def _solver(variant, x1, x2, d1, d2):
    x1 = np.asarray(x1, dtype=np.float64).reshape(1, 3, 3)
    x2 = np.asarray(x2, dtype=np.float64).reshape(1, 3, 3)
    models, counts = context(0).solve(variant, x1, x2, np.asarray(d1, dtype=np.float64).reshape(1, 3),
                                      np.asarray(d2, dtype=np.float64).reshape(1, 3))
    return [models[0, k] for k in range(int(counts[0]))]


def monodepth_pose_3pt(x1, x2, d1, d2):
    return [_geometry(m) for m in _solver(nv.CALIB_SHIFT, x1, x2, d1, d2)]


def shared_focal_monodepth_pose_3pt(x1, x2, d1, d2):
    return [MonoDepthImagePair(_geometry(m), Camera("SIMPLE_PINHOLE", [m["f1"], 0, 0]),
                               Camera("SIMPLE_PINHOLE", [m["f2"], 0, 0])) for m in _solver(nv.SHARED, x1, x2, d1, d2)]


def varying_focal_monodepth_pose_4pt(x1, x2, d1, d2):
    return [MonoDepthImagePair(_geometry(m), Camera("SIMPLE_PINHOLE", [m["f1"], 0, 0]),
                               Camera("SIMPLE_PINHOLE", [m["f2"], 0, 0])) for m in _solver(nv.VARYING, x1, x2, d1, d2)]
