"""Device-resident front end (SURVEY.md §8f item 2): torch CUDA tensors straight from the matcher / depth
network into the estimator, without the `.cpu().numpy()` round trip of /root/reference/make_pair.py:97-104.

torch is only plumbing here (device memory and the current stream); every computation is in
librepose_b200.so.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as nv
from . import api


def _ctx_for(t: torch.Tensor) -> nv.Context:
    if not t.is_cuda:
        raise ValueError("expected CUDA tensors (use mdrp_b200.api for host arrays)")
    return api.context(t.device.index or 0)


_GATHER_DTYPES = (torch.float64, torch.float32)


def _gather_fn(ctx, name, dtype, quality):
    if dtype not in _GATHER_DTYPES:
        raise ValueError("dtype must be torch.float64 or torch.float32")
    return getattr(ctx._lib, name + ("_f32" if dtype == torch.float32 else "") + ("_quality" if quality is not None else ""))


def _quality_buffers(quality, keypoints, n):
    """For a gather with a match quality: (the quality as contiguous float32 [n], its output tensor [n], and the two
    pointers the _quality entry point takes after kp2 and after d2, as one-element lists).  Without one: Nones and
    empty lists, so the twin's argument list is unchanged."""
    if quality is None:
        return None, None, [], []
    if not quality.is_cuda or quality.device != keypoints.device:
        raise ValueError("quality must be a CUDA tensor on the device of the keypoints")
    quality = quality.contiguous().to(torch.float32)
    if quality.shape != (n,):
        raise ValueError("quality must be [n], one value per keypoint row")
    q_out = torch.empty(n, dtype=torch.float32, device=keypoints.device)
    return quality, q_out, [quality.data_ptr()], [q_out.data_ptr()]


def gather_depths(depth_map1, depth_map2, keypoints1, keypoints2, dtype=torch.float64, quality=None):
    """depths at the matched keypoints + removal of rows whose depths are both inf (make_pair.py:97-106),
    on the device.  depth maps: [H,W] float32 CUDA; keypoints: [n,2] float32 CUDA (x, y).
    Returns (x1, x2, d1, d2) CUDA tensors of `dtype` (float64, or float32: the values unchanged, what `estimate_batch`
    takes without an FP64 copy) with the kept rows in order.
    `quality` (optional): CUDA tensor [n] of match qualities (converted to float32); the kept rows' qualities are then
    returned as a fifth element, float32 [m], bit for bit and aligned with the other outputs: the `quality` that
    `estimate_batch` takes for them."""
    ctx = _ctx_for(depth_map1)
    fn = _gather_fn(ctx, "rp_gather_depths_dev", dtype, quality)
    dm1 = depth_map1.contiguous().float()
    dm2 = depth_map2.contiguous().float()
    k1 = keypoints1.contiguous().float()
    k2 = keypoints2.contiguous().float()
    n = k1.shape[0]
    dev = dm1.device
    x1 = torch.empty(n, 2, dtype=dtype, device=dev)
    x2 = torch.empty(n, 2, dtype=dtype, device=dev)
    d1 = torch.empty(n, dtype=dtype, device=dev)
    d2 = torch.empty(n, dtype=dtype, device=dev)
    n_out = C.c_int64(0)
    q, q_out, q_in_p, q_out_p = _quality_buffers(quality, k1, n)
    stream = torch.cuda.current_stream(dev).cuda_stream
    ctx._call(fn, ctx._h, dm1.data_ptr(), dm1.shape[0], dm1.shape[1], dm2.data_ptr(),
              dm2.shape[0], dm2.shape[1], k1.data_ptr(), k2.data_ptr(), *q_in_p, n, x1.data_ptr(), x2.data_ptr(),
              d1.data_ptr(), d2.data_ptr(), *q_out_p, C.byref(n_out), stream)
    m = n_out.value
    return (x1[:m], x2[:m], d1[:m], d2[:m]) + (() if q_out is None else (q_out[:m],))


def gather_depths_batch(depth_maps, frame1, frame2, offsets, keypoints1, keypoints2, dtype=torch.float64, quality=None):
    """`gather_depths` for a batch of pairs in one call (a video: make_video.py:270-290).  depth_maps: [F,H,W] float32
    CUDA; frame1 / frame2: per-pair frame indices; offsets: [P+1] rows of the packed keypoints [N,2] float32 CUDA.
    Returns (out_offsets int64 numpy, x1, x2, d1, d2) — the packed CUDA tensors of `dtype` (float64 or float32)
    `estimate_batch` takes.  `quality` (optional): CUDA tensor [N] of match qualities; the packed float32 qualities of
    the kept rows are then returned as a sixth element, ready for `estimate_batch(..., quality=...)`."""
    ctx = _ctx_for(depth_maps)
    fn = _gather_fn(ctx, "rp_gather_depths_batch_dev", dtype, quality)
    dm = depth_maps.contiguous().float()
    k1, k2 = keypoints1.contiguous().float(), keypoints2.contiguous().float()
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    f1 = np.ascontiguousarray(frame1, dtype=np.int32)
    f2 = np.ascontiguousarray(frame2, dtype=np.int32)
    P, n, dev = len(offsets) - 1, k1.shape[0], dm.device
    if len(f1) != P or len(f2) != P or int(offsets[-1]) - int(offsets[0]) != n:
        raise ValueError("frame1 / frame2 need one entry per pair and offsets must cover the keypoints")
    x1 = torch.empty(n, 2, dtype=dtype, device=dev)
    x2 = torch.empty(n, 2, dtype=dtype, device=dev)
    d1 = torch.empty(n, dtype=dtype, device=dev)
    d2 = torch.empty(n, dtype=dtype, device=dev)
    out = np.zeros(P + 1, dtype=np.int64)
    q, q_out, q_in_p, q_out_p = _quality_buffers(quality, k1, n)
    ctx._call(fn, ctx._h, P, offsets.ctypes.data, dm.data_ptr(), dm.shape[0], dm.shape[1],
              dm.shape[2], f1.ctypes.data, f2.ctypes.data, k1.data_ptr(), k2.data_ptr(), *q_in_p, x1.data_ptr(),
              x2.data_ptr(), d1.data_ptr(), d2.data_ptr(), *q_out_p, out.ctypes.data, torch.cuda.current_stream(dev).cuda_stream)
    m = int(out[-1])
    return (out, x1[:m], x2[:m], d1[:m], d2[:m]) + (() if q_out is None else (q_out[:m],))


def estimate_batch(variant, offsets, x1, x2, d1, d2, cams, opt: nv.Options, quality=None):
    """Packed CUDA float64 tensors in (offsets: host int64 array), CUDA tensors out:
    models [P,12] float64, stats [P,5] (int64 view; columns 3,4 are float64 bit patterns — use
    `stats_to_numpy`), masks [N] uint8.  When x1, x2, d1, d2 are all float32 they are passed as they are to the
    float32 entry point (no FP64 copy of the batch; the same results as float64 tensors of the same values).
    `quality` (optional): CUDA tensor [N] of match qualities, converted to float32 on the device; each pair is then
    ordered by decreasing quality before the estimator runs (rp_estimate_batch_dev[_f32]_quality), and the masks come
    back in the caller's order."""
    ctx = _ctx_for(x1)
    dev = x1.device
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    P, N = len(offsets) - 1, int(offsets[-1])
    f32 = all(t.dtype == torch.float32 for t in (x1, x2, d1, d2))
    t64 = lambda t: t.contiguous().to(torch.float64)
    tin = (lambda t: t.contiguous()) if f32 else t64
    x1, x2, d1, d2 = tin(x1), tin(x2), tin(d1), tin(d2)
    if x1.shape != (N, 2) or x2.shape != (N, 2) or d1.shape != (N,) or d2.shape != (N,):
        raise ValueError("x1/x2 must be [N,2] and d1/d2 [N] with N = offsets[-1]")
    cams_t = t64(cams) if cams is not None else None
    if quality is not None:
        if not quality.is_cuda or quality.device != dev:
            raise ValueError("quality must be a CUDA tensor on the device of the points")
        quality = quality.contiguous().to(torch.float32)
        if quality.shape != (N,):
            raise ValueError("quality must be [N] with N = offsets[-1]")
    models = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    stats = torch.zeros(P, 5, dtype=torch.int64, device=dev)
    masks = torch.zeros(max(N, 1), dtype=torch.uint8, device=dev)
    outs = (models.data_ptr(), stats.data_ptr(), masks.data_ptr())
    stream = torch.cuda.current_stream(dev).cuda_stream
    cams_p = cams_t.data_ptr() if cams_t is not None else None
    if quality is not None:
        est = ctx.estimate_batch_dev_f32_quality if f32 else ctx.estimate_batch_dev_quality
        est(variant, offsets, x1.data_ptr(), x2.data_ptr(), d1.data_ptr(), d2.data_ptr(), cams_p, opt, *outs,
            quality.data_ptr(), stream)
    else:
        est = ctx.estimate_batch_dev_f32 if f32 else ctx.estimate_batch_dev
        est(variant, offsets, x1.data_ptr(), x2.data_ptr(), d1.data_ptr(), d2.data_ptr(), cams_p, opt, *outs, stream)
    return models, stats, masks[:N]


def refine_batch(variant, offsets, x1, x2, d1, d2, cams, init_models, opt: nv.Options, subset=None):
    """The estimator's final refinement from caller-supplied start models (rp_refine_pairs_dev[_f32]) on CUDA tensors:
    init_models [P,12] float64 (e.g. the `models` of a previous `estimate_batch` or `refine_batch`), `subset` (optional)
    [N] CUDA tensor, nonzero = used by the refinement.  Inputs as in `estimate_batch` (float32 passes through, anything
    else is converted to float64).  Returns (models [P,12] float64, bstats [P,7] (int64 view; columns 1-3, 5, 6 are
    float64 bit patterns — use `bstats_to_numpy`), num_inliers [P] int64, inliers [N] uint8), all on the device."""
    ctx = _ctx_for(x1)
    dev = x1.device
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    P, N = len(offsets) - 1, int(offsets[-1])
    f32 = all(t.dtype == torch.float32 for t in (x1, x2, d1, d2))
    t64 = lambda t: t.contiguous().to(torch.float64)
    tin = (lambda t: t.contiguous()) if f32 else t64
    x1, x2, d1, d2 = tin(x1), tin(x2), tin(d1), tin(d2)
    if x1.shape != (N, 2) or x2.shape != (N, 2) or d1.shape != (N,) or d2.shape != (N,):
        raise ValueError("x1/x2 must be [N,2] and d1/d2 [N] with N = offsets[-1]")
    init = t64(init_models)
    if init.shape != (P, 12) or not init.is_cuda or init.device != dev:
        raise ValueError("init_models must be a [P,12] CUDA tensor on the device of the points")
    if subset is not None:
        if not subset.is_cuda or subset.device != dev or subset.shape != (N,):
            raise ValueError("subset must be a CUDA tensor [N] on the device of the points")
        subset = (subset != 0).to(torch.uint8).contiguous()
    cams_t = t64(cams) if cams is not None else None
    models = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    bstats = torch.zeros(P, 7, dtype=torch.int64, device=dev)
    num_inliers = torch.zeros(P, dtype=torch.int64, device=dev)
    inliers = torch.zeros(max(N, 1), dtype=torch.uint8, device=dev)
    fn = ctx.refine_pairs_dev_f32 if f32 else ctx.refine_pairs_dev
    fn(variant, offsets, x1.data_ptr(), x2.data_ptr(), d1.data_ptr(), d2.data_ptr(),
       cams_t.data_ptr() if cams_t is not None else None, opt, init.data_ptr(),
       subset.data_ptr() if subset is not None else None, models.data_ptr(), bstats.data_ptr(), num_inliers.data_ptr(),
       inliers.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    return models, bstats, num_inliers, inliers[:N]


def bstats_to_numpy(bstats: torch.Tensor) -> np.ndarray:
    return bstats.cpu().numpy().view(nv.BSTATS_DTYPE).reshape(-1)


def stats_to_numpy(stats: torch.Tensor) -> np.ndarray:
    return stats.cpu().numpy().view(nv.STATS_DTYPE).reshape(-1)


def estimate_monodepth_relative_pose(points2D_1, points2D_2, depth_1, depth_2, camera1, camera2, ransac_opt={},
                                     bundle_opt={}, initial_pose=None, quality=None):
    """poselib.estimate_monodepth_relative_pose with CUDA tensor inputs; same return objects.  float32 points and
    depths take the float32 path of `estimate_batch`; `quality` (optional CUDA tensor [n]) is passed on to it."""
    opt = api.make_options(ransac_opt, bundle_opt, focal_variant=False)
    cams = torch.tensor([api.Camera.from_any(camera1).fxfycxcy() + api.Camera.from_any(camera2).fxfycxcy()],
                        dtype=torch.float64, device=points2D_1.device)
    n = points2D_1.shape[0]
    variant = nv.CALIB_SHIFT if opt.estimate_shift else nv.CALIB
    models, stats, masks = estimate_batch(variant, [0, n], points2D_1, points2D_2, depth_1, depth_2, cams, opt,
                                         quality=quality)
    m = models[0].cpu().numpy()
    st = stats_to_numpy(stats)[0]
    geom = api.MonoDepthTwoViewGeometry(api.CameraPose(m[:4], m[4:7]), m[7], m[8], m[9])
    return geom, api._info(st, masks.cpu().numpy())
