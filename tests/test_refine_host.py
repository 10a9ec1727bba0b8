"""CPU tier of the refinement of caller-supplied models (rp_refine_pairs_*): the C declarations and ctypes signatures,
which entry point `api` picks for which dtypes, how `api` turns geometries and image pairs into rp_model rows, and its
length checks (no device: recording stand-ins)."""
import ctypes as C

import numpy as np
import pytest

from test_quality_order_host import _RecordingCtx, _fake_load, _header, _params

EST_ARGS = ["rp_ctx *ctx", "int variant", "int64_t n_pairs", "const int64_t *offsets", "const {T} *x1", "const {T} *x2",
            "const {T} *d1", "const {T} *d2", "const double *cams", "const rp_options *opt"]
REFINE_TAIL = ["const rp_model *init", "const uint8_t *subset", "rp_model *models", "rp_bundle_stats *bstats",
               "int64_t *num_inliers", "uint8_t *inliers"]
REFINE = {"rp_refine_pairs_host": ("double", False), "rp_refine_pairs_dev": ("double", True),
          "rp_refine_pairs_host_f32": ("float", False), "rp_refine_pairs_dev_f32": ("float", True)}


def test_refine_declarations():
    header = _header()
    for name, (t, dev) in REFINE.items():
        want = [a.format(T=t) for a in EST_ARGS] + REFINE_TAIL + (["void *stream"] if dev else [])
        assert _params(header, name) == want, name


def test_refine_ctypes_signatures(monkeypatch):
    from mdrp_b200 import _native as nv
    L = _fake_load(monkeypatch)
    VP = C.c_void_p
    for name, (_, dev) in REFINE.items():
        assert name in nv.EXPORTS
        f = getattr(L, name)
        assert f.restype is C.c_int
        assert f.argtypes == [VP, C.c_int, C.c_int64, VP, VP, VP, VP, VP, VP, C.POINTER(nv.Options)] + [VP] * 6 + \
            ([VP] if dev else [])


class _RefineRecorder(_RecordingCtx):
    """Records the refine entry point, the input dtypes and the packed start models / subset."""

    def _refine(self, name, offsets, x1, x2, d1, d2, init, subset):
        from mdrp_b200 import _native as nv
        self.calls.append((name, x1.dtype, x2.dtype, d1.dtype, d2.dtype))
        self.init, self.subset = init, subset
        P, N = len(offsets) - 1, int(offsets[-1])
        return (np.array(init, nv.MODEL_DTYPE), np.zeros(P, nv.BSTATS_DTYPE), np.arange(P, dtype=np.int64),
                np.ones(N, np.uint8))

    def refine_pairs_host(self, variant, offsets, x1, x2, d1, d2, cams, opt, init, subset=None):
        self.variant, self.cams = variant, cams
        return self._refine("f64", offsets, x1, x2, d1, d2, init, subset)

    def refine_pairs_host_f32(self, variant, offsets, x1, x2, d1, d2, cams, opt, init, subset=None):
        self.variant, self.cams = variant, cams
        return self._refine("f32", offsets, x1, x2, d1, d2, init, subset)


@pytest.fixture
def rec(monkeypatch):
    from mdrp_b200 import api
    r = _RefineRecorder()
    monkeypatch.setattr(api, "context", lambda device=0: r)
    return r


def _geom(api, angle=0.3):
    q = np.array([np.cos(angle / 2), 0.0, np.sin(angle / 2), 0.0])
    return api.MonoDepthTwoViewGeometry(api.CameraPose(q, [0.1, -0.2, 0.3]), 1.5, 0.25, -0.5)


def test_api_refine_routes_by_dtype(rec):
    from mdrp_b200 import api, _native as nv
    f32 = lambda *s: np.ones(s, np.float32)
    f64 = lambda *s: np.ones(s)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    g = _geom(api)
    F, D = np.dtype(np.float32), np.dtype(np.float64)
    api.refine_monodepth_relative_pose_batch([f32(5, 2)], [f32(5, 2)], [f32(5)], [f32(5)], [cam], [cam], [g])
    api.refine_monodepth_relative_pose_batch([f32(5, 2)], [f64(5, 2)], [f32(5)], [f32(5)], [cam], [cam], [g])
    api.refine_monodepth_shared_focal_relative_pose_batch([f32(4, 2)], [f32(4, 2)], [f32(4)], [f32(4)],
                                                          [api.MonoDepthImagePair(g)])
    api.refine_monodepth_varying_focal_relative_pose_batch([f32(3, 2)], [f32(3, 2)], [f32(3)], [f64(3)],
                                                           [api.MonoDepthImagePair(g)])
    api.refine_monodepth_varying_focal_relative_pose(f64(3, 2), f64(3, 2), f64(3), f64(3), api.MonoDepthImagePair(g))
    assert rec.calls == [("f32", F, F, F, F), ("f64", D, D, D, D), ("f32", F, F, F, F), ("f64", D, D, D, D),
                         ("f64", D, D, D, D)]
    assert rec.variant == nv.VARYING and rec.cams is None
    api.refine_monodepth_relative_pose_batch([f64(5, 2)], [f64(5, 2)], [f64(5)], [f64(5)], [cam], [cam], [g],
                                             ransac_opt={"monodepth_estimate_shift": True})
    assert rec.variant == nv.CALIB_SHIFT
    assert rec.cams.tolist() == [[800.0, 800.0, 640.0, 480.0] * 2]


def test_api_refine_model_conversion(rec):
    from mdrp_b200 import api
    g = _geom(api)
    cam = {"model": "PINHOLE", "params": [700.0, 720.0, 640.0, 480.0]}
    pts = np.zeros((6, 2))
    res = api.refine_monodepth_relative_pose_batch([pts], [pts], [np.ones(6)], [np.ones(6)], [cam], [cam], [g],
                                                   subsets=[[1, 0, 2, 0, 1, 1]])
    m = rec.init[0]
    assert m["q"].tolist() == g.pose.q.tolist()   # w first, as the pose stores it
    assert m["t"].tolist() == [0.1, -0.2, 0.3]
    assert (m["scale"], m["shift1"], m["shift2"], m["f1"], m["f2"]) == (1.5, 0.25, -0.5, 1.0, 1.0)
    assert rec.subset.tolist() == [1, 0, 1, 0, 1, 1] and rec.subset.dtype == np.uint8
    # the returned geometry is the model row the entry point returned (here: the start model)
    geom, info = res[0]
    assert np.array_equal(geom.pose.R, g.pose.R) and geom.pose.q.tolist() == g.pose.q.tolist()
    assert (geom.scale, geom.shift1, geom.shift2) == (1.5, 0.25, -0.5)
    assert set(info) == {"iterations", "initial_cost", "cost", "lambda", "invalid_steps", "step_norm", "grad_norm",
                         "num_inliers", "inlier_ratio", "inliers"}
    assert info["num_inliers"] == 0 and info["inliers"] == [True] * 6
    # focal variants: f from camera.focal() of each camera; the result's cameras carry the returned f1 / f2
    pair = api.MonoDepthImagePair(g, api.Camera("PINHOLE", [700.0, 720.0, 0, 0]), api.Camera("SIMPLE_PINHOLE", [900.0, 0, 0]))
    out_pair, _ = api.refine_monodepth_varying_focal_relative_pose(pts, pts, np.ones(6), np.ones(6), pair)
    assert (rec.init[0]["f1"], rec.init[0]["f2"]) == (710.0, 900.0)
    assert out_pair.camera1.focal() == 710.0 and out_pair.camera2.focal() == 900.0
    assert rec.subset is None


def test_api_refine_length_mismatches(rec):
    from mdrp_b200 import api
    g = _geom(api)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    p5, d5 = np.zeros((5, 2)), np.ones(5)
    good = ([p5, p5], [p5, p5], [d5, d5], [d5, d5], [cam, cam], [cam, cam])
    with pytest.raises(ValueError):   # one start model for two pairs
        api.refine_monodepth_relative_pose_batch(*good, [g])
    with pytest.raises(ValueError):   # one subset for two pairs
        api.refine_monodepth_relative_pose_batch(*good, [g, g], subsets=[np.ones(5)])
    with pytest.raises(ValueError):   # a subset of the wrong length
        api.refine_monodepth_relative_pose_batch(*good, [g, g], subsets=[np.ones(5), np.ones(4)])
    with pytest.raises(ValueError):   # points and depths of different lengths
        api.refine_monodepth_relative_pose_batch([p5, p5], [p5, p5], [d5, np.ones(4)], [d5, d5], [cam, cam],
                                                 [cam, cam], [g, g])
    with pytest.raises(ValueError):   # one camera too few
        api.refine_monodepth_relative_pose_batch(*good[:4], [cam], [cam, cam], [g, g])
    with pytest.raises(ValueError):   # a depth list of another pair count
        api.refine_monodepth_shared_focal_relative_pose_batch([p5, p5], [p5, p5], [d5], [d5, d5],
                                                              [api.MonoDepthImagePair(g)] * 2)
    with pytest.raises(ValueError):   # distortion cameras are refused as for the estimator
        api.refine_monodepth_relative_pose_batch([p5], [p5], [d5], [d5], [{"model": "OPENCV", "params": [1] * 8}],
                                                 [cam], [g])
    with pytest.raises(NotImplementedError):
        api.refine_monodepth_relative_pose_batch([p5], [p5], [d5], [d5], [cam], [cam], [g],
                                                 bundle_opt={"loss_type": "TRUNCATED_LE_ZACH"})
    assert rec.calls == []
    # None entries of `subsets` select every correspondence of their pair
    api.refine_monodepth_relative_pose_batch(*good, [g, g], subsets=[None, np.arange(5) % 2 == 0])
    assert rec.subset.tolist() == [1] * 5 + [1, 0, 1, 0, 1]


def test_refine_names_stay_out_of_compat():
    import mdrp_b200.compat.poselib as compat
    assert not [n for n in dir(compat) if n.startswith("refine_monodepth")]


def test_torch_refine_routes_by_dtype(monkeypatch):
    torch = pytest.importorskip("torch")
    from mdrp_b200 import torch_frontend as tf, _native as nv

    class Rec:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            if not name.startswith("refine_pairs_dev"):
                raise AttributeError(name)
            return lambda *a: self.calls.append((name, a))
    rec = Rec()
    monkeypatch.setattr(tf, "_ctx_for", lambda t: rec)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: type("S", (), {"cuda_stream": 0})())
    real_zeros = torch.zeros
    monkeypatch.setattr(torch, "zeros", lambda *a, **k: real_zeros(*a, **{**k, "device": "cpu"}))
    offs = np.array([0, 3, 5], dtype=np.int64)
    x32, d32 = torch.ones(5, 2), torch.ones(5)
    init = torch.zeros(2, 12, dtype=torch.float64)
    o = nv.Options()
    tf.refine_batch(nv.SHARED, offs, x32, x32, d32, d32, None, init, o)
    tf.refine_batch(nv.SHARED, offs, x32.double(), x32, d32, d32, None, init, o, subset=torch.ones(5))
    names = [n for n, _ in rec.calls]
    assert names == ["refine_pairs_dev_f32", "refine_pairs_dev"]
    assert all(len(a) == 15 for _, a in rec.calls)
    assert rec.calls[0][1][9] is None   # no subset
    with pytest.raises(ValueError):
        tf.refine_batch(nv.SHARED, offs, x32, x32, d32, d32, None, init[:1], o)
    with pytest.raises(ValueError):
        tf.refine_batch(nv.SHARED, offs, x32, x32, d32, d32, None, init, o, subset=torch.ones(4))
