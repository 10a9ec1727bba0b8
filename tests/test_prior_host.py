"""CPU tier of estimation from a prior (rp_estimate_batch_*_init): the oracle's prior semantics (ro_ransac_prior /
ro_estimate_prior in tests/priororacle), the C declarations and ctypes signatures, and how `api` and `torch_frontend`
pack priors (no device: recording stand-ins)."""
import ctypes as C

import numpy as np
import pytest

from test_quality_order_host import _fake_load, _header, _params
import prior_oracle as po
from util import models_close

VARIANTS = (0, 1, 2, 3)
F = 800.0   # the scenes' focal length, f1 = f2 for the calibrated and shared variants


def _scene(variant, index, n=60, outliers=0.4):
    from mdrp_b200 import synth
    kw = dict(outlier_ratio=outliers)
    if variant == 1:
        kw.update(shift1=0.3, shift2=-0.2)
    if variant == 3:
        kw.update(f1=700.0, f2=900.0)
    return synth.make_scene(index, n, **kw)


def _normalised(sc):
    """Points in a normalised frame (principal point removed, divided by F): what ro_ransac expects."""
    return (sc.x1 - [640.0, 480.0]) / F, (sc.x2 - [640.0, 480.0]) / F


def _prior(port, variant, sc, rot_noise_deg, seed, frame_scale=F):
    from mdrp_b200 import synth
    v = synth.gt_model(sc, rot_noise_deg, seed)
    if variant < 2:
        v[10:] = 1.0
    else:
        v[10:] /= frame_scale
    return port.make_model(v[:4], v[4:7], *v[7:])


def _ransac_opt(port, variant, **kw):
    base = dict(max_iterations=60, min_iterations=60, max_epipolar_error=2.0 / F, max_reproj_error=16.0 / F, seed=7,
                estimate_shift=variant == 1)
    base.update(kw)
    return port.ransac_opt(**base)


def _same(a, b):
    (m1, s1, k1), (m2, s2, k2) = a, b
    return bytes(m1) == bytes(m2) and bytes(s1) == bytes(s2) and np.array_equal(k1, k2)


def _score(port, variant, m, x1, x2, sq_thr):
    if variant < 2:
        return port.msac_score_pose(m.q, m.t, x1, x2, sq_thr)
    return port.msac_score_F(port.fundamental_from_model(m), x1, x2, sq_thr)


def _lo(port, variant, m, x1, x2, d1, d2, ro):
    """The in-loop LO of ro_ransac: TRUNCATED, 25 iterations, the variant's LO loss scale."""
    sr = (ro.max_epipolar_error / ro.max_reproj_error) ** 2
    scale = 1.0 if variant == 3 else ro.max_epipolar_error
    out, _ = port.refine(variant, x1, x2, d1, d2, m, sr, ro.weight_sampson,
                         port.bundle_opt(max_iterations=25, loss_type="TRUNCATED", loss_scale=scale))
    return out


def test_no_prior_is_the_oracle_on_the_goldens(e2e_golden, port):
    """prior=None and an all-NaN prior through ro_estimate_prior give the reference's outputs on the golden cases, byte
    for byte the unchanged oracle's ro_estimate."""
    g = e2e_golden
    keys = sorted(k[:-6] for k in g.files if k.endswith("_model"))
    assert len(keys) >= 15
    nan = port.make_model(*([np.full(4, np.nan), np.full(3, np.nan)] + [np.nan] * 5))
    for key in keys:
        name = key.split("_cfg")[0].split("_hard")[0]
        variant = {"calib": 0, "calib_shift": 1, "shared": 2, "varying": 3, "calib_default_iters": 0}[name]
        iters = int(g[key + "_iters"][0])
        ro = port.ransac_opt(max_iterations=iters if iters > 0 else 5000, min_iterations=iters if iters > 0 else 100,
                             max_epipolar_error=2.0, max_reproj_error=16.0, seed=int(key[-1]), estimate_shift=variant == 1)
        f1, f2 = g[key + "_f"]
        cams = ([f1, f1, 640, 480], [f2, f2, 640, 480]) if variant < 2 else (None, None)
        bo = port.bundle_opt(loss_type="TRUNCATED_CAUCHY", loss_scale=1.0)
        args = (variant, g[key + "_x1"], g[key + "_x2"], g[key + "_d1"], g[key + "_d2"], *cams, ro, bo)
        m, st, mask = po.estimate(*args, prior=None)
        assert _same(port.estimate(*args), (m, st, mask)), key
        assert (st.refinements, st.iterations, st.num_inliers) == tuple(int(v) for v in g[key + "_stats"]), key
        assert (mask == g[key + "_mask"].astype(bool)).all(), key
        assert models_close(m, g[key + "_model"], rtol=1e-8, atol=1e-10), key
        assert _same(po.estimate(*args, prior=nan), (m, st, mask)), key


@pytest.mark.parametrize("variant", VARIANTS)
def test_nan_prior_is_no_prior(port, variant):
    sc = _scene(variant, 11)
    x1, x2 = _normalised(sc)
    ro = _ransac_opt(port, variant)
    plain = port.ransac(variant, x1, x2, sc.d1, sc.d2, ro)
    for field in ("q", "t", "scale", "shift2") + (("f1",) if variant >= 2 else ()):
        p = _prior(port, variant, sc, 2.0, 1)
        if field in ("q", "t"):
            getattr(p, field)[1 if field == "q" else 0] = np.nan
        else:
            setattr(p, field, np.nan)
        assert _same(po.ransac(variant, x1, x2, sc.d1, sc.d2, ro, prior=p), plain), field
    if variant < 2:
        # the calibrated variants do not read f1 / f2: a NaN there still is a prior
        p = _prior(port, variant, sc, 2.0, 1)
        p.f1 = np.nan
        _, st, _ = po.ransac(variant, x1, x2, sc.d1, sc.d2, ro, prior=p)
        assert st.refinements == po.ransac(variant, x1, x2, sc.d1, sc.d2, ro, prior=_prior(port, variant, sc, 2.0, 1))[1].refinements


@pytest.mark.parametrize("variant", VARIANTS)
def test_prior_invariants_on_random_scenes(port, variant):
    """model_score <= min(score(prior), score(LO(prior))); iterations count sampled iterations only; the prior's LO is one
    refinement more than a plain run sees before its first iteration.  Priors: perturbed ground truth, garbage, and the
    plain run's own result."""
    rng = np.random.default_rng(variant)
    for case in range(6):
        sc = _scene(variant, 100 + case, n=int(rng.choice([25, 60, 120])), outliers=float(rng.choice([0.2, 0.6])))
        x1, x2 = _normalised(sc)
        sq_thr = (2.0 / F) ** 2
        ro = _ransac_opt(port, variant, seed=int(rng.integers(0, 1000)))
        plain_model, plain_st, _ = port.ransac(variant, x1, x2, sc.d1, sc.d2, ro)
        garbage = port.make_model([0.6, 0.8, 0, 0], [1.0, 0, 0], 0.5, 0.0, 0.0, 1.3, 0.7)
        for prior in (_prior(port, variant, sc, 3.0, case), garbage, plain_model):
            m, st, mask = po.ransac(variant, x1, x2, sc.d1, sc.d2, ro, prior=prior)
            s0, _ = _score(port, variant, prior, x1, x2, sq_thr)
            s_lo, _ = _score(port, variant, _lo(port, variant, prior, x1, x2, sc.d1, sc.d2, ro), x1, x2, sq_thr)
            assert st.model_score <= min(s0, s_lo)
            assert st.refinements >= 2   # the prior's LO and the final LO
            assert st.iterations == ro.max_iterations   # fixed iterations: the prior is not an iteration
            assert mask.sum() == st.num_inliers or st.num_inliers <= 3
        # the estimator's own result as prior never makes the result worse
        _, st, _ = po.ransac(variant, x1, x2, sc.d1, sc.d2, ro, prior=plain_model)
        assert st.model_score <= plain_st.model_score


@pytest.mark.parametrize("variant", VARIANTS)
def test_zero_iterations_is_the_lo_of_the_prior(port, variant):
    sc = _scene(variant, 21)
    x1, x2 = _normalised(sc)
    ro = _ransac_opt(port, variant, max_iterations=0, min_iterations=0)
    p = _prior(port, variant, sc, 2.0, 5)
    m, st, _ = po.ransac(variant, x1, x2, sc.d1, sc.d2, ro, prior=p)
    assert (st.refinements, st.iterations) == (2, 0)
    lo = _lo(port, variant, p, x1, x2, sc.d1, sc.d2, ro)
    s0, _ = _score(port, variant, p, x1, x2, (2.0 / F) ** 2)
    s_lo, _ = _score(port, variant, lo, x1, x2, (2.0 / F) ** 2)
    assert st.model_score == min(s0, s_lo)
    # without a prior nothing is found: identity, no score
    _, st0, _ = port.ransac(variant, x1, x2, sc.d1, sc.d2, ro)
    assert (st0.refinements, st0.iterations, st0.model_score) == (1, 0, np.finfo(np.float64).max)
    # the same through ro_estimate, with the focal variants' f in pixels
    cam = [sc.f1, sc.f1, 640.0, 480.0] if variant < 2 else None
    a1, a2 = (sc.x1, sc.x2) if variant < 2 else (sc.x1 - [640.0, 480.0], sc.x2 - [640.0, 480.0])
    ro_px = port.ransac_opt(max_iterations=0, min_iterations=0, max_epipolar_error=2.0, max_reproj_error=16.0,
                            estimate_shift=variant == 1)
    from mdrp_b200 import synth
    v = synth.gt_model(sc, 0.02, 5)   # a prior close enough for inliers at 2 px
    m, st, _ = po.estimate(variant, a1, a2, sc.d1, sc.d2, cam, cam, ro_px, port.bundle_opt(),
                             prior=port.make_model(v[:4], v[4:7], *v[7:]))
    assert (st.refinements, st.iterations) == (2, 0) and st.num_inliers > 10


def test_degenerate_pairs_ignore_the_prior(port):
    sc = _scene(0, 3)
    x1, x2 = _normalised(sc)
    ro = _ransac_opt(port, 0)
    p = _prior(port, 0, sc, 1.0, 0)
    a = po.ransac(0, x1[:2], x2[:2], sc.d1[:2], sc.d2[:2], ro, prior=p)
    b = port.ransac(0, x1[:2], x2[:2], sc.d1[:2], sc.d2[:2], ro)
    assert _same(a, b) and a[1].iterations == 0 and models_close(a[0], port.make_model())


# ---- the C ABI and the Python packing --------------------------------------------------------------------------------
INIT = {"rp_estimate_batch_host_init": ("rp_estimate_batch_host_quality", False),
        "rp_estimate_batch_dev_init": ("rp_estimate_batch_dev_quality", True),
        "rp_estimate_batch_host_f32_init": ("rp_estimate_batch_host_f32_quality", False),
        "rp_estimate_batch_dev_f32_init": ("rp_estimate_batch_dev_f32_quality", True)}


def test_init_declarations_are_quality_twin_plus_init():
    header = _header()
    for name, (twin, _) in INIT.items():
        a, b = _params(header, name), _params(header, twin)
        i = b.index("const rp_options *opt")
        assert a == b[:i + 1] + ["const rp_model *init"] + b[i + 1:], (name, a, b)


def test_init_ctypes_signatures(monkeypatch):
    from mdrp_b200 import _native as nv
    L = _fake_load(monkeypatch)
    VP = C.c_void_p
    for name, (twin, dev) in INIT.items():
        assert name in nv.EXPORTS
        f = getattr(L, name)
        assert f.restype is C.c_int
        assert f.argtypes == [VP, C.c_int, C.c_int64, VP, VP, VP, VP, VP, VP, VP, C.POINTER(nv.Options), VP, VP, VP, VP] + \
            ([VP] if dev else [])


def test_init_symbols_exported():
    """The four entry points are in the built library (skipped where it has not been built)."""
    import os
    from mdrp_b200 import _native as nv
    if not os.path.exists(nv.SO_PATH):
        pytest.skip("library not built")
    lib = C.CDLL(nv.SO_PATH)
    for name in INIT:
        assert hasattr(lib, name), name


class _InitRecorder:
    """Stands in for nv.Context: records the prior calls' packed priors and quality."""

    def __init__(self):
        self.calls = []

    def estimate_batch_host_init(self, variant, offsets, x1, x2, d1, d2, cams, opt, init, quality=None):
        from mdrp_b200 import _native as nv
        self.calls.append((variant, x1.dtype, quality is not None))
        self.init = init
        P = len(offsets) - 1
        return np.zeros(P, nv.MODEL_DTYPE), np.zeros(P, nv.STATS_DTYPE), np.zeros(int(offsets[-1]), np.uint8)


@pytest.fixture
def rec(monkeypatch):
    from mdrp_b200 import api
    r = _InitRecorder()
    monkeypatch.setattr(api, "context", lambda device=0: r)
    return r


def test_api_packs_priors_with_nan_rows(rec):
    from mdrp_b200 import api, _native as nv
    q = np.array([np.cos(0.1), 0.0, np.sin(0.1), 0.0])
    g = api.MonoDepthTwoViewGeometry(api.CameraPose(q, [0.1, -0.2, 0.3]), 1.5, 0.25, -0.5)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    p5, d5 = np.zeros((5, 2)), np.ones(5)
    api.estimate_monodepth_relative_pose_batch([p5, p5], [p5, p5], [d5, d5], [d5, d5], [cam, cam], [cam, cam],
                                               initial_geometries=[None, g])
    assert rec.calls == [(nv.CALIB, np.dtype(np.float64), False)]
    assert rec.init.dtype == nv.MODEL_DTYPE and rec.init.shape == (2,)
    assert np.isnan(rec.init.view(np.float64).reshape(2, 12)[0]).all()
    row = rec.init[1]
    assert row["q"].tolist() == q.tolist() and row["t"].tolist() == [0.1, -0.2, 0.3]
    assert (row["scale"], row["shift1"], row["shift2"], row["f1"], row["f2"]) == (1.5, 0.25, -0.5, 1.0, 1.0)
    # focal variants: f from the cameras of the image pair; quality passes along
    pair = api.MonoDepthImagePair(g, api.Camera("SIMPLE_PINHOLE", [700.0, 0, 0]), api.Camera("PINHOLE", [880.0, 900.0, 0, 0]))
    api.estimate_monodepth_varying_focal_relative_pose_batch([p5], [p5], [d5], [d5], initial_image_pairs=[pair],
                                                             quality=[np.arange(5.0)])
    assert rec.calls[-1] == (nv.VARYING, np.dtype(np.float64), True)
    assert (rec.init[0]["f1"], rec.init[0]["f2"]) == (700.0, 890.0)
    api.estimate_monodepth_shared_focal_relative_pose_batch([p5.astype(np.float32)], [p5.astype(np.float32)],
                                                            [d5.astype(np.float32)], [d5.astype(np.float32)],
                                                            initial_image_pairs=[None])
    assert rec.calls[-1] == (nv.SHARED, np.dtype(np.float32), False)
    assert np.isnan(rec.init.view(np.float64)).all()


def test_api_prior_length_mismatch_raises(rec):
    from mdrp_b200 import api
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    p5, d5 = np.zeros((5, 2)), np.ones(5)
    with pytest.raises(ValueError):
        api.estimate_monodepth_relative_pose_batch([p5, p5], [p5, p5], [d5, d5], [d5, d5], [cam, cam], [cam, cam],
                                                   initial_geometries=[None])
    with pytest.raises(ValueError):
        api.estimate_monodepth_shared_focal_relative_pose_batch([p5], [p5], [d5], [d5], initial_image_pairs=[None, None])
    assert rec.calls == []


def test_native_host_init_checks_shape(monkeypatch):
    from mdrp_b200 import _native as nv
    ctx = nv.Context.__new__(nv.Context)
    with pytest.raises(ValueError):
        ctx.estimate_batch_host_init(0, [0, 3, 5], np.zeros((5, 2)), np.zeros((5, 2)), np.ones(5), np.ones(5), None,
                                     nv.Options(), np.zeros(1, nv.MODEL_DTYPE))


def test_single_pair_calls_keep_ignoring_initial_pose(monkeypatch):
    """The reference-signature single-pair functions accept and ignore initial_pose / initial_image_pair."""
    from mdrp_b200 import api

    class Plain(_InitRecorder):
        def estimate_batch_host(self, variant, offsets, x1, x2, d1, d2, cams, opt):
            self.calls.append("plain")
            return self.estimate_batch_host_init(variant, offsets, x1, x2, d1, d2, cams, opt, None)[:3]
    r = Plain()
    monkeypatch.setattr(api, "context", lambda device=0: r)
    p5, d5 = np.zeros((5, 2)), np.ones(5)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    api.estimate_monodepth_relative_pose(p5, p5, d5, d5, cam, cam, initial_pose=api.CameraPose())
    api.estimate_monodepth_shared_focal_relative_pose(p5, p5, d5, d5, initial_image_pair=api.MonoDepthImagePair())
    api.estimate_monodepth_varying_focal_relative_pose(p5, p5, d5, d5, initial_image_pair=api.MonoDepthImagePair())
    assert [c for c in r.calls if c == "plain"] == ["plain"] * 3 and len(r.calls) == 6


def test_torch_estimate_routes_priors(monkeypatch):
    torch = pytest.importorskip("torch")
    from mdrp_b200 import torch_frontend as tf, _native as nv

    class Rec:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            if not name.startswith("estimate_batch_dev"):
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
    init = torch.full((2, 12), float("nan"), dtype=torch.float64)
    o = nv.Options()
    tf.estimate_batch(nv.SHARED, offs, x32, x32, d32, d32, None, o, init_models=init)
    tf.estimate_batch(nv.SHARED, offs, x32.double(), x32, d32, d32, None, o, quality=torch.ones(5), init_models=init)
    tf.estimate_batch(nv.SHARED, offs, x32.double(), x32, d32, d32, None, o)
    assert [n for n, _ in rec.calls] == ["estimate_batch_dev_f32_init", "estimate_batch_dev_init", "estimate_batch_dev"]
    assert rec.calls[0][1][8] == init.data_ptr() and rec.calls[0][1][12] is None
    assert rec.calls[1][1][12] is not None
    with pytest.raises(ValueError):
        tf.estimate_batch(nv.SHARED, offs, x32, x32, d32, d32, None, o, init_models=init[:1])
    with pytest.raises(ValueError):
        tf.estimate_batch(nv.SHARED, offs, x32, x32, d32, d32, None, o, init_models=init.float())
