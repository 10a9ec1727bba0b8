"""GPU tier: float32 keypoints and depths (rp_estimate_batch_*_f32, rp_gather_depths_*_f32 and the Python / torch
surfaces that route float32 arrays to them).

float -> double is exact, so every comparison here is against the FP64 path on `astype(float64)` of the same float32
values, as BYTES: models, stats, masks and rp_pair_status."""
import ctypes as C

import numpy as np
import pytest

from mdrp_b200 import _native as nv, api, synth

pytestmark = pytest.mark.gpu

SIZES = [400, 0, 150, 2, 3, 900, 1, 250]   # ragged, with empty pairs and pairs of fewer than 3 correspondences


def _ragged(cfg, base, sizes=SIZES):
    """float32 packed batch of `cfg` scenes (pixel coordinates; principal-point-centred for the focal variants)."""
    c = synth.CONFIGS[cfg]
    scs = [synth.scene_for(cfg, base + i, n=max(n, 3)) for i, n in enumerate(sizes)]
    focal = c["variant"] != "calib"
    x1 = np.concatenate([(s.centred()[0] if focal else s.x1)[:n] for s, n in zip(scs, sizes)])
    x2 = np.concatenate([(s.centred()[1] if focal else s.x2)[:n] for s, n in zip(scs, sizes)])
    d1 = np.concatenate([s.d1[:n] for s, n in zip(scs, sizes)])
    d2 = np.concatenate([s.d2[:n] for s, n in zip(scs, sizes)])
    offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    cams = None if focal else np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
    variant = {"calib": nv.CALIB_SHIFT if c["shift"] else nv.CALIB, "shared": nv.SHARED, "varying": nv.VARYING}[c["variant"]]
    f = lambda a: a.astype(np.float32)
    return variant, offs, f(x1), f(x2), f(d1), f(d2), cams


def _options(iters, shift=False, min_iters=None):
    o = nv.default_options()
    o.max_iterations = iters
    o.min_iterations = iters if min_iters is None else min_iters
    o.max_epipolar_error, o.max_reproj_error, o.estimate_shift = 2.0, 16.0, int(shift)
    o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    return o


def _both(ctx, variant, offs, x1, x2, d1, d2, cams, o):
    """(float32 path, FP64 path on the widened values), each with its rp_pair_status."""
    P = len(offs) - 1
    a = ctx.estimate_batch_host_f32(variant, offs, x1, x2, d1, d2, cams, o)
    sa = ctx.pair_status(P)
    w = lambda v: v.astype(np.float64)
    b = ctx.estimate_batch_host(variant, offs, w(x1), w(x2), w(d1), w(d2), cams, o)
    sb = ctx.pair_status(P)
    return (a, sa), (b, sb)


def _assert_same(r32, r64):
    (a, sa), (b, sb) = r32, r64
    for u, v in zip(a, b):
        assert u.tobytes() == v.tobytes()
    assert sa.tobytes() == sb.tobytes()


@pytest.mark.parametrize("cfg", ["cfg1_calib_scale", "cfg2_calib_shift", "cfg3_shared_focal", "cfg4_varying_focal",
                                 "hard_calib"])
def test_float32_host_path_equals_fp64_bytes(ctx, cfg):
    variant, offs, x1, x2, d1, d2, cams = _ragged(cfg, 40)
    r32, r64 = _both(ctx, variant, offs, x1, x2, d1, d2, cams, _options(600, shift=synth.CONFIGS[cfg]["shift"]))
    _assert_same(r32, r64)
    st = r32[1]
    assert (st[np.diff(offs) < 3] == nv.PAIR_DEGENERATE).all() and (st[np.diff(offs) >= 3] == nv.PAIR_OK).all()
    ms, _ = ctx.last_timing()   # of the FP64 call: no widening
    assert ms["widen"] == 0.0


def test_float32_timing_slot_reports_widening(ctx):
    variant, offs, x1, x2, d1, d2, cams = _ragged("cfg2_calib_shift", 50)
    ctx.estimate_batch_host_f32(variant, offs, x1, x2, d1, d2, cams, _options(200, shift=True))
    ms, cn = ctx.last_timing()
    assert ms["widen"] > 0.0 and ms["h2d"] > 0.0 and ms["device_total"] > 0.0 and cn["chunks"] >= 1


def test_float32_prosac_early_termination(ctx):
    variant, offs, x1, x2, d1, d2, cams = _ragged("cfg1_calib_scale", 60)
    o = _options(5000, min_iters=100)
    o.progressive_sampling = 1
    r32, r64 = _both(ctx, variant, offs, x1, x2, d1, d2, cams, o)
    _assert_same(r32, r64)


def test_float32_event_list_rerun(monkeypatch):
    """RP_EV_CAP=4 sends most pairs through the per-pair re-run (its sub-batch gather reads the widened chunk)."""
    variant, offs, x1, x2, d1, d2, cams = _ragged("cfg2_calib_shift", 70, sizes=[400, 150, 3, 900] * 6)
    monkeypatch.setenv("RP_EV_CAP", "4")
    small = nv.Context(0)
    r32, r64 = _both(small, variant, offs, x1, x2, d1, d2, cams, _options(2000, shift=True))
    small.close()
    _assert_same(r32, r64)
    assert ((r32[1] & nv.PAIR_EVENTS_RERUN) != 0).sum() >= 12


def test_float32_default_options_hard_pair(ctx):
    """PoseLib's default early termination with one 2 %-inlier pair that is run again on its own (RP_PAIR_CONTINUED)."""
    P, n, hard = 512, 300, 77
    scs = [synth.scene_for("cfg1_calib_scale", 9000 + i, n=n) for i in range(P)]
    scs[hard] = synth.make_scene(424242, n, outlier_ratio=0.98)
    f = lambda k: np.concatenate([getattr(s, k) for s in scs]).astype(np.float32)
    offs = np.arange(P + 1, dtype=np.int64) * n
    cams = np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
    o = nv.default_options()
    o.max_epipolar_error, o.max_reproj_error = 2.0, 16.0
    o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    r32, r64 = _both(ctx, nv.CALIB, offs, f("x1"), f("x2"), f("d1"), f("d2"), cams, o)
    _assert_same(r32, r64)
    assert r32[1][hard] & nv.PAIR_CONTINUED


def test_float32_several_chunks_and_lead_chunk(ctx, monkeypatch):
    """A small workspace on a fresh context splits the batch into a lead chunk and several more (host path: double-
    buffered float staging; device path: one widening per chunk): the same bytes as one FP64 chunk."""
    import torch
    P, n = 1100, 120
    b = synth.make_batch("cfg1_calib_scale", P, seed=3, n=n)
    offs = b["offsets"]
    x1, x2, d1, d2 = (b[k].astype(np.float32) for k in ("x1", "x2", "d1", "d2"))
    o = _options(200)
    w = lambda v: v.astype(np.float64)
    ref = ctx.estimate_batch_host(nv.CALIB, offs, w(x1), w(x2), w(d1), w(d2), b["cams"], o)
    assert ctx.last_timing()[1]["chunks"] <= 2   # the lead chunk and the rest
    monkeypatch.setenv("RP_WORKSPACE_GB", "0.1")
    small = nv.Context(0)
    got = small.estimate_batch_host_f32(nv.CALIB, offs, x1, x2, d1, d2, b["cams"], o)
    chunks = small.last_timing()[1]["chunks"]
    assert chunks >= 4
    for u, v in zip(got, ref):
        assert u.tobytes() == v.tobytes()
    # a second call sizes its lead chunk from the measured upload + widening / kernel times of the first
    again = small.estimate_batch_host_f32(nv.CALIB, offs, x1, x2, d1, d2, b["cams"], o)
    for u, v in zip(again, ref):
        assert u.tobytes() == v.tobytes()
    # device path, several chunks
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dm = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    ds = torch.zeros(P, 5, dtype=torch.int64, device=dev)
    dk = torch.zeros(int(offs[-1]), dtype=torch.uint8, device=dev)
    tx1, tx2, td1, td2, tc = t(x1), t(x2), t(d1), t(d2), t(b["cams"])
    small.estimate_batch_dev_f32(nv.CALIB, offs, tx1.data_ptr(), tx2.data_ptr(), td1.data_ptr(), td2.data_ptr(),
                                 tc.data_ptr(), o, dm.data_ptr(), ds.data_ptr(), dk.data_ptr(),
                                 torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize()
    assert small.last_timing()[1]["chunks"] >= 4 and small.last_timing()[0]["widen"] > 0.0
    small.close()
    assert dm.cpu().numpy().tobytes() == ref[0].tobytes() and ds.cpu().numpy().tobytes() == ref[1].tobytes()
    assert dk.cpu().numpy().tobytes() == ref[2].tobytes()


def test_torch_float32_tensors_without_fp64_copy(ctx):
    import torch
    from mdrp_b200 import torch_frontend as tf
    P, n = 16, 6000
    b = synth.make_batch("cfg2_calib_shift", P, seed=9, n=n)
    offs, N = b["offsets"], P * n
    dev = torch.device("cuda", 0)
    t32 = {k: torch.from_numpy(b[k].astype(np.float32)).to(dev) for k in ("x1", "x2", "d1", "d2")}
    t64 = {k: v.double() for k, v in t32.items()}
    cams = torch.from_numpy(b["cams"]).to(dev)
    o = _options(300, shift=True)
    ref = tf.estimate_batch(nv.CALIB_SHIFT, offs, t64["x1"], t64["x2"], t64["d1"], t64["d2"], cams, o)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    got = tf.estimate_batch(nv.CALIB_SHIFT, offs, t32["x1"], t32["x2"], t32["d1"], t32["d2"], cams, o)
    torch.cuda.synchronize()
    grew = torch.cuda.max_memory_allocated(dev) - base
    # outputs (models, stats, masks) only; an FP64 copy of the inputs would be N * 48 bytes
    assert grew < P * (96 + 40) + N + 64 * 1024 < N * 48
    for u, v in zip(got, ref):
        assert torch.equal(u, v)


def _maps_and_keypoints(seed=5):
    """Two depth maps with inf and NaN pixels and keypoints on a synthetic scene (a few outside the map)."""
    rng = np.random.default_rng(seed)
    sc = synth.scene_for("cfg1_calib_scale", 31, n=700)
    H, W = 960, 1280
    dm1 = rng.uniform(1, 9, size=(H, W)).astype(np.float32)
    dm2 = rng.uniform(1, 9, size=(H, W)).astype(np.float32)
    kp1, kp2 = sc.x1.astype(np.float32), sc.x2.astype(np.float32)
    inside = lambda kp: (np.clip(kp[:, 1].astype(int), 0, H - 1), np.clip(kp[:, 0].astype(int), 0, W - 1))
    dm1[inside(kp1)] = sc.d1.astype(np.float32)
    dm2[inside(kp2)] = sc.d2.astype(np.float32)
    both, one, nan = rng.choice(700, 60, replace=False).reshape(3, 20)
    r1, c1 = inside(kp1)
    r2, c2 = inside(kp2)
    dm1[r1[both], c1[both]] = np.inf
    dm2[r2[both], c2[both]] = np.inf
    dm1[r1[one], c1[one]] = np.inf
    dm2[r2[nan], c2[nan]] = np.nan
    return sc, dm1, dm2, kp1, kp2


def test_gather_f32_then_estimate_equals_fp64_chain(ctx):
    import torch
    from mdrp_b200 import torch_frontend as tf
    sc, dm1, dm2, kp1, kp2 = _maps_and_keypoints()
    g = lambda a: torch.from_numpy(a).cuda()
    a = tf.gather_depths(g(dm1), g(dm2), g(kp1), g(kp2), dtype=torch.float32)
    b = tf.gather_depths(g(dm1), g(dm2), g(kp1), g(kp2))
    assert all(u.dtype == torch.float32 for u in a) and all(v.dtype == torch.float64 for v in b)
    # both-inf rows dropped, one-inf and NaN rows kept (make_pair.py:106)
    H, W = dm1.shape
    at = lambda dm, kp: dm[np.clip(kp[:, 1].astype(int), 0, H - 1), np.clip(kp[:, 0].astype(int), 0, W - 1)]
    keep = ~(np.isinf(at(dm1, kp1)) & np.isinf(at(dm2, kp2)))
    assert a[0].shape[0] == b[0].shape[0] == keep.sum() < len(kp1)
    assert np.array_equal(a[0].cpu().numpy(), kp1[keep]) and np.isnan(a[3].cpu().numpy()).any()
    for u, v in zip(a, b):
        assert torch.equal(torch.isnan(u), torch.isnan(v)) and torch.equal(torch.nan_to_num(u.double()), torch.nan_to_num(v))
    # the estimate of the pair from each chain (rows with a non-finite depth left in: the reference does the same)
    c1, c2 = sc.camera_dicts()
    ro = {"max_iterations": 500, "min_iterations": 500, "max_epipolar_error": 2.0, "max_reproj_error": 16.0}
    bo = {"loss_type": "TRUNCATED_CAUCHY"}
    ga, ia = tf.estimate_monodepth_relative_pose(*a, c1, c2, ro, bo)
    gb, ib = tf.estimate_monodepth_relative_pose(*b, c1, c2, ro, bo)
    assert ia == ib and ia["iterations"] == 500
    assert ga.pose.q.tobytes() == gb.pose.q.tobytes() and ga.pose.t.tobytes() == gb.pose.t.tobytes()
    assert (ga.scale, ga.shift1, ga.shift2) == (gb.scale, gb.shift1, gb.shift2)


def test_batched_gather_f32_then_estimate_equals_fp64_chain(ctx):
    import torch
    from mdrp_b200 import torch_frontend as tf
    rng = np.random.default_rng(8)
    F, H, W = 4, 960, 1280
    sizes = [700, 0, 2, 1025, 256]
    f1, f2 = [0, 1, 2, 3, 0], [1, 2, 3, 0, 2]
    scs = [synth.scene_for("cfg1_calib_scale", 300 + i, n=max(s, 3)) for i, s in enumerate(sizes)]
    maps = rng.uniform(1, 9, size=(F, H, W)).astype(np.float32)
    maps[rng.uniform(size=maps.shape) < 0.05] = np.inf
    maps[rng.uniform(size=maps.shape) < 0.01] = np.nan
    kp1 = np.concatenate([s.x1[:n] for s, n in zip(scs, sizes)]).astype(np.float32)
    kp2 = np.concatenate([s.x2[:n] for s, n in zip(scs, sizes)]).astype(np.float32)
    offs = np.r_[0, np.cumsum(sizes)]
    g = torch.from_numpy(maps).cuda()
    k1, k2 = torch.from_numpy(kp1).cuda(), torch.from_numpy(kp2).cuda()
    oa, *a = tf.gather_depths_batch(g, f1, f2, offs, k1, k2, dtype=torch.float32)
    ob, *b = tf.gather_depths_batch(g, f1, f2, offs, k1, k2)
    assert np.array_equal(oa, ob) and oa[-1] < offs[-1]
    for u, v in zip(a, b):
        assert u.dtype == torch.float32 and torch.equal(torch.isnan(u), torch.isnan(v))
        assert torch.equal(torch.nan_to_num(u.double()), torch.nan_to_num(v))
    cams = torch.tensor([[800.0, 800, 640, 480, 800, 800, 640, 480]] * len(sizes), dtype=torch.float64).cuda()
    o = _options(300)
    ra = tf.estimate_batch(nv.CALIB, oa, *a, cams, o)
    sa = ctx.pair_status(len(sizes))
    rb = tf.estimate_batch(nv.CALIB, ob, *b, cams, o)
    sb = ctx.pair_status(len(sizes))
    for u, v in zip(ra, rb):
        assert u.cpu().numpy().tobytes() == v.cpu().numpy().tobytes()
    assert sa.tobytes() == sb.tobytes()


def test_api_float32_numpy_batch_and_single_pair(ctx, monkeypatch):
    cfg = "cfg2_calib_shift"
    scs = [synth.scene_for(cfg, 80 + i, n=n) for i, n in enumerate([300, 2, 500])]
    p1 = [s.x1.astype(np.float32) for s in scs]
    p2 = [s.x2.astype(np.float32) for s in scs]
    e1 = [s.d1.astype(np.float32) for s in scs]
    e2 = [s.d2.astype(np.float32) for s in scs]
    cams = [s.camera_dicts() for s in scs]
    ro = {"max_iterations": 400, "min_iterations": 400, "max_epipolar_error": 2.0, "max_reproj_error": 16.0,
          "monodepth_estimate_shift": True}
    bo = {"loss_type": "TRUNCATED_CAUCHY"}
    calls = []
    real = api.context(0)
    for name in ("estimate_batch_host", "estimate_batch_host_f32"):
        fn = getattr(real, name)
        monkeypatch.setattr(real, name, lambda *a, _fn=fn, _name=name: (calls.append(_name), _fn(*a))[1])
    w = lambda xs: [x.astype(np.float64) for x in xs]

    def same(r, q):
        for (ga, ia), (gb, ib) in zip(r, q):
            assert ia == ib
            assert ga.pose.q.tobytes() == gb.pose.q.tobytes() and ga.pose.t.tobytes() == gb.pose.t.tobytes()
            assert (ga.scale, ga.shift1, ga.shift2) == (gb.scale, gb.shift1, gb.shift2)

    r32 = api.estimate_monodepth_relative_pose_batch(p1, p2, e1, e2, [c[0] for c in cams], [c[1] for c in cams], ro, bo)
    r64 = api.estimate_monodepth_relative_pose_batch(w(p1), w(p2), w(e1), w(e2), [c[0] for c in cams],
                                                     [c[1] for c in cams], ro, bo)
    assert calls == ["estimate_batch_host_f32", "estimate_batch_host"]
    same(r32, r64)
    # one float64 array in the batch: the FP64 path
    calls.clear()
    mixed = api.estimate_monodepth_relative_pose_batch(p1, p2, e1[:2] + w(e1[2:]), e2, [c[0] for c in cams],
                                                       [c[1] for c in cams], ro, bo)
    assert calls == ["estimate_batch_host"]
    same(mixed, r64)
    # single pair, calibrated and focal
    calls.clear()
    same([api.estimate_monodepth_relative_pose(p1[0], p2[0], e1[0], e2[0], *cams[0], ro, bo)],
         [api.estimate_monodepth_relative_pose(*w([p1[0], p2[0], e1[0], e2[0]]), *cams[0], ro, bo)])
    ro_f = {"max_iterations": 400, "min_iterations": 400, "max_epipolar_error": 2.0}
    a1, a2 = (c.astype(np.float32) for c in scs[0].centred())
    fa = api.estimate_monodepth_varying_focal_relative_pose(a1, a2, e1[0], e2[0], ro_f, bo)
    fb = api.estimate_monodepth_varying_focal_relative_pose(*w([a1, a2, e1[0], e2[0]]), ro_f, bo)
    assert calls == ["estimate_batch_host_f32", "estimate_batch_host", "estimate_batch_host_f32", "estimate_batch_host"]
    assert fa[1] == fb[1] and (fa[0].camera1.params, fa[0].camera2.params) == (fb[0].camera1.params, fb[0].camera2.params)
    assert fa[0].pose.q.tobytes() == fb[0].pose.q.tobytes() and fa[0].pose.t.tobytes() == fb[0].pose.t.tobytes()


def test_non_finite_inputs(ctx):
    variant, offs, x1, x2, d1, d2, cams = _ragged("cfg2_calib_shift", 90)
    x1[5] = np.nan
    x2[17, 1] = np.inf
    d1[33] = -np.inf
    d2[40:60] = np.nan
    d1[offs[5] + 3] = np.inf
    r32, r64 = _both(ctx, variant, offs, x1, x2, d1, d2, cams, _options(400, shift=True))
    _assert_same(r32, r64)


def _codes(ctx, call):
    """(return code, rp_last_error) of `call(f32)` for the float32 and the FP64 entry point."""
    out = []
    for f32 in (True, False):
        rc = call(f32)
        out.append((rc, ctx._lib.rp_last_error(ctx._h).decode() if rc else ""))
    return out


def test_argument_errors_match_fp64_entry_points(ctx):
    L, h = ctx._lib, ctx._h
    n = 10
    x = np.zeros((n, 2)), np.zeros((n, 2), dtype=np.float32)
    d = np.ones(n), np.ones(n, dtype=np.float32)
    cams = np.tile(np.array([800.0, 800, 640, 480, 800, 800, 640, 480]), (1, 1))
    good, bad = np.array([0, n], dtype=np.int64), np.array([0, n, 4], dtype=np.int64)
    models = np.zeros(2, dtype=nv.MODEL_DTYPE)
    stats = np.zeros(2, dtype=nv.STATS_DTYPE)
    masks = np.zeros(n, dtype=np.uint8)
    opt = _options(100)
    opt_bad = _options(100)
    opt_bad.max_iterations = opt_bad.min_iterations = (1 << 24) + 1
    P = lambda a: a.ctypes.data if a is not None else None
    cases = {   # name -> (ctx handle, variant, n_pairs, offsets, data given, cams, opt)
        "null ctx": (None, 0, 1, good, True, cams, opt), "variant": (h, 7, 1, good, True, cams, opt),
        "negative n_pairs": (h, 0, -1, good, True, cams, opt), "null offsets": (h, 0, 1, None, True, cams, opt),
        "null opt": (h, 0, 1, good, True, cams, None), "iterations": (h, 0, 1, good, True, cams, opt_bad),
        "offsets decrease": (h, 0, 2, bad, True, np.tile(cams, (2, 1)), opt), "null data": (h, 0, 1, good, False, cams, opt),
        "no cams": (h, 0, 1, good, True, None, opt), "ok, zero pairs": (h, 0, 0, good[:1], False, None, opt),
    }
    for name, (hh, var, npairs, offs, data, cm, o) in cases.items():
        for dev in (False, True):
            def call(f32, hh=hh, var=var, npairs=npairs, offs=offs, data=data, cm=cm, o=o, dev=dev):
                k = int(f32)
                ptrs = [P(x[k]), P(x[k]), P(d[k]), P(d[k])] if data else [None] * 4
                args = [hh, var, npairs, P(offs)] + ptrs + [P(cm), C.byref(o) if o is not None else None,
                                                            P(models), P(stats), P(masks)]
                if dev:
                    # the argument checks come before any device pointer is touched: host arrays stand in for them
                    return (L.rp_estimate_batch_dev_f32 if f32 else L.rp_estimate_batch_dev)(*args, None)
                return (L.rp_estimate_batch_host_f32 if f32 else L.rp_estimate_batch_host)(*args)
            a, b = _codes(ctx, call)
            assert a == b, (name, dev, a, b)
            assert a[0] == (0 if name == "ok, zero pairs" else -1), (name, dev, a)
    # gathers
    f = np.zeros((4, 4), dtype=np.float32)
    out32, out64 = np.zeros(8, dtype=np.float32), np.zeros(8)
    n_out = C.c_int64(0)
    for args in ((h, P(f), 0, 4, P(f), 4, 4), (h, P(f), 4, 4, None, 4, 4), (None, P(f), 4, 4, P(f), 4, 4)):
        rc = [fn(*args, P(f), P(f), 4, P(o), P(o), P(o), P(o), C.byref(n_out), None)
              for fn, o in ((L.rp_gather_depths_dev_f32, out32), (L.rp_gather_depths_dev, out64))]
        assert rc[0] == rc[1] == -1
    off_bad = np.array([0, 3, 1], dtype=np.int64)
    fr = np.array([0, 5], dtype=np.int32)
    oo = np.zeros(3, dtype=np.int64)
    rc = [fn(h, 2, P(off_bad), P(f), 1, 4, 4, P(fr), P(fr), P(f), P(f), P(o), P(o), P(o), P(o), P(oo), None)
          for fn, o in ((L.rp_gather_depths_batch_dev_f32, out32), (L.rp_gather_depths_batch_dev, out64))]
    assert rc[0] == rc[1] == -1
