"""GPU tier: per-correspondence match quality (rp_order_by_quality, rp_estimate_batch_*_quality and the Python / torch
surfaces that route a quality to them).

The quality entry points are defined by a reordering: their outputs are, as BYTES, those of the unscored twin called with
every pair reordered by (float32 quality descending, original index ascending; NaN as -inf, -0 as +0), with the masks
scattered back to the caller's order.  Every end-to-end test here builds that definition on the host and compares."""
import ctypes as C

import numpy as np
import pytest

from mdrp_b200 import _native as nv, api, synth

pytestmark = pytest.mark.gpu

SIZES = [400, 0, 150, 2, 3, 900, 1, 250]   # ragged, with empty pairs and pairs of fewer than 3 correspondences
CAP = nv.ORDER_SMEM_CAP


def ref_order(offs, q):
    """The defining order, per pair: np.lexsort((index, -key)) with key = float32 quality, NaN -> -inf, -0 -> +0."""
    key = np.asarray(q, dtype=np.float32).astype(np.float64)
    key[np.isnan(key)] = -np.inf
    key = key + 0.0
    perm = np.zeros(len(key), dtype=np.int32)
    for p in range(len(offs) - 1):
        o, e = int(offs[p]), int(offs[p + 1])
        perm[o:e] = np.lexsort((np.arange(e - o), -key[o:e]))
    return perm


def reorder(offs, perm, *arrays):
    """Each pair's rows in the order `perm`."""
    src = np.concatenate([int(offs[p]) + perm[offs[p]:offs[p + 1]] for p in range(len(offs) - 1)] + [np.zeros(0, int)])
    return [a[src] for a in arrays], src


def _ragged(cfg, base, sizes=SIZES, dtype=np.float64):
    c = synth.CONFIGS[cfg]
    scs = [synth.scene_for(cfg, base + i, n=max(n, 3)) for i, n in enumerate(sizes)]
    focal = c["variant"] != "calib"
    x1 = np.concatenate([(s.centred()[0] if focal else s.x1)[:n] for s, n in zip(scs, sizes)])
    x2 = np.concatenate([(s.centred()[1] if focal else s.x2)[:n] for s, n in zip(scs, sizes)])
    d1 = np.concatenate([s.d1[:n] for s, n in zip(scs, sizes)])
    d2 = np.concatenate([s.d2[:n] for s, n in zip(scs, sizes)])
    inl = np.concatenate([s.inlier_mask[:n] for s, n in zip(scs, sizes)])
    offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    cams = None if focal else np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
    variant = {"calib": nv.CALIB_SHIFT if c["shift"] else nv.CALIB, "shared": nv.SHARED, "varying": nv.VARYING}[c["variant"]]
    # quality correlated with being an inlier, with overlap, and a few ties
    rng = np.random.default_rng(base)
    q = np.where(inl, rng.uniform(0.3, 1.0, len(inl)), rng.uniform(0.0, 0.7, len(inl))).astype(np.float32)
    q[::17] = 0.5
    f = lambda a: a.astype(dtype)
    return variant, offs, f(x1), f(x2), f(d1), f(d2), cams, q


def _options(iters, shift=False, min_iters=None, prosac=True, max_prosac=None):
    o = nv.default_options()
    o.max_iterations = iters
    o.min_iterations = iters if min_iters is None else min_iters
    o.max_epipolar_error, o.max_reproj_error, o.estimate_shift = 2.0, 16.0, int(shift)
    o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    o.progressive_sampling = int(prosac)
    if max_prosac is not None:
        o.max_prosac_iterations = max_prosac
    return o


def definition(ctx, variant, offs, x1, x2, d1, d2, cams, o, q):
    """(models, stats, masks in the caller's order), rp_pair_status of the unscored call on the reordered batch."""
    perm = ref_order(offs, q)
    (a1, a2, b1, b2), src = reorder(offs, perm, x1, x2, d1, d2)
    fn = ctx.estimate_batch_host_f32 if x1.dtype == np.float32 else ctx.estimate_batch_host
    m, s, k = fn(variant, offs, a1, a2, b1, b2, cams, o)
    st = ctx.pair_status(len(offs) - 1)
    out = np.zeros_like(k)
    out[src] = k
    return (m, s, out), st


def _host_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q):
    r = ctx.estimate_batch_host_quality(variant, offs, x1, x2, d1, d2, cams, o, q)
    return r, ctx.pair_status(len(offs) - 1)


def _dev_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q):
    import torch
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    P, N = len(offs) - 1, int(offs[-1])
    dm = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    ds = torch.zeros(P, 5, dtype=torch.int64, device=dev)
    dk = torch.zeros(max(N, 1), dtype=torch.uint8, device=dev)
    tx1, tx2, td1, td2, tq = t(x1), t(x2), t(d1), t(d2), t(q)
    tc = t(cams) if cams is not None else None
    est = ctx.estimate_batch_dev_f32_quality if x1.dtype == np.float32 else ctx.estimate_batch_dev_quality
    est(variant, offs, tx1.data_ptr(), tx2.data_ptr(), td1.data_ptr(), td2.data_ptr(),
        tc.data_ptr() if tc is not None else None, o, dm.data_ptr(), ds.data_ptr(), dk.data_ptr(), tq.data_ptr(),
        torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize()
    return (dm.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1), ds.cpu().numpy().view(nv.STATS_DTYPE).reshape(-1),
            dk.cpu().numpy()[:N]), ctx.pair_status(P)


def _assert_same(got, ref):
    (a, sa), (b, sb) = got, ref
    for u, v in zip(a, b):
        assert u.tobytes() == v.tobytes()
    assert sa.tobytes() == sb.tobytes()


# ---- the sort alone -------------------------------------------------------------------------------
def _keys(kind, n, rng):
    if kind == "random":
        return rng.standard_normal(n).astype(np.float32)
    if kind == "ties3":
        return rng.choice(np.array([0.25, 0.5, 0.75], np.float32), n)
    if kind == "equal":
        return np.full(n, 0.5, np.float32)
    if kind == "special":
        vals = np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, 3e-39, -3e-39, 1.0, -1.0,
                         np.float32(np.finfo(np.float32).max), np.float32(-np.finfo(np.float32).max)], np.float32)
        out = rng.choice(vals, n).astype(np.float32)
        out.view(np.uint32)[rng.uniform(size=n) < 0.05] = 0x7fc01234   # NaN with a payload
        return out
    if kind == "sorted":
        return np.sort(rng.uniform(size=n).astype(np.float32))[::-1].copy()
    if kind == "reverse":
        return np.sort(rng.uniform(size=n).astype(np.float32))
    raise ValueError(kind)


KINDS = ["random", "ties3", "equal", "special", "sorted", "reverse"]
SORT_SIZES = [0, 1, 2, 3, 31, 32, 33, 255, 256, 257, 2000, 10000, CAP - 1, CAP, CAP + 1]


@pytest.mark.parametrize("kind", KINDS)
def test_order_alone_every_size(ctx, kind):
    rng = np.random.default_rng(KINDS.index(kind))
    for n in SORT_SIZES:
        q = _keys(kind, n, rng)
        offs = np.array([0, n], dtype=np.int64)
        assert np.array_equal(ctx.order(offs, q), ref_order(offs, q)), (kind, n)


@pytest.mark.parametrize("kind", ["random", "special", "ties3"])
def test_order_alone_large_pair(ctx, kind):
    rng = np.random.default_rng(11)
    n = (1 << 20) + 3
    q = _keys(kind, n, rng)
    offs = np.array([0, n], dtype=np.int64)
    assert np.array_equal(ctx.order(offs, q), ref_order(offs, q))


def test_order_alone_mixed_sizes_and_offset_base(ctx):
    rng = np.random.default_rng(5)
    sizes = [0, 1, 3, 33, CAP + 1, 257, 0, 2000, CAP, 2, 70000, 10000, 31]
    kinds = [KINDS[i % len(KINDS)] for i in range(len(sizes))]
    q = np.concatenate([_keys(k, n, rng) for k, n in zip(kinds, sizes)])
    offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    assert np.array_equal(ctx.order(offs, q), ref_order(offs, q))
    # offsets that start inside the arrays: quality and perm are indexed by the offsets as they are
    sub = offs[3:9]
    perm = np.full(len(q), -7, dtype=np.int32)
    L = ctx._lib
    assert L.rp_order_by_quality(ctx._h, len(sub) - 1, sub.ctypes.data, q.ctypes.data, perm.ctypes.data) == 0
    want = ref_order(sub - sub[0], q[sub[0]:sub[-1]])
    assert np.array_equal(perm[sub[0]:sub[-1]], want)
    assert (perm[:sub[0]] == -7).all() and (perm[sub[-1]:] == -7).all()


def test_order_alone_argument_errors(ctx):
    L, h = ctx._lib, ctx._h
    q = np.zeros(4, np.float32)
    perm = np.zeros(4, np.int32)
    P = lambda a: a.ctypes.data
    good, dec, big = (np.array(v, dtype=np.int64) for v in ([0, 4], [0, 3, 1], [0, 1 << 24]))
    assert L.rp_order_by_quality(None, 1, P(good), P(q), P(perm)) == -1
    assert L.rp_order_by_quality(h, -1, P(good), P(q), P(perm)) == -1
    assert L.rp_order_by_quality(h, 1, None, P(q), P(perm)) == -1
    assert L.rp_order_by_quality(h, 1, P(good), None, P(perm)) == -1
    assert L.rp_order_by_quality(h, 1, P(good), P(q), None) == -1
    assert L.rp_order_by_quality(h, 2, P(dec), P(q), P(perm)) == -1
    assert L.rp_order_by_quality(h, 1, P(big), P(q), P(perm)) == -1
    assert L.rp_order_by_quality(h, 0, P(good), None, None) == 0


# ---- end to end, as bytes ---------------------------------------------------------------------------
CFGS = ["cfg1_calib_scale", "cfg2_calib_shift", "cfg3_shared_focal", "cfg4_varying_focal", "hard_calib"]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("cfg", CFGS)
def test_quality_host_and_device_equal_definition(ctx, cfg, dtype):
    variant, offs, x1, x2, d1, d2, cams, q = _ragged(cfg, 40 + CFGS.index(cfg), dtype=dtype)
    o = _options(600, shift=synth.CONFIGS[cfg]["shift"], max_prosac=300)
    ref = definition(ctx, variant, offs, x1, x2, d1, d2, cams, o, q)
    st = ref[1]
    assert (st[np.diff(offs) < 3] == nv.PAIR_DEGENERATE).all() and (st[np.diff(offs) >= 3] == nv.PAIR_OK).all()
    assert ctx.last_timing()[0]["order"] == 0.0   # an unscored call
    _assert_same(_host_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), ref)
    ms, _ = ctx.last_timing()
    assert ms["order"] > 0.0 and ms["widen"] == 0.0
    _assert_same(_dev_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), ref)
    ms, _ = ctx.last_timing()
    assert ms["order"] > 0.0 and ms["widen"] == 0.0


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_quality_prosac_default_max_and_uniform(ctx, dtype):
    variant, offs, x1, x2, d1, d2, cams, q = _ragged("cfg2_calib_shift", 55, dtype=dtype)
    for o in (_options(800, shift=True), _options(800, shift=True, prosac=False)):
        ref = definition(ctx, variant, offs, x1, x2, d1, d2, cams, o, q)
        _assert_same(_host_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), ref)
        _assert_same(_dev_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), ref)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_quality_prosac_early_termination(ctx, dtype):
    variant, offs, x1, x2, d1, d2, cams, q = _ragged("cfg1_calib_scale", 60, dtype=dtype)
    o = _options(5000, min_iters=100, max_prosac=1000)
    ref = definition(ctx, variant, offs, x1, x2, d1, d2, cams, o, q)
    _assert_same(_host_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), ref)
    _assert_same(_dev_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), ref)


def test_quality_default_options_continued_pair(ctx):
    """PoseLib's default early termination with one 2 %-inlier pair that is run again on its own (RP_PAIR_CONTINUED)."""
    P, n, hard = 512, 300, 77
    scs = [synth.scene_for("cfg1_calib_scale", 9000 + i, n=n) for i in range(P)]
    scs[hard] = synth.make_scene(424242, n, outlier_ratio=0.98)
    f = lambda k: np.concatenate([getattr(s, k) for s in scs])
    offs = np.arange(P + 1, dtype=np.int64) * n
    cams = np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
    rng = np.random.default_rng(3)
    inl = f("inlier_mask")
    q = np.where(inl, rng.uniform(0.3, 1.0, len(inl)), rng.uniform(0.0, 0.7, len(inl))).astype(np.float32)
    o = nv.default_options()
    o.max_epipolar_error, o.max_reproj_error = 2.0, 16.0
    o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    o.progressive_sampling = 1
    args = (nv.CALIB, offs, f("x1"), f("x2"), f("d1"), f("d2"), cams, o, q)
    ref = definition(ctx, *args)
    got = _host_quality(ctx, *args)
    _assert_same(got, ref)
    assert got[1][hard] & nv.PAIR_CONTINUED
    _assert_same(_dev_quality(ctx, *args), ref)


def test_quality_event_list_rerun(monkeypatch):
    """RP_EV_CAP=4 sends most pairs through the per-pair re-run, whose masks land in the ordered layout first."""
    variant, offs, x1, x2, d1, d2, cams, q = _ragged("cfg2_calib_shift", 70, sizes=[400, 150, 3, 900] * 6)
    monkeypatch.setenv("RP_EV_CAP", "4")
    small = nv.Context(0)
    o = _options(2000, shift=True)
    ref = definition(small, variant, offs, x1, x2, d1, d2, cams, o, q)
    got = _host_quality(small, variant, offs, x1, x2, d1, d2, cams, o, q)
    _assert_same(got, ref)
    assert ((got[1] & nv.PAIR_EVENTS_RERUN) != 0).sum() >= 12
    _assert_same(_dev_quality(small, variant, offs, x1, x2, d1, d2, cams, o, q), ref)
    small.close()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_quality_several_chunks_and_lead_chunk(ctx, monkeypatch, dtype):
    """A small workspace on a fresh context: a lead chunk and several more (host path: double-buffered staging, sort and
    gather on the copy stream; device path: one sort and gather per chunk).  The same bytes as the definition run as
    one chunk."""
    P, n = 1100, 120
    b = synth.make_batch("cfg1_calib_scale", P, seed=3, n=n)
    offs = b["offsets"]
    x1, x2, d1, d2 = (b[k].astype(dtype) for k in ("x1", "x2", "d1", "d2"))
    q = np.random.default_rng(4).uniform(size=int(offs[-1])).astype(np.float32)
    q[::5] = 0.25
    o = _options(200)
    ref = definition(ctx, nv.CALIB, offs, x1, x2, d1, d2, b["cams"], o, q)
    assert ctx.last_timing()[1]["chunks"] <= 2
    monkeypatch.setenv("RP_WORKSPACE_GB", "0.1")
    small = nv.Context(0)
    for _ in range(2):   # the second call sizes its lead chunk from the first one's times
        got = _host_quality(small, nv.CALIB, offs, x1, x2, d1, d2, b["cams"], o, q)
        assert small.last_timing()[1]["chunks"] >= 4
        _assert_same(got, ref)
    got = _dev_quality(small, nv.CALIB, offs, x1, x2, d1, d2, b["cams"], o, q)
    assert small.last_timing()[1]["chunks"] >= 4 and small.last_timing()[0]["order"] > 0.0
    small.close()
    _assert_same(got, ref)


def test_quality_in_descending_order_is_the_unscored_call(ctx):
    variant, offs, x1, x2, d1, d2, cams, _ = _ragged("cfg2_calib_shift", 90)
    q = np.concatenate([np.linspace(1.0, 0.0, int(n), dtype=np.float32) for n in np.diff(offs)])
    q[offs[0] + 10:offs[0] + 20] = q[offs[0] + 10]   # ties keep index order
    o = _options(500, shift=True)
    plain = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, o)
    sp = ctx.pair_status(len(offs) - 1)
    _assert_same(_host_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), (plain, sp))
    _assert_same(_dev_quality(ctx, variant, offs, x1, x2, d1, d2, cams, o, q), (plain, sp))


def test_torch_frontend_quality(ctx):
    import torch
    from mdrp_b200 import torch_frontend as tf
    o = _options(400)
    dev = torch.device("cuda", 0)
    for dt, npdt in ((torch.float32, np.float32), (torch.float64, np.float64)):
        variant, offs, x1, x2, d1, d2, cams, q = _ragged("cfg3_shared_focal", 100, dtype=npdt)
        ref = definition(ctx, variant, offs, x1, x2, d1, d2, cams, o, q)
        t = lambda a: torch.from_numpy(a).to(dev)
        args = [t(x1), t(x2), t(d1), t(d2)]
        # the quality as given (float32) and as float64 of the same values
        tq = t(q) if dt == torch.float32 else t(q.astype(np.float64))
        m, s, k = tf.estimate_batch(variant, offs, *args, None, o, quality=tq)
        torch.cuda.synchronize()
        got = ((m.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1), tf.stats_to_numpy(s), k.cpu().numpy()),
               ctx.pair_status(len(offs) - 1))
        _assert_same(got, ref)


def test_api_batch_functions_quality(ctx):
    cfg = "cfg2_calib_shift"
    scs = [synth.scene_for(cfg, 120 + i, n=n) for i, n in enumerate([300, 2, 500])]
    rng = np.random.default_rng(6)
    quality = [np.where(s.inlier_mask, rng.uniform(0.3, 1, len(s.d1)), rng.uniform(0, 0.7, len(s.d1))) for s in scs]
    ro = {"max_iterations": 400, "min_iterations": 400, "max_epipolar_error": 2.0, "max_reproj_error": 16.0,
          "monodepth_estimate_shift": True, "progressive_sampling": True}
    bo = {"loss_type": "TRUNCATED_CAUCHY"}
    for dt in (np.float64, np.float32):
        p1, p2 = [s.x1.astype(dt) for s in scs], [s.x2.astype(dt) for s in scs]
        e1, e2 = [s.d1.astype(dt) for s in scs], [s.d2.astype(dt) for s in scs]
        cams = [s.camera_dicts() for s in scs]
        got = api.estimate_monodepth_relative_pose_batch(p1, p2, e1, e2, [c[0] for c in cams], [c[1] for c in cams], ro, bo,
                                                         quality=quality)
        # the definition through the same surface: each pair reordered on the host, inlier lists scattered back
        perms = [ref_order(np.array([0, len(qq)]), qq) for qq in quality]
        ref = api.estimate_monodepth_relative_pose_batch([a[p] for a, p in zip(p1, perms)], [a[p] for a, p in zip(p2, perms)],
                                                         [a[p] for a, p in zip(e1, perms)], [a[p] for a, p in zip(e2, perms)],
                                                         [c[0] for c in cams], [c[1] for c in cams], ro, bo)
        for (ga, ia), (gb, ib), p in zip(got, ref, perms):
            inl = np.zeros(len(p), bool)
            inl[p] = ib["inliers"]
            assert ia == {**ib, "inliers": inl.tolist()}
            assert ga.pose.q.tobytes() == gb.pose.q.tobytes() and ga.pose.t.tobytes() == gb.pose.t.tobytes()
            assert (ga.scale, ga.shift1, ga.shift2) == (gb.scale, gb.shift1, gb.shift2)
    # focal variants
    ro_f = {"max_iterations": 300, "min_iterations": 300, "max_epipolar_error": 2.0, "progressive_sampling": True}
    c1 = [s.centred()[0] for s in scs]
    c2 = [s.centred()[1] for s in scs]
    perms = [ref_order(np.array([0, len(qq)]), qq) for qq in quality]
    for fn in (api.estimate_monodepth_shared_focal_relative_pose_batch, api.estimate_monodepth_varying_focal_relative_pose_batch):
        got = fn(c1, c2, [s.d1 for s in scs], [s.d2 for s in scs], ro_f, bo, quality=quality)
        ref = fn([a[p] for a, p in zip(c1, perms)], [a[p] for a, p in zip(c2, perms)], [s.d1[p] for s, p in zip(scs, perms)],
                 [s.d2[p] for s, p in zip(scs, perms)], ro_f, bo)
        for (ga, ia), (gb, ib), p in zip(got, ref, perms):
            inl = np.zeros(len(p), bool)
            inl[p] = ib["inliers"]
            assert ia == {**ib, "inliers": inl.tolist()}
            assert ga.pose.q.tobytes() == gb.pose.q.tobytes() and ga.camera1.params == gb.camera1.params


def test_argument_errors_match_twins(ctx):
    L, h = ctx._lib, ctx._h
    n = 10
    x = np.zeros((n, 2)), np.zeros((n, 2), dtype=np.float32)
    d = np.ones(n), np.ones(n, dtype=np.float32)
    q = np.ones(n, dtype=np.float32)
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
        for f32 in (False, True):
            for dev in (False, True):
                k = int(f32)
                ptrs = [P(x[k]), P(x[k]), P(d[k]), P(d[k])] if data else [None] * 4
                tail = [P(cm), C.byref(o) if o is not None else None, P(models), P(stats), P(masks)]
                suffix = ("_f32" if f32 else "")
                twin = getattr(L, ("rp_estimate_batch_dev" if dev else "rp_estimate_batch_host") + suffix)
                qual = getattr(L, ("rp_estimate_batch_dev" if dev else "rp_estimate_batch_host") + suffix + "_quality")
                extra = [None] if dev else []
                # the argument checks come before any device pointer is touched: host arrays stand in for them
                rc_t = twin(hh, var, npairs, P(offs), *ptrs, *tail, *extra)
                e_t = L.rp_last_error(hh).decode() if rc_t and hh else ""
                rc_q = qual(hh, var, npairs, P(offs), *ptrs, P(q) if data else None, *tail, *extra)
                e_q = L.rp_last_error(hh).decode() if rc_q and hh else ""
                assert (rc_q, e_q) == (rc_t, e_t), (name, f32, dev)
                assert rc_q == (0 if name == "ok, zero pairs" else -1), (name, f32, dev)
    # a null quality with a non-empty batch, everything else valid
    for f32 in (False, True):
        for dev in (False, True):
            k = int(f32)
            qual = getattr(L, ("rp_estimate_batch_dev" if dev else "rp_estimate_batch_host") + ("_f32" if f32 else "") + "_quality")
            rc = qual(h, 0, 1, P(good), P(x[k]), P(x[k]), P(d[k]), P(d[k]), None, P(cams), C.byref(opt), P(models), P(stats),
                      P(masks), *([None] if dev else []))
            assert rc == -1 and "quality" in L.rp_last_error(h).decode()
