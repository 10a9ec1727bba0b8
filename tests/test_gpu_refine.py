"""GPU tier: refinement of caller-supplied models (rp_refine_pairs_{host,dev}[_f32], api.refine_*, torch_frontend.refine_batch).

The call is defined as what the estimator does after RANSAC, with the caller's start model in place of the RANSAC model and
the caller's subset in place of the RANSAC inlier mask.  The tests hold it to that definition three ways: against the
estimator itself (bytes for the calibrated variants), against the stage entry point rp_refine_batch fed with the
estimator's pre-processing restated on the host (bytes, all variants), and against the oracle (DESIGN §3 LM contract)."""
import ctypes as C
import math

import numpy as np
import pytest

from mdrp_b200 import _native as nv, synth

pytestmark = pytest.mark.gpu

SIZES = [300, 0, 120, 2, 3, 4, 250, 1, 180]   # ragged, with pairs of 0, 1, 2, 3 and 4 correspondences
CFG = {nv.CALIB: "cfg1_calib_scale", nv.CALIB_SHIFT: "cfg2_calib_shift", nv.SHARED: "cfg3_shared_focal",
       nv.VARYING: "cfg4_varying_focal"}
FOCAL = (nv.SHARED, nv.VARYING)


def _ragged(variant, base, sizes=SIZES):
    cfg = CFG[variant]
    focal = variant in FOCAL
    scs = [synth.scene_for(cfg, base + i, n=max(n, 3)) for i, n in enumerate(sizes)]
    x1 = np.concatenate([(s.centred()[0] if focal else s.x1)[:n] for s, n in zip(scs, sizes)])
    x2 = np.concatenate([(s.centred()[1] if focal else s.x2)[:n] for s, n in zip(scs, sizes)])
    d1 = np.concatenate([s.d1[:n] for s, n in zip(scs, sizes)])
    d2 = np.concatenate([s.d2[:n] for s, n in zip(scs, sizes)])
    offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    cams = None if focal else np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
    return offs, x1, x2, d1, d2, cams


def _options(variant, bundle_iters=100, iters=200):
    o = nv.default_options()
    o.max_iterations = o.min_iterations = iters
    o.max_epipolar_error, o.max_reproj_error = 2.0, 16.0
    o.estimate_shift = int(variant == nv.CALIB_SHIFT)
    o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    o.loss_scale = 1.0 if variant in FOCAL else 0.7   # the calibrated variants ignore it
    o.bundle_max_iterations = bundle_iters
    return o


def _f32(*arrays):
    return [a.astype(np.float32).astype(np.float64) for a in arrays]


def _dev_refine(ctx, variant, offs, x1, x2, d1, d2, cams, o, init, subset):
    import torch
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    P, N = len(offs) - 1, int(offs[-1])
    dm = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    db = torch.zeros(P, 7, dtype=torch.int64, device=dev)
    dn = torch.zeros(P, dtype=torch.int64, device=dev)
    dk = torch.zeros(max(N, 1), dtype=torch.uint8, device=dev)
    tx = [t(a) for a in (x1, x2, d1, d2)]
    ti = t(np.ascontiguousarray(init).view(np.float64).reshape(P, 12))
    ts = t(subset) if subset is not None else None
    tc = t(cams) if cams is not None else None
    fn = ctx.refine_pairs_dev_f32 if x1.dtype == np.float32 else ctx.refine_pairs_dev
    fn(variant, offs, *[a.data_ptr() for a in tx], tc.data_ptr() if tc is not None else None, o, ti.data_ptr(),
       ts.data_ptr() if ts is not None else None, dm.data_ptr(), db.data_ptr(), dn.data_ptr(), dk.data_ptr(),
       torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize()
    return (dm.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1), db.cpu().numpy().view(nv.BSTATS_DTYPE).reshape(-1),
            dn.cpu().numpy(), dk.cpu().numpy()[:N])


def refine(ctx, path, variant, offs, x1, x2, d1, d2, cams, o, init, subset=None, dtype=np.float64):
    a = [v.astype(dtype) for v in (x1, x2, d1, d2)]
    if path == "dev":
        return _dev_refine(ctx, variant, offs, *a, cams, o, init, subset)
    fn = ctx.refine_pairs_host_f32 if dtype == np.float32 else ctx.refine_pairs_host
    return fn(variant, offs, *a, cams, o, init, subset)


def _same(a, b):
    for u, v in zip(a, b):
        assert np.ascontiguousarray(u).tobytes() == np.ascontiguousarray(v).tobytes()


# ---- 1. against the estimator, calibrated variants: bytes ---------------------------------------------------------
@pytest.mark.parametrize("variant", [nv.CALIB, nv.CALIB_SHIFT])
def test_calibrated_equals_estimator_bytes(ctx, variant):
    offs, x1, x2, d1, d2, cams = _ragged(variant, 40)
    x1, x2, d1, d2 = _f32(x1, x2, d1, d2)   # float32-representable, so the float32 entry points see the same values
    o0, o = _options(variant, bundle_iters=0), _options(variant)
    m0, s0, k0 = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, o0)
    m, _, _ = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, o)
    for path in ("host", "dev"):
        for dtype in (np.float64, np.float32):
            got = refine(ctx, path, variant, offs, x1, x2, d1, d2, cams, o, m0, k0, dtype)
            assert got[0].tobytes() == m.tobytes(), (path, dtype)
            g0 = refine(ctx, path, variant, offs, x1, x2, d1, d2, cams, o0, m0, k0, dtype)
            assert g0[0].tobytes() == m0.tobytes()
            assert g0[3].tobytes() == k0.tobytes()
            assert g0[2].tolist() == s0["num_inliers"].tolist()


# ---- 2. against the estimator, focal variants: DESIGN §3 LM contract ------------------------------------------------
def _pose_close(a, b, tol=1e-6):
    q, r = np.asarray(a["q"]), np.asarray(b["q"])
    if np.dot(q, r) < 0:
        r = -r
    rel = lambda u, v: abs(u - v) <= tol * max(1.0, abs(v))
    return (np.allclose(q, r, rtol=0, atol=tol) and np.allclose(a["t"], b["t"], rtol=tol, atol=tol) and
            all(rel(a[k], b[k]) for k in ("scale", "shift1", "shift2", "f1", "f2")))


@pytest.mark.parametrize("variant", FOCAL)
def test_focal_matches_estimator(ctx, variant):
    offs, x1, x2, d1, d2, cams = _ragged(variant, 60)
    o0, o = _options(variant, bundle_iters=0), _options(variant)
    m0, s0, k0 = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, o0)
    m, _, _ = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, o)
    got, bs, _, _ = refine(ctx, "host", variant, offs, x1, x2, d1, d2, cams, o, m0, k0)
    # the estimator's final cost: its model evaluated by the same LM kernel with no iteration
    _, est_bs, _, _ = refine(ctx, "host", variant, offs, x1, x2, d1, d2, cams, o0, m, k0)
    for p in range(len(m)):
        if s0["num_inliers"][p] > 3:
            assert _pose_close(got[p], m[p]), p
            assert bs[p]["cost"] <= est_bs[p]["cost"] * (1 + 1e-9), p
        else:
            assert got[p].tobytes() == m0[p].tobytes()


# ---- 3. against the stage entry point, all variants: bytes ----------------------------------------------------------
def host_prepare(variant, x1, x2, cam, o):
    """The estimator's P1/P2 for one pair, restated with the same IEEE operations as prepare_kernel (oracle ro_estimate):
    (normalised x1, x2, scale_reproj, final loss scale, nscale)."""
    if variant in FOCAL:
        s = 0.0
        for k in range(len(x1)):
            s += math.sqrt(x1[k, 0] * x1[k, 0] + x1[k, 1] * x1[k, 1])
            s += math.sqrt(x2[k, 0] * x2[k, 0] + x2[k, 1] * x2[k, 1])
        nscale = s / (math.sqrt(2.0) * len(x1))
        thr, rep = o.max_epipolar_error / nscale, o.max_reproj_error / nscale
        ls = o.loss_scale / nscale
        a, b = x1 / nscale, x2 / nscale
    else:
        fx1, fy1, cx1, cy1, fx2, fy2, cx2, cy2 = cam
        a = np.stack([(x1[:, 0] - cx1) / fx1, (x1[:, 1] - cy1) / fy1], axis=1)
        b = np.stack([(x2[:, 0] - cx2) / fx2, (x2[:, 1] - cy2) / fy2], axis=1)
        k = 0.5 * (1.0 / (0.5 * (fx1 + fy1)) + 1.0 / (0.5 * (fx2 + fy2)))
        thr, rep = o.max_epipolar_error * k, o.max_reproj_error * k
        ls, nscale = 0.5 * thr, 1.0
    sr = (thr * thr) / (rep * rep) if rep > 0.0 else 0.0
    return a, b, sr, ls, nscale


def _subsets(offs, k0):
    """The estimator's masks, with pair 0 cut to its first half and pair 6 to 3 correspondences (not refined)."""
    s = k0.copy()
    s[offs[0] + (offs[1] - offs[0]) // 2:offs[1]] = 0
    s[offs[6]:offs[7]] = 0
    s[offs[6]:offs[6] + 3] = 1
    return s


@pytest.mark.parametrize("variant", [nv.CALIB, nv.CALIB_SHIFT, nv.SHARED, nv.VARYING])
def test_equals_stage_entry_point_bytes(ctx, port, variant):
    offs, x1, x2, d1, d2, cams = _ragged(variant, 80)
    m0, _, k0 = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, _options(variant, bundle_iters=0))
    subset = _subsets(offs, k0)
    o = _options(variant)
    got, bs, _, _ = refine(ctx, "host", variant, offs, x1, x2, d1, d2, cams, o, m0, subset)
    refined = 0
    for p in range(len(offs) - 1):
        sl = slice(offs[p], offs[p + 1])
        if subset[sl].sum() <= 3:
            assert got[p].tobytes() == m0[p].tobytes() and not bs[p].tobytes().strip(b"\0")
            continue
        refined += 1
        a, b, sr, ls, nscale = host_prepare(variant, x1[sl], x2[sl], cams[p] if cams is not None else None, o)
        start = m0[p:p + 1].copy()
        if variant in FOCAL:
            start["f1"] /= nscale
            start["f2"] /= nscale
        bopt = nv.bundle_options(o.bundle_max_iterations, o.loss_type, ls, o.gradient_tol, o.step_tol, o.initial_lambda,
                                 o.min_lambda, o.max_lambda)
        ref, rst = ctx.refine(variant, start, a, b, d1[sl], d2[sl], sr, o.weight_sampson, bopt, mask=subset[sl])
        # 4. the oracle on the same normalised subset, DESIGN §3 LM contract
        s = subset[sl].astype(bool)
        pm = port.make_model(*[start[0][k] for k in ("q", "t", "scale", "shift1", "shift2", "f1", "f2")])
        om, ost = port.refine(variant, a[s], b[s], d1[sl][s], d2[sl][s], pm, sr, o.weight_sampson,
                              port.bundle_opt(o.bundle_max_iterations, "TRUNCATED_CAUCHY", ls, o.gradient_tol, o.step_tol,
                                              o.initial_lambda, o.min_lambda, o.max_lambda))
        assert rst[0]["cost"] <= ost.cost * (1 + 1e-9)
        if variant in FOCAL:
            ref["f1"] *= nscale
            ref["f2"] *= nscale
        assert got[p].tobytes() == ref[0].tobytes(), p
        assert bs[p].tobytes() == rst[0].tobytes(), p
        oq, ot, osc, os1, os2, of1, of2 = om.as_tuple()
        orow = np.zeros((), nv.MODEL_DTYPE)
        orow["q"], orow["t"], orow["scale"], orow["shift1"], orow["shift2"] = oq, ot, osc, os1, os2
        orow["f1"], orow["f2"] = (of1 * nscale, of2 * nscale) if variant in FOCAL else (of1, of2)
        assert _pose_close(ref[0], orow), p
        if variant == nv.CALIB:   # 7 parameters: the shifts are held
            assert (got[p]["shift1"], got[p]["shift2"]) == (m0[p]["shift1"], m0[p]["shift2"])
        if variant not in FOCAL:   # f1 / f2 are returned as given
            assert (got[p]["f1"], got[p]["f2"]) == (m0[p]["f1"], m0[p]["f2"])
    assert refined >= 3


# ---- 5. independence of the batch and of the chunking; null subset ---------------------------------------------------
def _gt_models(b, P):
    from scipy.spatial.transform import Rotation as Rot
    q = Rot.from_matrix(b["R"]).as_quat()   # x, y, z, w
    m = np.zeros(P, nv.MODEL_DTYPE)
    m["q"] = np.c_[q[:, 3], q[:, :3]]
    m["t"] = b["t"] * 1.05
    m["scale"], m["f1"], m["f2"] = 1.6, 1.0, 1.0
    return m


def test_independent_of_batch_and_chunking(ctx, monkeypatch):
    P, n = 1100, 1500   # 1.65 M correspondences: several chunks on both paths in a 0.1 GB workspace
    b = synth.make_batch("cfg1_calib_scale", P, seed=5, n=n)
    offs, cams = b["offsets"], b["cams"]
    x1, x2, d1, d2 = (b[k] for k in ("x1", "x2", "d1", "d2"))
    init, subset = _gt_models(b, P), b["inliers"].astype(np.uint8)
    o = _options(nv.CALIB)
    ref = refine(ctx, "dev", nv.CALIB, offs, x1, x2, d1, d2, cams, o, init, subset)
    _same(refine(ctx, "host", nv.CALIB, offs, x1, x2, d1, d2, cams, o, init, subset), ref)
    for p in (0, 517, P - 1):
        sl = slice(offs[p], offs[p + 1])
        alone = refine(ctx, "host", nv.CALIB, np.array([0, n]), x1[sl], x2[sl], d1[sl], d2[sl], cams[p:p + 1], o,
                       init[p:p + 1], subset[sl])
        _same(alone, (ref[0][p:p + 1], ref[1][p:p + 1], ref[2][p:p + 1], ref[3][sl]))
    monkeypatch.setenv("RP_WORKSPACE_GB", "0.1")
    small = nv.Context(0)
    try:
        for path in ("host", "dev"):
            _same(refine(small, path, nv.CALIB, offs, x1, x2, d1, d2, cams, o, init, subset), ref)
    finally:
        small.close()


@pytest.mark.parametrize("variant", [nv.CALIB_SHIFT, nv.VARYING])
def test_null_subset_is_all_ones(ctx, variant):
    offs, x1, x2, d1, d2, cams = _ragged(variant, 100)
    m0, _, _ = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, _options(variant, bundle_iters=0))
    o = _options(variant)
    for path in ("host", "dev"):
        a = refine(ctx, path, variant, offs, x1, x2, d1, d2, cams, o, m0, None)
        _same(a, refine(ctx, path, variant, offs, x1, x2, d1, d2, cams, o, m0, np.ones(int(offs[-1]), np.uint8)))


# ---- 6. pairs that are not refined ------------------------------------------------------------------------------------
def test_pairs_not_refined_keep_init_bytes(ctx):
    variant = nv.SHARED
    offs, x1, x2, d1, d2, cams = _ragged(variant, 120)
    P = len(offs) - 1
    init = np.zeros(P, nv.MODEL_DTYPE)
    init["q"] = [0.9, 0.1, -0.3, 0.2]   # not normalised: bytes must survive untouched
    init["t"], init["scale"], init["shift1"], init["shift2"] = [0.1, 0.2, 0.3], 1.3, 0.1, -0.1
    init["f1"], init["f2"] = 1e-7 + np.arange(P), 3.0   # values whose f / nscale * nscale round trip would show
    subset = np.zeros(int(offs[-1]), np.uint8)
    subset[offs[6]:offs[6] + 3] = 1         # 3 selected of 250: not refined
    subset[offs[5]:offs[6]] = 1             # the pair of 4 correspondences: refined
    for path in ("host", "dev"):
        m, bs, ni, inl = refine(ctx, path, variant, offs, x1, x2, d1, d2, cams, _options(variant), init, subset)
        for p in range(P):
            if p == 5:   # refined: its bundle stats are written
                assert bs[p].tobytes().strip(b"\0")
                continue
            assert m[p].tobytes() == init[p].tobytes() and not bs[p].tobytes().strip(b"\0"), p
            if offs[p + 1] - offs[p] < 3:
                assert ni[p] == 0 and not inl[offs[p]:offs[p + 1]].any()
        assert ni.tolist() == [int(inl[offs[p]:offs[p + 1]].sum()) for p in range(P)]


# ---- 7. state of the last estimate call -------------------------------------------------------------------------------
def test_state_of_last_estimate_is_kept(ctx):
    variant = nv.CALIB
    offs, x1, x2, d1, d2, cams = _ragged(variant, 140)
    m0, _, k0 = ctx.estimate_batch_host(variant, offs, x1, x2, d1, d2, cams, _options(variant))
    P = len(offs) - 1
    st, tm = ctx.pair_status(P), ctx.last_timing()
    refine(ctx, "host", variant, offs, x1, x2, d1, d2, cams, _options(variant), m0, k0)
    refine(ctx, "dev", variant, offs[:3], x1[:offs[2]], x2[:offs[2]], d1[:offs[2]], d2[:offs[2]], cams[:2],
           _options(variant), m0[:2], None)
    assert ctx.pair_status(P).tolist() == st.tolist()
    assert ctx.last_timing() == tm


# ---- 8. argument errors -----------------------------------------------------------------------------------------------
def test_argument_errors_are_the_estimators(ctx):
    L, h = ctx._lib, ctx._h
    offs, x1, x2, d1, d2, cams = _ragged(nv.CALIB, 160, sizes=[5, 6])
    P, N = 2, 11
    o = _options(nv.CALIB)
    init = np.zeros(P, nv.MODEL_DTYPE)
    out_m, out_s, out_k = np.zeros(P, nv.MODEL_DTYPE), np.zeros(P, nv.STATS_DTYPE), np.zeros(N, np.uint8)
    out_b, out_n = np.zeros(P, nv.BSTATS_DTYPE), np.zeros(P, np.int64)
    p = lambda a: a.ctypes.data if a is not None else None
    bad_o = _options(nv.CALIB)
    bad_o.max_iterations = -1
    cases = [  # (variant, n_pairs, offsets, x1, cams, opt)
        (7, P, offs, x1, cams, o), (nv.CALIB, P, None, x1, cams, o), (nv.CALIB, P, np.array([0, 6, 5], np.int64), x1, cams, o),
        (nv.CALIB, P, offs, None, cams, o), (nv.CALIB, P, offs, x1, None, o), (nv.CALIB, P, offs, x1, cams, bad_o),
        (nv.CALIB, P, offs, x1, cams, None), (nv.CALIB, -1, offs, x1, cams, o)]
    for v, n, of, a1, cm, op in cases:
        oref = C.byref(op) if op is not None else None
        est = L.rp_estimate_batch_host(h, v, n, p(of), p(a1), p(x2), p(d1), p(d2), p(cm), oref, p(out_m), p(out_s), p(out_k))
        got = L.rp_refine_pairs_host(h, v, n, p(of), p(a1), p(x2), p(d1), p(d2), p(cm), oref, p(init), None, p(out_m),
                                     p(out_b), p(out_n), p(out_k))
        assert est < 0 and got == est, (v, n, est, got)
    for bad_init, bad_models in ((None, out_m), (init, None)):
        assert L.rp_refine_pairs_host(h, nv.CALIB, P, p(offs), p(x1), p(x2), p(d1), p(d2), p(cams), C.byref(o), p(bad_init),
                                      None, p(bad_models), None, None, None) == -1
    # an empty batch is fine with null data pointers
    assert L.rp_refine_pairs_host(h, nv.CALIB, 0, p(np.zeros(1, np.int64)), None, None, None, None, None, C.byref(o),
                                  None, None, None, None, None, None) == 0


# ---- 9. torch ---------------------------------------------------------------------------------------------------------
def test_torch_refine_batch_equals_host(ctx):
    import torch
    from mdrp_b200 import torch_frontend as tf
    variant = nv.VARYING
    offs, x1, x2, d1, d2, cams = _ragged(variant, 180)
    o = _options(variant)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    em, _, ek = tf.estimate_batch(variant, offs, t(x1), t(x2), t(d1), t(d2), None, _options(variant, bundle_iters=0))
    host = ctx.refine_pairs_host(variant, offs, x1, x2, d1, d2, None, o, em.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1),
                                 ek.cpu().numpy())
    for dtype in (torch.float64, torch.float32):
        c = lambda a: t(a).to(dtype)
        m, bs, ni, inl = tf.refine_batch(variant, offs, c(x1.astype(np.float32)), c(x2.astype(np.float32)),
                                         c(d1.astype(np.float32)), c(d2.astype(np.float32)), None, em, o, subset=ek)
        ref = ctx.refine_pairs_host_f32(variant, offs, x1.astype(np.float32), x2.astype(np.float32),
                                        d1.astype(np.float32), d2.astype(np.float32), None, o,
                                        em.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1), ek.cpu().numpy())
        _same((m.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1), tf.bstats_to_numpy(bs), ni.cpu().numpy(),
               inl.cpu().numpy()), ref)
    m, bs, ni, inl = tf.refine_batch(variant, offs, t(x1), t(x2), t(d1), t(d2), None, em, o, subset=ek)
    _same((m.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1), tf.bstats_to_numpy(bs), ni.cpu().numpy(), inl.cpu().numpy()),
          host)


def test_torch_tracking_chain(ctx):
    """gather_depths_batch -> estimate_batch on frame pairs (f, f+1) -> refine_batch of the next pairs (f+1, f+2) from the
    previous models, as a tracker does; pairs whose inlier count drops would go back to estimate_batch."""
    import torch
    from mdrp_b200 import torch_frontend as tf
    dev = torch.device("cuda", 0)
    g = torch.Generator(device="cpu").manual_seed(0)
    F, H, W, n = 5, 96, 128, 400
    depth = (2.0 + 6.0 * torch.rand(F, H, W, generator=g)).to(dev)
    kp1 = (torch.rand(4 * n, 2, generator=g) * torch.tensor([W - 1.0, H - 1.0])).to(dev)
    kp2 = (kp1 + 0.5 * torch.randn(4 * n, 2, generator=g).to(dev)).clamp(0, W - 1)
    offs = np.arange(4 + 1, dtype=np.int64) * n
    cams = torch.tensor([[100.0, 100.0, 64.0, 48.0] * 2] * 3, dtype=torch.float64, device=dev)
    o = _options(nv.CALIB)
    first = tf.gather_depths_batch(depth, [0, 1, 2], [1, 2, 3], offs[:4], kp1[:3 * n], kp2[:3 * n], dtype=torch.float32)
    models, stats, masks = tf.estimate_batch(nv.CALIB, first[0], *first[1:], cams, o)
    nxt = tf.gather_depths_batch(depth, [1, 2, 3], [2, 3, 4], offs[:4], kp1[n:], kp2[n:], dtype=torch.float32)
    m, bs, ni, inl = tf.refine_batch(nv.CALIB, nxt[0], *nxt[1:], cams, models, o)
    assert m.shape == (3, 12) and ni.shape == (3,) and ni.dtype == torch.int64
    assert inl.shape == (int(nxt[0][-1]),)
    assert ni.cpu().tolist() == [int(inl[int(nxt[0][p]):int(nxt[0][p + 1])].sum()) for p in range(3)]


# ---- api ----------------------------------------------------------------------------------------------------------
def test_api_refine_batch_equals_context(ctx):
    from mdrp_b200 import api
    variant = nv.SHARED
    offs, x1, x2, d1, d2, _ = _ragged(variant, 200, sizes=[200, 150])
    res = api.estimate_monodepth_shared_focal_relative_pose_batch(
        [x1[:200], x1[200:]], [x2[:200], x2[200:]], [d1[:200], d1[200:]], [d2[:200], d2[200:]],
        ransac_opt={"max_iterations": 200, "min_iterations": 200, "max_epipolar_error": 2.0},
        bundle_opt={"max_iterations": 0})
    pairs = [r[0] for r in res]
    out = api.refine_monodepth_shared_focal_relative_pose_batch(
        [x1[:200], x1[200:]], [x2[:200], x2[200:]], [d1[:200], d1[200:]], [d2[:200], d2[200:]], pairs,
        ransac_opt={"max_epipolar_error": 2.0}, bundle_opt={"loss_type": "TRUNCATED_CAUCHY"},
        subsets=[r[1]["inliers"] for r in res])
    for (pair, info), (_, info0) in zip(out, res):
        assert info["iterations"] > 0 and info["cost"] <= info["initial_cost"]
        assert info["num_inliers"] == sum(info["inliers"]) and abs(pair.camera1.focal() / 800.0 - 1) < 0.2
