"""GPU tier: the match quality through the depth gathers (rp_gather_depths_*_quality, `torch_frontend.gather_depths*`
with `quality=`) and through the sharded entry points.

The _quality gathers are defined against their twins: x1, x2, d1, d2 and the kept count / packed offsets are the twin's
bytes, and quality_out is quality[keep] (input order, 32-bit patterns) under the twin's keep rule.  Every test here
compares with the twin and with the host recipe of the reference's callers: depth_map[(int)y, (int)x] with the index
clamped to the map, rows whose two depths are both infinite dropped."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from mdrp_b200 import _native as nv, api, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = ["float64", "float32"]


def _torch():
    import torch
    return torch


def special_quality(n, rng):
    """float32 qualities with NaNs (one with a payload), -0, +-inf, subnormals and ordinary values."""
    vals = np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-45, -1e-45, 3e-39, -3e-39, 0.5, 1.0, -1.0],
                    np.float32)
    q = np.where(rng.uniform(size=n) < 0.5, rng.choice(vals, n), rng.standard_normal(n)).astype(np.float32)
    q.view(np.uint32)[rng.uniform(size=n) < 0.05] = 0x7fc01234
    q.view(np.uint32)[rng.uniform(size=n) < 0.05] = 0xffa00001   # a signalling-NaN pattern
    return q


def recipe(dm1, dm2, kp1, kp2):
    """(keep, d1, d2) of the reference's host recipe: (int) truncation, border clamp, both-inf rows dropped."""
    def look(dm, kp):
        h, w = dm.shape
        r = np.clip(kp[:, 1].astype(np.int64), 0, h - 1)
        c = np.clip(kp[:, 0].astype(np.int64), 0, w - 1)
        return dm[r, c]
    d1, d2 = look(dm1, kp1), look(dm2, kp2)
    return ~(np.isinf(d1) & np.isinf(d2)), d1, d2


def _maps_and_keypoints(rng, F, H, W, n, inf_frac=0.2):
    maps = rng.uniform(1, 9, size=(F, H, W)).astype(np.float32)
    maps[rng.uniform(size=maps.shape) < inf_frac] = np.inf
    # some outside the map on every side (clamped), some with small negative coordinates ((int) truncates towards 0)
    kp1 = rng.uniform(-4, [W + 4, H + 4], size=(n, 2)).astype(np.float32)
    kp2 = rng.uniform(-4, [W + 4, H + 4], size=(n, 2)).astype(np.float32)
    kp1[::7] = -rng.uniform(0, 1, size=kp1[::7].shape).astype(np.float32)
    return maps, kp1, kp2


def _np(t):
    return t.cpu().numpy()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


# ---- single pair ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
def test_single_gather_quality_equals_twin_and_recipe(ctx, dtype):
    torch = _torch()
    from mdrp_b200 import torch_frontend as tf
    dt = getattr(torch, dtype)
    rng = np.random.default_rng(21)
    H, W = 120, 160
    for n in (0, 1, 600, 1025):
        maps, kp1, kp2 = _maps_and_keypoints(rng, 2, H, W, n)
        if n == 600:   # both-inf rows (dropped) and single-inf rows (kept) at known keypoints
            maps[0, kp1[:40, 1].astype(int).clip(0, H - 1), kp1[:40, 0].astype(int).clip(0, W - 1)] = np.inf
            maps[1, kp2[:20, 1].astype(int).clip(0, H - 1), kp2[:20, 0].astype(int).clip(0, W - 1)] = np.inf
        q = special_quality(n, rng)
        g = torch.from_numpy(maps).cuda()
        k1, k2, tq = torch.from_numpy(kp1).cuda(), torch.from_numpy(kp2).cuda(), torch.from_numpy(q).cuda()
        twin = tf.gather_depths(g[0], g[1], k1, k2, dtype=dt)
        got = tf.gather_depths(g[0], g[1], k1, k2, dtype=dt, quality=tq)
        assert len(got) == 5 and got[4].dtype == torch.float32 and got[4].is_cuda
        for a, b in zip(got[:4], twin):
            assert a.dtype == dt and _np(a).tobytes() == _np(b).tobytes(), n
        keep, d1, d2 = recipe(maps[0], maps[1], kp1, kp2)
        npdt = np.dtype(dtype)
        assert _np(got[0]).tobytes() == kp1[keep].astype(npdt).tobytes()
        assert _np(got[1]).tobytes() == kp2[keep].astype(npdt).tobytes()
        assert _np(got[2]).tobytes() == d1[keep].astype(npdt).tobytes()
        assert _np(got[3]).tobytes() == d2[keep].astype(npdt).tobytes()
        assert np.array_equal(_bits(_np(got[4])), _bits(q[keep])), n
        if n == 600:
            assert 0 < keep.sum() < n and (np.isinf(d1[keep]) | np.isinf(d2[keep])).any()


@pytest.mark.parametrize("dtype", DTYPES)
def test_single_gather_quality_every_row_dropped(ctx, dtype):
    torch = _torch()
    from mdrp_b200 import torch_frontend as tf
    rng = np.random.default_rng(22)
    maps, kp1, kp2 = _maps_and_keypoints(rng, 2, 30, 40, 300)
    maps[:] = np.inf
    g = torch.from_numpy(maps).cuda()
    q = torch.from_numpy(special_quality(300, rng)).cuda()
    got = tf.gather_depths(g[0], g[1], torch.from_numpy(kp1).cuda(), torch.from_numpy(kp2).cuda(),
                           dtype=getattr(torch, dtype), quality=q)
    assert [t.shape[0] for t in got] == [0] * 5


def test_single_gather_float64_quality_is_converted(ctx):
    torch = _torch()
    from mdrp_b200 import torch_frontend as tf
    rng = np.random.default_rng(23)
    maps, kp1, kp2 = _maps_and_keypoints(rng, 2, 50, 60, 200)
    g = torch.from_numpy(maps).cuda()
    k1, k2 = torch.from_numpy(kp1).cuda(), torch.from_numpy(kp2).cuda()
    q64 = rng.uniform(size=200)
    got = tf.gather_depths(g[0], g[1], k1, k2, quality=torch.from_numpy(q64).cuda())
    keep = recipe(maps[0], maps[1], kp1, kp2)[0]
    assert np.array_equal(_bits(_np(got[4])), _bits(q64.astype(np.float32)[keep]))
    with pytest.raises(ValueError):
        tf.gather_depths(g[0], g[1], k1, k2, quality=torch.from_numpy(q64[:-1]).cuda())
    with pytest.raises(ValueError):
        tf.gather_depths(g[0], g[1], k1, k2, quality=torch.from_numpy(q64))   # host tensor


# ---- batch ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
def test_batch_gather_quality_equals_twin_and_recipe(ctx, dtype):
    torch = _torch()
    from mdrp_b200 import torch_frontend as tf
    dt = getattr(torch, dtype)
    rng = np.random.default_rng(31)
    F, H, W = 5, 120, 160
    sizes = [700, 0, 33, 1025, 256, 40, 1, 300, 0, 90]
    f1 = [0, 1, 2, 3, 0, 0, 2, 4, 3, 1]   # repeated frames, a frame paired with itself
    f2 = [1, 2, 3, 0, 2, 0, 2, 4, 3, 1]
    offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    maps, kp1, kp2 = _maps_and_keypoints(rng, F, H, W, int(offs[-1]))
    maps[4] = np.inf   # pair 7 reads frame 4 on both sides: every row dropped
    q = special_quality(int(offs[-1]), rng)
    g = torch.from_numpy(maps).cuda()
    k1, k2, tq = torch.from_numpy(kp1).cuda(), torch.from_numpy(kp2).cuda(), torch.from_numpy(q).cuda()
    twin = tf.gather_depths_batch(g, f1, f2, offs, k1, k2, dtype=dt)
    got = tf.gather_depths_batch(g, f1, f2, offs, k1, k2, dtype=dt, quality=tq)
    assert len(got) == 6 and np.array_equal(got[0], twin[0])
    for a, b in zip(got[1:5], twin[1:]):
        assert a.dtype == dt and _np(a).tobytes() == _np(b).tobytes()
    out, qo = got[0], _np(got[5])
    assert qo.shape == (out[-1],)
    npdt = np.dtype(dtype)
    for p in range(len(sizes)):
        sl, o = slice(offs[p], offs[p + 1]), slice(out[p], out[p + 1])
        keep, d1, d2 = recipe(maps[f1[p]], maps[f2[p]], kp1[sl], kp2[sl])
        assert out[p + 1] - out[p] == keep.sum(), p
        assert _np(got[1][o]).tobytes() == kp1[sl][keep].astype(npdt).tobytes()
        assert _np(got[2][o]).tobytes() == kp2[sl][keep].astype(npdt).tobytes()
        assert _np(got[3][o]).tobytes() == d1[keep].astype(npdt).tobytes()
        assert _np(got[4][o]).tobytes() == d2[keep].astype(npdt).tobytes()
        assert np.array_equal(_bits(qo[o]), _bits(q[sl][keep])), p
    assert out[8] == out[7] and sizes[7] > 0


def test_batch_gather_quality_all_pairs_empty(ctx):
    torch = _torch()
    from mdrp_b200 import torch_frontend as tf
    g = torch.ones(2, 10, 10, device="cuda")
    e = torch.zeros(0, 2, device="cuda")
    got = tf.gather_depths_batch(g, [0, 1], [1, 0], [0, 0, 0], e, e, quality=torch.zeros(0, device="cuda"))
    assert list(got[0]) == [0, 0, 0] and [t.shape[0] for t in got[1:]] == [0] * 5


# ---- the chain: gather_depths_batch(quality) -> estimate_batch(quality) ----------------------------------------------
def _video_like(seed, sizes, H=960, W=1280):
    """Per pair its own two frames, with the scene's depths written at its keypoints; some both-inf and single-inf rows."""
    rng = np.random.default_rng(seed)
    P = len(sizes)
    maps = rng.uniform(1, 9, size=(2 * P, H, W)).astype(np.float32)
    kp1s, kp2s, qs, cams, scs = [], [], [], [], []
    for p, n in enumerate(sizes):
        sc = synth.scene_for("cfg2_calib_shift", 300 + p, n=max(n, 3))
        k1 = np.clip(sc.x1[:n], 0, [W - 1.001, H - 1.001]).astype(np.float32)
        k2 = np.clip(sc.x2[:n], 0, [W - 1.001, H - 1.001]).astype(np.float32)
        maps[2 * p][k1[:, 1].astype(int), k1[:, 0].astype(int)] = sc.d1[:n].astype(np.float32)
        maps[2 * p + 1][k2[:, 1].astype(int), k2[:, 0].astype(int)] = sc.d2[:n].astype(np.float32)
        if n >= 50:
            maps[2 * p][k1[:10, 1].astype(int), k1[:10, 0].astype(int)] = np.inf       # both inf: dropped
            maps[2 * p + 1][k2[:10, 1].astype(int), k2[:10, 0].astype(int)] = np.inf
            maps[2 * p][k1[40:45, 1].astype(int), k1[40:45, 0].astype(int)] = np.inf   # one inf: kept
        inl = sc.inlier_mask[:n]
        q = np.where(inl, rng.uniform(0.3, 1.0, n), rng.uniform(0.0, 0.7, n)).astype(np.float32)
        q[::17] = 0.5
        kp1s.append(k1), kp2s.append(k2), qs.append(q), scs.append(sc)
        cams.append(sc.camera_dicts())
    offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    f1, f2 = np.arange(P) * 2, np.arange(P) * 2 + 1
    return maps, f1, f2, offs, np.concatenate(kp1s), np.concatenate(kp2s), np.concatenate(qs), cams


@pytest.mark.parametrize("dtype", DTYPES)
def test_chain_equals_host_recipe(ctx, dtype):
    torch = _torch()
    from mdrp_b200 import torch_frontend as tf
    dt, npdt = getattr(torch, dtype), np.dtype(dtype)
    sizes = [600, 0, 2, 450, 1200, 80]
    maps, f1, f2, offs, kp1, kp2, q, cams = _video_like(41, sizes)
    ro = {"max_iterations": 500, "min_iterations": 500, "max_epipolar_error": 2.0, "max_reproj_error": 16.0,
          "monodepth_estimate_shift": True, "progressive_sampling": True, "max_prosac_iterations": 300}
    bo = {"loss_type": "TRUNCATED_CAUCHY"}
    P = len(sizes)

    # device chain
    g = torch.from_numpy(maps).cuda()
    out, x1, x2, d1, d2, qo = tf.gather_depths_batch(g, f1, f2, offs, torch.from_numpy(kp1).cuda(),
                                                     torch.from_numpy(kp2).cuda(), dtype=dt,
                                                     quality=torch.from_numpy(q).cuda())
    finite = torch.isfinite(d1) & torch.isfinite(d2)
    pair_of = np.repeat(np.arange(P), np.diff(out))
    fin = _np(finite)
    offs2 = np.r_[0, np.cumsum(np.bincount(pair_of[fin], minlength=P))].astype(np.int64)
    x1, x2, d1, d2, qo = x1[finite], x2[finite], d1[finite], d2[finite], qo[finite]
    opt = api.make_options(ro, bo, focal_variant=False)
    tcams = torch.tensor([api.Camera.from_any(a).fxfycxcy() + api.Camera.from_any(b).fxfycxcy() for a, b in cams],
                         dtype=torch.float64, device="cuda")
    m, s, k = tf.estimate_batch(nv.CALIB_SHIFT, offs2, x1, x2, d1, d2, tcams, opt, quality=qo)
    torch.cuda.synchronize()
    st_dev = api.context(0).pair_status(P)
    m, s, k = _np(m), tf.stats_to_numpy(s), _np(k)

    # host recipe: compact in numpy, drop the non-finite rows, then the api batch call with per-pair q[keep]
    p1, p2, e1, e2, pq = [], [], [], [], []
    for p in range(P):
        sl = slice(offs[p], offs[p + 1])
        keep, a1, a2 = recipe(maps[f1[p]], maps[f2[p]], kp1[sl], kp2[sl])
        keep &= np.isfinite(a1) & np.isfinite(a2)
        p1.append(kp1[sl][keep].astype(npdt)), p2.append(kp2[sl][keep].astype(npdt))
        e1.append(a1[keep].astype(npdt)), e2.append(a2[keep].astype(npdt)), pq.append(q[sl][keep])
    assert [len(a) for a in p1] == list(np.diff(offs2))
    res = api.estimate_monodepth_relative_pose_batch(p1, p2, e1, e2, [c[0] for c in cams], [c[1] for c in cams], ro, bo,
                                                     quality=pq)
    st_host = api.context(0).pair_status(P)
    assert st_dev.tobytes() == st_host.tobytes()
    assert (st_host[np.diff(offs2) < 3] == nv.PAIR_DEGENERATE).all()
    for p, (geom, info) in enumerate(res):
        ref = np.r_[geom.pose.q, geom.pose.t, geom.scale, geom.shift1, geom.shift2, 1.0, 1.0]
        assert m[p].tobytes()[:80] == ref[:10].tobytes(), p
        row = np.array([(info["refinements"], info["iterations"], info["num_inliers"], info["inlier_ratio"],
                         info["model_score"])], dtype=nv.STATS_DTYPE)
        assert s[p:p + 1].tobytes() == row.tobytes(), p
        assert k[offs2[p]:offs2[p + 1]].tobytes() == np.array(info["inliers"], dtype=np.uint8).tobytes(), p
    assert s["num_inliers"].max() > 100


# ---- argument errors ------------------------------------------------------------------------------------------------
def test_gather_quality_argument_errors_match_twins(ctx):
    torch = _torch()
    L, h = ctx._lib, ctx._h
    n = 16
    dm = torch.ones(2, 8, 8, device="cuda")
    kp = torch.ones(n, 2, device="cuda")
    q = torch.ones(n, device="cuda")
    outs = {np.float64: [torch.zeros(n, 2, dtype=torch.float64, device="cuda") for _ in range(2)] +
            [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(2)],
            np.float32: [torch.zeros(n, 2, device="cuda") for _ in range(2)] + [torch.zeros(n, device="cuda") for _ in range(2)]}
    q_out = torch.zeros(n, device="cuda")
    D, K, Q, QO = dm.data_ptr(), kp.data_ptr(), q.data_ptr(), q_out.data_ptr()
    n_out = C.c_int64(0)
    N_OUT = C.byref(n_out)

    def err(rc):
        return L.rp_last_error(h).decode() if rc else ""

    single = {   # name -> (ctx, depth1, h1, w1, depth2, h2, w2, kp1, kp2, n, outputs given, n_out)
        "null ctx": (None, D, 8, 8, D, 8, 8, K, K, n, True, N_OUT), "negative n": (h, D, 8, 8, D, 8, 8, K, K, -1, True, N_OUT),
        "null n_out": (h, D, 8, 8, D, 8, 8, K, K, n, True, None), "h1": (h, D, 0, 8, D, 8, 8, K, K, n, True, N_OUT),
        "w2": (h, D, 8, 8, D, 8, -1, K, K, n, True, N_OUT), "null depth": (h, None, 8, 8, D, 8, 8, K, K, n, True, N_OUT),
        "null kp2": (h, D, 8, 8, D, 8, 8, K, None, n, True, N_OUT), "null outputs": (h, D, 8, 8, D, 8, 8, K, K, n, False, N_OUT),
        "ok, empty": (h, None, 8, 8, None, 8, 8, None, None, 0, False, N_OUT), "ok": (h, D, 8, 8, D, 8, 8, K, K, n, True, N_OUT),
    }
    for name, (hh, d1p, h1, w1, d2p, h2, w2, k1p, k2p, nn, given, no) in single.items():
        for npdt, suffix in ((np.float64, ""), (np.float32, "_f32")):
            o = [t.data_ptr() for t in outs[npdt]] if given else [None] * 4
            twin = getattr(L, "rp_gather_depths_dev" + suffix)
            qual = getattr(L, "rp_gather_depths_dev" + suffix + "_quality")
            rc_t = twin(hh, d1p, h1, w1, d2p, h2, w2, k1p, k2p, nn, *o, no, None)
            e_t = err(rc_t) if hh else ""
            rc_q = qual(hh, d1p, h1, w1, d2p, h2, w2, k1p, k2p, Q if nn else None, nn, *o, QO if nn else None, no, None)
            e_q = err(rc_q) if hh else ""
            assert (rc_q, e_q) == (rc_t, e_t), (name, suffix)
            assert rc_q == (0 if name.startswith("ok") else -1), (name, suffix)
    for suffix in ("", "_f32"):
        qual = getattr(L, "rp_gather_depths_dev" + suffix + "_quality")
        o = [t.data_ptr() for t in outs[np.float32 if suffix else np.float64]]
        for qq, qqo in ((None, QO), (Q, None), (None, None)):
            rc = qual(h, D, 8, 8, D, 8, 8, K, K, qq, n, *o, qqo, N_OUT, None)
            assert rc == -1 and "quality" in err(rc), suffix

    good = np.array([0, 6, 16], dtype=np.int64)
    dec = np.array([0, 9, 4], dtype=np.int64)
    empty = np.array([0, 0, 0], dtype=np.int64)
    fr0, fr1, fr_bad = np.array([0, 1], np.int32), np.array([1, 0], np.int32), np.array([0, 2], np.int32)
    out_off = np.zeros(3, dtype=np.int64)
    P = lambda a: a.ctypes.data if a is not None else None   # noqa: E731
    batch = {   # name -> (ctx, n_pairs, in_offsets, depth_maps, n_frames, h, w, frame1, frame2, kp, outputs given, out_offsets)
        "null ctx": (None, 2, good, D, 2, 8, 8, fr0, fr1, K, True, out_off),
        "negative n_pairs": (h, -1, good, D, 2, 8, 8, fr0, fr1, K, True, out_off),
        "null offsets": (h, 2, None, D, 2, 8, 8, fr0, fr1, K, True, out_off),
        "null out_offsets": (h, 2, good, D, 2, 8, 8, fr0, fr1, K, True, None),
        "h": (h, 2, good, D, 2, 0, 8, fr0, fr1, K, True, out_off),
        "n_frames": (h, 2, good, D, 0, 8, 8, fr0, fr1, K, True, out_off),
        "null depth_maps": (h, 2, good, None, 2, 8, 8, fr0, fr1, K, True, out_off),
        "null frame2": (h, 2, good, D, 2, 8, 8, fr0, None, K, True, out_off),
        "offsets decrease": (h, 2, dec, D, 2, 8, 8, fr0, fr1, K, True, out_off),
        "frame out of range": (h, 2, good, D, 2, 8, 8, fr0, fr_bad, K, True, out_off),
        "null data": (h, 2, good, D, 2, 8, 8, fr0, fr1, None, True, out_off),
        "null outputs": (h, 2, good, D, 2, 8, 8, fr0, fr1, K, False, out_off),
        "ok, zero pairs": (h, 0, good[:1], None, 2, 8, 8, None, None, None, False, out_off),
        "ok, empty pairs": (h, 2, empty, D, 2, 8, 8, fr0, fr1, None, False, out_off),
        "ok": (h, 2, good, D, 2, 8, 8, fr0, fr1, K, True, out_off),
    }
    for name, (hh, npairs, offs, dmp, nf, hh_, ww, a, b, kpp, given, oo) in batch.items():
        for npdt, suffix in ((np.float64, ""), (np.float32, "_f32")):
            o = [t.data_ptr() for t in outs[npdt]] if given else [None] * 4
            twin = getattr(L, "rp_gather_depths_batch_dev" + suffix)
            qual = getattr(L, "rp_gather_depths_batch_dev" + suffix + "_quality")
            nonempty = offs is not None and npairs > 0 and offs[npairs] > offs[0]
            rc_t = twin(hh, npairs, P(offs), dmp, nf, hh_, ww, P(a), P(b), kpp, kpp, *o, P(oo), None)
            e_t = err(rc_t) if hh else ""
            ref_out = out_off.copy()
            rc_q = qual(hh, npairs, P(offs), dmp, nf, hh_, ww, P(a), P(b), kpp, kpp, Q if nonempty else None, *o,
                        QO if nonempty else None, P(oo), None)
            e_q = err(rc_q) if hh else ""
            assert (rc_q, e_q) == (rc_t, e_t), (name, suffix)
            assert rc_q == (0 if name.startswith("ok") else -1), (name, suffix)
            if rc_q == 0:
                assert np.array_equal(out_off, ref_out), name
    for suffix in ("", "_f32"):
        qual = getattr(L, "rp_gather_depths_batch_dev" + suffix + "_quality")
        o = [t.data_ptr() for t in outs[np.float32 if suffix else np.float64]]
        for qq, qqo in ((None, QO), (Q, None)):
            rc = qual(h, 2, P(good), D, 2, 8, 8, P(fr0), P(fr1), K, K, qq, *o, qqo, P(out_off), None)
            assert rc == -1 and "quality" in err(rc), suffix


# ---- sharding -------------------------------------------------------------------------------------------------------
def test_sharded_quality_equals_unsharded_on_two_gpus():
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tools", "sharded_check.py"), "--quality"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SHARDED_CHECK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("(quality)") == 6
