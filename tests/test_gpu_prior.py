"""GPU tier: estimation from a prior (rp_estimate_batch_*_init and the Python / torch surfaces that route priors to them).

A prior is scored and locally optimised before RANSAC's first iteration (include/repose_b200.h); a NaN row is no prior.
The tests compare against the plain and _quality twins (NaN priors), the oracle started from a prior (ro_estimate_prior, tests/priororacle), and the
call itself across paths, dtypes, event capacities and batch compositions."""
import os
import sys

import numpy as np
import pytest

import prior_oracle as po
from mdrp_b200 import _native as nv, synth
from test_gpu_quality_order import _options, _ragged, definition

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import fuzz_parity  # noqa: E402

pytestmark = pytest.mark.gpu

CFGS = ["cfg1_calib_scale", "cfg2_calib_shift", "cfg3_shared_focal", "cfg4_varying_focal"]
SIZES = [300, 0, 150, 2, 3, 500, 1, 250]


def nan_rows(P):
    m = np.zeros(P, nv.MODEL_DTYPE)
    m.view(np.float64).reshape(P, 12)[:] = np.nan
    return m


def priors_for(cfg, base, P, kinds=("gt", "nan", "noisy", "garbage")):
    """Per pair: ground truth, no prior, ground truth turned by 3 degrees, or a wrong model (cycled)."""
    out = nan_rows(P)
    v = out.view(np.float64).reshape(P, 12)
    c = synth.CONFIGS[cfg]
    for i in range(P):
        sc = synth.scene_for(cfg, base + i, n=3)
        k = kinds[i % len(kinds)]
        if k == "gt":
            v[i] = synth.gt_model(sc, 0.01, i)
        elif k == "noisy":
            v[i] = synth.gt_model(sc, 3.0, i)
        elif k == "garbage":
            v[i] = [0.6, 0.8, 0, 0, 1.0, 0, 0, 0.5, 0, 0, 300.0, 2000.0]
        if k != "nan" and c["variant"] == "calib":
            v[i, 10:] = 1.0
    return out


def same(a, b):
    return all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(a, b))


@pytest.fixture(scope="module")
def ctx2():
    """A second context with an event list of two (every pair with three LO triggers takes the re-run path)."""
    old = os.environ.get("RP_EV_CAP")
    os.environ["RP_EV_CAP"] = "2"
    try:
        return nv.Context(0)
    finally:
        if old is None:
            del os.environ["RP_EV_CAP"]
        else:
            os.environ["RP_EV_CAP"] = old


@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("f32", [False, True])
def test_nan_priors_are_the_twins(ctx, cfg, f32):
    """All-NaN priors: the plain twin's bytes (models, stats, masks, rp_pair_status) and, with quality, the _quality
    twin's; host and device paths."""
    torch = pytest.importorskip("torch")
    from mdrp_b200 import torch_frontend as tf
    variant, offs, x1, x2, d1, d2, cams, q = _ragged(cfg, 40, SIZES, np.float32 if f32 else np.float64)
    o = _options(300, shift=variant == nv.CALIB_SHIFT, min_iters=30, prosac=True)
    P = len(offs) - 1
    plain_fn = ctx.estimate_batch_host_f32 if f32 else ctx.estimate_batch_host
    plain = plain_fn(variant, offs, x1, x2, d1, d2, cams, o)
    plain_st = ctx.pair_status(P)
    got = ctx.estimate_batch_host_init(variant, offs, x1, x2, d1, d2, cams, o, nan_rows(P))
    assert same(got, plain) and np.array_equal(ctx.pair_status(P), plain_st)
    qual = ctx.estimate_batch_host_quality(variant, offs, x1, x2, d1, d2, cams, o, q)
    qual_st = ctx.pair_status(P)
    got = ctx.estimate_batch_host_init(variant, offs, x1, x2, d1, d2, cams, o, nan_rows(P), q)
    assert same(got, qual) and np.array_equal(ctx.pair_status(P), qual_st)
    # device path
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    init = torch.full((P, 12), float("nan"), dtype=torch.float64, device="cuda")
    ct = T(cams) if cams is not None else None
    m, s, k = tf.estimate_batch(variant, offs, T(x1), T(x2), T(d1), T(d2), ct, o, init_models=init)
    torch.cuda.synchronize()
    assert np.array_equal(m.cpu().numpy().view(np.uint8).reshape(-1), plain[0].view(np.uint8))
    assert np.array_equal(s.cpu().numpy().view(np.uint8).reshape(-1), plain[1].view(np.uint8))
    assert np.array_equal(k.cpu().numpy(), plain[2])
    m, s, k = tf.estimate_batch(variant, offs, T(x1), T(x2), T(d1), T(d2), ct, o, quality=T(q), init_models=init)
    torch.cuda.synchronize()
    assert np.array_equal(k.cpu().numpy(), qual[2])
    assert np.array_equal(m.cpu().numpy().view(np.uint8).reshape(-1), qual[0].view(np.uint8))


def _oracle_prior(port, row):
    return port.make_model(row["q"], row["t"], row["scale"], row["shift1"], row["shift2"], row["f1"], row["f2"])


def run_parity(ctx, port, cases, seed, kind):
    """fuzz_parity's cases with a prior per case through rp_estimate_batch_host_init and ro_estimate_prior.  kind:
    "gt" (ground truth turned by 0.01 degrees), "noisy" (3 degrees), "garbage", "own" (the plain GPU call's result),
    "zero" (ground truth, max_iterations = 0)."""
    rng = np.random.default_rng(seed)
    bad, total = [], 0
    for variant in (0, 1, 2, 3):
        for _ in range(cases // 4):
            sc, x1, x2, d1, d2, o = fuzz_parity.random_case(rng, variant)
            n = len(d1)
            iters = 0 if kind == "zero" else o["iters"]
            opt = nv.default_options()
            opt.max_iterations = iters
            opt.min_iterations = iters if o["min_iters"] is None or kind == "zero" else o["min_iters"]
            opt.progressive_sampling, opt.max_prosac_iterations = int(o["prosac"]), o["max_prosac"]
            opt.max_epipolar_error, opt.max_reproj_error, opt.seed = o["t_epi"], o["t_rep"], o["seed"]
            opt.estimate_shift = int(variant == 1)
            opt.weight_sampson = o["weight_sampson"]
            opt.loss_type = nv.LOSS[o["loss"]]
            opt.loss_scale = 0.5 * o["t_epi"]
            opt.bundle_max_iterations = o["bundle_iters"]
            if variant < 2:
                a1, a2 = x1, x2
                cams = np.array([[sc.f1, sc.f1, 640, 480, sc.f2, sc.f2, 640, 480]])
                cam = ([sc.f1, sc.f1, 640, 480], [sc.f2, sc.f2, 640, 480])
            else:
                a1, a2 = x1 - [640.0, 480.0], x2 - [640.0, 480.0]
                cams, cam = None, (None, None)
            prior = np.zeros(1, nv.MODEL_DTYPE)
            pv = prior.view(np.float64)
            if kind == "own":
                prior[:] = ctx.estimate_batch_host(variant, [0, n], a1, a2, d1, d2, cams, opt)[0]
            elif kind == "garbage":
                pv[:] = [0.6, 0.8, 0, 0, 1.0, 0, 0, 0.5, 0, 0, 300.0, 2000.0]
            else:
                pv[:] = synth.gt_model(sc, 3.0 if kind == "noisy" else 0.01, int(rng.integers(0, 1000)))
            if variant < 2:
                pv[10:] = 1.0
            models, stats, masks = ctx.estimate_batch_host_init(variant, [0, n], a1, a2, d1, d2, cams, opt, prior)
            ro = port.ransac_opt(max_iterations=iters, min_iterations=int(opt.min_iterations),
                                 max_epipolar_error=o["t_epi"], max_reproj_error=o["t_rep"], seed=o["seed"],
                                 estimate_shift=variant == 1, weight_sampson=o["weight_sampson"],
                                 progressive_sampling=o["prosac"], max_prosac_iterations=o["max_prosac"])
            bo = port.bundle_opt(max_iterations=o["bundle_iters"], loss_type=o["loss"], loss_scale=0.5 * o["t_epi"])
            m, st, mask = po.estimate(variant, a1, a2, d1, d2, cam[0], cam[1], ro, bo, prior=_oracle_prior(port, prior[0]))
            total += 1
            got_st = (int(stats[0]["refinements"]), int(stats[0]["iterations"]), int(stats[0]["num_inliers"]))
            ref_st = (st.refinements, st.iterations, st.num_inliers)
            same_mask = np.array_equal(masks.astype(bool), mask)
            ref = np.r_[np.array(m.q), np.array(m.t), m.scale, m.shift1, m.shift2, m.f1, m.f2]
            got = np.r_[models[0]["q"], models[0]["t"], models[0]["scale"], models[0]["shift1"], models[0]["shift2"],
                        models[0]["f1"], models[0]["f2"]]
            if got[:4] @ ref[:4] < 0:
                got[:4] = -got[:4]
            finite = np.isfinite(ref).all() and np.isfinite(got).all()
            same_model = bool(np.allclose(got, ref, rtol=1e-6, atol=1e-8)) if finite else bool(
                np.array_equal(np.isnan(got), np.isnan(ref)))
            if not (got_st == ref_st and same_mask and same_model):
                bad.append(dict(variant=variant, n=n, kind=kind, opts=o, stats_gpu=got_st, stats_ref=ref_st,
                                same_mask=same_mask, same_model=same_model))
    return total, bad


@pytest.mark.parametrize("kind", ["gt", "noisy", "garbage", "own", "zero"])
def test_prior_parity_with_the_oracle(ctx, port, kind):
    """Under test_gpu_fuzz's rules: iterations always equal; masks and num_inliers equal where there is consensus;
    refinements differ only with the same model (a tie decided by summation order); the model differs only when the
    final refinement is under-determined.  PROSAC and early termination are on in a quarter of the cases each."""
    total, bad = run_parity(ctx, port, 240, {"gt": 21, "noisy": 22, "garbage": 23, "own": 24, "zero": 25}[kind], kind)
    assert total == 240
    for b in bad:
        assert b["stats_gpu"][1] == b["stats_ref"][1], b
        if b["stats_ref"][2] > 5:
            assert b["same_mask"] and b["stats_gpu"][2] == b["stats_ref"][2], b
            if b["stats_gpu"][0] != b["stats_ref"][0]:
                assert b["same_model"] and abs(b["stats_gpu"][0] - b["stats_ref"][0]) == 1, b
        if not b["same_model"]:
            assert b["stats_ref"][2] < 10, b
    assert len(bad) <= 0.02 * total, bad


def test_zero_iterations_stats(ctx):
    variant, offs, x1, x2, d1, d2, cams, _ = _ragged("cfg2_calib_shift", 60, [200, 2, 150])
    o = _options(0, shift=True, prosac=False)
    init = priors_for("cfg2_calib_shift", 60, 3, kinds=("gt",))
    _, stats, _ = ctx.estimate_batch_host_init(variant, offs, x1, x2, d1, d2, cams, o, init)
    assert [(int(s["refinements"]), int(s["iterations"])) for s in stats] == [(2, 0), (0, 0), (2, 0)]
    assert stats[0]["num_inliers"] > 100


@pytest.mark.parametrize("cfg", CFGS)
def test_rerun_path_and_batch_independence(ctx, ctx2, cfg):
    """An event list of two (re-runs carry the priors into their sub-batches) gives the default capacity's bytes; a
    pair's bytes alone equal its bytes inside a mixed batch of thousands; float32 gives the FP64 bytes; the host path
    gives the device path's bytes."""
    torch = pytest.importorskip("torch")
    from mdrp_b200 import torch_frontend as tf
    variant, offs, x1, x2, d1, d2, cams, _ = _ragged(cfg, 80, SIZES, np.float32)
    P = len(offs) - 1
    init = priors_for(cfg, 80, P)
    o = _options(400, shift=variant == nv.CALIB_SHIFT, min_iters=20, prosac=False)
    ref = ctx.estimate_batch_host_init(variant, offs, *(a.astype(np.float64) for a in (x1, x2, d1, d2)), cams, o, init)
    ref_st = ctx.pair_status(P)
    assert ctx.last_timing()[0]["r15"] > 0
    assert same(ctx.estimate_batch_host_init(variant, offs, x1, x2, d1, d2, cams, o, init), ref)   # float32
    assert same(ctx2.estimate_batch_host_init(variant, offs, x1, x2, d1, d2, cams, o, init), ref)  # re-run path
    assert (ctx2.pair_status(P) & nv.PAIR_EVENTS_RERUN).any()
    assert np.array_equal(ctx2.pair_status(P) & ~nv.PAIR_EVENTS_RERUN, ref_st & ~nv.PAIR_EVENTS_RERUN)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    m, s, k = tf.estimate_batch(variant, offs, T(x1), T(x2), T(d1), T(d2), T(cams) if cams is not None else None, o,
                                init_models=T(init.view(np.float64).reshape(P, 12)))
    torch.cuda.synchronize()
    assert same((m.cpu().numpy().reshape(-1).view(nv.MODEL_DTYPE), s.cpu().numpy().reshape(-1).view(nv.STATS_DTYPE),
                 k.cpu().numpy()), ref)
    # each pair alone, and the batch tiled to 2 400 pairs
    for p in (0, 2, 5):
        sl = slice(int(offs[p]), int(offs[p + 1]))
        one = ctx.estimate_batch_host_init(variant, [0, int(offs[p + 1] - offs[p])], x1[sl], x2[sl], d1[sl], d2[sl],
                                           cams[p:p + 1] if cams is not None else None, o, init[p:p + 1])
        assert same(one, (ref[0][p:p + 1], ref[1][p:p + 1], ref[2][sl])), p
    reps = 300
    n = np.diff(offs)
    big_offs = np.r_[0, np.cumsum(np.tile(n, reps))].astype(np.int64)
    tile = lambda a: np.concatenate([a] * reps)
    big = ctx.estimate_batch_host_init(variant, big_offs, tile(x1), tile(x2), tile(d1), tile(d2),
                                       tile(cams) if cams is not None else None, o, tile(init))
    for r in (0, 137, reps - 1):
        ps = slice(r * P, (r + 1) * P)
        assert same((big[0][ps], big[1][ps], big[2][int(big_offs[r * P]):int(big_offs[(r + 1) * P])]), ref), r


@pytest.mark.parametrize("cfg", CFGS)
def test_prior_with_quality_is_prior_on_reordered_pairs(ctx, cfg):
    variant, offs, x1, x2, d1, d2, cams, q = _ragged(cfg, 120, SIZES)
    P = len(offs) - 1
    init = priors_for(cfg, 120, P)
    o = _options(300, shift=variant == nv.CALIB_SHIFT, min_iters=30, prosac=True)

    class WithPrior:
        """definition()'s context: the unscored calls with the same priors."""
        def estimate_batch_host(self, *a):
            return ctx.estimate_batch_host_init(*a, init)
        estimate_batch_host_f32 = estimate_batch_host

        def pair_status(self, P):
            return ctx.pair_status(P)
    want, want_st = definition(WithPrior(), variant, offs, x1, x2, d1, d2, cams, o, q)
    got = ctx.estimate_batch_host_init(variant, offs, x1, x2, d1, d2, cams, o, init, q)
    assert same(got, want) and np.array_equal(ctx.pair_status(P), want_st)


def test_api_priors_end_to_end():
    """api: a ground-truth prior with max_iterations 0 returns the refined prior; None entries are plain pairs."""
    from mdrp_b200 import api
    scs = [synth.scene_for("cfg1_calib_scale", 200 + i, n=300) for i in range(2)]
    c1, c2 = scs[0].camera_dicts()
    v = synth.gt_model(scs[0], 0.01, 0)
    g = api.MonoDepthTwoViewGeometry(api.CameraPose(v[:4], v[4:7]), v[7], v[8], v[9])
    args = ([s.x1 for s in scs], [s.x2 for s in scs], [s.d1 for s in scs], [s.d2 for s in scs], [c1, c1], [c2, c2])
    res = api.estimate_monodepth_relative_pose_batch(*args, ransac_opt={"max_iterations": 0, "min_iterations": 0},
                                                     initial_geometries=[g, None])
    assert (res[0][1]["refinements"], res[0][1]["iterations"]) == (2, 0) and res[0][1]["num_inliers"] > 150
    assert synth.rotation_error_deg(res[0][0].pose.R, scs[0].R) < 0.5
    assert (res[1][1]["refinements"], res[1][1]["iterations"]) == (1, 0)
    plain = api.estimate_monodepth_relative_pose_batch(*args, ransac_opt={"max_iterations": 200, "min_iterations": 200})
    nan_prior = api.estimate_monodepth_relative_pose_batch(*args, ransac_opt={"max_iterations": 200, "min_iterations": 200},
                                                         initial_geometries=[None, None])
    assert [r[1] for r in plain] == [r[1] for r in nan_prior]
