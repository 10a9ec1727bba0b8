#!/usr/bin/env python
"""Estimation from a prior (rp_estimate_batch_*_init) on one GPU: what the prior stage costs, and what a prior changes
on a tracker-like workload.

Overhead: the cfg2 shape (10 000 pairs x 2 000 correspondences, RP_CALIB_SHIFT) and the cfg5 shape (4 000 x 10 000,
RP_CALIB), synth.make_batch, the configs' fixed iteration counts, inputs resident in HBM.  Two arms alternate: the plain
call (rp_estimate_batch_dev) and the prior call (rp_estimate_batch_dev_init, ground truth turned by 2 degrees).  Each
call is timed by a host clock around it (the call returns after its stream has finished); pairs/s is the median over
`--steps` calls after `--warmup`.  rp_last_timing slot [15] (the prior stage) is reported as a share of [8] (device
total).  With fixed iterations the prior changes no iteration count, so this is the cost of the stage and of one more
LO problem per pair.

Tracker-like: cfg1 (30 % outliers) and hard_calib (60 % outliers, 2 px noise, 10 % depth noise), 2 000 pairs x 1 000
correspondences, PoseLib's default early termination (min_iterations 1 000, max_iterations 100 000,
dyn_num_trials_mult 3, success_prob 0.9999), from host buffers (rp_estimate_batch_host[_init]).  Priors: the
ground truth with rotation and translation direction each turned by `--perturb-deg` degrees about random axes, as a
tracker's previous pose would be off.  Reported with and without priors: mean stats.iterations, the fraction of pairs
re-run because early termination needed more than min_iterations + 1 iterations (RP_PAIR_CONTINUED), median rotation
and translation-direction errors (degrees), mean refinements, and the call's wall time.

The GPU's name, power limit and SM clocks are read in the same run and stored beside the numbers.

  python tools/prior_bench.py --steps 3 --warmup 1 --out profiles/r07_prior.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OVERHEAD = {"cfg2_calib_shift": 10000, "cfg5_roma_calib": 4000}
TRACKER = {"cfg1_calib_scale": 2000, "hard_calib": 2000}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [f.strip() for f in out.split(",")]))
    except Exception as e:   # the record says so instead of guessing
        return {"error": str(e)}


def priors(b, deg, seed, shift):
    """Ground truth of every pair of a make_batch batch, rotation and t direction turned by `deg` degrees."""
    from mdrp_b200 import _native as nv, synth
    rng = np.random.default_rng(seed)
    P = len(b["R"])
    out = np.zeros(P, nv.MODEL_DTYPE)
    v = out.view(np.float64).reshape(P, 12)
    for i in range(P):
        dR = synth.rodrigues(rng.normal(size=3), np.deg2rad(deg))
        t = synth.rodrigues(rng.normal(size=3), np.deg2rad(deg)) @ b["t"][i]
        v[i] = np.r_[synth.quat_from_rotmat(dR @ b["R"][i]), t, 1.7, shift[0], shift[1], 1.0, 1.0]
    return out


def options(cfg, fixed):
    from mdrp_b200 import _native as nv, synth
    c = synth.CONFIGS[cfg]
    o = nv.default_options()
    if fixed:
        o.max_iterations = o.min_iterations = c["iters"]
    o.max_epipolar_error, o.max_reproj_error, o.seed = 2.0, 16.0, 0
    o.estimate_shift = int(c["shift"])
    o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    return o


def overhead(ctx, cfg, P, steps, warmup, deg):
    import torch
    from mdrp_b200 import _native as nv, synth
    c = synth.CONFIGS[cfg]
    variant = nv.CALIB_SHIFT if c["shift"] else nv.CALIB
    b = synth.make_batch(cfg, P, seed=1)
    o = options(cfg, True)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    x1, x2, d1, d2, cams = T(b["x1"]), T(b["x2"]), T(b["d1"]), T(b["d2"]), T(b["cams"])
    init = T(priors(b, deg, 2, (c.get("shift1", 0.0), c.get("shift2", 0.0))).view(np.float64).reshape(P, 12))
    N = int(b["offsets"][-1])
    models = torch.zeros(P, 12, dtype=torch.float64, device="cuda")
    stats = torch.zeros(P, 5, dtype=torch.int64, device="cuda")
    masks = torch.zeros(N, dtype=torch.uint8, device="cuda")
    outs = (models.data_ptr(), stats.data_ptr(), masks.data_ptr())
    args = (variant, b["offsets"], x1.data_ptr(), x2.data_ptr(), d1.data_ptr(), d2.data_ptr(), cams.data_ptr(), o)
    arms = {"plain": lambda: ctx.estimate_batch_dev(*args, *outs),
            "prior": lambda: ctx.estimate_batch_dev_init(*args, init.data_ptr(), *outs)}
    times = {k: [] for k in arms}
    share = []
    for step in range(warmup + steps):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            if step >= warmup:
                times[name].append(dt)
                if name == "prior":
                    ms, _ = ctx.last_timing()
                    share.append(ms["r15"] / ms["device_total"])
    rec = {k: {"pairs_per_s": P / float(np.median(v)), "call_s": [round(x, 4) for x in v]} for k, v in times.items()}
    rec["prior_stage_share_of_device_total"] = float(np.median(share))
    rec["prior_over_plain_time"] = float(np.median(times["prior"]) / np.median(times["plain"]))
    rec.update(pairs=P, correspondences=int(c["n"]), iterations=int(c["iters"]), perturb_deg=deg)
    return rec


def tracker(ctx, cfg, P, deg):
    from mdrp_b200 import _native as nv, synth
    c = synth.CONFIGS[cfg]
    variant = nv.CALIB_SHIFT if c["shift"] else nv.CALIB
    b = synth.make_batch(cfg, P, seed=3)
    o = options(cfg, False)
    init = priors(b, deg, 4, (c.get("shift1", 0.0), c.get("shift2", 0.0)))
    args = (variant, b["offsets"], b["x1"], b["x2"], b["d1"], b["d2"], b["cams"], o)
    rec = {"pairs": P, "correspondences": int(c["n"]), "outlier_ratio": c["outlier_ratio"], "perturb_deg": deg,
           "min_iterations": int(o.min_iterations), "max_iterations": int(o.max_iterations)}
    ctx.estimate_batch_host(*args)   # warm-up of this shape
    for name in ("plain", "prior"):
        t0 = time.perf_counter()
        models, stats, _ = ctx.estimate_batch_host(*args) if name == "plain" else ctx.estimate_batch_host_init(*args, init)
        dt = time.perf_counter() - t0
        st = ctx.pair_status(P)
        rot, tra = [], []
        for i in range(P):
            w, x, y, z = models[i]["q"]
            R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                          [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                          [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
            rot.append(synth.rotation_error_deg(R, b["R"][i]))
            tra.append(synth.translation_error_deg(models[i]["t"], b["t"][i]))
        rec[name] = {"mean_iterations": float(stats["iterations"].mean()),
                     "mean_refinements": float(stats["refinements"].mean()),
                     "rerun_fraction": float(((st & nv.PAIR_CONTINUED) != 0).mean()),
                     "median_rot_err_deg": float(np.median(rot)), "median_trans_err_deg": float(np.median(tra)),
                     "call_s": round(dt, 4)}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--perturb-deg", type=float, default=2.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_prior.json"))
    a = ap.parse_args()
    from mdrp_b200 import _native as nv
    ctx = nv.Context(0)
    rec = {"gpu": gpu_info(), "overhead_fixed_iterations": {}, "tracker_early_termination": {}}
    for cfg, P in OVERHEAD.items():
        rec["overhead_fixed_iterations"][cfg] = overhead(ctx, cfg, P, a.steps, a.warmup, a.perturb_deg)
        print(cfg, json.dumps(rec["overhead_fixed_iterations"][cfg]), flush=True)
    for cfg, P in TRACKER.items():
        rec["tracker_early_termination"][cfg] = tracker(ctx, cfg, P, a.perturb_deg)
        print(cfg, json.dumps(rec["tracker_early_termination"][cfg]), flush=True)
    rec["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
