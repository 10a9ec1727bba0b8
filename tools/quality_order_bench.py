#!/usr/bin/env python
"""Quality-ordered estimation (rp_estimate_batch_*_quality) on one GPU: what the ordering costs, and what PROSAC on the
quality order buys under early termination.

Cost.  cfg2 and cfg5 at full size (10 000 x 2 000 and 4 000 x 10 000 correspondences), fixed iterations, PROSAC on,
FP64 inputs.  Two arms compute the same thing:
  quality    rp_estimate_batch_{host,dev}_quality with a random float32 quality per correspondence
  presorted  rp_estimate_batch_{host,dev} on the same batch sorted on the host beforehand, in the order the definition
             gives (quality descending, index ascending); its masks are compared in that order
The outputs of the two arms are compared as bytes.  Per arm: pairs/s from a host clock around the call (it returns after
its last read-back / its stream has finished), the rp_last_timing slots ordering [14] and device total [8] per step.
The host-buffer arm reads pinned host memory; the resident arm has every input in HBM.  Blocks of `--warmup` + `--steps`
steps alternate presorted, quality, presorted, quality.

Value.  PoseLib's default early termination (min_iterations 1 000, max_iterations 100 000, success_prob 0.9999) on a
high-outlier calibrated set: `--value-pairs` scenes of 1 000 correspondences with 80 % outliers (synth.make_scene).
Quality rule: inliers U(0.3, 1), outliers U(0, 0.7), drawn from a seeded generator.  Uniform sampling on the caller's
order against PROSAC on the quality order (the same quality call with progressive_sampling 0 and 1).  Reported: mean
RANSAC iterations, pairs/s, median rotation and translation errors in degrees and mAA over 1..10 degrees of
max(rotation, translation error) against the ground truth (benchmark_reader metrics).

The GPU's name, power limit and SM clocks are read in the same run and stored beside the numbers.

  python tools/quality_order_bench.py --steps 3 --warmup 1 --out profiles/r04_quality_order.json
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

DEFAULT_PAIRS = {"cfg2_calib_shift": 10000, "cfg5_roma_calib": 4000}   # bench.py's single-GPU lines of DESIGN §6


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [f.strip() for f in out.split(",")]))
    except Exception as e:   # the record says so instead of guessing
        return {"error": str(e)}


def host_order(offs, q):
    """Source index of every position of the ordered batch (quality descending, index ascending per pair; no NaN here)."""
    P = len(offs) - 1
    n = np.diff(offs)
    pair = np.repeat(np.arange(P), n)
    idx = np.lexsort((np.arange(len(q)), -q.astype(np.float64), pair))
    return idx


def run_cost(cfg, P, steps, warmup):
    import torch
    from mdrp_b200 import _native as nv, synth
    c = synth.CONFIGS[cfg]
    variant = nv.CALIB_SHIFT if c["shift"] else nv.CALIB
    opt = nv.default_options()
    opt.max_iterations = opt.min_iterations = c["iters"]
    opt.max_epipolar_error, opt.max_reproj_error, opt.seed = 2.0, 16.0, 0
    opt.estimate_shift = int(c["shift"])
    opt.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    opt.progressive_sampling = 1
    batch = synth.make_batch(cfg, P, seed=1000)
    offs = batch["offsets"]
    N = int(offs[-1])
    q = np.random.default_rng(7).uniform(size=N).astype(np.float32)
    src = host_order(offs, q)
    dev = torch.device("cuda", 0)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    raw = {k: pin(batch[k]) for k in ("x1", "x2", "d1", "d2")}
    srt = {k: pin(batch[k][src]) for k in ("x1", "x2", "d1", "d2")}
    del batch["x1"], batch["x2"], batch["d1"], batch["d2"]
    h_q = pin(q)
    d_raw = {k: v.to(dev) for k, v in raw.items()}
    d_srt = {k: v.to(dev) for k, v in srt.items()}
    d_q = h_q.to(dev)
    h_cams = pin(batch["cams"])
    d_cams = h_cams.to(dev)
    outs = lambda d: (torch.zeros(P, 12, dtype=torch.float64, device=d), torch.zeros(P, 5, dtype=torch.int64, device=d),
                      torch.zeros(max(N, 1), dtype=torch.uint8, device=d))
    h_out = {a: tuple(t.pin_memory() for t in outs("cpu")) for a in ("quality", "presorted")}
    d_out = {a: outs(dev) for a in ("quality", "presorted")}
    ctx = nv.Context(0)
    stream = torch.cuda.current_stream(dev).cuda_stream
    L = ctx._lib
    import ctypes as C

    def step(arm, path):
        t0 = time.perf_counter()
        if path == "host":
            h = srt if arm == "presorted" else raw
            ptrs = [h[k].data_ptr() for k in ("x1", "x2", "d1", "d2")]
            o = [t.data_ptr() for t in h_out[arm]]
            if arm == "quality":
                ctx._check(L.rp_estimate_batch_host_quality(ctx._h, variant, P, offs.ctypes.data, *ptrs, h_q.data_ptr(),
                                                            h_cams.data_ptr(), C.byref(opt), *o))
            else:
                ctx._check(L.rp_estimate_batch_host(ctx._h, variant, P, offs.ctypes.data, *ptrs, h_cams.data_ptr(),
                                                    C.byref(opt), *o))
        else:
            d = d_srt if arm == "presorted" else d_raw
            ptrs = [d[k].data_ptr() for k in ("x1", "x2", "d1", "d2")]
            o = [t.data_ptr() for t in d_out[arm]]
            if arm == "quality":
                ctx.estimate_batch_dev_quality(variant, offs, *ptrs, d_cams.data_ptr(), opt, *o, d_q.data_ptr(), stream)
            else:
                ctx.estimate_batch_dev(variant, offs, *ptrs, d_cams.data_ptr(), opt, *o, stream)
        dt = time.perf_counter() - t0
        ms, cn = ctx.last_timing()
        return dt, ms, cn

    rec = {"pairs": P, "matches_per_pair": c["n"], "ransac_iterations": c["iters"], "correspondences": N,
           "input": "float64", "progressive_sampling": 1}
    rounds = 2
    for path in ("host", "dev"):
        got = {a: {"s": [], "order": [], "device": [], "chunks": 0} for a in ("presorted", "quality")}
        for _ in range(rounds):
            for arm in ("presorted", "quality"):
                for _ in range(warmup):
                    step(arm, path)
                for _ in range(steps):
                    dt, ms, cn = step(arm, path)
                    g = got[arm]
                    g["s"].append(dt)
                    g["order"].append(ms["order"])
                    g["device"].append(ms["device_total"])
                    g["chunks"] = cn["chunks"]
        out = {}
        for arm, g in got.items():
            n, tot = len(g["s"]), sum(g["s"])
            out[arm] = {"pairs_per_s": P * n / tot, "ms_per_step": 1000.0 * tot / n,
                        "ms_each_step": [round(1000.0 * s, 2) for s in g["s"]],
                        "pairs_per_s_by_round": [P * steps / sum(g["s"][r * steps:(r + 1) * steps]) for r in range(rounds)],
                        "order_ms_per_step": float(np.mean(g["order"])), "device_ms_per_step": float(np.mean(g["device"])),
                        "order_ms_each_step": [round(v, 3) for v in g["order"]], "chunks_per_call": g["chunks"]}
        out["order_share_of_device_total"] = out["quality"]["order_ms_per_step"] / out["quality"]["device_ms_per_step"]
        out["quality_over_presorted"] = out["quality"]["pairs_per_s"] / out["presorted"]["pairs_per_s"]
        res = h_out if path == "host" else d_out
        a = [t.cpu().numpy() for t in res["quality"]]
        b = [t.cpu().numpy() for t in res["presorted"]]
        mask_sorted_to_caller = np.zeros_like(b[2][:N])
        mask_sorted_to_caller[src] = b[2][:N]
        out["outputs_identical"] = bool(a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes() and
                                        a[2][:N].tobytes() == mask_sorted_to_caller.tobytes())
        rec["host_buffers" if path == "host" else "resident"] = out
    ctx.close()
    return rec


def run_value(P, n, outlier_ratio, seed):
    from mdrp_b200 import _native as nv, api, synth, benchmark_reader as br
    scs = [synth.make_scene(seed + i, n, outlier_ratio=outlier_ratio) for i in range(P)]
    rng = np.random.default_rng(seed)
    f = lambda k: np.concatenate([getattr(s, k) for s in scs])
    inl = f("inlier_mask")
    q = np.where(inl, rng.uniform(0.3, 1.0, len(inl)), rng.uniform(0.0, 0.7, len(inl))).astype(np.float32)
    offs = np.arange(P + 1, dtype=np.int64) * n
    cams = np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
    x1, x2, d1, d2 = f("x1"), f("x2"), f("d1"), f("d2")
    ctx = nv.Context(0)
    rec = {"pairs": P, "matches_per_pair": n, "outlier_ratio": outlier_ratio,
           "quality_rule": "inliers U(0.3, 1), outliers U(0, 0.7), float32, numpy default_rng(%d)" % seed,
           "options": "PoseLib defaults: min_iterations 1000, max_iterations 100000, success_prob 0.9999, "
                      "dyn_num_trials_mult 3; max_epipolar_error 2, max_reproj_error 16, TRUNCATED_CAUCHY",
           "pose_error": "max(rotation, translation direction) error in degrees; mAA over thresholds 1..10 degrees"}
    for name, prosac in (("uniform", 0), ("prosac_on_quality", 1)):
        o = nv.default_options()
        o.max_epipolar_error, o.max_reproj_error = 2.0, 16.0
        o.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
        o.progressive_sampling = prosac
        ctx.estimate_batch_host_quality(nv.CALIB, offs, x1, x2, d1, d2, cams, o, q)   # warm-up
        times = []
        for _ in range(2):
            t0 = time.perf_counter()
            models, stats, masks = ctx.estimate_batch_host_quality(nv.CALIB, offs, x1, x2, d1, d2, cams, o, q)
            times.append(time.perf_counter() - t0)
        ms, _ = ctx.last_timing()
        re, te = [], []
        for m, s in zip(models, scs):
            R = api.CameraPose(m["q"], m["t"]).R
            re.append(br.rotation_error_deg(R, s.R))
            te.append(br.translation_error_deg(m["t"], s.t))
        re, te = np.array(re), np.array(te)
        rec[name] = {"mean_iterations": float(stats["iterations"].mean()),
                     "median_iterations": float(np.median(stats["iterations"])),
                     "pairs_per_s": P * len(times) / sum(times), "s_each_call": [round(t, 3) for t in times],
                     "order_ms": ms["order"], "device_ms": ms["device_total"],
                     "median_rot_err_deg": float(np.median(re)), "median_t_err_deg": float(np.median(te)),
                     "mAA_10deg": br.pose_maa(np.maximum(re, te)),
                     "mean_inlier_ratio": float(stats["inlier_ratio"].mean())}
    rec["prosac_over_uniform_pairs_per_s"] = rec["prosac_on_quality"]["pairs_per_s"] / rec["uniform"]["pairs_per_s"]
    ctx.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg2_calib_shift,cfg5_roma_calib")
    ap.add_argument("--pairs", type=int, default=0, help="pairs per step of the cost part (0: 10 000 for cfg2, 4 000 for cfg5)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--value-pairs", type=int, default=2000)
    ap.add_argument("--value-outliers", type=float, default=0.8)
    ap.add_argument("--out", help="write the record here (JSON); printed to stdout as well")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("quality_order_bench.py needs a CUDA device")
    record = {"what": "rp_estimate_batch_*_quality: ordering cost against a host-presorted unscored call, and PROSAC on "
                      "the quality order against uniform sampling under early termination; one GPU",
              "gpu_before": gpu_info(), "steps": args.steps, "warmup": args.warmup, "cost": {}}
    for cfg in args.configs.split(","):
        P = args.pairs or DEFAULT_PAIRS.get(cfg, 10000)
        record["cost"][cfg] = run_cost(cfg, P, args.steps, args.warmup)
        print(cfg, json.dumps(record["cost"][cfg]), file=sys.stderr, flush=True)
    record["value"] = run_value(args.value_pairs, 1000, args.value_outliers, 5000)
    print("value", json.dumps(record["value"]), file=sys.stderr, flush=True)
    record["gpu_after"] = gpu_info()
    text = json.dumps(record, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
