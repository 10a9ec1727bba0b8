#!/usr/bin/env python
"""Refinement of caller-supplied models (rp_refine_pairs_*) on one GPU: pairs/s, and how its device time compares with the
estimator's own final refinement on the same batch.

Workloads: cfg2 shape (10 000 pairs x 2 000 correspondences, calibrated with shifts, RP_CALIB_SHIFT) and cfg5 shape
(4 000 x 10 000, calibrated, RP_CALIB), synth.make_batch, the configs' RANSAC iterations, TRUNCATED_CAUCHY bundle options
(100 iterations).  Start models and subsets come from the estimator run with bundle_max_iterations = 0, as a pipeline
that re-refines a RANSAC result would hold them.

Arms, each timed by a host clock around the call (the call returns after its last read-back / after its stream has
finished): FP64 and float32 inputs, from pinned host buffers (rp_refine_pairs_host[_f32]) and with every input resident
in HBM (rp_refine_pairs_dev[_f32]).  Blocks of `--warmup` + `--steps` calls alternate the four arms.  The resident FP64
arm is also timed with CUDA events on its stream.  For comparison the estimator (resident FP64 inputs, the same bundle
options) is run `--steps` times and its rp_last_timing slots [0] prepare (with the tensor-core feature rows, which the
refine call does not build), [7] final refinement (enable, LM, finalize) and [8] device total are reported; the refine
call does prepare, the LM launch of slot [7] and one get_inliers scoring launch, so its device time should be close to
[0] + [7] + one scoring launch.  The FP64 arms' refined models are compared as bytes with the estimator's, the float32
arms' with each other (their inputs are the FP64 values rounded to float32, so they are not the estimator's inputs).

The GPU's name, power limit and SM clocks are read in the same run and stored beside the numbers.

  python tools/refine_bench.py --steps 5 --warmup 2 --out profiles/r06_refine.json
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

WORKLOADS = {"cfg2_calib_shift": 10000, "cfg5_roma_calib": 4000}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [f.strip() for f in out.split(",")]))
    except Exception as e:   # the record says so instead of guessing
        return {"error": str(e)}


def run(cfg, P, steps, warmup):
    import torch
    from mdrp_b200 import _native as nv, synth
    c = synth.CONFIGS[cfg]
    variant = nv.CALIB_SHIFT if c["shift"] else nv.CALIB
    opt = nv.default_options()
    opt.max_iterations = opt.min_iterations = c["iters"]
    opt.max_epipolar_error, opt.max_reproj_error, opt.seed = 2.0, 16.0, 0
    opt.estimate_shift = int(c["shift"])
    opt.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    opt.bundle_max_iterations = 100
    opt0 = nv.Options.from_buffer_copy(opt)
    opt0.bundle_max_iterations = 0
    b = synth.make_batch(cfg, P, seed=1000)
    offs, N = b["offsets"], int(b["offsets"][-1])
    ctx = nv.Context(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h64 = {k: pin(b[k]) for k in ("x1", "x2", "d1", "d2")}
    h32 = {k: pin(b[k].astype(np.float32)) for k in ("x1", "x2", "d1", "d2")}
    cams = pin(b["cams"])
    d64 = {k: v.to(dev) for k, v in h64.items()}
    d32 = {k: v.to(dev) for k, v in h32.items()}
    dcams = cams.to(dev)
    xs = lambda d: [d[k].data_ptr() for k in ("x1", "x2", "d1", "d2")]
    # start models and subsets: the estimator with no final refinement
    m0 = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    s0 = torch.zeros(P, 5, dtype=torch.int64, device=dev)
    k0 = torch.zeros(N, dtype=torch.uint8, device=dev)
    ctx.estimate_batch_dev(variant, offs, *xs(d64), dcams.data_ptr(), opt0, m0.data_ptr(), s0.data_ptr(), k0.data_ptr(),
                           stream.cuda_stream)
    hm0 = m0.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1)
    hk0 = k0.cpu().numpy()
    # the estimator with the bundle options: its final models and its stage times
    em = torch.zeros_like(m0)
    es, ek = torch.zeros_like(s0), torch.zeros_like(k0)
    est_slots = []
    for _ in range(steps):
        ctx.estimate_batch_dev(variant, offs, *xs(d64), dcams.data_ptr(), opt, em.data_ptr(), es.data_ptr(), ek.data_ptr(),
                               stream.cuda_stream)
        ms, _ = ctx.last_timing()
        est_slots.append([ms["prepare"], ms["final_refine"], ms["device_total"]])
    est_slots = np.median(np.array(est_slots), axis=0)
    # refine arms
    rm = torch.zeros_like(m0)
    rb = torch.zeros(P, 7, dtype=torch.int64, device=dev)
    rn = torch.zeros(P, dtype=torch.int64, device=dev)
    rk = torch.zeros(N, dtype=torch.uint8, device=dev)
    outs = [rm.data_ptr(), rb.data_ptr(), rn.data_ptr(), rk.data_ptr()]
    host_np = lambda d: [d[k].numpy() for k in ("x1", "x2", "d1", "d2")]
    arms = {
        "host_fp64": lambda: ctx.refine_pairs_host(variant, offs, *host_np(h64), cams.numpy(), opt, hm0, hk0),
        "host_f32": lambda: ctx.refine_pairs_host_f32(variant, offs, *host_np(h32), cams.numpy(), opt, hm0, hk0),
        "resident_fp64": lambda: ctx.refine_pairs_dev(variant, offs, *xs(d64), dcams.data_ptr(), opt, m0.data_ptr(),
                                                      k0.data_ptr(), *outs, stream.cuda_stream),
        "resident_f32": lambda: ctx.refine_pairs_dev_f32(variant, offs, *xs(d32), dcams.data_ptr(), opt, m0.data_ptr(),
                                                         k0.data_ptr(), *outs, stream.cuda_stream),
    }
    times = {k: [] for k in arms}
    results = {}
    for i in range(warmup + steps):
        for name, fn in arms.items():
            t0 = time.perf_counter()
            r = fn()
            t1 = time.perf_counter()
            if i >= warmup:
                times[name].append(t1 - t0)
            if i == 0:
                results[name] = r if r is not None else (rm.cpu().numpy().view(nv.MODEL_DTYPE).reshape(-1).copy(),)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dev_ms = []
    for _ in range(steps):
        ev0.record(stream)
        arms["resident_fp64"]()
        ev1.record(stream)
        ev1.synchronize()
        dev_ms.append(ev0.elapsed_time(ev1))
    est_models = em.cpu().numpy().tobytes()
    rec = {"pairs": P, "correspondences_per_pair": int(N // P), "variant": int(variant), "ransac_iterations": c["iters"],
           "bundle_max_iterations": 100, "loss": "TRUNCATED_CAUCHY",
           "fp64_models_equal_estimator": all(results[k][0].tobytes() == est_models for k in ("host_fp64", "resident_fp64")),
           "f32_host_equals_resident": results["host_f32"][0].tobytes() == results["resident_f32"][0].tobytes(),
           "refined_pairs": int((s0.cpu().numpy()[:, 2] > 3).sum()),
           "estimator_ms": {"prepare_0": est_slots[0], "final_refine_7": est_slots[1], "device_total_8": est_slots[2]},
           "refine_resident_fp64_device_ms_median": float(np.median(dev_ms))}
    for name, ts in times.items():
        med = float(np.median(ts))
        rec[name] = {"ms_median": 1e3 * med, "ms_min": 1e3 * float(np.min(ts)), "pairs_per_s": P / med}
    ctx.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_refine.json"))
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of each workload's pairs (rehearsal)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    out = {"gpu": gpu_info(), "steps": a.steps, "warmup": a.warmup, "timer": "host clock around each call (median)",
           "workloads": {}}
    for cfg, P in WORKLOADS.items():
        out["workloads"][cfg] = run(cfg, max(1, int(P * a.scale)), a.steps, a.warmup)
        print(cfg, json.dumps(out["workloads"][cfg]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
