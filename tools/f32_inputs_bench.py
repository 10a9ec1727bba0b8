#!/usr/bin/env python
"""float32 vs FP64 inputs of the batched estimator, end to end and resident, on one GPU.

The inputs are `synth.make_batch` of each config rounded to float32; the FP64 arm gets the same values widened to
float64, so both arms compute the same thing (checked: the outputs of the two arms are compared as bytes).  Per config:

  host  rp_estimate_batch_host vs rp_estimate_batch_host_f32 from pinned host buffers, results read back into pinned
        buffers; pairs/s from a host clock around the call (it returns after the last read-back has finished)
  dev   rp_estimate_batch_dev vs rp_estimate_batch_dev_f32 with the inputs resident in HBM; the same clock (the call
        returns after its stream has finished)

Both arms share one context (one workspace: cfg2 at 10 000 pairs runs as one ~71 GB chunk).  Timed steps come in
blocks: `--warmup` steps of an arm, then `--steps` timed steps of it, so that the lead chunk of a host-path call is sized
from that arm's previous call (rp_last_timing of the same context); the blocks go f64, f32, f64, f32 so that drift of the
machine shows as a difference between the two rounds.  Reported per arm: pairs/s,
ms per step (mean and every step), the rp_last_timing slots H2D [9], widening [13] and device total [8] per step, chunks
per call, and the bytes uploaded per step computed from the shapes.  The GPU's name, power limit and SM clocks are read
in the same run and stored beside the numbers.

  python tools/f32_inputs_bench.py --steps 5 --warmup 3 --out record.json
"""
import argparse
import ctypes as C
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


def upload_bytes(N, P, in_bytes, pose):
    """Host-to-device bytes of one host-path call: points and depths, cams, offsets (as bench.py counts them)."""
    return N * in_bytes + (P * 64 if pose else 0) + (P + 1) * 8


def run_config(cfg, P, steps, warmup):
    import torch
    from mdrp_b200 import _native as nv, synth
    c = synth.CONFIGS[cfg]
    variant = {"calib": nv.CALIB_SHIFT if c["shift"] else nv.CALIB, "shared": nv.SHARED, "varying": nv.VARYING}[c["variant"]]
    opt = nv.default_options()
    opt.max_iterations = opt.min_iterations = c["iters"]
    opt.max_epipolar_error, opt.max_reproj_error, opt.seed = 2.0, 16.0, 0
    opt.estimate_shift = int(c["shift"])
    opt.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    opt.loss_scale = 1.0
    batch = synth.make_batch(cfg, P, seed=1000)
    offs = batch["offsets"]
    N = int(offs[-1])
    pose = batch["cams"] is not None
    dev = torch.device("cuda", 0)
    ctx = nv.Context(0)
    arms = {}
    for name, dt in (("f64", np.float64), ("f32", np.float32)):
        host = {k: torch.from_numpy(np.ascontiguousarray(batch[k].astype(np.float32).astype(dt))).pin_memory()
                for k in ("x1", "x2", "d1", "d2")}
        arms[name] = dict(host=host, devt={k: v.to(dev) for k, v in host.items()},
                          h_out=(torch.zeros(P, 12, dtype=torch.float64).pin_memory(),
                                 torch.zeros(P, 5, dtype=torch.int64).pin_memory(),
                                 torch.zeros(max(N, 1), dtype=torch.uint8).pin_memory()),
                          d_out=(torch.zeros(P, 12, dtype=torch.float64, device=dev),
                                 torch.zeros(P, 5, dtype=torch.int64, device=dev),
                                 torch.zeros(max(N, 1), dtype=torch.uint8, device=dev)))
    del batch["x1"], batch["x2"], batch["d1"], batch["d2"]
    h_cams = torch.from_numpy(batch["cams"]).pin_memory() if pose else None
    d_cams = h_cams.to(dev) if pose else None
    stream = torch.cuda.current_stream(dev).cuda_stream

    def step(name, path):
        a = arms[name]
        L = ctx._lib
        t0 = time.perf_counter()
        if path == "host":
            fn = L.rp_estimate_batch_host_f32 if name == "f32" else L.rp_estimate_batch_host
            h = a["host"]
            ctx._check(fn(ctx._h, variant, P, offs.ctypes.data, h["x1"].data_ptr(), h["x2"].data_ptr(), h["d1"].data_ptr(),
                          h["d2"].data_ptr(), h_cams.data_ptr() if pose else None, C.byref(opt),
                          *(t.data_ptr() for t in a["h_out"])))
        else:
            est = ctx.estimate_batch_dev_f32 if name == "f32" else ctx.estimate_batch_dev
            d = a["devt"]
            est(variant, offs, d["x1"].data_ptr(), d["x2"].data_ptr(), d["d1"].data_ptr(), d["d2"].data_ptr(),
                d_cams.data_ptr() if pose else None, opt, *(t.data_ptr() for t in a["d_out"]), stream)
        dt = time.perf_counter() - t0
        ms, cn = ctx.last_timing()
        return dt, ms, cn

    rec = {"pairs": P, "matches_per_pair": c["n"], "ransac_iterations": c["iters"], "correspondences": N}
    rounds = 2
    for path in ("host", "dev"):
        got = {n: {"s": [], "h2d": 0.0, "widen": 0.0, "device": 0.0, "chunks": 0} for n in ("f64", "f32")}
        for _ in range(rounds):
            for name in ("f64", "f32"):
                for _ in range(warmup):
                    step(name, path)
                for _ in range(steps):
                    dt, ms, cn = step(name, path)
                    g = got[name]
                    g["s"].append(dt)
                    g["h2d"] += ms["h2d"]
                    g["widen"] += ms["widen"]
                    g["device"] += ms["device_total"]
                    g["chunks"] = cn["chunks"]
        out = {}
        for name, g in got.items():
            n = len(g["s"])
            tot = sum(g["s"])
            u, w, d = g["h2d"] / n, g["widen"] / n, g["device"] / n
            out[name] = {"pairs_per_s": P * n / tot, "ms_per_step": 1000.0 * tot / n,
                         "ms_each_step": [round(1000.0 * s, 2) for s in g["s"]],
                         "pairs_per_s_by_round": [P * steps / sum(g["s"][r * steps:(r + 1) * steps]) for r in range(rounds)],
                         "h2d_ms_per_step": u, "widen_ms_per_step": w, "device_ms_per_step": d, "chunks_per_call": g["chunks"]}
            if path == "host":
                out[name]["h2d_bytes_per_step"] = upload_bytes(N, P, 48 if name == "f64" else 24, pose)
                # the share of the batch the next call's lead chunk gets, U / (U + C) clamped to [1/32, 1/3], with U = H2D +
                # the widening of the batch extrapolated from chunk 0's: between these two bounds (without any widening,
                # and with all of [13], which on this path includes waiting for SMs)
                clamp = lambda f: min(1 / 3, max(1 / 32, f))
                out[name]["lead_chunk_fraction_of_next_call_bounds"] = [clamp(u / (u + d)), clamp((u + w) / (u + w + d))]
        out["f32_over_f64"] = out["f32"]["pairs_per_s"] / out["f64"]["pairs_per_s"]
        key = "h_out" if path == "host" else "d_out"
        out["outputs_identical"] = all(x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()
                                       for x, y in zip(arms["f64"][key], arms["f32"][key]))
        rec["host_buffers" if path == "host" else "resident"] = out
    ctx.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg2_calib_shift,cfg5_roma_calib")
    ap.add_argument("--pairs", type=int, default=0, help="pairs per step (0: 10 000 for cfg2, 4 000 for cfg5)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="write the record here (JSON); printed to stdout as well")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("f32_inputs_bench.py needs a CUDA device")
    record = {"what": "float32 vs FP64 inputs (same values), one GPU: host buffers end to end and inputs resident",
              "gpu_before": gpu_info(), "steps": args.steps, "warmup": args.warmup, "configs": {}}
    for cfg in args.configs.split(","):
        P = args.pairs or DEFAULT_PAIRS.get(cfg, 10000)
        record["configs"][cfg] = run_config(cfg, P, args.steps, args.warmup)
        print(cfg, json.dumps(record["configs"][cfg]), file=sys.stderr, flush=True)
    record["gpu_after"] = gpu_info()
    text = json.dumps(record, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
