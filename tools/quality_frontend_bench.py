#!/usr/bin/env python
"""Match quality through the depth gathers on one GPU: what carrying it costs, and the chain against the workaround it
replaces.

Data: the video shape.  A 501-frame 480x640 float32 depth stack (616 MB, larger than L2), 500 frame pairs (p, p+1),
10 000 matches per pair (5 M rows).  The matches are cfg5 scenes (synth.make_batch, 30 % outliers) at half resolution
(keypoints and intrinsics halved), with each scene's depths written into its two frames at its keypoints (where a
neighbouring pair writes the same pixel, the later value wins: a few rows get a wrong depth and act as outliers).  About
5 % of the rows are made both-inf (dropped by the gather).  Quality: inliers U(0.3, 1), outliers U(0, 0.7), float32.

Gather.  rp_gather_depths_batch_dev[_f32] (twin) against rp_gather_depths_batch_dev[_f32]_quality on the same inputs,
outputs preallocated.  Each call ends in a device synchronise (the call synchronises before it returns); it is timed
with a host clock.  After a warm-up of both arms, steps alternate twin / quality (the order swapped every step).
Reported: median and spread of each arm, the ratio of medians, and the logical bytes per kept row from the shapes
(pass 1 reads 16 B of keypoints and 8 B of depth per input row and writes 6 values per kept row; pass 2 copies those;
the quality adds 4 B read + 4 B written per kept row in each pass).  The twin's outputs are compared with the quality
call's as bytes.

Chain vs workaround, at cfg5 options (1 000 iterations, PROSAC on, float32).  Chain: gather_depths_batch(quality=q) ->
estimate_batch(quality=q_out).  Workaround: gather_depths_batch() -> the lookup repeated in torch to find the kept rows
((int) truncation, border clamp, both-inf test) -> q[keep] -> estimate_batch(quality=...).  Each step ends with the
estimator's read-back of its stream.  The outputs of the two are compared as bytes.

The GPU's name, power limit and SM clocks are read in the same run and stored beside the numbers.

  python tools/quality_frontend_bench.py --steps 20 --warmup 3 --out profiles/r05_quality_frontend.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from quality_order_bench import gpu_info  # noqa: E402

F, H, W = 501, 480, 640


def make_video(P, n, seed):
    from mdrp_b200 import synth
    b = synth.make_batch("cfg5_roma_calib", P, seed=seed, n=n)
    rng = np.random.default_rng(seed + 1)
    kp1 = np.clip(b["x1"] / 2, 0, [W - 1.001, H - 1.001]).astype(np.float32)
    kp2 = np.clip(b["x2"] / 2, 0, [W - 1.001, H - 1.001]).astype(np.float32)
    maps = rng.uniform(1, 9, size=(F, H, W)).astype(np.float32)
    pair = np.repeat(np.arange(P), n)
    r1, c1 = kp1[:, 1].astype(np.int64), kp1[:, 0].astype(np.int64)
    r2, c2 = kp2[:, 1].astype(np.int64), kp2[:, 0].astype(np.int64)
    maps[pair, r1, c1] = b["d1"].astype(np.float32)
    maps[pair + 1, r2, c2] = b["d2"].astype(np.float32)
    both = rng.uniform(size=len(pair)) < 0.05
    maps[pair[both], r1[both], c1[both]] = np.inf
    maps[pair[both] + 1, r2[both], c2[both]] = np.inf
    inl = b["inliers"]
    q = np.where(inl, rng.uniform(0.3, 1.0, len(inl)), rng.uniform(0.0, 0.7, len(inl))).astype(np.float32)
    cams = b["cams"] / np.array([2.0] * 8)
    return maps, kp1, kp2, q, b["offsets"], cams


def _summary(ts):
    a = np.asarray(ts) * 1e3
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()),
            "p25_ms": float(np.percentile(a, 25)), "p75_ms": float(np.percentile(a, 75)), "n": len(a)}


def bench_gather(ctx, g, k1, k2, tq, offs, f1, f2, dtype, steps, warmup):
    import torch
    P, N, dev = len(offs) - 1, k1.shape[0], g.device
    L = ctx._lib
    suffix = "_f32" if dtype == torch.float32 else ""
    twin, qual = getattr(L, "rp_gather_depths_batch_dev" + suffix), getattr(L, "rp_gather_depths_batch_dev" + suffix + "_quality")
    bufs = {a: ([torch.empty(N, 2, dtype=dtype, device=dev) for _ in range(2)] +
                [torch.empty(N, dtype=dtype, device=dev) for _ in range(2)]) for a in ("twin", "quality")}
    q_out = torch.empty(N, dtype=torch.float32, device=dev)
    outs = {a: np.zeros(P + 1, dtype=np.int64) for a in ("twin", "quality")}
    stream = torch.cuda.current_stream(dev).cuda_stream
    head = [ctx._h, P, offs.ctypes.data, g.data_ptr(), F, H, W, f1.ctypes.data, f2.ctypes.data, k1.data_ptr(), k2.data_ptr()]

    def call(arm):
        o = [t.data_ptr() for t in bufs[arm]]
        t0 = time.perf_counter()
        if arm == "twin":
            rc = twin(*head, *o, outs[arm].ctypes.data, stream)
        else:
            rc = qual(*head, tq.data_ptr(), *o, q_out.data_ptr(), outs[arm].ctypes.data, stream)
        dt = time.perf_counter() - t0
        ctx._check(rc)
        return dt

    for _ in range(warmup):
        call("twin"), call("quality")
    ts = {"twin": [], "quality": []}
    for s in range(steps):
        for arm in (("twin", "quality") if s % 2 == 0 else ("quality", "twin")):
            ts[arm].append(call(arm))
    kept = int(outs["twin"][-1])
    same = bool(np.array_equal(outs["twin"], outs["quality"]) and
                all(torch.equal(a[:kept].view(torch.uint8), b[:kept].view(torch.uint8))
                    for a, b in zip(bufs["twin"], bufs["quality"])))
    s = 8 if dtype == torch.float64 else 4
    # logical bytes from the shapes (the depth reads are random 4 B reads: a 32 B sector each on the device)
    twin_bytes = N * 24 + kept * 6 * s * 3
    qual_bytes = twin_bytes + kept * 16
    rec = {"output": str(dtype).replace("torch.", ""), "rows": N, "kept_rows": kept, "kept_fraction": kept / N,
           "twin": _summary(ts["twin"]), "quality": _summary(ts["quality"]),
           "quality_over_twin_median": float(np.median(ts["quality"]) / np.median(ts["twin"])),
           "bytes_per_kept_row": {"twin": twin_bytes / kept, "quality": qual_bytes / kept},
           "logical_GBps_at_median": {"twin": twin_bytes / np.median(ts["twin"]) / 1e9,
                                      "quality": qual_bytes / np.median(ts["quality"]) / 1e9},
           "twin_outputs_identical": same}
    return rec


def bench_chain(g, k1, k2, tq, offs, f1, f2, cams, steps, warmup):
    import torch
    from mdrp_b200 import _native as nv, torch_frontend as tf
    dev = g.device
    opt = nv.default_options()
    opt.max_iterations = opt.min_iterations = 1000
    opt.max_epipolar_error, opt.max_reproj_error, opt.seed = 2.0, 16.0, 0
    opt.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    opt.progressive_sampling = 1
    tcams = torch.from_numpy(cams).to(dev)
    P = len(offs) - 1
    t_f1 = torch.from_numpy(f1.astype(np.int64)).to(dev)
    t_f2 = torch.from_numpy(f2.astype(np.int64)).to(dev)
    counts = torch.from_numpy(np.diff(offs)).to(dev)
    N = k1.shape[0]

    def chain():
        out, x1, x2, d1, d2, qk = tf.gather_depths_batch(g, f1, f2, offs, k1, k2, dtype=torch.float32, quality=tq)
        return tf.estimate_batch(nv.CALIB, out, x1, x2, d1, d2, tcams, opt, quality=qk)

    def workaround():
        out, x1, x2, d1, d2 = tf.gather_depths_batch(g, f1, f2, offs, k1, k2, dtype=torch.float32)
        # the kernel's keep rule repeated in torch: (int) truncation, border clamp, both-inf rows dropped
        fr1 = torch.repeat_interleave(t_f1, counts, output_size=N)
        fr2 = torch.repeat_interleave(t_f2, counts, output_size=N)
        r1, c1 = k1[:, 1].to(torch.int32).clamp(0, H - 1), k1[:, 0].to(torch.int32).clamp(0, W - 1)
        r2, c2 = k2[:, 1].to(torch.int32).clamp(0, H - 1), k2[:, 0].to(torch.int32).clamp(0, W - 1)
        keep = ~(torch.isinf(g[fr1, r1, c1]) & torch.isinf(g[fr2, r2, c2]))
        return tf.estimate_batch(nv.CALIB, out, x1, x2, d1, d2, tcams, opt, quality=tq[keep])

    arms = {"chain": chain, "workaround": workaround}
    res = {}

    def call(arm):
        t0 = time.perf_counter()
        r = arms[arm]()
        torch.cuda.synchronize(dev)
        res[arm] = r
        return time.perf_counter() - t0

    for _ in range(warmup):
        call("chain"), call("workaround")
    ts = {"chain": [], "workaround": []}
    for s in range(steps):
        for arm in (("chain", "workaround") if s % 2 == 0 else ("workaround", "chain")):
            ts[arm].append(call(arm))
    same = all(torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))
               for a, b in zip(res["chain"], res["workaround"]))
    return {"options": "cfg5: CALIB, 1000 iterations (min = max), PROSAC on, TRUNCATED_CAUCHY, float32 gather", "pairs": P,
            "chain": _summary(ts["chain"]), "workaround": _summary(ts["workaround"]),
            "chain_over_workaround_median": float(np.median(ts["chain"]) / np.median(ts["workaround"])),
            "pairs_per_s_at_median": {a: P / float(np.median(v)) for a, v in ts.items()},
            "outputs_identical": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=500)
    ap.add_argument("--matches", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chain-steps", type=int, default=10)
    ap.add_argument("--out", help="write the record here (JSON); printed to stdout as well")
    a = ap.parse_args()
    import torch
    from mdrp_b200 import _native as nv
    if not torch.cuda.is_available():
        sys.exit("quality_frontend_bench.py needs a CUDA device")
    assert a.pairs + 1 <= F
    maps, kp1, kp2, q, offs, cams = make_video(a.pairs, a.matches, seed=500)
    dev = torch.device("cuda", 0)
    g = torch.from_numpy(maps).to(dev)
    k1, k2, tq = torch.from_numpy(kp1).to(dev), torch.from_numpy(kp2).to(dev), torch.from_numpy(q).to(dev)
    f1 = np.arange(a.pairs, dtype=np.int32)
    f2 = f1 + 1
    ctx = nv.Context(0)
    record = {"gpu": gpu_info(), "shape": {"frames": F, "height": H, "width": W, "pairs": a.pairs,
                                           "matches_per_pair": a.matches, "depth_stack_MB": maps.nbytes / 1e6},
              "gather": [bench_gather(ctx, g, k1, k2, tq, offs, f1, f2, dt, a.steps, a.warmup)
                         for dt in (torch.float64, torch.float32)]}
    for r in record["gather"]:
        print("gather", json.dumps(r), file=sys.stderr, flush=True)
    record["chain_vs_workaround"] = bench_chain(g, k1, k2, tq, offs, f1, f2, cams, a.chain_steps, a.warmup)
    print("chain", json.dumps(record["chain_vs_workaround"]), file=sys.stderr, flush=True)
    ctx.close()
    text = json.dumps(record, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    ok = all(r["twin_outputs_identical"] for r in record["gather"]) and record["chain_vs_workaround"]["outputs_identical"]
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
