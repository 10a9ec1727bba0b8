#!/usr/bin/env python
"""bench.py — image pairs/s (and hypothesis-scores/s) of the batched RePoseD LO-RANSAC on B200.

A "step" = one pass of the hot path over one batch of synthetic two-view scenes.  Workload at
N=1 = BASELINE.json configs[1]: calibrated scale+shift (monodepth_estimate_shift=True), 2 000
matches per pair, 10 000 RANSAC iterations (min = max), 30 % outliers, truncated-Cauchy final
refinement; `--pairs` pairs per GPU per step (default 10 000 = the config's batch).

  value     whole-job pairs/s with the inputs already resident in HBM (rp_estimate_batch_dev),
            CUDA events on the launching stream, max over ranks
  e2e       the same through the reference-facing entry point with HOST buffers
            (rp_estimate_batch_host): pinned host -> device copies and result read-back inside
            the timed region
  roofline  dominant kernel (score_kernel over the minimal models): 34 algorithmic FP64 flops per
            point-score (SURVEY.md §8d) over its device time measured live with CUDA events,
            against the FP64 FMA pipe peak measured on this device by rp_measure_pipes
  cpu_baseline  the reference's own CPU implementation (oracle/_ref wheel, else the C port) on a
            bounded sample of the same workload on all host cores

Launch: python bench.py --gpus N --steps K --warmup W   (N>1 under torchrun, one rank per GPU)
        python bench.py --impl reference …              (the reference arm: CPU path only)
        python bench.py … --dump-outputs DIR            (also writes the last timed step's results, see dump_outputs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_POINT_SCORE = 34.0  # SURVEY.md §8d


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2_calib_shift")
    ap.add_argument("--pairs", type=int, default=10000, help="image pairs per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0's pairs when --gpus > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    return args


def bench_config(cfg_name, c, pairs, world):
    """`config` of the JSON line: identical keys and values in both arms (ours / --impl reference)."""
    return {"workload": workload_name(cfg_name, c, pairs), "pairs_per_gpu_per_step": pairs,
            "l2": "inputs_larger_than_l2 (%.0f MB per step)" % (pairs * c["n"] * 48 / 1e6),
            "parallelism": f"pairs sharded x{world}, no collective"}


def workload_name(cfg_name, c, pairs):
    return (f"{cfg_name}: {c['variant']}{'+shift' if c['shift'] else ''}, {pairs} pairs x {c['n']} matches, "
            f"{c['iters']} RANSAC iters (min=max), {int(c['outlier_ratio'] * 100)}% outliers, "
            "t=2px r=16px, TRUNCATED_CAUCHY final refinement")


# ---- clocks ---------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_timed=None):
        """Samples that arrived after `t_timed` (the start of the timed region); the sampler is started before the
        warm-up steps — the same load — so that a short timed region (N ranks each spawning nvidia-smi take ~0.5 s to
        deliver the first line) still has samples: if none arrived inside it, the warm-up's are reported."""
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        inside = [ln for t, ln in self.lines if t_timed is None or t >= t_timed]
        window = "timed region" if inside else "warm-up steps (none arrived inside the timed region)"
        for ln in (inside or [ln for _, ln in self.lines]):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ---- CPU reference arm --------------------------------------------------------------------------------
def _ref_options(c):
    iters = c["iters"]
    ro = {"max_iterations": iters, "min_iterations": iters, "max_epipolar_error": 2.0, "max_reproj_error": 16.0, "seed": 0}
    bo = {"loss_type": "TRUNCATED_CAUCHY"}
    if c["variant"] != "calib":
        bo["loss_scale"] = 1.0  # the binding's default for the focal variants: 0.5 * max_epipolar_error
    return ro, bo


def cpu_pairs_per_s(cfg_name, n_sample, seed=12345, keep=False):
    """The reference's CPU path on `n_sample` pairs of the workload, all host cores (GIL released).
    keep=True also returns the batch and the reference's outputs (the parity leg compares the GPU path with them)."""
    from mdrp_b200 import synth
    from oracle import parity
    c = synth.CONFIGS[cfg_name]
    batch = synth.make_batch(cfg_name, n_sample, seed=seed)
    ro, bo = _ref_options(c)
    ref = parity.run_reference(c["variant"], c["shift"], batch, ro, bo)
    out = (n_sample / ref["seconds"], ref["cores"], ref["kind"], ref["seconds"])
    return out + (batch, ref) if keep else out


def reference_arm(args, c, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_sample = args.cpu_sample or max(16 * cores, 64)   # ~3 s of wall clock per step on 16 cores
    for _ in range(args.warmup):
        cpu_pairs_per_s(args.config, max(2, min(n_sample, cores)), seed=1)
    t_tot, n_tot, kind = 0.0, 0, "port"
    for k in range(args.steps):
        pps, cores, kind, dt = cpu_pairs_per_s(args.config, n_sample, seed=100 + k)
        t_tot += dt
        n_tot += n_sample
    value = n_tot / t_tot
    sample = f"{n_sample} pairs per step of the workload, per-pair calls from a {cores}-thread pool"
    line = {"impl": "reference", "metric": "image_pairs_per_sec", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * t_tot / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.config, c, args.pairs, args.gpus),
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


def _ncu_traffic(kernel, pairs_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum of `kernel` from the committed `ncu --set full` capture
    (profiles/rNN_dram_traffic_bytes.json: one launch over `pairs_in_launch` pairs of this workload), scaled
    to the pairs one launch of this run processes; None when no capture is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_dram_traffic_bytes.json")))
    if not files:
        return None
    try:
        d = json.load(open(files[-1]))
        return d[kernel] / d["pairs_in_launch"] * pairs_per_launch
    except Exception:
        return None


# ---- the GPU arm ------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line.  Libraries write banners to fd 1 (NCCL prints its version there at
    the first communicator): park the real stdout and point fd 1 at stderr until the line is emitted."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


DUMP_BYTES = 64_000_000   # --dump-outputs writes at most this much, .npy headers included


def dump_outputs(out_dir, offsets, models, stats, masks):
    """What one estimate call returned, as float arrays two builds can be compared by:
      models.npy      [P,12] f64  q (4), t (3), scale, shift1, shift2, f1, f2
      stats.npy       [P,5]  f64  refinements, iterations, num_inliers, inlier_ratio, model_score
      masks.npy       [M]    f32  inlier masks of the pairs in mask_pairs.npy, concatenated
      mask_pairs.npy  [K]    f64  those pairs: all of them, or a fixed seeded sample when all masks (one value per match)
                                  would not fit in DUMP_BYTES"""
    from mdrp_b200 import _native as nv
    st = stats.view(nv.STATS_DTYPE).reshape(-1)
    out = {"models": np.ascontiguousarray(models, dtype=np.float64),
           "stats": np.stack([st[f].astype(np.float64) for f in nv.STATS_DTYPE.names], axis=1)}
    P = len(offsets) - 1
    lens = np.diff(offsets)
    budget = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 8 * P - 4 * 1024
    order = np.random.default_rng(0).permutation(P)
    pairs = np.sort(order[:int(np.searchsorted(np.cumsum(4 * lens[order]), budget, side="right"))])
    out["masks"] = np.concatenate([masks[offsets[i]:offsets[i + 1]] for i in pairs] or [masks[:0]]).astype(np.float32)
    out["mask_pairs"] = pairs.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    args = parse_args()
    _claim_stdout()
    from mdrp_b200 import synth
    c = synth.CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, c, rank, world)
        return

    import torch
    import torch.distributed as dist
    from mdrp_b200 import _native as nv
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = nv.Context(local_rank)
    variant = {"calib": nv.CALIB_SHIFT if c["shift"] else nv.CALIB, "shared": nv.SHARED, "varying": nv.VARYING}[c["variant"]]
    opt = nv.default_options()
    opt.max_iterations = opt.min_iterations = c["iters"]
    opt.max_epipolar_error, opt.max_reproj_error, opt.seed = 2.0, 16.0, 0
    opt.estimate_shift = int(c["shift"])
    opt.loss_type = nv.LOSS["TRUNCATED_CAUCHY"]
    opt.loss_scale = 1.0  # binding default 0.5*max_epipolar_error for the focal variants

    P = args.pairs
    batch = synth.make_batch(args.config, P, seed=1000 + rank)
    offs = batch["offsets"]
    N = int(offs[-1])
    # pinned host buffers (e2e leg) and device-resident copies (value leg)
    host = {k: torch.from_numpy(np.ascontiguousarray(batch[k])).pin_memory() for k in ("x1", "x2", "d1", "d2")}
    host_cams = torch.from_numpy(batch["cams"]).pin_memory() if batch["cams"] is not None else None
    devt = {k: v.to(dev) for k, v in host.items()}
    dev_cams = host_cams.to(dev) if host_cams is not None else None
    d_models = torch.zeros(P, 12, dtype=torch.float64, device=dev)
    d_stats = torch.zeros(P, 5, dtype=torch.int64, device=dev)
    d_masks = torch.zeros(max(N, 1), dtype=torch.uint8, device=dev)
    h_models = torch.zeros(P, 12, dtype=torch.float64).pin_memory()
    h_stats = torch.zeros(P, 5, dtype=torch.int64).pin_memory()
    h_masks = torch.zeros(max(N, 1), dtype=torch.uint8).pin_memory()
    stream = torch.cuda.current_stream()

    def step_dev():
        ctx.estimate_batch_dev(variant, offs, devt["x1"].data_ptr(), devt["x2"].data_ptr(), devt["d1"].data_ptr(),
                               devt["d2"].data_ptr(), dev_cams.data_ptr() if dev_cams is not None else None, opt,
                               d_models.data_ptr(), d_stats.data_ptr(), d_masks.data_ptr(), stream.cuda_stream)

    import ctypes as C

    def step_host():
        L = ctx._lib
        rc = L.rp_estimate_batch_host(ctx._h, variant, P, offs.ctypes.data, host["x1"].data_ptr(), host["x2"].data_ptr(),
                                      host["d1"].data_ptr(), host["d2"].data_ptr(),
                                      host_cams.data_ptr() if host_cams is not None else None, C.byref(opt),
                                      h_models.data_ptr(), h_stats.data_ptr(), h_masks.data_ptr())
        ctx._check(rc)

    fp64_tf, fp32_tf = ctx.measure_pipes()

    # ---- value: inputs resident in HBM ------------------------------------------------------------
    clocks = ClockSampler(local_rank)
    clocks.start()
    for _ in range(args.warmup):
        step_dev()
    barrier()
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms = {}
    counters = {}
    barrier()
    t_timed = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step_dev()
        tm, cn = ctx.last_timing()
        for k, v in tm.items():
            stage_ms[k] = stage_ms.get(k, 0.0) + v
        for k, v in cn.items():
            counters[k] = v if k == "head_models" else counters.get(k, 0) + v
    e1.record(stream)
    barrier()
    elapsed = e0.elapsed_time(e1) / 1000.0
    launches = ctx.launch_count - launches0
    clk = clocks.stop(t_timed)
    # the last timed step's results, read back after the timed region; the legs below write other buffers
    last_outputs = (d_models.cpu().numpy(), d_stats.cpu().numpy(), d_masks[:N].cpu().numpy()) if args.dump_outputs else None
    t = torch.tensor([elapsed], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_max = float(t.item())
    value = world * P * args.steps / elapsed_max

    # sanity of what was timed: every pair produced a model with a plausible inlier count
    ninl = d_stats[:, 2].float().mean().item()
    assert ninl > 0.5 * c["n"] * (1 - c["outlier_ratio"]), f"implausible result (mean inliers {ninl})"

    # ---- e2e: host buffers through the C ABI, copies inside the timed region --------------------------
    # At N > 1 the job is not done until rank 0 holds everybody's results: the gather of the sharded product path
    # (mdrp_b200.sharding.gather_results: preallocated byte tensors over NCCL / NVLink, one read-back on rank 0) is
    # inside the timed region.
    from mdrp_b200 import sharding
    np_models = h_models.numpy().view(nv.MODEL_DTYPE).reshape(-1)
    np_stats = h_stats.numpy().view(nv.STATS_DTYPE).reshape(-1)
    np_masks = h_masks.numpy()[:N]
    gathered = [None]

    def step_e2e():
        step_host()
        if world > 1:
            gathered[0] = sharding.gather_results(h_models, h_stats, h_masks[:N], rank, world, device=dev)

    for _ in range(max(1, min(args.warmup, 3))):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_elapsed = time.perf_counter() - t0
    if world > 1 and rank == 0:
        assert len(gathered[0][0]) == world * P and gathered[0][0][:P].tobytes() == np_models.tobytes()
    t = torch.tensor([e2e_elapsed], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * P * args.steps / float(t.item())
    assert torch.equal(h_stats.to(dev), d_stats), "host-buffer and device-buffer paths disagree"
    h2d = N * 48 + (P * 64 if host_cams is not None else 0) + (P + 1) * 8
    d2h = P * (96 + 40) + N
    gather_bytes = (world - 1) * d2h if world > 1 else 0   # what rank 0 receives over NVLink and reads back per step

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, offs, *last_outputs)

    # ---- rooflines ---------------------------------------------------------------------------------------------
    # Every kernel that holds > 10 % of the step gets an entry: its algorithmic work (stated in DESIGN.md §5, counted by
    # device counters) over its own CUDA-event time, against the measured peak of the pipe that bounds it.  `roofline`
    # (the contract's key) is the entry of the kernel with the largest share of the step.
    dev_s = stage_ms["device_total"] / 1000.0
    hyps = counters["hypotheses"]
    n_chunk_launches = max(1, int(counters["chunks"]))
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        bf16_tf, bf16_src = float(peaks["bf16_tflops_sustained"]), "MEASURED_PEAKS.json bf16_tflops_sustained"
    except Exception:
        hbm_peak, hbm_src, bf16_tf, bf16_src = 6650.0, "fallback of B200_PROFILING.md", 1400.0, "fallback of B200_PROFILING.md (sustained)"
    pipes_src = "rp_measure_pipes on this device (FMA chains; MEASURED_PEAKS.json has no FP32 / FP64 figure)"
    entries = []
    # (1) tensor-core count tier: 96 tensor flop per point-score (48 TF32 MACs: hi/lo-split C 32, den 16)
    tc_s = stage_ms.get("tc_kernel", 0.0) / 1000.0
    if tc_s > 0:
        tc_ps = counters["tc_evaluated"]
        tf32_peak = bf16_tf / 2.0
        entries.append({"kernel": "tc_count_kernel (tcgen05.mma kind::tf32 + TMEM epilogue: certain-outlier count of every minimal model)",
                        "bound": "tensor", "achieved": 96.0 * tc_ps / tc_s / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                        "frac": 96.0 * tc_ps / tc_s / 1e12 / tf32_peak,
                        "peak_source": bf16_src + " / 2 (dense TF32 runs at half the bf16 rate; no TF32 figure is measured)",
                        "work": "point-scores evaluated (device counter) x 96 tensor flop",
                        "traffic": _ncu_traffic("tc", P * args.steps / n_chunk_launches),
                        "point_scores_per_s": tc_ps / tc_s, "launches": n_chunk_launches,
                        "ms_per_launch": 1000.0 * tc_s / n_chunk_launches, "share_of_step": tc_s / dev_s,
                        "passed_on_fraction": counters["tc_selected"] / max(hyps, 1),
                        "hbm": {"bound": "hbm", "achieved": (args.steps * N * 128 + hyps * 100) / tc_s / 1e9, "peak": hbm_peak,
                                "unit": "GB/s", "frac": (args.steps * N * 128 + hyps * 100) / tc_s / 1e9 / hbm_peak,
                                "peak_source": hbm_src, "note": "feature rows once per pair + model in / count out: this roof does not bind"}})
    # (2) FP32 bound kernel over the survivors of (1): 41 FP32 flop per evaluated point-score
    bound_s = stage_ms["bound_kernel"] / 1000.0
    if bound_s > 0:
        evaluated = counters["bound_evaluated"]
        entries.append({"kernel": "bound_kernel (FP32 outlier-count / score-bound tier, packed f32x2)", "bound": "fp32_pipe",
                        "achieved": 41.0 * evaluated / bound_s / 1e12, "peak": fp32_tf, "unit": "TFLOP/s",
                        "frac": 41.0 * evaluated / bound_s / 1e12 / fp32_tf if fp32_tf else None, "peak_source": pipes_src,
                        "work": "evaluated point-scores (device counter) x 41 FP32 flop",
                        "traffic": _ncu_traffic("bound", P * args.steps / n_chunk_launches),
                        "evaluated_fraction": evaluated / max(counters["point_scores"], 1), "launches": n_chunk_launches,
                        "ms_per_launch": 1000.0 * bound_s / n_chunk_launches, "share_of_step": bound_s / dev_s})
    # (3) LM kernel (LO refinement of every trigger, final LO, final refinement): FP64 flops from device counters x the
    # per-row counts of rp_lm.cuh (LM_FLOPS)
    lm_s = (stage_ms["lo_refine"] + stage_ms["final_refine"]) / 1000.0
    if lm_s > 0 and counters.get("lm_flops", 0):
        entries.append({"kernel": "lm_warp_kernel + lm_kernel (Levenberg-Marquardt: LO of every trigger, one warp per problem; final LO and final refinement, one block per problem)", "bound": "fp64_pipe",
                        "achieved": counters["lm_flops"] / lm_s / 1e12, "peak": fp64_tf, "unit": "TFLOP/s",
                        "frac": counters["lm_flops"] / lm_s / 1e12 / fp64_tf if fp64_tf else None, "peak_source": pipes_src,
                        "work": "device counters: correspondences evaluated, rows accumulated x the FP64 flop table LM_FLOPS (DESIGN.md §5)",
                        "traffic": _ncu_traffic("lm", P * args.steps / n_chunk_launches),
                        "share_of_step": lm_s / dev_s, "lm_iterations": counters["lm_iterations"],
                        "lm_problems": counters["lm_problems"], "note": "includes the LO / final score+merge kernels between the two LM launches: "
                        "stage timers, not per-kernel"})
    entries.sort(key=lambda e: -e["share_of_step"])
    roofline = dict(entries[0]) if entries else {}
    roofline["exact_models_fraction"] = counters["exact_models"] / max(hyps, 1)
    roofline["score_stage_share_of_step"] = stage_ms["score_minimal"] / 1000.0 / dev_s
    ps = hyps * c["n"]   # point-scores the reference would compute for these minimal models

    line = {"metric": "image_pairs_per_sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * elapsed_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.config, c, P, world),
            "secondary": {"hypothesis_scores_per_sec": world * hyps / elapsed_max, "point_scores_per_sec": world * ps / elapsed_max,
                          "models_per_iteration": hyps / (args.steps * P * c["iters"])},
            "stage_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "gathered_to_rank0_bytes_per_step": gather_bytes},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "rooflines": entries}
    if not args.no_cpu_baseline and world == 1:   # the CPU baseline is reported at N = 1 only
        cores = os.cpu_count() or 1
        n_sample = args.cpu_sample or max(64 * cores, 256)   # ~11 s of wall clock on 16 cores
        pps, cores, kind, dt, cb, ref = cpu_pairs_per_s(args.config, n_sample, keep=True)
        line["cpu_baseline"] = {"value": pps, "unit": "pairs/s", "cores": cores, "kind": kind,
                                "sample": f"{n_sample} pairs of the workload, per-pair calls from a {cores}-thread pool, {dt:.1f} s"}
        # parity on the timed workload: the same sample through the GPU path (host entry point), compared with
        # what the reference just returned for it (oracle/parity.py; untimed)
        from oracle import parity
        gm, gs, gk = ctx.estimate_batch_host(variant, cb["offsets"], cb["x1"], cb["x2"], cb["d1"], cb["d2"], cb["cams"], opt)
        rec, _ = parity.compare(ref, cb["offsets"], gm, gs, gk)
        line["parity"] = rec
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
