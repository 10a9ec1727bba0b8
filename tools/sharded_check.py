#!/usr/bin/env python
"""Sharded == unsharded, on real GPUs (launched under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/sharded_check.py

Every rank builds the same ragged batch, runs its shard through the CUDA estimator (mdrp_b200.sharding over NCCL) and
rank 0 compares the gathered result with the whole batch run on its own GPU: bytes must be identical.

--quality: the same batches with one match quality per correspondence and PROSAC on, through both sharded entry points
(each rank gets its slice of the quality); rank 0 compares with the unsharded estimate_batch_host_quality call."""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mdrp_b200 import _native as nv, sharding, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quality", action="store_true", help="per-correspondence match quality, PROSAC on")
    with_q = ap.parse_args().quality
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ctx = nv.Context(local)
    ok = True
    for cfg, variant in (("cfg2_calib_shift", nv.CALIB_SHIFT), ("cfg3_shared_focal", nv.SHARED), ("cfg5_roma_calib", nv.CALIB)):
        c = synth.CONFIGS[cfg]
        sizes = [c["n"], 37, 3, c["n"] // 2, 1000, 0, 64, 513, 129, 2000, 5, 700, 64]
        scs = [synth.scene_for(cfg, 100 + i, n=max(n, 1)) for i, n in enumerate(sizes)]
        for sc_, n_ in zip(scs, sizes):   # an empty pair: scene_for treats n = 0 as 'default size'
            if n_ == 0:
                sc_.x1, sc_.x2, sc_.d1, sc_.d2 = sc_.x1[:0], sc_.x2[:0], sc_.d1[:0], sc_.d2[:0]
        offs = np.r_[0, np.cumsum(sizes)].astype(np.int64)
        focal = variant >= 2
        x1 = np.concatenate([(s.centred()[0] if focal else s.x1).reshape(-1, 2) for s in scs])
        x2 = np.concatenate([(s.centred()[1] if focal else s.x2).reshape(-1, 2) for s in scs])
        d1, d2 = np.concatenate([s.d1 for s in scs]), np.concatenate([s.d2 for s in scs])
        cams = None if focal else np.array([[s.f1, s.f1, 640, 480, s.f2, s.f2, 640, 480] for s in scs], dtype=np.float64)
        o = nv.default_options()
        o.max_iterations = o.min_iterations = min(c["iters"], 2000)
        o.max_epipolar_error, o.max_reproj_error, o.estimate_shift = 2.0, 16.0, int(c["shift"])
        o.loss_type, o.loss_scale = nv.LOSS["TRUNCATED_CAUCHY"], 1.0
        p0, p1, n0, n1, loc = sharding.shard_of(offs, rank, world)
        if with_q:
            # quality correlated with being an inlier, with ties and a NaN every 101st
            rng = np.random.default_rng(7)
            inl = np.concatenate([s.inlier_mask[:n] for s, n in zip(scs, sizes)])
            q = np.where(inl, rng.uniform(0.3, 1.0, len(inl)), rng.uniform(0.0, 0.7, len(inl))).astype(np.float32)
            q[::13], q[::101] = 0.5, np.nan
            o.progressive_sampling = 1
            fn = lambda of, a, b, e, f, k, qq: ctx.estimate_batch_host_quality(variant, of, a, b, e, f, k, o, qq)  # noqa: E731
            got = sharding.estimate_sharded(fn, offs, x1, x2, d1, d2, cams, rank, world, device=dev, quality=q)
            got2 = sharding.estimate_local_shard(ctx, variant, loc, x1[n0:n1], x2[n0:n1], d1[n0:n1], d2[n0:n1],
                                                 None if cams is None else cams[p0:p1], o, rank, world, device=dev,
                                                 quality=q[n0:n1])
            unsharded = lambda: fn(offs, x1, x2, d1, d2, cams, q)  # noqa: E731
        else:
            fn = lambda of, a, b, e, f, k: ctx.estimate_batch_host(variant, of, a, b, e, f, k, o)  # noqa: E731
            got = sharding.estimate_sharded(fn, offs, x1, x2, d1, d2, cams, rank, world, device=dev)
            # the local-shard entry point (each rank holds only its shard)
            got2 = sharding.estimate_local_shard(ctx, variant, loc, x1[n0:n1], x2[n0:n1], d1[n0:n1], d2[n0:n1],
                                                 None if cams is None else cams[p0:p1], o, rank, world, device=dev)
            unsharded = lambda: fn(offs, x1, x2, d1, d2, cams)  # noqa: E731
        if rank == 0:
            ref = unsharded()
            for g in (got, got2):
                same = all(a.tobytes() == b.tobytes() for a, b in zip(g, ref))
                ok = ok and same
                print(f"{cfg}{' (quality)' if with_q else ''}: {len(sizes)} pairs over {world} GPUs, sharded == unsharded "
                      f"bytes: {same}", flush=True)
        else:
            assert got is None and got2 is None
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("SHARDED_CHECK", "OK" if ok else "FAILED", flush=True)
        sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
