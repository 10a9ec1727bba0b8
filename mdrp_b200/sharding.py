"""Multi-GPU data parallelism over image pairs (SURVEY.md §8e).

Pairs are independent (no cross-pair state, per-pair RNG seeded from opt.seed), so the batch is
partitioned by pair index across ranks, one process per GPU (the reference's parallelism is a process
pool over pairs, /root/reference/eval.py:355-359).  No data-path collective exists; torch.distributed is
only plumbing: a barrier around timed regions and ONE gather of the result arrays to rank 0 —
preallocated byte tensors through `dist.gather` (96 B model + 40 B stats + N mask bytes per pair),
never pickled objects.  With the NCCL backend the gather runs device to device over NVLink and rank 0
reads the concatenation back once.
"""
import numpy as np


def shard_bounds(n_pairs: int, world_size: int):
    """Contiguous, balanced partition: rank r owns pairs [b[r], b[r+1])."""
    base, rem = divmod(n_pairs, world_size)
    b = [0]
    for r in range(world_size):
        b.append(b[-1] + base + (1 if r < rem else 0))
    return b


def shard_of(offsets, rank: int, world_size: int):
    """(pair_start, pair_end, point_start, point_end, local offsets) of this rank's shard."""
    offsets = np.asarray(offsets, dtype=np.int64)
    b = shard_bounds(len(offsets) - 1, world_size)
    p0, p1 = b[rank], b[rank + 1]
    return p0, p1, int(offsets[p0]), int(offsets[p1]), offsets[p0:p1 + 1] - offsets[p0]


def _as_bytes(a):
    """Zero-copy uint8 torch view of a numpy array or CPU torch tensor."""
    import torch
    if isinstance(a, torch.Tensor):
        return a.contiguous().view(torch.uint8).reshape(-1)
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.view(np.uint8).reshape(-1))


class ResultGatherer:
    """Gathers per-rank result arrays on rank 0 through preallocated buffers (no pickling, no per-call allocation once
    warm).  gloo: CPU tensors.  NCCL (`device` given): each array is staged to the rank's GPU, gathered device to
    device over NVLink into one contiguous buffer on rank 0 and read back once into pinned host memory."""

    def __init__(self, rank: int, world_size: int, device=None):
        self.rank, self.world, self.device = rank, world_size, device
        self._bufs = {}

    def _buf(self, key, nbytes, device, pinned=False):
        import torch
        t = self._bufs.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device, pin_memory=pinned)
            self._bufs[key] = t
        return t

    def gather(self, arrays):
        """arrays: list of numpy arrays / CPU tensors of this rank.  Returns on rank 0 a list of uint8 numpy arrays (the
        byte concatenation over ranks, in rank order; views into buffers that the next call reuses), elsewhere None."""
        import torch
        import torch.distributed as dist
        dev = torch.device("cpu") if self.device is None else self.device
        views = [_as_bytes(a) for a in arrays]
        mine = torch.tensor([v.numel() for v in views], dtype=torch.int64, device=dev)
        sizes = torch.empty(self.world * len(views), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(sizes, mine)
        sizes = sizes.cpu().numpy().reshape(self.world, len(views))
        out = []
        for i, v in enumerate(views):
            nmax = max(int(sizes[:, i].max()), 1)
            send = self._buf(("send", i), nmax, dev)
            send[:v.numel()].copy_(v, non_blocking=True)
            bucket = None
            if self.rank == 0:
                recv = self._buf(("recv", i), self.world * nmax, dev)
                bucket = [recv[r * nmax:(r + 1) * nmax] for r in range(self.world)]
            dist.gather(send[:nmax], bucket, dst=0)
            if self.rank != 0:
                continue
            if self.device is not None:
                host = self._buf(("host", i), self.world * nmax, torch.device("cpu"), pinned=True)
                host[:self.world * nmax].copy_(recv[:self.world * nmax])
            else:
                host = recv
            h = host.numpy()
            if (sizes[:, i] == nmax).all():
                out.append(h[:self.world * nmax])
            else:
                out.append(np.concatenate([h[r * nmax:r * nmax + int(sizes[r, i])] for r in range(self.world)]))
        return out if self.rank == 0 else None


_gatherers = {}


def gather_results(models, stats, masks, rank: int, world_size: int, device=None, gather_masks: bool = True):
    """This rank's (models, stats, masks) — numpy structured arrays, or CPU torch tensors holding the same bytes — ->
    on rank 0 the concatenation over ranks in pair order as numpy arrays (None elsewhere).  `device`: the rank's
    torch CUDA device when the process group is NCCL; None for gloo."""
    from . import _native as nv
    if world_size == 1:
        return models, stats, masks
    key = (rank, world_size, str(device))
    if key not in _gatherers:
        _gatherers[key] = ResultGatherer(rank, world_size, device)
    got = _gatherers[key].gather([models, stats] + ([masks] if gather_masks else []))
    if got is None:
        return None
    return got[0].view(nv.MODEL_DTYPE), got[1].view(nv.STATS_DTYPE), (got[2] if gather_masks else None)


def estimate_sharded(estimate_fn, offsets, x1, x2, d1, d2, cams, rank: int, world_size: int, gather: bool = True,
                     device=None, quality=None):
    """Every rank holds (or maps) the whole batch: run `estimate_fn(offsets, x1, x2, d1, d2, cams) -> (models, stats,
    masks)` on this rank's shard and gather the results on rank 0 in pair order (other ranks get None).  With a
    `quality` ([N], one match quality per correspondence) the shard's slice of it is passed as a seventh argument."""
    p0, p1, n0, n1, loc = shard_of(offsets, rank, world_size)
    args = (loc, x1[n0:n1], x2[n0:n1], d1[n0:n1], d2[n0:n1], None if cams is None else cams[p0:p1])
    res = estimate_fn(*args) if quality is None else estimate_fn(*args, quality[n0:n1])
    if world_size == 1 or not gather:
        return res
    return gather_results(res[0], res[1], res[2], rank, world_size, device=device)


def estimate_local_shard(ctx, variant, offsets, x1, x2, d1, d2, cams, opt, rank: int, world_size: int, device=None,
                         gather_masks: bool = True, quality=None):
    """Every rank holds only ITS shard (local offsets and arrays): run it on this rank's GPU (`ctx`: an
    mdrp_b200._native.Context) and gather on rank 0.  This is what bench.py times at N > 1.  float32 numpy points and
    depths go through the float32 entry point (half the upload, the same results), everything else through FP64.
    `quality` (optional): the shard's match qualities [N], one per correspondence; each pair is then ordered by it
    (the quality entry point of the same dtype)."""
    from .api import _estimate_host
    models, stats, masks = _estimate_host(ctx, variant, offsets, x1, x2, d1, d2, cams, opt, quality)
    return gather_results(models, stats, masks, rank, world_size, device=device, gather_masks=gather_masks)
