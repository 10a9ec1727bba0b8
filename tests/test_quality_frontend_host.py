"""CPU tier of the match quality through the depth gathers and the sharded entry points: the C declarations and ctypes
signatures of rp_gather_depths_*_quality, which gather `torch_frontend` calls with which arguments (CPU stand-ins for
CUDA tensors), and the quality slice each rank of `sharding` receives (a recording context, and world size 2 over
gloo)."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

from test_quality_order_host import _RecordingCtx, _fake_load, _header, _params

GATHER_TWINS = {"rp_gather_depths_dev_quality": "rp_gather_depths_dev",
                "rp_gather_depths_dev_f32_quality": "rp_gather_depths_dev_f32",
                "rp_gather_depths_batch_dev_quality": "rp_gather_depths_batch_dev",
                "rp_gather_depths_batch_dev_f32_quality": "rp_gather_depths_batch_dev_f32"}


def test_gather_quality_declarations_are_twin_plus_quality():
    header = _header()
    for q, twin in GATHER_TWINS.items():
        a, b = _params(header, q), _params(header, twin)
        i = b.index(next(p for p in b if p.endswith("kp2")))
        j = b.index(next(p for p in b if p.endswith("d2")))
        assert a == b[:i + 1] + ["const float *quality"] + b[i + 1:j + 1] + ["float *quality_out"] + b[j + 1:], (q, a, b)


def test_gather_quality_ctypes_signatures(monkeypatch):
    from mdrp_b200 import _native as nv
    L = _fake_load(monkeypatch)
    for q, twin in GATHER_TWINS.items():
        assert q in nv.EXPORTS
        assert getattr(L, q).restype is C.c_int
        t = getattr(L, twin).argtypes
        names = _params(_header(), twin)
        i = names.index(next(p for p in names if p.endswith("kp2")))
        j = names.index(next(p for p in names if p.endswith("d2")))
        assert len(t) == len(names)
        assert getattr(L, q).argtypes == t[:i + 1] + [C.c_void_p] + t[i + 1:j + 1] + [C.c_void_p] + t[j + 1:]


def _floats_at(ptr, n):
    return np.ctypeslib.as_array((C.c_float * n).from_address(ptr)).copy()


class _GatherLib:
    """Records (symbol, args) of every gather call and, for the _quality gathers, the input quality as the call sees it
    (the converted tensor lives only as long as the call).  Reports every row as kept."""

    def __init__(self):
        self.log, self.quality = [], []

    def __getattr__(self, name):
        def fn(*args):
            self.log.append((name, args))
            q = name.endswith("_quality")
            if "batch" in name:
                offs = np.ctypeslib.as_array((C.c_int64 * (args[1] + 1)).from_address(args[2]))
                np.ctypeslib.as_array((C.c_int64 * (args[1] + 1)).from_address(args[-2]))[:] = offs - offs[0]
                if q:   # quality after kp2: argument 11
                    self.quality.append(_floats_at(args[11], int(offs[-1] - offs[0])))
            else:
                n = args[10] if q else args[9]
                args[-2]._obj.value = n
                if q:   # quality after kp2: argument 9
                    self.quality.append(_floats_at(args[9], n))
            return 0
        return fn


class _GatherCtx:
    def __init__(self):
        self._lib, self._h = _GatherLib(), C.c_void_p(1)

    def _call(self, fn, *args):
        assert fn(*args) == 0


@pytest.fixture
def cpu_frontend(monkeypatch):
    """torch_frontend with CPU tensors standing in for CUDA ones and a recording context."""
    torch = pytest.importorskip("torch")
    from mdrp_b200 import torch_frontend as tf
    ctx = _GatherCtx()
    monkeypatch.setattr(tf, "_ctx_for", lambda t: ctx)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: type("S", (), {"cuda_stream": 0})())
    return torch, tf, ctx._lib


def test_gather_depths_routes_quality(cpu_frontend):
    torch, tf, lib = cpu_frontend
    log = lib.log
    dm, kp = torch.ones(4, 6), torch.ones(5, 2)
    q64 = torch.tensor([0.5, 1 / 3, float("nan"), -0.0, 1e-40], dtype=torch.float64)
    out = tf.gather_depths(dm, dm, kp, kp)
    assert len(out) == 4
    out = tf.gather_depths(dm, dm, kp, kp, quality=q64)
    assert len(out) == 5 and out[4].dtype == torch.float32 and out[0].dtype == torch.float64
    qa = log[-1][1]
    # float64 quality is converted to float32 before the call (the values the kernel copies)
    assert lib.quality[-1].tobytes() == q64.float().numpy().tobytes()
    # quality after kp2, quality_out after d2, the twin's arguments around them
    plain = log[0][1]
    assert len(plain) == 16 and len(qa) == 18
    assert qa[:9] == plain[:9] and qa[10] == plain[9] == 5 and qa[-1] == plain[-1]
    assert qa[11] == out[0].data_ptr() and qa[14] == out[3].data_ptr() and qa[15] == out[4].data_ptr()
    out = tf.gather_depths(dm, dm, kp, kp, dtype=torch.float32, quality=q64.float())
    assert len(out) == 5 and out[0].dtype == torch.float32 and len(log[-1][1]) == 18
    names = [n for n, _ in log]
    assert names == ["rp_gather_depths_dev", "rp_gather_depths_dev_quality", "rp_gather_depths_dev_f32_quality"]
    for bad in (torch.ones(4), torch.ones(5, 1), torch.ones(5, device="meta")):
        with pytest.raises(ValueError):
            tf.gather_depths(dm, dm, kp, kp, quality=bad)
    assert len(log) == 3


def test_gather_depths_batch_routes_quality(cpu_frontend):
    torch, tf, lib = cpu_frontend
    log = lib.log
    maps, kp = torch.ones(3, 4, 6), torch.ones(7, 2)
    offs, f1, f2 = np.array([0, 3, 3, 7]), [0, 1, 2], [1, 2, 0]
    q64 = torch.linspace(0, 1, 7, dtype=torch.float64)
    out = tf.gather_depths_batch(maps, f1, f2, offs, kp, kp)
    assert len(out) == 5
    out = tf.gather_depths_batch(maps, f1, f2, offs, kp, kp, quality=q64)
    assert len(out) == 6 and out[5].dtype == torch.float32
    qa = log[-1][1]
    assert lib.quality[-1].tobytes() == q64.float().numpy().tobytes()
    plain = log[0][1]
    assert len(plain) == 17 and len(qa) == 19
    assert qa[:2] == plain[:2] and qa[3:7] == plain[3:7] and qa[-1] == plain[-1]
    assert qa[12] == out[1].data_ptr() and qa[15] == out[4].data_ptr() and qa[16] == out[5].data_ptr()
    tf.gather_depths_batch(maps, f1, f2, offs, kp, kp, dtype=torch.float32, quality=q64.float())
    names = [n for n, _ in log]
    assert names == ["rp_gather_depths_batch_dev", "rp_gather_depths_batch_dev_quality",
                     "rp_gather_depths_batch_dev_f32_quality"]
    for bad in (torch.ones(6), torch.ones(7, device="meta")):
        with pytest.raises(ValueError):
            tf.gather_depths_batch(maps, f1, f2, offs, kp, kp, quality=bad)
    assert len(log) == 3


def test_single_pair_torch_estimate_forwards_quality(cpu_frontend, monkeypatch):
    torch, tf, _ = cpu_frontend
    from mdrp_b200 import api, _native as nv
    monkeypatch.setattr(api, "make_options", lambda *a, **k: nv.Options())
    seen = []

    def fake_estimate_batch(variant, offsets, x1, x2, d1, d2, cams, opt, quality=None):
        seen.append(quality)
        n = int(offsets[-1])
        return torch.zeros(1, 12, dtype=torch.float64), torch.zeros(1, 5, dtype=torch.int64), torch.zeros(n, dtype=torch.uint8)
    monkeypatch.setattr(tf, "estimate_batch", fake_estimate_batch)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    x, d, q = torch.ones(6, 2), torch.ones(6), torch.arange(6.0)
    tf.estimate_monodepth_relative_pose(x, x, d, d, cam, cam)
    tf.estimate_monodepth_relative_pose(x, x, d, d, cam, cam, quality=q)
    assert seen[0] is None and seen[1] is q


def test_local_shard_passes_its_quality():
    from mdrp_b200 import sharding
    rec = _RecordingCtx()
    offs = np.array([0, 4, 9], dtype=np.int64)
    x, d = np.ones((9, 2), np.float32), np.ones(9, np.float32)
    q = np.linspace(0, 1, 9).astype(np.float32)
    sharding.estimate_local_shard(rec, 0, offs, x, x, d, d, None, None, 0, 1, quality=q)
    assert rec.quality.tobytes() == q.tobytes()
    sharding.estimate_local_shard(rec, 0, offs, x.astype(np.float64), x, d, d, None, None, 0, 1, quality=q)
    sharding.estimate_local_shard(rec, 0, offs, x, x, d, d, None, None, 0, 1)
    F, D = np.dtype(np.float32), np.dtype(np.float64)
    assert rec.calls == [("quality", F, F, F, F, F), ("quality", D, F, F, F, F), ("f32", F, F, F, F, None)]


def _fake_estimate_q(offsets, x1, x2, d1, d2, cams, quality):
    """Stand-in for the GPU quality call: per pair, shift1 = sum of the pair's quality, num_inliers = its length;
    mask = quality > 0.5."""
    from mdrp_b200 import _native as nv
    assert len(quality) == len(d1) == int(offsets[-1])
    n = len(offsets) - 1
    models = np.zeros(n, dtype=nv.MODEL_DTYPE)
    stats = np.zeros(n, dtype=nv.STATS_DTYPE)
    for i in range(n):
        models["shift1"][i] = quality[offsets[i]:offsets[i + 1]].astype(np.float64).sum()
        models["scale"][i] = x1[offsets[i]:offsets[i + 1]].sum()
        stats["num_inliers"][i] = offsets[i + 1] - offsets[i]
    return models, stats, (quality > 0.5).astype(np.uint8)


def _worker(rank, world, port, out_q):
    import torch.distributed as dist
    from mdrp_b200 import sharding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(1)
    sizes = rng.integers(0, 30, size=11)
    offsets = np.r_[0, np.cumsum(sizes)]
    n = int(offsets[-1])
    x1, x2 = rng.normal(size=(n, 2)), rng.normal(size=(n, 2))
    d1, d2 = rng.normal(size=n), rng.normal(size=n)
    quality = rng.uniform(size=n).astype(np.float32)
    got = sharding.estimate_sharded(_fake_estimate_q, offsets, x1, x2, d1, d2, None, rank, world, quality=quality)
    mine = sharding.estimate_sharded(_fake_estimate_q, offsets, x1, x2, d1, d2, None, rank, world, gather=False,
                                     quality=quality)
    _, _, n0, n1, loc = sharding.shard_of(offsets, rank, world)
    own = _fake_estimate_q(loc, x1[n0:n1], x2[n0:n1], d1[n0:n1], d2[n0:n1], None, quality[n0:n1])
    ok = all(a.tobytes() == b.tobytes() for a, b in zip(mine, own))
    dist.barrier()
    if rank == 0:
        ref = _fake_estimate_q(offsets, x1, x2, d1, d2, None, quality)
        ok = ok and all(a.tobytes() == b.tobytes() for a, b in zip(got, ref))
    else:
        ok = ok and got is None
    out_q.put((rank, ok))
    dist.destroy_process_group()


def test_two_ranks_get_their_quality_slices():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert sorted(q.get(timeout=5) for _ in range(2)) == [(0, True), (1, True)]
