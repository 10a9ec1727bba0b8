"""CPU tier of the float32 inputs: the C declarations and ctypes signatures of the float32 entry points, float32 packing
of the Python surface, and which entry point `api` and `sharding` pick for which dtypes (no device: the context is a
recording stand-in)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32_TWINS = {"rp_estimate_batch_host_f32": "rp_estimate_batch_host", "rp_estimate_batch_dev_f32": "rp_estimate_batch_dev",
             "rp_gather_depths_dev_f32": "rp_gather_depths_dev",
             "rp_gather_depths_batch_dev_f32": "rp_gather_depths_batch_dev"}


def _params(header, name):
    m = re.search(r"RP_API\s+int\s+" + name + r"\s*\(([^)]*)\)", header)
    return [re.sub(r"\s+", " ", p.strip()) for p in m.group(1).split(",")]


def test_f32_declarations_differ_from_fp64_twins_only_in_input_type():
    header = open(os.path.join(ROOT, "include", "repose_b200.h")).read()
    for f32, f64 in F32_TWINS.items():
        a, b = _params(header, f32), _params(header, f64)
        assert len(a) == len(b), f32
        changed = [(p, q) for p, q in zip(a, b) if p != q]
        names = {q.split("*")[-1].strip() for _, q in changed}
        assert names == {"x1", "x2", "d1", "d2"}, (f32, changed)
        for p, q in changed:
            assert p.replace("float", "double") == q, (f32, p, q)


def test_f32_ctypes_signatures(monkeypatch):
    """load() gives each float32 symbol the argtypes of its FP64 twin (all pointers are void *) and an int result."""
    from mdrp_b200 import _native as nv

    class FakeFn:
        restype = argtypes = None

    class FakeLib:
        def __getattr__(self, name):
            f = FakeFn()
            setattr(self, name, f)
            return f
    monkeypatch.setattr(nv, "_lib", None)
    monkeypatch.setattr(nv.os.path, "exists", lambda p: True)
    monkeypatch.setattr(nv.C, "CDLL", lambda p: FakeLib())
    L = nv.load()
    monkeypatch.setattr(nv, "_lib", None)
    for f32, f64 in F32_TWINS.items():
        assert f32 in nv.EXPORTS
        assert getattr(L, f32).restype is C.c_int
        assert getattr(L, f32).argtypes == getattr(L, f64).argtypes and getattr(L, f32).argtypes is not None


def test_pack_f32_keeps_dtype_and_offsets():
    from mdrp_b200 import api
    p1 = [np.arange(8, dtype=np.float32).reshape(4, 2), np.zeros((0, 2), np.float32), np.ones((2, 2), np.float32)]
    p2 = [a + 1 for a in p1]
    e1 = [np.arange(4, dtype=np.float32), np.zeros(0, np.float32), np.full(2, 7, np.float32)]
    e2 = [a * 2 for a in e1]
    assert api._all_float32(p1, p2, e1, e2)
    off, x1, x2, d1, d2 = api._pack_auto(p1, p2, e1, e2)
    assert off.tolist() == [0, 4, 4, 6]
    assert all(a.dtype == np.float32 for a in (x1, x2, d1, d2))
    assert x1.shape == (6, 2) and d2.shape == (6,)
    ref = api._pack(p1, p2, e1, e2)
    for a, b in zip((off, x1, x2, d1, d2), ref):
        assert np.array_equal(a, b)
    with pytest.raises(TypeError):
        api._pack_f32([np.zeros((4, 3), np.float32)], [np.zeros((4, 3), np.float32)], [np.ones(4, np.float32)],
                      [np.ones(4, np.float32)])
    with pytest.raises(ValueError):
        api._pack_f32([np.zeros((4, 2), np.float32)], [np.zeros((4, 2), np.float32)], [np.ones(3, np.float32)],
                      [np.ones(4, np.float32)])


def test_mixed_or_other_dtypes_pack_as_float64():
    from mdrp_b200 import api
    f32 = lambda *s: np.zeros(s, np.float32)
    cases = [([f32(3, 2)], [f32(3, 2)], [f32(3)], [np.zeros(3)]),            # one float64 array
             ([f32(3, 2)], [f32(3, 2)], [[1.0, 2.0, 3.0]], [f32(3)]),        # a list
             ([f32(3, 2).astype(np.float16)], [f32(3, 2)], [f32(3)], [f32(3)]),
             ([], [], [], [])]                                               # empty batch
    for c in cases:
        assert not api._all_float32(*c)
        off, x1, x2, d1, d2 = api._pack_auto(*c)
        assert all(a.dtype == np.float64 for a in (x1, x2, d1, d2))


class _RecordingCtx:
    """Stands in for nv.Context: records which estimate entry point was called with which dtypes."""

    def __init__(self):
        self.calls = []

    def _out(self, name, offsets, x1, x2, d1, d2):
        from mdrp_b200 import _native as nv
        self.calls.append((name, x1.dtype, x2.dtype, d1.dtype, d2.dtype))
        P = len(offsets) - 1
        return np.zeros(P, nv.MODEL_DTYPE), np.zeros(P, nv.STATS_DTYPE), np.zeros(int(offsets[-1]), np.uint8)

    def estimate_batch_host(self, variant, offsets, x1, x2, d1, d2, cams, opt):
        return self._out("f64", offsets, x1, x2, d1, d2)

    def estimate_batch_host_f32(self, variant, offsets, x1, x2, d1, d2, cams, opt):
        return self._out("f32", offsets, x1, x2, d1, d2)


def test_api_routes_by_dtype(monkeypatch):
    from mdrp_b200 import api, _native as nv
    rec = _RecordingCtx()
    monkeypatch.setattr(api, "context", lambda device=0: rec)
    monkeypatch.setattr(api, "make_options", lambda *a, **k: nv.Options())
    f32 = lambda *s: np.ones(s, np.float32)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    api.estimate_monodepth_relative_pose(f32(5, 2), f32(5, 2), f32(5), f32(5), cam, cam)
    api.estimate_monodepth_relative_pose(f32(5, 2), f32(5, 2), f32(5), np.ones(5), cam, cam)
    api.estimate_monodepth_shared_focal_relative_pose(f32(5, 2), f32(5, 2), f32(5), f32(5))
    api.estimate_monodepth_varying_focal_relative_pose_batch([f32(5, 2), f32(3, 2)], [f32(5, 2), f32(3, 2)],
                                                             [f32(5), f32(3)], [f32(5), f32(3)])
    api.estimate_monodepth_varying_focal_relative_pose(f32(5, 2).tolist(), f32(5, 2), f32(5), f32(5))
    F, D = np.dtype(np.float32), np.dtype(np.float64)
    assert rec.calls == [("f32", F, F, F, F), ("f64", D, D, D, D), ("f32", F, F, F, F), ("f32", F, F, F, F),
                         ("f64", D, D, D, D)]


def test_sharding_routes_by_dtype():
    from mdrp_b200 import sharding, _native as nv
    rec = _RecordingCtx()
    offs = np.array([0, 4, 6], dtype=np.int64)
    f32 = lambda *s: np.ones(s, np.float32)
    sharding.estimate_local_shard(rec, nv.CALIB, offs, f32(6, 2), f32(6, 2), f32(6), f32(6), None, None, 0, 1)
    sharding.estimate_local_shard(rec, nv.CALIB, offs, np.ones((6, 2)), np.ones((6, 2)), np.ones(6), np.ones(6), None,
                                  None, 0, 1)
    sharding.estimate_local_shard(rec, nv.CALIB, offs, f32(6, 2), np.ones((6, 2)), f32(6), f32(6), None, None, 0, 1)
    assert [c[0] for c in rec.calls] == ["f32", "f64", "f64"]
    # float64 arrays reach the FP64 entry point as they are (what bench.py's multi-GPU line feeds it)
    assert rec.calls[1][1:] == (np.dtype(np.float64),) * 4
    assert rec.calls[2][1:] == (np.dtype(np.float32), np.dtype(np.float64), np.dtype(np.float32), np.dtype(np.float32))
