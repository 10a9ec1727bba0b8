"""CPU tier of the quality-ordered entry points: the C declarations and ctypes signatures of rp_estimate_batch_*_quality
and rp_order_by_quality, the packing of ragged quality lists, and which entry point `api`, `Context` and
`torch_frontend` pick for which dtypes (no device: recording stand-ins)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QUALITY_TWINS = {"rp_estimate_batch_host_quality": "rp_estimate_batch_host",
                 "rp_estimate_batch_dev_quality": "rp_estimate_batch_dev",
                 "rp_estimate_batch_host_f32_quality": "rp_estimate_batch_host_f32",
                 "rp_estimate_batch_dev_f32_quality": "rp_estimate_batch_dev_f32"}


def _header():
    return open(os.path.join(ROOT, "include", "repose_b200.h")).read()


def _params(header, name):
    m = re.search(r"RP_API\s+int\s+" + name + r"\s*\(([^)]*)\)", header)
    return [re.sub(r"\s+", " ", p.strip()) for p in m.group(1).split(",")]


def test_quality_declarations_are_twin_plus_quality():
    header = _header()
    for q, twin in QUALITY_TWINS.items():
        a, b = _params(header, q), _params(header, twin)
        i = b.index(next(p for p in b if p.endswith("d2")))
        assert a == b[:i + 1] + ["const float *quality"] + b[i + 1:], (q, a, b)
    assert _params(header, "rp_order_by_quality") == ["rp_ctx *ctx", "int64_t n_pairs", "const int64_t *offsets",
                                                      "const float *quality", "int32_t *perm"]


def test_smem_cap_matches_header():
    from mdrp_b200 import _native as nv
    m = re.search(r"#define\s+RP_ORDER_SMEM_CAP\s+(\d+)", _header())
    assert int(m.group(1)) == nv.ORDER_SMEM_CAP


def _fake_load(monkeypatch):
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
    return L


def test_quality_ctypes_signatures(monkeypatch):
    from mdrp_b200 import _native as nv
    L = _fake_load(monkeypatch)
    for q, twin in QUALITY_TWINS.items():
        assert q in nv.EXPORTS
        assert getattr(L, q).restype is C.c_int
        t = getattr(L, twin).argtypes
        assert getattr(L, q).argtypes == t[:8] + [C.c_void_p] + t[8:]
    assert "rp_order_by_quality" in nv.EXPORTS
    assert L.rp_order_by_quality.restype is C.c_int
    assert L.rp_order_by_quality.argtypes == [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    assert nv.TIMING_KEYS[13:15] == ["widen", "order"]


def test_pack_quality_converts_to_float32_and_checks_lengths():
    from mdrp_b200 import api
    offs = np.array([0, 3, 3, 5], dtype=np.int64)
    q64 = [np.array([0.1, 1 / 3, np.nan]), np.zeros(0), [2.0, -0.0]]
    q = api._pack_quality(q64, offs)
    assert q.dtype == np.float32 and q.shape == (5,)
    assert q[1] == np.float32(1 / 3) and np.isnan(q[2]) and np.signbit(q[4])
    # float64 values that differ only below float32 precision become ties
    q = api._pack_quality([np.array([1.0, 1.0 + 1e-12, 1.0 - 1e-12])], np.array([0, 3]))
    assert len(set(q.tolist())) == 1
    with pytest.raises(ValueError):
        api._pack_quality([np.zeros(3), np.zeros(1), np.zeros(2)], offs)   # pair 1 has no correspondences
    with pytest.raises(ValueError):
        api._pack_quality([np.zeros(3), np.zeros(0)], offs)                # one array per pair
    assert api._pack_quality([], np.array([0])).shape == (0,)


class _RecordingCtx:
    """Stands in for nv.Context: records which estimate entry point was called with which dtypes."""

    def __init__(self):
        self.calls = []

    def _out(self, name, offsets, x1, x2, d1, d2, quality=None):
        from mdrp_b200 import _native as nv
        self.calls.append((name, x1.dtype, x2.dtype, d1.dtype, d2.dtype, None if quality is None else quality.dtype))
        self.quality = quality
        P = len(offsets) - 1
        return np.zeros(P, nv.MODEL_DTYPE), np.zeros(P, nv.STATS_DTYPE), np.zeros(int(offsets[-1]), np.uint8)

    def estimate_batch_host(self, variant, offsets, x1, x2, d1, d2, cams, opt):
        return self._out("f64", offsets, x1, x2, d1, d2)

    def estimate_batch_host_f32(self, variant, offsets, x1, x2, d1, d2, cams, opt):
        return self._out("f32", offsets, x1, x2, d1, d2)

    def estimate_batch_host_quality(self, variant, offsets, x1, x2, d1, d2, cams, opt, quality):
        return self._out("quality", offsets, x1, x2, d1, d2, quality)


def test_api_batch_functions_route_quality(monkeypatch):
    from mdrp_b200 import api, _native as nv
    rec = _RecordingCtx()
    monkeypatch.setattr(api, "context", lambda device=0: rec)
    monkeypatch.setattr(api, "make_options", lambda *a, **k: nv.Options())
    f32 = lambda *s: np.ones(s, np.float32)
    f64 = lambda *s: np.ones(s)
    cam = {"model": "SIMPLE_PINHOLE", "params": [800.0, 640.0, 480.0]}
    F, D = np.dtype(np.float32), np.dtype(np.float64)
    api.estimate_monodepth_relative_pose_batch([f32(5, 2)], [f32(5, 2)], [f32(5)], [f32(5)], [cam], [cam],
                                               quality=[np.linspace(0, 1, 5)])
    assert rec.quality.tolist() == np.linspace(0, 1, 5).astype(np.float32).tolist()
    api.estimate_monodepth_relative_pose_batch([f64(5, 2)], [f64(5, 2)], [f64(5)], [f64(5)], [cam], [cam],
                                               quality=[f32(5)])
    api.estimate_monodepth_shared_focal_relative_pose_batch([f32(4, 2), f32(2, 2)], [f32(4, 2), f32(2, 2)],
                                                            [f32(4), f32(2)], [f32(4), f32(2)], quality=[f64(4), f64(2)])
    api.estimate_monodepth_varying_focal_relative_pose_batch([f32(3, 2)], [f32(3, 2)], [f32(3)], [f64(3)],
                                                             quality=[[3, 2, 1]])
    api.estimate_monodepth_varying_focal_relative_pose_batch([f32(3, 2)], [f32(3, 2)], [f32(3)], [f32(3)])
    assert rec.calls == [("quality", F, F, F, F, F), ("quality", D, D, D, D, F), ("quality", F, F, F, F, F),
                         ("quality", D, D, D, D, F), ("f32", F, F, F, F, None)]
    with pytest.raises(ValueError):
        api.estimate_monodepth_relative_pose_batch([f32(5, 2)], [f32(5, 2)], [f32(5)], [f32(5)], [cam], [cam],
                                                   quality=[f32(4)])
    # the single-pair functions keep their signatures
    import inspect
    assert "quality" not in inspect.signature(api.estimate_monodepth_relative_pose).parameters


class _FakeFn:
    def __init__(self, name, log):
        self.name, self.log = name, log

    def __call__(self, *args):
        self.log.append((self.name, args))
        return 0


class _FakeLib:
    def __init__(self):
        self.log = []

    def __getattr__(self, name):
        f = _FakeFn(name, self.log)
        setattr(self, name, f)
        return f


def _fake_context():
    from mdrp_b200 import _native as nv
    ctx = object.__new__(nv.Context)
    ctx._lib = _FakeLib()
    ctx._h = C.c_void_p(1)
    import threading
    ctx._lock = threading.RLock()
    return ctx


def test_context_host_quality_routes_by_dtype():
    from mdrp_b200 import _native as nv
    ctx = _fake_context()
    offs = np.array([0, 4, 6], dtype=np.int64)
    f32 = lambda *s: np.ones(s, np.float32)
    o = nv.Options()
    ctx.estimate_batch_host_quality(nv.SHARED, offs, f32(6, 2), f32(6, 2), f32(6), f32(6), None, o, np.arange(6.0))
    ctx.estimate_batch_host_quality(nv.SHARED, offs, f32(6, 2), np.ones((6, 2)), f32(6), f32(6), None, o, f32(6))
    ctx.estimate_batch_host_quality(nv.SHARED, offs, [[0, 0]] * 6, f32(6, 2), f32(6), f32(6), None, o, f32(6))
    names = [n for n, _ in ctx._lib.log]
    assert names == ["rp_estimate_batch_host_f32_quality", "rp_estimate_batch_host_quality", "rp_estimate_batch_host_quality"]
    args = ctx._lib.log[0][1]
    assert len(args) == 14 and args[2] == 2   # ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, 3 outputs
    with pytest.raises(ValueError):
        ctx.estimate_batch_host_quality(nv.SHARED, offs, f32(6, 2), f32(6, 2), f32(6), f32(6), None, o, f32(5))
    # the device methods put the quality pointer after d2 and the stream last
    ctx._lib.log.clear()
    ctx.estimate_batch_dev_quality(nv.SHARED, offs, 1, 2, 3, 4, None, o, 5, 6, 7, 8, stream=9)
    ctx.estimate_batch_dev_f32_quality(nv.SHARED, offs, 1, 2, 3, 4, None, o, 5, 6, 7, 8)
    (n1, a1), (n2, a2) = ctx._lib.log
    assert (n1, n2) == ("rp_estimate_batch_dev_quality", "rp_estimate_batch_dev_f32_quality")
    assert a1[4:9] == (1, 2, 3, 4, 8) and a1[-4:] == (5, 6, 7, 9) and a2[-1] is None


def test_torch_frontend_routes_quality(monkeypatch):
    torch = pytest.importorskip("torch")
    from mdrp_b200 import torch_frontend as tf, _native as nv

    class Rec:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            if not name.startswith("estimate_batch_dev"):
                raise AttributeError(name)
            return lambda *a: self.calls.append((name, a))
    rec = Rec()
    monkeypatch.setattr(tf, "_ctx_for", lambda t: rec)
    # CPU tensors stand in for CUDA ones: only the routing and the conversions are checked here
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: type("S", (), {"cuda_stream": 0})())
    real_zeros = torch.zeros
    monkeypatch.setattr(torch, "zeros", lambda *a, **k: real_zeros(*a, **{**k, "device": "cpu"}))
    offs = np.array([0, 3, 5], dtype=np.int64)
    x32, d32 = torch.ones(5, 2), torch.ones(5)
    x64, d64 = x32.double(), d32.double()
    q64 = torch.tensor([0.5, 0.25, 1.0, 0.0, 1 / 3], dtype=torch.float64)
    o = nv.Options()
    tf.estimate_batch(nv.SHARED, offs, x32, x32, d32, d32, None, o, quality=q64)
    tf.estimate_batch(nv.SHARED, offs, x64, x64, d64, d64, None, o, quality=q64.float())
    tf.estimate_batch(nv.SHARED, offs, x32, x32, d32, d32, None, o)
    names = [n for n, _ in rec.calls]
    assert names == ["estimate_batch_dev_f32_quality", "estimate_batch_dev_quality", "estimate_batch_dev_f32"]
    assert all(len(a) == 13 for _, a in rec.calls[:2]) and len(rec.calls[2][1]) == 12
    with pytest.raises(ValueError):
        tf.estimate_batch(nv.SHARED, offs, x32, x32, d32, d32, None, o, quality=torch.ones(4))
