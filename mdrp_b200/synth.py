"""Synthetic two-view scenes with monocular depths (SURVEY.md §8d).

The reference publishes no dataset that is available offline, so every config
of BASELINE.json is realised as seeded synthetic scenes:
image 1280x960, pp=(640,480); R = Rodrigues(random axis, 20deg*U(0.2,1));
|t| = 0.5; x1 ~ U(image), z1 ~ U(2,8); pixel noise sigma px on both images;
d1 = z1(1+dn*eps) - shift1, d2 = (z2/scale)(1+dn*eps) - shift2; a random subset
of rows gets x2 ~ U(image) (outliers).  RNG = numpy default_rng(1000+index).
"""
from dataclasses import dataclass

import numpy as np

W, H = 1280.0, 960.0
PP = np.array([640.0, 480.0])


@dataclass
class Scene:
    x1: np.ndarray       # [N,2] pixels (full image coordinates)
    x2: np.ndarray       # [N,2]
    d1: np.ndarray       # [N]
    d2: np.ndarray       # [N]
    R: np.ndarray        # ground truth, X2 = R X1 + t
    t: np.ndarray
    scale: float
    shift1: float
    shift2: float
    f1: float
    f2: float
    inlier_mask: np.ndarray

    def camera_dicts(self):
        c1 = {"model": "SIMPLE_PINHOLE", "width": int(W), "height": int(H),
              "params": [self.f1, PP[0], PP[1]]}
        c2 = {"model": "SIMPLE_PINHOLE", "width": int(W), "height": int(H),
              "params": [self.f2, PP[0], PP[1]]}
        return c1, c2

    def centred(self):
        """Points with the principal point subtracted (focal variants' input)."""
        return self.x1 - PP, self.x2 - PP


def rodrigues(axis, angle):
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)


def make_scene(index: int, n: int, f1: float = 800.0, f2: float = 800.0,
               outlier_ratio: float = 0.3, scale: float = 1.7, shift1: float = 0.0,
               shift2: float = 0.0, sigma_px: float = 0.5, depth_noise: float = 0.01) -> Scene:
    rng = np.random.default_rng(1000 + index)
    axis = rng.normal(size=3)
    angle = np.deg2rad(20.0) * rng.uniform(0.2, 1.0)
    R = rodrigues(axis, angle)
    t = rng.normal(size=3)
    t = 0.5 * t / np.linalg.norm(t)
    x1 = np.stack([rng.uniform(0, W, n), rng.uniform(0, H, n)], axis=1)
    z1 = rng.uniform(2.0, 8.0, n)
    X1 = np.concatenate([(x1 - PP) / f1, np.ones((n, 1))], axis=1) * z1[:, None]
    X2 = X1 @ R.T + t
    z2 = X2[:, 2]
    x2 = X2[:, :2] / z2[:, None] * f2 + PP
    x1n = x1 + sigma_px * rng.normal(size=(n, 2))
    x2n = x2 + sigma_px * rng.normal(size=(n, 2))
    d1 = z1 * (1 + depth_noise * rng.normal(size=n)) - shift1
    d2 = (z2 / scale) * (1 + depth_noise * rng.normal(size=n)) - shift2
    n_out = int(round(outlier_ratio * n))
    out_idx = rng.permutation(n)[:n_out]
    x2n[out_idx] = np.stack([rng.uniform(0, W, n_out), rng.uniform(0, H, n_out)], axis=1)
    mask = np.ones(n, dtype=bool)
    mask[out_idx] = False
    return Scene(x1n, x2n, d1, d2, R, t, scale, shift1, shift2, f1, f2, mask)


# BASELINE.json configs as generator arguments (SURVEY.md §8d items 1-5 + hard variant)
CONFIGS = {
    "cfg1_calib_scale": dict(n=1000, iters=1000, f1=800.0, f2=800.0, outlier_ratio=0.3,
                             variant="calib", shift=False),
    "cfg2_calib_shift": dict(n=2000, iters=10000, f1=800.0, f2=800.0, outlier_ratio=0.3,
                             shift1=0.3, shift2=-0.2, variant="calib", shift=True),
    "cfg3_shared_focal": dict(n=2000, iters=10000, f1=800.0, f2=800.0, outlier_ratio=0.3,
                              variant="shared", shift=False),
    "cfg4_varying_focal": dict(n=2000, iters=10000, f1=700.0, f2=900.0, outlier_ratio=0.5,
                               variant="varying", shift=False),
    "cfg5_roma_calib": dict(n=10000, iters=1000, f1=800.0, f2=800.0, outlier_ratio=0.3,
                            variant="calib", shift=False),
    "hard_calib": dict(n=1000, iters=1000, f1=800.0, f2=800.0, outlier_ratio=0.6,
                       sigma_px=2.0, depth_noise=0.1, variant="calib", shift=False),
}


def scene_for(config: str, index: int, n: int | None = None) -> Scene:
    c = CONFIGS[config]
    kw = {k: c[k] for k in ("f1", "f2", "outlier_ratio", "shift1", "shift2", "sigma_px",
                            "depth_noise") if k in c}
    return make_scene(index, n or c["n"], **kw)


def rotation_error_deg(R, R_gt):
    c = (np.trace(R_gt.T @ R) - 1.0) / 2.0
    return float(np.degrees(np.arccos(np.clip(c, -1.0, 1.0))))


def translation_error_deg(t, t_gt):
    """Angle between translation directions (/root/reference/utils/data.py:64-80)."""
    n = np.linalg.norm(t) * np.linalg.norm(t_gt)
    if n < 1e-12:
        return 180.0
    c = np.clip(np.dot(t, t_gt) / n, -1.0, 1.0)
    return float(np.degrees(np.arccos(c)))


def make_batch(config: str, n_pairs: int, seed: int = 0, n: int | None = None):
    """Vectorised generator for the benchmark: the same scene model as make_scene for `n_pairs`
    pairs at once (one RNG stream for the whole batch, so individual scenes differ from
    make_scene(index) — parity tests use make_scene, the bench only needs data of this shape).
    Returns dict(offsets, x1, x2, d1, d2, cams, R, t) with packed [n_pairs*n, …] arrays; x are full
    pixel coordinates for the calibrated variants and principal-point-centred for the focal ones."""
    c = CONFIGS[config]
    n = n or c["n"]
    f1, f2 = c["f1"], c["f2"]
    out_ratio, scale = c["outlier_ratio"], 1.7
    shift1, shift2 = c.get("shift1", 0.0), c.get("shift2", 0.0)
    sigma, dn = c.get("sigma_px", 0.5), c.get("depth_noise", 0.01)
    rng = np.random.default_rng(seed)
    P = n_pairs
    axis = rng.normal(size=(P, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    ang = np.deg2rad(20.0) * rng.uniform(0.2, 1.0, size=P)
    K = np.zeros((P, 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 0] = -axis[:, 2], axis[:, 1], axis[:, 2]
    K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -axis[:, 0], -axis[:, 1], axis[:, 0]
    R = np.eye(3)[None] + np.sin(ang)[:, None, None] * K + (1 - np.cos(ang))[:, None, None] * (K @ K)
    t = rng.normal(size=(P, 3))
    t = 0.5 * t / np.linalg.norm(t, axis=1, keepdims=True)
    x1 = np.stack([rng.uniform(0, W, (P, n)), rng.uniform(0, H, (P, n))], axis=2)
    z1 = rng.uniform(2.0, 8.0, (P, n))
    X1 = np.concatenate([(x1 - PP) / f1, np.ones((P, n, 1))], axis=2) * z1[..., None]
    X2 = np.einsum("pij,pnj->pni", R, X1) + t[:, None, :]
    z2 = X2[..., 2]
    x2 = X2[..., :2] / z2[..., None] * f2 + PP
    x1n = x1 + sigma * rng.normal(size=(P, n, 2))
    x2n = x2 + sigma * rng.normal(size=(P, n, 2))
    d1 = z1 * (1 + dn * rng.normal(size=(P, n))) - shift1
    d2 = (z2 / scale) * (1 + dn * rng.normal(size=(P, n))) - shift2
    outl = rng.uniform(size=(P, n)) < out_ratio
    rnd = np.stack([rng.uniform(0, W, (P, n)), rng.uniform(0, H, (P, n))], axis=2)
    x2n = np.where(outl[..., None], rnd, x2n)
    focal = c["variant"] in ("shared", "varying")
    if focal:
        x1n, x2n = x1n - PP, x2n - PP
    cams = None if focal else np.tile(np.array([f1, f1, PP[0], PP[1], f2, f2, PP[0], PP[1]]), (P, 1))
    return dict(offsets=np.arange(P + 1, dtype=np.int64) * n, x1=x1n.reshape(-1, 2), x2=x2n.reshape(-1, 2),
                d1=d1.reshape(-1), d2=d2.reshape(-1), cams=cams, R=R, t=t, inliers=~outl.reshape(-1))


def quat_from_rotmat(R):
    """w-first unit quaternion of a rotation matrix (w >= 0)."""
    R = np.asarray(R, dtype=np.float64)
    w = np.sqrt(max(0.0, 1.0 + R[0, 0] + R[1, 1] + R[2, 2])) / 2.0
    x = np.copysign(np.sqrt(max(0.0, 1.0 + R[0, 0] - R[1, 1] - R[2, 2])) / 2.0, R[2, 1] - R[1, 2])
    y = np.copysign(np.sqrt(max(0.0, 1.0 - R[0, 0] + R[1, 1] - R[2, 2])) / 2.0, R[0, 2] - R[2, 0])
    z = np.copysign(np.sqrt(max(0.0, 1.0 - R[0, 0] - R[1, 1] + R[2, 2])) / 2.0, R[1, 0] - R[0, 1])
    q = np.array([w, x, y, z])
    return q / np.linalg.norm(q)


def gt_model(sc: Scene, rot_noise_deg: float = 0.0, seed: int = 0) -> np.ndarray:
    """The scene's ground truth as a 12-vector model row (q, t, scale, shift1, shift2, f1, f2; f in pixels), with the
    rotation turned by `rot_noise_deg` about a random axis and t turned by as much (a tracker-like prior)."""
    rng = np.random.default_rng(seed)
    dR = rodrigues(rng.normal(size=3), np.deg2rad(rot_noise_deg))
    t = rodrigues(rng.normal(size=3), np.deg2rad(rot_noise_deg)) @ sc.t
    return np.r_[quat_from_rotmat(dR @ sc.R), t, sc.scale, sc.shift1, sc.shift2, sc.f1, sc.f2]
