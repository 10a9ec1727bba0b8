"""The LM kernels against an extended-precision reference with exact derivatives.

The reference below writes the refinement problem of rp_lm.cuh from its formulas, not from the device code:
  cost = sum_k  w_s rho(r_s^2) + rho(s_r |pi(R (d1+u) p1 + t) - x2|^2)[Z.z > 0] + rho(s_r |pi(R^T (sigma (d2+v) p2 - t)) - x1|^2)[Y.z > 0]
with r_s the Sampson residual of F = K2^-T [t]x R K1^-1, parameters (w, t, scale, then (shift1, shift2) | f | (f1, f2))
and the update R <- R exp([w]x).  It runs in numpy.longdouble (64-bit mantissa) and takes its Jacobians by complex
step in clongdouble, so its values and derivatives are exact to ~1e-18, far below the FP64 kernels' rounding.  The
losses, IRLS weights and the reference's quirks (DESIGN.md §3, oracle/repose_oracle.c) are encoded as such:
  - the Sampson row enters the normal equations with weight_sampson^2 and the cost with weight_sampson;
  - the focal variants evaluate the Sampson robust weight at weight_sampson * r^2;
  - TRUNCATED is min(r^2, t^2), so a NaN residual stays NaN.

The final-refinement kernels are reached through rp_refine_batch; the LO configuration (use_final = 0: lm_warp_kernel
and the block kernel with the TRUNCATED loss) only through tests/lmcheck, a harness built with the product's own
repose_lm.cu.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from mdrp_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "mdrp_b200", "csrc")
LMC_SRC = os.path.join(HERE, "lmcheck", "lmcheck.cu")
LMC_SO = os.path.join(HERE, "lmcheck", "liblmcheck.so")

LD, CLD = np.longdouble, np.clongdouble
U = np.finfo(np.float64).eps / 2            # unit roundoff of FP64
NPAR = {0: 7, 1: 9, 2: 8, 3: 9}
VARIANTS = [0, 1, 2, 3]
TRIVIAL, TRUNCATED, HUBER, CAUCHY, TRUNCATED_CAUCHY = range(5)
LOSSES = [TRIVIAL, TRUNCATED, HUBER, CAUCHY, TRUNCATED_CAUCHY]
LOSS_NAMES = ["TRIVIAL", "TRUNCATED", "HUBER", "CAUCHY", "TRUNCATED_CAUCHY"]
THRESHOLD_LOSSES = (TRUNCATED, HUBER, TRUNCATED_CAUCHY)
SR = (2.0 / 16.0) ** 2
# (weight_sampson, scale_reproj): every combination except both terms off
TERM_COMBOS = [(ws, sr) for ws in (1.0, 0.37, 0.0) for sr in (SR, 0.0) if ws > 0 or sr > 0]
SIZES = [0, 1, 3, 31, 32, 33, 63, 64, 65, 127, 128, 129, 1000, 16384, 23000]
MARGIN = 1e-9                               # decisions closer than this (relative) may go either way in FP64
COST_RTOL = 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# reference

def _re(a):
    return np.real(a) if a.dtype != object else np.array([float(v.real) if hasattr(v, "real") else float(v) for v in a])


def _skew(v):
    z = v[0] * 0
    return np.array([[z, -v[2], v[1]], [v[2], z, -v[0]], [-v[1], v[0], z]], dtype=v.dtype)


def _rotmat(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]], dtype=q.dtype)


def residuals(v, m, x1, x2, d1, d2, dp, sqrt=np.sqrt):
    """Residuals of every correspondence at the model m (12-vector) moved by the parameter vector dp (the rotation
    enters to first order, R (I + [w]x), which is exact for the first derivative).  Works on longdouble,
    clongdouble and mpmath object arrays.  Returns rs [n], r12 [n,2], r21 [n,2], the gates Z.z > 0, Y.z > 0 and the
    Sampson denominator."""
    dt = dp.dtype
    one = dp[0] * 0 + 1
    R = _rotmat(m[:4].astype(dt)) @ (np.eye(3, dtype=dt) * one + _skew(dp[:3]))
    t = m[4:7].astype(dt) + dp[3:6]
    scale, sh1, sh2, f1, f2 = (m[7] + dp[6], m[8] * one, m[9] * one, m[10] * one, m[11] * one)
    if v == 1:
        sh1, sh2 = sh1 + dp[7], sh2 + dp[8]
    elif v == 2:
        f1, f2 = f1 + dp[7], f2 + dp[7]
    elif v == 3:
        f1, f2 = f1 + dp[7], f2 + dp[8]
    E = _skew(t) @ R
    K1i = np.array([[1 / f1, 0 * one, 0 * one], [0 * one, 1 / f1, 0 * one], [0 * one, 0 * one, one]], dtype=dt)
    K2i = np.array([[1 / f2, 0 * one, 0 * one], [0 * one, 1 / f2, 0 * one], [0 * one, 0 * one, one]], dtype=dt)
    F = K2i.T @ E @ K1i
    h1 = np.concatenate([x1.astype(dt), np.ones((len(x1), 1), dtype=dt) * one], axis=1)
    h2 = np.concatenate([x2.astype(dt), np.ones((len(x2), 1), dtype=dt) * one], axis=1)
    Fx1, Ftx2 = h1 @ F.T, h2 @ F
    Cs = (h2 * Fx1).sum(axis=1)
    sden = sqrt(Fx1[:, 0] ** 2 + Fx1[:, 1] ** 2 + Ftx2[:, 0] ** 2 + Ftx2[:, 1] ** 2)
    rs = Cs / sden
    p1, p2 = h1 @ K1i.T, h2 @ K2i.T
    Z = ((d1.astype(dt) + sh1)[:, None] * p1) @ R.T + t
    r12 = f2 * Z[:, :2] / Z[:, 2:3] - x2
    Y = (scale * (d2.astype(dt) + sh2)[:, None] * p2 - t) @ R
    r21 = f1 * Y[:, :2] / Y[:, 2:3] - x1
    return rs, r12, r21, _re(Z[:, 2]) > 0, _re(Y[:, 2]) > 0, sden


def rho(loss, t2, r2):
    if loss == TRIVIAL:
        return r2
    if loss == TRUNCATED:
        return np.where(t2 < r2, t2, r2)
    if loss == HUBER:
        r = np.sqrt(r2)
        return np.where(r <= np.sqrt(t2), r2, np.sqrt(t2) * (2 * r - np.sqrt(t2)))
    if loss == CAUCHY:
        return t2 * np.log1p(r2 / t2)
    return np.where(r2 > t2, t2 * np.log1p(LD(1)), t2 * np.log1p(r2 / t2))


def rho_weight(loss, t2, r2):
    if loss == TRIVIAL:
        return np.ones_like(r2)
    if loss == TRUNCATED:
        return np.where(r2 < t2, LD(1), LD(0))
    if loss == HUBER:
        r = np.sqrt(r2)
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(r <= np.sqrt(t2), LD(1), np.sqrt(t2) / r)
    if loss == CAUCHY:
        return 1 / (1 + r2 / t2)
    return np.where(r2 > t2, LD(0), 1 / (1 + r2 / t2))


class Problem:
    """One refinement problem: data in longdouble plus the options the cost depends on."""

    def __init__(self, v, x1, x2, d1, d2, ws, sr, loss, t):
        self.v, self.np = v, NPAR[v]
        self.x1, self.x2 = np.asarray(x1, dtype=LD).reshape(-1, 2), np.asarray(x2, dtype=LD).reshape(-1, 2)
        self.d1, self.d2 = np.asarray(d1, dtype=LD), np.asarray(d2, dtype=LD)
        self.ws, self.sr, self.loss, self.t2 = LD(ws), LD(sr), loss, LD(t) * LD(t)

    def _res(self, m, dp):
        with np.errstate(all="ignore"):
            return residuals(self.v, np.asarray(m, dtype=LD), self.x1, self.x2, self.d1, self.d2, dp)

    def rows(self, m, jac=True):
        """Per residual kind: (cost term factor, r^2 argument of the loss, gate, weight argument, row weight factor,
        residual rows [n,k], Jacobian [n,k,NP] or None, FP64 rounding scale of the residual [n])."""
        rs, r12, r21, v12, v21, sden = self._res(m, np.zeros(self.np, dtype=LD))
        J = None
        if jac:
            h = LD("1e-30")
            Js, J12, J21 = (np.zeros((len(rs), k, self.np), dtype=LD) for k in (1, 2, 2))
            for i in range(self.np):
                dp = np.zeros(self.np, dtype=CLD)
                dp[i] = 1j * h
                a, b, c = self._res(m, dp)[:3]
                Js[:, 0, i], J12[:, :, i], J21[:, :, i] = a.imag / h, b.imag / h, c.imag / h
            J = (Js, J12, J21)
        mm = np.asarray(m, dtype=LD)
        f1, f2 = mm[10], mm[11]
        # magnitude of the FP64 quantities each residual is computed from (for the rounding allowance)
        n1 = np.abs(self.x1).sum(axis=1) / abs(f1) + 1
        n2 = np.abs(self.x2).sum(axis=1) / abs(f2) + 1
        out = []
        foc = self.v in (2, 3)
        if self.ws > 0:
            r2 = rs * rs
            # p2^T E p1 sums products of magnitude |p1| |E| |p2|, |E| <= 2 |t|
            scale_s = np.abs(rs) + 2 * n1 * n2 * np.sqrt((mm[4:7] ** 2).sum()) * (1 + 1 / abs(f1)) * (1 + 1 / abs(f2)) / sden
            out.append(("s", self.ws, r2, np.ones(len(rs), bool), self.ws * r2 if foc else r2, self.ws * self.ws,
                        rs[:, None], None if J is None else J[0], scale_s))
        if self.sr > 0:
            for name, r, gate, jj, xs in (("12", r12, v12, None if J is None else J[1], self.x2),
                                          ("21", r21, v21, None if J is None else J[2], self.x1)):
                r2 = self.sr * (r ** 2).sum(axis=1)
                out.append((name, LD(1), r2, gate, r2, self.sr, r, jj, np.abs(r).sum(axis=1) + 2 * np.abs(xs).sum(axis=1) + 1))
        return out

    def point_costs(self, m):
        """Per correspondence: cost, sum of |terms|, FP64 rounding allowance of the cost, smallest threshold margin
        |x - 1| of its residuals (cost and weight arguments)."""
        n = len(self.d1)
        c, a_abs, allow = (np.zeros(n, dtype=LD) for _ in range(3))
        marg = np.full(n, LD(np.inf))
        for name, fac, r2, gate, warg, rwf, r, J, sc in self.rows(m, jac=False):
            with np.errstate(all="ignore"):
                tk = fac * rho(self.loss, self.t2, r2)
                wk = rho_weight(self.loss, self.t2, r2)
                rr = np.sqrt(r2 / (self.sr if name != "s" else 1))
                dr = 64 * LD(U) * sc
                a = fac * np.where(np.isfinite(wk), wk, 0) * (self.sr if name != "s" else 1) * (2 * rr * dr + dr * dr)
                c += np.where(gate, tk, 0)
                a_abs += np.where(gate, np.abs(tk), 0)
                allow += np.where(gate & np.isfinite(a), a, 0)
                if self.loss in THRESHOLD_LOSSES:
                    for arg in ((r2, warg) if name == "s" and self.v in (2, 3) else (r2,)):
                        mk = np.abs(arg / self.t2 - 1)
                        marg = np.where(gate & np.isfinite(mk) & (mk < marg), mk, marg)
        return c, a_abs, allow, marg

    def cost(self, m):
        """cost, sum |terms|, the FP64 rounding allowance of the sum, and the smallest threshold margin |x - 1|."""
        c, a_abs, allow, marg = self.point_costs(m)
        return c.sum(), a_abs.sum(), allow.sum(), (marg.min() if len(marg) else LD(np.inf))

    def normal(self, m):
        """A = sum w J^T J and g = sum w J^T r (the oracle's normal equations, quirks included)."""
        A = np.zeros((self.np, self.np), dtype=LD)
        g = np.zeros(self.np, dtype=LD)
        for name, fac, r2, gate, warg, rwf, r, J, sc in self.rows(m):
            with np.errstate(all="ignore"):
                w = rwf * rho_weight(self.loss, self.t2, warg)
            use = gate & (w != 0)
            if not use.any():
                continue
            Jw, rw, ww = J[use], r[use], w[use]
            A += np.einsum("n,nki,nkj->ij", ww, Jw, Jw)
            g += np.einsum("n,nki,nk->i", ww, Jw, rw)
        return A, g


def solve_ld(A, b):
    """(A) x = b by Cholesky in longdouble (numpy.linalg rejects longdouble)."""
    n = len(b)
    L = np.zeros((n, n), dtype=LD)
    for j in range(n):
        s = A[j, j] - (L[j, :j] ** 2).sum()
        L[j, j] = np.sqrt(s)
        for i in range(j + 1, n):
            L[i, j] = (A[i, j] - (L[i, :j] * L[j, :j]).sum()) / L[j, j]
    y = np.zeros(n, dtype=LD)
    for i in range(n):
        y[i] = (b[i] - (L[i, :i] * y[:i]).sum()) / L[i, i]
    x = np.zeros(n, dtype=LD)
    for i in reversed(range(n)):
        x[i] = (y[i] - (L[i + 1:, i] * x[i + 1:]).sum()) / L[i, i]
    return x


def lm_step(A, g, lam):
    return -solve_ld(A + LD(lam) * np.eye(len(g), dtype=LD), g)


def _qmul(a, b):
    return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3],
                     a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                     a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1],
                     a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]], dtype=LD)


def model_step(v, m, x):
    m = np.asarray(m, dtype=LD).copy()
    w = np.asarray(x[:3], dtype=LD)
    th = np.sqrt((w * w).sum())
    if th > 1e-6:
        dq = np.r_[np.cos(th / 2), np.sin(th / 2) / th * w]
    else:
        a2 = th * th / 4
        dq = np.r_[1 - a2 / 2 + a2 * a2 / 24, (LD(0.5) - a2 / 12 + a2 * a2 / 240) * w]
    m[:4] = _qmul(m[:4], dq.astype(LD))
    m[4:7] += x[3:6]
    m[7] += x[6]
    if v == 1:
        m[8] += x[7]
        m[9] += x[8]
    elif v == 2:
        m[10] += x[7]
        m[11] = m[10]
    elif v == 3:
        m[10] += x[7]
        m[11] += x[8]
    return m


def step_from_models(v, m0, m1):
    """The parameter step that model_step applied to m0 to give m1: log map of q0^-1 q1, differences elsewhere."""
    m0, m1 = np.asarray(m0, dtype=LD), np.asarray(m1, dtype=LD)
    q0c = m0[:4] * np.array([1, -1, -1, -1], dtype=LD)
    dq = _qmul(q0c, m1[:4]) / (m0[:4] ** 2).sum()
    if dq[0] < 0:
        dq = -dq
    s = np.sqrt((dq[1:] ** 2).sum())
    w = dq[1:] * (2 * np.arctan2(s, dq[0]) / s) if s > 0 else dq[1:] * 2
    rest = [m1[4] - m0[4], m1[5] - m0[5], m1[6] - m0[6], m1[7] - m0[7]]
    if v == 1:
        rest += [m1[8] - m0[8], m1[9] - m0[9]]
    elif v == 2:
        rest += [m1[10] - m0[10]]
    elif v == 3:
        rest += [m1[10] - m0[10], m1[11] - m0[11]]
    return np.r_[w, np.array(rest, dtype=LD)].astype(LD)


def lm_run(pb, m0, max_it, gtol, stol, lam0, lmin, lmax):
    """lm_impl of the kernels, in longdouble; lambda stays float64 exactly as the kernels keep it.  Records the
    smallest relative margin of every decision: the accept test (relative to sum |terms|), the gradient and step
    tolerances, and every residual's threshold test."""
    m = np.asarray(m0, dtype=LD)
    cost, terms, _, tm = pb.cost(m)
    init = cost
    hist = []                       # (iteration, |g|, smallest margin so far) at every gradient check
    shist = []                      # (iteration, |step|, smallest margin so far) at every step check
    accepted = 0
    lam = float(lam0)
    margin = float(tm)
    it, inv, gn, sn = 0, 0, -1.0, -1.0
    A = g = None
    if max_it > 0:
        A, g = pb.normal(m)
    recompute = True
    while it < max_it:
        if recompute:
            gn = np.sqrt((g * g).sum())
            hist.append((it, float(gn), margin))
            if gtol > 0:
                margin = min(margin, float(abs(gn - LD(gtol)) / LD(gtol)))
            if gn < gtol:
                break
        x = lm_step(A, g, lam)
        sn = np.sqrt((x * x).sum())
        shist.append((it, float(sn), margin))
        if stol > 0:
            margin = min(margin, float(abs(sn - LD(stol)) / LD(stol)))
        if sn < stol:
            break
        mn = model_step(pb.v, m, x)
        cn, tn, _, tm = pb.cost(mn)
        margin = min(margin, float(tm), float(abs(cn - cost) / max(tn, terms)))
        if cn < cost:
            m, cost, terms = mn, cn, tn
            accepted += 1
            lam = max(lmin, lam / 10)
            if it < max_it - 1:
                A, g = pb.normal(m)
            recompute = True
        else:
            inv += 1
            lam = min(lmax, lam * 10)
            recompute = False
        it += 1
    return dict(model=m, cost=cost, terms=terms, initial_cost=init, lam=lam, iterations=it, invalid_steps=inv,
                step_norm=sn, grad_norm=gn, margin=margin, hist=hist, shist=shist, accepted=accepted)


# ---------------------------------------------------------------------------------------------------------------------
# data

def gt_model(sc, v, ns=1.0):
    from scipy.spatial.transform import Rotation as Rot
    qq = Rot.from_matrix(sc.R).as_quat()
    foc = v in (2, 3)
    return np.r_[qq[3], qq[0], qq[1], qq[2], sc.t, sc.scale, sc.shift1 if v == 1 else 0.0, sc.shift2 if v == 1 else 0.0,
                 sc.f1 / ns if foc else 1.0, (sc.f1 if v == 2 else sc.f2) / ns if foc else 1.0]


def make_data(v, n, seed, huge=False, inliers_only=False):
    """Normalised correspondences mixing, point by point: inliers at 0.5 px and at 0 px, outliers, points behind
    camera 2 (d1 < 0) and behind camera 1 (d2 < 0); with `huge`, outliers whose r^2 / t^2 reaches 1e120.  Returns
    x1, x2, d1, d2, the ground-truth model and a loss scale of 2 px."""
    f2 = 900.0 if v == 3 else 800.0
    kw = dict(f1=700.0 if v == 3 else 800.0, f2=f2, outlier_ratio=0.0, sigma_px=0.0,
              shift1=0.3 if v == 1 else 0.0, shift2=-0.2 if v == 1 else 0.0)
    sc = synth.make_scene(seed, max(n, 1), **kw)
    rng = np.random.default_rng(seed + 77)
    cat = rng.choice(6, size=max(n, 1), p=[0.55, 0.15, 0.1, 0.07, 0.07, 0.06])
    if inliers_only:
        cat[:] = 0
    x1, x2, d1, d2 = sc.x1.copy(), sc.x2.copy(), sc.d1.copy(), sc.d2.copy()
    k = cat == 0
    x1[k] += 0.5 * rng.normal(size=(k.sum(), 2))
    x2[k] += 0.5 * rng.normal(size=(k.sum(), 2))
    k = cat == 2
    x2[k] = rng.uniform(0, 1000, size=(k.sum(), 2))
    d1[cat == 3] = -d1[cat == 3] - 1.0
    d2[cat == 4] = -d2[cat == 4] - 1.0
    k = cat == 5
    x2[k] += (10.0 ** rng.uniform(0, 57 if huge else 3, size=k.sum()))[:, None] * rng.normal(size=(k.sum(), 2))
    if v in (0, 1):
        x1, x2, ns = (x1 - synth.PP) / sc.f1, (x2 - synth.PP) / sc.f2, 1.0
    else:
        x1, x2 = x1 - synth.PP, x2 - synth.PP
        ns = 1.6 * 400.0
        x1, x2 = x1 / ns, x2 / ns
    m = gt_model(sc, v, ns)
    t = 2.0 / (sc.f1 if v in (0, 1) else ns)
    return x1[:n], x2[:n], d1[:n], d2[:n], m, t


def perturb(m, v, rng, rot_deg=0.5, dt=0.02, ds=0.03, dsh=0.05, df=0.02):
    from scipy.spatial.transform import Rotation as Rot
    a = rng.normal(size=3)
    a *= np.deg2rad(rot_deg) / np.linalg.norm(a)
    q = Rot.from_quat([m[1], m[2], m[3], m[0]]) * Rot.from_rotvec(a)
    qq = q.as_quat()
    o = m.copy()
    o[:4] = [qq[3], qq[0], qq[1], qq[2]]
    o[4:7] = m[4:7] * (1 + dt * rng.normal(size=3))
    o[7] = m[7] * (1 + ds * rng.normal())
    if v == 1:
        o[8:10] = m[8:10] + dsh * rng.normal(size=2)
    if v in (2, 3):
        o[10] = m[10] * (1 + df * rng.normal())
        o[11] = o[10] if v == 2 else m[11] * (1 + df * rng.normal())
    return o


# ---------------------------------------------------------------------------------------------------------------------
# reference self-check (CPU)

def test_longdouble_has_extended_mantissa():
    assert np.finfo(np.longdouble).nmant >= 63


@pytest.mark.parametrize("v", VARIANTS)
def test_reference_against_mpmath(v):
    """Terms and complex-step Jacobian of the longdouble reference against mpmath at 40 digits, with the
    derivatives taken independently by mpmath's numerical differentiation."""
    import mpmath as mp
    mp.mp.dps = 40
    x1, x2, d1, d2, m, t = make_data(v, 40, 5 + v)
    idx = [i for i in range(40) if d1[i] > 0 and d2[i] > 0][:4]
    m = perturb(m, v, np.random.default_rng(v))
    pb = Problem(v, x1[idx], x2[idx], d1[idx], d2[idx], 0.37, SR, CAUCHY, t)
    rows = pb.rows(m)
    ob = lambda a: np.array([mp.mpf(float(z)) for z in np.ravel(a)], dtype=object).reshape(np.shape(a))

    def mres(dp):
        rs, r12, r21 = residuals(v, ob(m), ob(x1[idx]), ob(x2[idx]), ob(d1[idx]), ob(d2[idx]), dp, sqrt=np.vectorize(mp.sqrt, otypes=[object]))[:3]
        return [rs[:, None], r12, r21]

    z = np.array([mp.mpf(0)] * pb.np, dtype=object)
    base = mres(z)
    by_name = {"s": 0, "12": 1, "21": 2}
    for name, fac, r2, gate, warg, rwf, r, J, sc in rows:
        k = by_name[name]
        for i in range(len(idx)):
            for c in range(r.shape[1]):
                # two orders of magnitude below the FP64 rounding of the same residual
                assert abs(float(LD(str(base[k][i, c])) - r[i, c])) <= 1e-18 * float(sc[i])
        for p in range(pb.np):
            def f(h, p=p, k=k):
                dp = z.copy()
                dp[p] = h
                return mres(dp)[k]
            # first order in the rotation: d/dh of R (I + h [e_p]x) at h = 0
            for i in range(len(idx)):
                for c in range(r.shape[1]):
                    d = mp.diff(lambda h: f(h)[i, c], 0)
                    assert abs(float(LD(str(d)) - J[i, c, p])) <= 1e-17 * max(1.0, abs(float(d)))


@pytest.mark.parametrize("v", VARIANTS)
@pytest.mark.parametrize("ws", [1.0, 0.5])
def test_reference_normal_equations_equal_oracle(port, v, ws):
    """The reference's A, g and cost agree with the C oracle (independent code, same quirks) to FP64 rounding; at
    weight_sampson = 1 with the TRIVIAL loss, g is half the gradient of the cost."""
    x1, x2, d1, d2, m, t = make_data(v, 300, 11 + v)
    m = perturb(m, v, np.random.default_rng(3))
    for loss in LOSSES:
        pb = Problem(v, x1, x2, d1, d2, ws, SR, loss, t)
        A, g = pb.normal(m)
        om = port.make_model(m[:4], m[4:7], *m[7:])
        JtJ, Jtr = port.accumulate(v, x1, x2, d1, d2, om, SR, ws, LOSS_NAMES[loss], t)
        n = pb.np
        Af = np.asarray(A, dtype=np.float64)
        assert np.abs(JtJ[:n, :n] - Af).max() <= 1e-9 * np.abs(Af).max()
        assert np.abs(Jtr[:n] - np.asarray(g, dtype=np.float64)).max() <= 1e-9 * np.abs(np.asarray(g, dtype=np.float64)).max()
        c, cabs, _, _ = pb.cost(m)
        oc = port.cost(v, x1, x2, d1, d2, om, SR, ws, LOSS_NAMES[loss], t)
        assert abs(float(c) - oc) <= 1e-12 * float(cabs)
    if ws == 1.0:
        pb = Problem(v, x1, x2, d1, d2, ws, SR, TRIVIAL, t)
        _, g = pb.normal(m)
        for p in range(pb.np):
            h = 1e-7
            dp = np.zeros(pb.np)
            dp[p] = h
            num = (pb.cost(model_step(v, m, dp))[0] - pb.cost(model_step(v, m, -dp))[0]) / (2 * h)
            assert abs(float(num) / 2 - float(g[p])) <= 1e-6 * float(np.abs(g).max())


# ---------------------------------------------------------------------------------------------------------------------
# device side

def _newer_than(path, sources):
    return os.path.exists(path) and os.path.getmtime(path) >= max(os.path.getmtime(f) for f in sources)


@pytest.fixture(scope="module")
def lmc():
    """tests/lmcheck/liblmcheck.so: the harness and the product's repose_lm.cu, built with the product's flags."""
    from mdrp_b200 import build as b
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [LMC_SRC]
    if not _newer_than(LMC_SO, srcs):
        extra = dict(b.SOURCES)["repose_lm.cu"]
        subprocess.check_call([os.environ.get("NVCC", "nvcc")] + b.NVCC_FLAGS + extra +
                              ["-shared", "-o", LMC_SO, LMC_SRC, os.path.join(CSRC, "repose_lm.cu")])
    L = C.CDLL(LMC_SO)
    L.lmc_run.restype = C.c_int
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def run_harness(lmc, v, pairs, models, *, ws, prob_list=None, prob_per_pair=1, enable=None, mask=None, warp=0, single=0,
                use_final=0, max_it=25, loss=TRUNCATED, gtol=0.0, stol=0.0, lam=1e-3, lmin=1e-10, lmax=1e10,
                loss_override=-1.0, sr_override=-1.0, stats=None):
    """pairs: list of (x1, x2, d1, d2, scale_reproj, lo_loss_scale, valid); returns models and stats."""
    from mdrp_b200 import _native as nv
    off = np.cumsum([0] + [len(p[2]) for p in pairs[:-1]]).astype(np.int64)
    cnt = np.array([len(p[2]) for p in pairs], dtype=np.int32)
    pts = np.ascontiguousarray(np.concatenate([np.c_[p[0], p[1]].reshape(-1, 4) for p in pairs] + [np.zeros((0, 4))]), dtype=np.float64)
    d1 = np.ascontiguousarray(np.concatenate([p[2] for p in pairs] + [np.zeros(0)]), dtype=np.float64)
    d2 = np.ascontiguousarray(np.concatenate([p[3] for p in pairs] + [np.zeros(0)]), dtype=np.float64)
    valid = np.array([p[6] for p in pairs], dtype=np.int32)
    srs = np.array([p[4] for p in pairs], dtype=np.float64)
    lts = np.array([p[5] for p in pairs], dtype=np.float64)
    mo = np.zeros(len(models), dtype=nv.MODEL_DTYPE)
    mv = np.asarray(models, dtype=np.float64).reshape(-1, 12)
    mo["q"], mo["t"], mo["scale"], mo["shift1"], mo["shift2"], mo["f1"], mo["f2"] = (
        mv[:, :4], mv[:, 4:7], mv[:, 7], mv[:, 8], mv[:, 9], mv[:, 10], mv[:, 11])
    st = np.zeros(len(models), dtype=nv.BSTATS_DTYPE) if stats is None else stats.copy()
    pl = None if prob_list is None else np.ascontiguousarray(prob_list, dtype=np.int32)
    n_prob = len(models) if pl is None else len(pl)
    en = None if enable is None else np.ascontiguousarray(enable, dtype=np.int32)
    mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
    iopt = np.array([use_final, warp, single, max_it, loss, prob_per_pair], dtype=np.int32)
    dopt = np.array([ws, gtol, stol, lam, lmin, lmax, loss_override, sr_override], dtype=np.float64)
    err = lmc.lmc_run(v, len(pairs), _ptr(off), _ptr(cnt), _ptr(valid), _ptr(srs), _ptr(lts), _ptr(lts), C.c_longlong(len(d1)),
                      _ptr(pts), _ptr(d1), _ptr(d2), _ptr(mk), _ptr(en), n_prob, _ptr(pl), len(models), _ptr(mo), _ptr(st),
                      _ptr(iopt), _ptr(dopt))
    assert err == 0, f"CUDA error {err}"
    return mo, st


def mvec(m):
    return np.r_[m["q"], m["t"], m["scale"], m["shift1"], m["shift2"], m["f1"], m["f2"]].astype(np.float64)


def refine_final(ctx, v, x1, x2, d1, d2, models, ws, sr, loss, t, mask=None, **kw):
    from mdrp_b200 import _native as nv
    from util import struct_models
    bo = nv.bundle_options(loss_type=loss, loss_scale=t, **kw)
    return ctx.refine(v, struct_models(np.asarray(models).reshape(-1, 12)), x1, x2, d1, d2, sr, ws, bo, mask=mask)


LO_KERNELS = [pytest.param(dict(warp=1, single=1), id="warp"), pytest.param(dict(warp=0), id="block")]


def _assert_cost(dev, ref, cabs, allow, what):
    ref, cabs, allow = float(ref), float(cabs), float(allow)
    assert np.isnan(dev) == np.isnan(ref), what
    if not np.isnan(ref):
        assert abs(dev - ref) <= COST_RTOL * cabs + allow, (what, dev, ref, (dev - ref) / max(cabs, 1e-300))


# (a) cost of every kernel and loss ----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("v", VARIANTS)
def test_cost_final_kernels(ctx, v, loss):
    """rp_refine_batch with max_iterations = 0 reports the cost of the start model as cost and initial_cost."""
    x1, x2, d1, d2, m, t = make_data(v, max(SIZES), 100 + v, huge=loss in (TRUNCATED, CAUCHY, TRUNCATED_CAUCHY))
    starts = [m, perturb(m, v, np.random.default_rng(v))]
    for ws, sr in TERM_COMBOS:
        pb = Problem(v, x1, x2, d1, d2, ws, sr, loss, t)
        pcs = [[np.r_[LD(0), np.cumsum(a)] for a in pb.point_costs(s)[:3]] for s in starts]
        for n in SIZES:
            _, st = refine_final(ctx, v, x1[:n], x2[:n], d1[:n], d2[:n], starts, ws, sr, LOSS_NAMES[loss], t, max_iterations=0)
            for k, (c, a, al) in enumerate(pcs):
                assert st[k]["iterations"] == 0
                assert st[k]["cost"] == st[k]["initial_cost"] or np.isnan(st[k]["cost"])
                _assert_cost(st[k]["cost"], c[n], a[n], al[n], (ws, sr, n, k))


@pytest.mark.gpu
@pytest.mark.parametrize("kern", LO_KERNELS)
@pytest.mark.parametrize("v", VARIANTS)
def test_cost_lo_kernels(lmc, v, kern):
    """The LO kernels' initial_cost (TRUNCATED at lo_loss_scale); one pair per size in one launch."""
    x1, x2, d1, d2, m, t = make_data(v, max(SIZES), 200 + v, huge=True)
    for ws, sr in TERM_COMBOS:
        pb = Problem(v, x1, x2, d1, d2, ws, sr, TRUNCATED, t)
        c, a, al = (np.r_[LD(0), np.cumsum(z)] for z in pb.point_costs(m)[:3])
        pairs = [(x1[:n], x2[:n], d1[:n], d2[:n], sr, t, 1) for n in SIZES]
        _, st = run_harness(lmc, v, pairs, [m] * len(SIZES), ws=ws, gtol=np.inf, **kern)
        for k, n in enumerate(SIZES):
            assert st[k]["iterations"] == 0
            _assert_cost(st[k]["initial_cost"], c[n], a[n], al[n], (ws, sr, n))


@pytest.mark.gpu
@pytest.mark.parametrize("loss", [CAUCHY, TRUNCATED_CAUCHY])
@pytest.mark.parametrize("v", VARIANTS)
def test_cauchy_cost_small_residuals(ctx, v, loss):
    """Inliers only, loss scales from 1 to 1e8 times the residuals: r^2 / t^2 runs from ~1e-1 down to ~1e-17, where a
    cost accumulated as a running product of (1 + x) loses every term below an ulp of the product."""
    x1, x2, d1, d2, m, t = make_data(v, 3000, 300 + v, inliers_only=True)
    for ts in (1.0, 1e2, 1e4, 1e6, 1e8):
        for ws, sr in ((1.0, SR), (1.0, 0.0), (0.0, SR)):
            pb = Problem(v, x1, x2, d1, d2, ws, sr, loss, t * ts)
            c, a, al, _ = pb.cost(m)
            _, st = refine_final(ctx, v, x1, x2, d1, d2, [m], ws, sr, LOSS_NAMES[loss], t * ts, max_iterations=0)
            _assert_cost(st[0]["cost"], c, a, al, (ts, ws, sr))


@pytest.mark.gpu
@pytest.mark.parametrize("v", VARIANTS)
def test_cost_nan_inputs(ctx, lmc, v):
    """A NaN depth removes the reprojection it gates on both sides; a NaN keypoint makes both costs NaN."""
    x1, x2, d1, d2, m, t = make_data(v, 200, 400 + v)
    for loss in LOSSES:
        for what in ("depth", "keypoint"):
            y1, e1 = x1.copy(), d1.copy()
            if what == "depth":
                e1[17] = np.nan
            else:
                y1[17, 0] = np.nan
            pb = Problem(v, y1, x2, e1, d2, 1.0, SR, loss, t)
            c, a, al, _ = pb.cost(m)
            assert np.isnan(float(c)) == (what == "keypoint")
            _, st = refine_final(ctx, v, y1, x2, e1, d2, [m], 1.0, SR, LOSS_NAMES[loss], t, max_iterations=0)
            _assert_cost(st[0]["cost"], c, a, al, (loss, what))
            if loss == TRUNCATED:
                for kern in ({"warp": 1, "single": 1}, {"warp": 0}):
                    _, sl = run_harness(lmc, v, [(y1, x2, e1, d2, SR, t, 1)], [m], ws=1.0, gtol=np.inf, **kern)
                    _assert_cost(sl[0]["initial_cost"], c, a, al, ("lo", what, kern))


# (b) normal equations through one step ------------------------------------------------------------------------------

LAMBDA_FACTORS = (1e-3, 1.0, 1e3, 1e12)


def _one_step_reference(pb, m0, lam):
    A, g = pb.normal(m0)
    x = lm_step(A, g, lam)
    m1 = model_step(pb.v, m0, x)
    c0, a0, _, _ = pb.cost(m0)
    c1, a1, _, tm1 = pb.cost(m1)
    margin = min(float(abs(c1 - c0) / max(a0, a1)), float(tm1), float(pb.cost(m0)[3]))
    return A, g, x, m1, bool(c1 < c0), margin


def _check_recovered_step(pb, m0, lam, A, g, dev_model):
    """The step recovered from the returned model solves the reference's damped normal equations."""
    xd = step_from_models(pb.v, m0, dev_model)
    M = A + LD(lam) * np.eye(pb.np, dtype=LD)
    nM = np.linalg.norm(np.asarray(M, dtype=np.float64), 2)
    gn = float(np.sqrt((g * g).sum()))
    # the returned model is rounded to FP64: a step below that resolution is not recoverable from it
    dx = 4 * U * (np.abs(np.asarray(m0, dtype=np.float64)) + 1).max()
    res = np.linalg.norm(np.asarray(M @ xd + g, dtype=np.float64))
    assert res <= 1e-10 * (nM * float(np.sqrt((xd * xd).sum())) + gn) + nM * dx * np.sqrt(pb.np), (res, gn)


def _check_step(pb, m0, lam, A, g, x, accept, dev_model, st):
    """grad_norm, step_norm, accept decision (None: not decided by the reference) and the step taken."""
    gn, sn = float(np.sqrt((g * g).sum())), float(np.sqrt((x * x).sum()))
    assert abs(st["grad_norm"] - gn) <= 1e-9 * gn, (st["grad_norm"], gn)
    assert abs(st["step_norm"] - sn) <= 1e-8 * sn, (st["step_norm"], sn)
    if accept is None:          # accept margin below MARGIN: either decision is admissible
        return
    assert st["invalid_steps"] == (0 if accept else 1)
    if accept:
        _check_recovered_step(pb, m0, lam, A, g, dev_model)
    else:
        assert np.array_equal(dev_model, np.asarray(m0, dtype=np.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("v", VARIANTS)
def test_one_step_final_kernels(ctx, v, loss):
    x1, x2, d1, d2, m, t = make_data(v, 1000, 500 + v)
    checked = total = 0
    for ws in (1.0, 0.37):
        pb = Problem(v, x1, x2, d1, d2, ws, SR, loss, t)
        for seed in range(2):
            m0 = perturb(m, v, np.random.default_rng(10 * v + seed))
            A0, _ = pb.normal(m0)
            for f in LAMBDA_FACTORS:
                lam = f * float(np.trace(np.asarray(A0, dtype=np.float64))) / pb.np
                A, g, x, m1, accept, margin = _one_step_reference(pb, m0, lam)
                out, st = refine_final(ctx, v, x1, x2, d1, d2, [m0], ws, SR, LOSS_NAMES[loss], t, max_iterations=1,
                                       initial_lambda=lam, gradient_tol=0.0, step_tol=0.0)
                _check_step(pb, m0, lam, A, g, x, accept if margin >= MARGIN else None, mvec(out[0]), st[0])
                # at lambda = 1e12 tr(A) / NP the step is ~1e-12 of an undamped one and its cost change is below
                # any FP64 accept test: only grad_norm and step_norm are checked there
                if f < 1e12:
                    total += 1
                    checked += margin >= MARGIN
    assert checked >= 0.9 * total, (checked, total)


@pytest.mark.gpu
@pytest.mark.parametrize("kern", [pytest.param(dict(warp=1, single=1), id="warp_single"),
                                  pytest.param(dict(warp=1, list=True), id="warp_list"),
                                  pytest.param(dict(warp=0), id="block"),
                                  pytest.param(dict(warp=0, list=True), id="block_list")])
@pytest.mark.parametrize("v", VARIANTS)
def test_one_step_lo_kernels(lmc, v, kern):
    """gradient_tol between |g0| and |g1| of the reference (or step_tol between the step norms): one accepted step,
    after any rejected ones, then stop."""
    kern = dict(kern)
    use_list = kern.pop("list", False)
    x1, x2, d1, d2, m, t = make_data(v, 1000, 600 + v)
    checked = total = 0
    for ws in (1.0, 0.37):
        pb = Problem(v, x1, x2, d1, d2, ws, SR, TRUNCATED, t)
        for seed in range(4):
            m0 = perturb(m, v, np.random.default_rng(20 * v + seed))
            A0, _ = pb.normal(m0)
            for f in LAMBDA_FACTORS:
                lam = f * float(np.trace(np.asarray(A0, dtype=np.float64))) / pb.np
                if f < 1e12:
                    total += 1
                r = lm_run(pb, m0, 25, 0.0, 0.0, lam, 1e-10, 1e10)
                # stop right after the first accepted step: by gradient_tol when |g1| < |g0|, else by step_tol when
                # the step after it is shorter than every step before
                ref = None
                if len(r["hist"]) > 1 and r["hist"][1][1] < r["hist"][0][1]:
                    gtol, stol = float(np.sqrt(r["hist"][0][1] * r["hist"][1][1])), 0.0
                    ref = lm_run(pb, m0, 25, gtol, stol, lam, 1e-10, 1e10)
                elif len(r["hist"]) > 1:
                    it1 = r["hist"][1][0]
                    before = [h[1] for h in r["shist"] if h[0] < it1]
                    after = [h[1] for h in r["shist"] if h[0] == it1]
                    if after and after[0] < min(before):
                        gtol, stol = 0.0, float(np.sqrt(after[0] * min(before)))
                        ref = lm_run(pb, m0, 25, gtol, stol, lam, 1e-10, 1e10)
                if ref is None or ref["margin"] < MARGIN or ref["accepted"] != 1:
                    continue
                out, st = run_harness(lmc, v, [(x1, x2, d1, d2, SR, t, 1)], [m0], ws=ws, gtol=gtol, stol=stol, lam=lam,
                                      prob_list=[0] if use_list else None, **kern)
                st = st[0]
                lam_acc = lam
                for _ in range(ref["invalid_steps"]):
                    lam_acc = min(1e10, lam_acc * 10)
                A, g = pb.normal(m0)
                _check_recovered_step(pb, m0, lam_acc, A, g, mvec(out[0]))
                assert st["iterations"] == ref["iterations"] and st["invalid_steps"] == ref["invalid_steps"]
                assert st["lam"] == ref["lam"]
                assert abs(st["grad_norm"] - ref["grad_norm"]) <= 1e-9 * ref["grad_norm"]
                assert abs(st["step_norm"] - ref["step_norm"]) <= 1e-8 * ref["step_norm"]
                checked += f < 1e12
    # the first TRUNCATED step moves residuals across the threshold, so |g| and |step| need not fall after it: up to
    # about half of the starts cannot be stopped after exactly one step by either tolerance
    assert checked >= max(6, 0.4 * total), (checked, total)


# (c) full runs -------------------------------------------------------------------------------------------------------

def _decisive_gtol(r):
    """A gradient_tol that ends the reference run at its last gradient check that every earlier decision clears by
    MARGIN and whose |g| is below every earlier one (a converged run ends in accept tests closer than any FP64
    evaluation resolves); None when there is none."""
    best = None
    for i, (it, gn, mg) in enumerate(r["hist"]):
        if mg < MARGIN:
            break
        if i > 0:
            prev = min(h[1] for h in r["hist"][:i])
            if gn < prev:
                best = float(np.sqrt(gn * prev))
    return best


def _compare_run(ref, st, model):
    assert st["iterations"] == ref["iterations"] and st["invalid_steps"] == ref["invalid_steps"], (st, ref["iterations"])
    assert st["lam"] == ref["lam"]
    mr = np.asarray(ref["model"], dtype=np.float64)
    md = np.where(np.dot(model[:4], mr[:4]) < 0, -1, 1) * np.r_[np.ones(4), np.zeros(8)] * model + np.r_[np.zeros(4), np.ones(8)] * model
    assert np.all(np.abs(md - mr) <= 1e-9 * np.maximum(np.abs(mr), 1)), (md - mr)


DEFAULT_BUNDLE = dict(max_it=100, stol=1e-8, lam=1e-3, lmin=1e-10, lmax=1e10)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("v", VARIANTS)
def test_full_runs_final_kernels(ctx, v, loss):
    x1, x2, d1, d2, m, t = make_data(v, 300, 700 + v)
    compared = total = 0
    for ws in (1.0, 0.37):
        for seed in range(3):
            m0 = perturb(m, v, np.random.default_rng(30 * v + seed))
            pb = Problem(v, x1, x2, d1, d2, ws, SR, loss, t)
            o = DEFAULT_BUNDLE
            total += 1
            gtol = _decisive_gtol(lm_run(pb, m0, o["max_it"], 0.0, o["stol"], o["lam"], o["lmin"], o["lmax"]))
            if gtol is None:
                continue
            ref = lm_run(pb, m0, o["max_it"], gtol, o["stol"], o["lam"], o["lmin"], o["lmax"])
            if ref["margin"] < MARGIN:
                continue
            out, st = refine_final(ctx, v, x1, x2, d1, d2, [m0], ws, SR, LOSS_NAMES[loss], t, gradient_tol=gtol)
            _compare_run(ref, st[0], mvec(out[0]))
            _, cabs, allow, _ = pb.cost(ref["model"])
            _assert_cost(st[0]["cost"], ref["cost"], cabs, allow, "final cost")
            compared += 1
    assert compared >= 0.9 * total, (compared, total)


@pytest.mark.gpu
@pytest.mark.parametrize("kern", LO_KERNELS)
@pytest.mark.parametrize("v", VARIANTS)
def test_full_runs_lo_kernels(lmc, v, kern):
    x1, x2, d1, d2, m, t = make_data(v, 300, 800 + v)
    compared = total = 0
    for ws in (1.0, 0.37):
        for seed in range(3):
            m0 = perturb(m, v, np.random.default_rng(40 * v + seed))
            pb = Problem(v, x1, x2, d1, d2, ws, SR, TRUNCATED, t)
            total += 1
            gtol = _decisive_gtol(lm_run(pb, m0, 25, 0.0, 0.0, 1e-3, 1e-10, 1e10))
            if gtol is None:
                continue
            ref = lm_run(pb, m0, 25, gtol, 0.0, 1e-3, 1e-10, 1e10)
            if ref["margin"] < MARGIN:
                continue
            out, st = run_harness(lmc, v, [(x1, x2, d1, d2, SR, t, 1)], [m0], ws=ws, gtol=gtol, **kern)
            _compare_run(ref, st[0], mvec(out[0]))
            _, cabs, allow, _ = pb.cost(ref["model"])
            _assert_cost(st[0]["cost"], ref["cost"], cabs, allow, "LO cost")
            compared += 1
    assert compared >= 0.9 * total, (compared, total)


# (d) masks and scheduling --------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n", [16384, 16385, 40000])
@pytest.mark.parametrize("v", [1, 3])
def test_mask_equals_subset(ctx, v, n):
    """Masked problems: the compacted inlier list (n <= 16384) and the mask read on the fly (n > 16384) both equal
    the reference on the subset."""
    x1, x2, d1, d2, m, t = make_data(v, n, 900 + v)
    mask = np.random.default_rng(n).random(n) < 0.7
    for loss in (TRUNCATED_CAUCHY, HUBER):
        pb = Problem(v, x1[mask], x2[mask], d1[mask], d2[mask], 1.0, SR, loss, t)
        m0 = perturb(m, v, np.random.default_rng(v))
        c, cabs, allow, _ = pb.cost(m0)
        _, st = refine_final(ctx, v, x1, x2, d1, d2, [m0], 1.0, SR, LOSS_NAMES[loss], t, mask=mask.astype(np.uint8),
                             max_iterations=0)
        _assert_cost(st[0]["cost"], c, cabs, allow, "masked cost")
        A0, _ = pb.normal(m0)
        lam = 1e-3 * float(np.trace(np.asarray(A0, dtype=np.float64))) / pb.np
        A, g, x, m1, accept, margin = _one_step_reference(pb, m0, lam)
        assert margin >= MARGIN
        out, st = refine_final(ctx, v, x1, x2, d1, d2, [m0], 1.0, SR, LOSS_NAMES[loss], t, mask=mask.astype(np.uint8),
                               max_iterations=1, initial_lambda=lam, gradient_tol=0.0, step_tol=0.0)
        _check_step(pb, m0, lam, A, g, x, accept, mvec(out[0]), st[0])
    # an empty subset: nothing to refine, zero cost, the model comes back unchanged
    m0 = perturb(m, v, np.random.default_rng(v))
    out, st = refine_final(ctx, v, x1, x2, d1, d2, [m0], 1.0, SR, "CAUCHY", t, mask=np.zeros(n, np.uint8))
    assert np.array_equal(mvec(out[0]), m0)
    assert st[0]["cost"] == 0.0 and st[0]["initial_cost"] == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("kern", LO_KERNELS)
def test_problem_scheduling(lmc, kern):
    """Several pairs, three problems per pair, a permuted problem list; pairs switched off by `enable` or `valid`
    leave their models and stats (sentinels) untouched, and every problem returns the bytes it returns alone."""
    v = 1
    sizes = [300, 0, 57, 1000, 129, 40]
    pairs, models = [], []
    for p, n in enumerate(sizes):
        x1, x2, d1, d2, m, t = make_data(v, n, 1000 + p)
        pairs.append((x1, x2, d1, d2, SR, t, 0 if p == 2 else 1))
        models += [perturb(m, v, np.random.default_rng(50 + 3 * p + k)) for k in range(3)]
    enable = [1, 0, 1, 1, 0, 1]
    from mdrp_b200 import _native as nv
    sentinel = np.zeros(len(models), dtype=nv.BSTATS_DTYPE)
    for f in sentinel.dtype.names:
        sentinel[f] = -7
    plist = np.random.default_rng(1).permutation(len(models))
    out, st = run_harness(lmc, v, pairs, models, ws=1.0, prob_list=plist, prob_per_pair=3, enable=enable, gtol=1e-12,
                          stats=sentinel, **kern)
    for p in range(len(models)):
        pair = p // 3
        if not enable[pair] or not pairs[pair][6]:
            assert np.array_equal(mvec(out[p]), models[p])
            assert st[p].tobytes() == sentinel[p].tobytes()
            continue
        assert st[p]["iterations"] > 0 or sizes[pair] == 0
        o1, s1 = run_harness(lmc, v, pairs, models, ws=1.0, prob_list=[p], prob_per_pair=3, enable=enable, gtol=1e-12,
                             stats=sentinel, **kern)
        assert o1[p].tobytes() == out[p].tobytes() and s1[p].tobytes() == st[p].tobytes(), p


# (e) threshold edges -------------------------------------------------------------------------------------------------

def _edge_cases(v, loss):
    """(problem, the residual's x, first-order g and cost with the residual inside and outside the threshold)."""
    x1, x2, d1, d2, m, t = make_data(v, 40, 1100 + v, inliers_only=True)
    for ws, sr in ((1.0, 0.0), (0.0, SR)):
        for i in range(3):
            sl = slice(i, i + 1)
            pb = Problem(v, x1[sl], x2[sl], d1[sl], d2[sl], ws, sr, loss, t)
            r2 = pb.rows(m, jac=False)[0][2][0]           # Sampson r^2, or the 1->2 reprojection's s_r |r|^2
            yield pb, m, x1[sl], x2[sl], d1[sl], d2[sl], ws, sr, r2


def _grad_cost(pb, m):
    A, g = pb.normal(m)
    c, cabs, allow, marg = pb.cost(m)
    return float(np.sqrt((g * g).sum())), float(c), float(allow), float(marg)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", THRESHOLD_LOSSES)
@pytest.mark.parametrize("v", VARIANTS)
def test_threshold_edges(ctx, lmc, v, loss):
    """Residuals at t (1 +- 1e-9) land on the reference's side; within a few ulps of t either side is accepted (the
    kernels decide on r^2 (1 / t^2) > 1 or r^2 < t^2, the oracle on r^2 > t^2), but nothing in between."""
    def device(m, x1, x2, d1, d2, ws, sr, t):
        out = []
        _, st = refine_final(ctx, v, x1, x2, d1, d2, [m], ws, sr, LOSS_NAMES[loss], t, max_iterations=1,
                             gradient_tol=np.inf)
        out.append((st[0]["grad_norm"], st[0]["initial_cost"]))
        if loss == TRUNCATED:
            for kern in ({"warp": 1, "single": 1}, {"warp": 0}):
                _, sl = run_harness(lmc, v, [(x1, x2, d1, d2, sr, t, 1)], [m], ws=ws, gtol=np.inf, **kern)
                out.append((sl[0]["grad_norm"], sl[0]["initial_cost"]))
        return out

    def matches(dev, ref):
        return abs(dev[0] - ref[0]) <= 1e-11 * ref[0] and abs(dev[1] - ref[1]) <= 1e-12 * abs(ref[1]) + ref[2]

    for pb, m, x1, x2, d1, d2, ws, sr, r2 in _edge_cases(v, loss):
        r = float(np.sqrt(r2))
        for f in (1 - 1e-9, 1 + 1e-9):
            t = r / f                                   # x = r^2 / t^2 = f^2
            pbt = Problem(v, x1, x2, d1, d2, ws, sr, loss, t)
            ref = _grad_cost(pbt, m)
            if ref[3] < 1e-10:
                continue
            for dev in device(m, x1, x2, d1, d2, ws, sr, t):
                assert matches(dev, ref[:3]), (f, dev, ref)
        # the two admissible outcomes: the reference at a loss scale just inside / outside the residual
        sides = [_grad_cost(Problem(v, x1, x2, d1, d2, ws, sr, loss, r * (1 + s * 1e-13)), m) for s in (-1, 1)]
        sides = [s[:3] for s in sides]
        for k in range(-4, 5):
            t = r * (1 + k * U)
            for dev in device(m, x1, x2, d1, d2, ws, sr, t):
                assert any(matches(dev, s) for s in sides), (k, dev, sides)
