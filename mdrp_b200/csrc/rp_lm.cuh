// rp_lm.cuh — residuals and Jacobians of the hybrid monodepth refinement.
//
//   L2  refine_monodepth_relpose so@0x261030 (7 params, 9 with shifts),
//       refine_monodepth_shared_focal_relpose so@0x2592e0 (8), …_varying_focal_… so@0x260fa0 (9)
//       = lm_impl<MonoDepth*JacobianAccumulator<Loss,Weights>> of PoseLib bundle.cc/jacobian_impl.h
//
// cost = sum_k  w_s rho(r_s^2) + rho(s_r |pi(R (d1+u) p1 + t) - x2|^2)[z>0]
//                              + rho(s_r |pi(R^T (sigma (d2+v) p2 - t)) - x1|^2)[z>0]
// with p_i = K_i^-1 (x_i, 1) and r_s the Sampson residual of F = K2^-T [t]x R K1^-1.
// Parameter order: rotation tangent w (R <- R exp([w]x)), t, scale, then (shift1, shift2) | f | (f1, f2).
// SURVEY.md §8a rows L1/L2.  One residual row at a time is pushed into a packed lower-triangular
// J^T J held in registers (explicit FMAs: this path is not bit-pinned, the oracle comparison is
// cost <= oracle*(1+1e-9) and pose within 1e-6).
#pragma once
#include "rp_common.cuh"

namespace rp {

RP_HD double loss_eval(int type, double thr, double r2) {
    const double t2 = thr * thr;
    switch (type) {
    case RP_LOSS_TRIVIAL: return r2;
    case RP_LOSS_TRUNCATED: return t2 < r2 ? t2 : r2;  // std::min(r2, t2) of the reference: a NaN residual stays NaN
    case RP_LOSS_HUBER: { const double r = sqrt(r2); return r <= thr ? r2 : thr * (2.0 * r - thr); }
    case RP_LOSS_CAUCHY: return t2 * log1p(r2 / t2);
    case RP_LOSS_TRUNCATED_CAUCHY: return r2 > t2 ? t2 * log1p(1.0) : t2 * log1p(r2 / t2);
    default: return r2 < t2 ? r2 : t2;
    }
}
RP_HD double loss_weight(int type, double thr, double r2) {
    const double t2 = thr * thr;
    switch (type) {
    case RP_LOSS_TRIVIAL: return 1.0;
    case RP_LOSS_TRUNCATED: return r2 < t2 ? 1.0 : 0.0;
    case RP_LOSS_HUBER: { const double r = sqrt(r2); return r <= thr ? 1.0 : thr / r; }
    case RP_LOSS_CAUCHY: return 1.0 / (1.0 + r2 / t2);
    case RP_LOSS_TRUNCATED_CAUCHY: return r2 > t2 ? 0.0 : 1.0 / (1.0 + r2 / t2);
    default: return r2 < t2 ? 1.0 : 0.0;
    }
}

// 1/x and 1/sqrt(x) for the point loop of the LM kernel.  The IEEE division / sqrt+division sequences cost
// ~15 / ~35 instructions with a slow-path branch each; on the device these use the hardware approximations
// refined by Newton steps (<= 1-2 ulp, this path is not bit-pinned).  Arguments are positive and normal here
// (projective depths behind `z > 0`, Sampson denominators); anything else falls back to the exact sequence.
RP_HD double lm_rcp(double x) {
#ifdef __CUDA_ARCH__
    if (!(x > 1e-300 && x < 1e300)) return 1.0 / x;  // (never taken on sane data: a real branch, not a select)
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    y = ::fma(::fma(-x, y, 1.0), y, y);
    y = ::fma(::fma(-x, y, 1.0), y, y);
    return y;
#else
    return 1.0 / x;
#endif
}
RP_HD double lm_rsqrt(double x) {
#ifdef __CUDA_ARCH__
    if (!(x > 1e-300 && x < 1e300)) return 1.0 / sqrt(x);
    return rsqrt(x);
#else
    return 1.0 / sqrt(x);
#endif
}

struct LMParams {
    double scale_reproj, weight_sampson, loss_scale;
    double inv_t2;      // 1 / loss_scale^2
    int loss_type;
};

// Cost of the Cauchy losses, sum_k t^2 log1p(r_k^2 / t^2), accumulated as t^2 log1p(q) with q = prod_k (1 + r_k^2 / t^2) - 1:
// one FMA and one add per residual instead of a 45-instruction FP64 log1p (the final refinement evaluates three of them
// per correspondence per pass).  Carrying q rather than the product itself keeps residuals far below an ulp of 1
// (near-exact data, r^2 / t^2 down to 1e-20 and less) at full relative accuracy: q <- (1 + q)(1 + x) - 1 = fma(q, x, q + x).
// Two running values (the Sampson terms carry weight_sampson), folded into `acc` every 512 factors (TRUNCATED_CAUCHY:
// factors <= 2, so the product stays below 2^512) or when q passes 1e150 (CAUCHY).
// log1p(q), q >= 0, from log: log(u) with u = 1 + q, plus the first-order correction (q - (u - 1)) / u for the rounding
// of u (the numerator is exact and at most half an ulp of u, so a rough reciprocal suffices), within a few ulps.  The
// library log1p, inlined at every fold, would add ~1 800 instructions to each Cauchy kernel, and the final-refinement
// launch is sensitive to instruction fetch.
RP_HD double log1p_q(double q) {
    const double u = 1.0 + q;
#ifdef __CUDA_ARCH__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(u));
#else
    const double r = 1.0 / u;
#endif
    return log(u) + (q - (u - 1.0)) * r;
}
struct LogProd {
    double qs, qr, acc;
    int cnt;
    RP_HD void init() { qs = 0.0; qr = 0.0; acc = 0.0; cnt = 0; }
    RP_HD void fold(double ws) { acc += ws * log1p_q(qs) + log1p_q(qr); qs = 0.0; qr = 0.0; cnt = 0; }
    // the accumulated cost, in units of t^2
    RP_HD double total(double ws) const { return acc + ws * log1p_q(qs) + log1p_q(qr); }
    template <bool SAMPSON>
    RP_HD void add(int type, double x, double ws) {
        if (type == RP_LOSS_TRUNCATED_CAUCHY) x = x > 1.0 ? 1.0 : x;   // (a NaN residual stays NaN, as in loss_eval)
        else if (!(x < 1e100)) { acc += (SAMPSON ? ws : 1.0) * log1p(x); return; }
        if (SAMPSON) qs = fma_(qs, x, qs + x); else qr = fma_(qr, x, qr + x);
        if (++cnt >= 512 || (type == RP_LOSS_CAUCHY && (qs > 1e150 || qr > 1e150))) fold(ws);
    }
};

// LOSS template argument of the LM code: >= 0 fixes the robust loss at compile time, < 0 reads it from LMParams.  The
// Cauchy losses (compile-time or run-time) take the log-product path on the device.
RP_HD constexpr bool lm_loss_may_be_cauchy(int LOSS) { return LOSS < 0 || LOSS == RP_LOSS_CAUCHY || LOSS == RP_LOSS_TRUNCATED_CAUCHY; }

// one robustified residual of the LM cost: returns its contribution, or parks it in `lp` (device, Cauchy losses)
template <int LOSS, bool SAMPSON>
RP_HD double robust_cost(const LMParams &P, int loss_type, double r2, LogProd &lp) {
#ifdef __CUDA_ARCH__
    if (lm_loss_may_be_cauchy(LOSS) && (loss_type == RP_LOSS_CAUCHY || loss_type == RP_LOSS_TRUNCATED_CAUCHY)) {
        lp.template add<SAMPSON>(loss_type, r2 * P.inv_t2, P.weight_sampson);
        return 0.0;
    }
#endif
    return (SAMPSON ? P.weight_sampson : 1.0) * loss_eval(loss_type, P.loss_scale, r2);
}
// IRLS weight; on the device the Cauchy weights 1 / (1 + r^2 / t^2) use the Newton-refined reciprocal instead of two
// IEEE divisions
template <int LOSS>
RP_HD double robust_weight(const LMParams &P, int loss_type, double r2) {
#ifdef __CUDA_ARCH__
    if (lm_loss_may_be_cauchy(LOSS) && (loss_type == RP_LOSS_CAUCHY || loss_type == RP_LOSS_TRUNCATED_CAUCHY)) {
        const double x = r2 * P.inv_t2;
        if (loss_type == RP_LOSS_TRUNCATED_CAUCHY && x > 1.0) return 0.0;
        return lm_rcp(1.0 + x);
    }
#endif
    return loss_weight(loss_type, P.loss_scale, r2);
}

// everything about the current model that is constant across points
struct LMFrame {
    M3 R, E;
    V3 t, Rt;   // Rt = R^T t
    double scale, shift1, shift2, f1, f2, if1, if2, if1sq, if2sq;
};

RP_HD LMFrame make_frame(const Model &m) {
    LMFrame F;
    F.R = quat_to_rotmat(m.q);
    F.E = essential_from_motion(m.q, m.t);
    F.t = m.t;
    F.Rt = mulT(F.R, m.t);
    F.scale = m.scale; F.shift1 = m.shift1; F.shift2 = m.shift2;
    F.f1 = m.f1; F.f2 = m.f2;
    F.if1 = 1.0 / m.f1;
    F.if2 = 1.0 / m.f2;
    F.if1sq = 1.0 / (m.f1 * m.f1);
    F.if2sq = 1.0 / (m.f2 * m.f2);
    return F;
}

template <int NP>
struct NormalEq {
    double A[NP * (NP + 1) / 2];  // packed lower triangle, row-major: (i,j<=i) at i(i+1)/2+j
    double g[NP];
    RP_HD void clear() {
#pragma unroll
        for (int i = 0; i < NP * (NP + 1) / 2; ++i) A[i] = 0.0;
#pragma unroll
        for (int i = 0; i < NP; ++i) g[i] = 0.0;
    }
    // rank-1 update restricted to the columns whose bit is set in MASK (structural zeros of the row)
    template <unsigned MASK>
    RP_HD void add_row(double w, const double (&J)[NP], double r) {
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            if (!((MASK >> i) & 1u)) continue;
            const double wi = w * J[i];
            g[i] = fma_(wi, r, g[i]);
#pragma unroll
            for (int j = 0; j <= i; ++j) {
                if (!((MASK >> j) & 1u)) continue;
                A[i * (i + 1) / 2 + j] = fma_(wi, J[j], A[i * (i + 1) / 2 + j]);
            }
        }
    }
};

RP_HD V3 unit(int i) { return v3(i == 0 ? 1.0 : 0.0, i == 1 ? 1.0 : 0.0, i == 2 ? 1.0 : 0.0); }
RP_HD double comp(V3 v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }
RP_HD V3 row(const M3 &M, int i) { return i == 0 ? M.r0 : (i == 1 ? M.r1 : M.r2); }

// cost contribution of one correspondence
// LOSS >= 0 fixes the robust loss at compile time (the LO refinement always uses TRUNCATED: the per-residual
// switch disappears); LOSS < 0 reads it from P.
template <int VARIANT, int LOSS = -1>
RP_HD double point_cost(const LMFrame &F, const LMParams &P, double x1_0, double x1_1, double x2_0, double x2_1,
                        double d1, double d2, LogProd &lp) {
    constexpr bool FOCAL_ = (VARIANT == RP_SHARED || VARIANT == RP_VARYING);
    const int loss_type = LOSS >= 0 ? LOSS : P.loss_type;
    // calibrated variants carry f1 = f2 = 1: literal ones let the compiler drop the multiplications
    const double f1 = FOCAL_ ? F.f1 : 1.0, f2 = FOCAL_ ? F.f2 : 1.0;
    const double if1sq = FOCAL_ ? F.if1sq : 1.0, if2sq = FOCAL_ ? F.if2sq : 1.0;
    const V3 p1 = FOCAL_ ? v3(x1_0 * F.if1, x1_1 * F.if1, 1.0) : v3(x1_0, x1_1, 1.0);
    const V3 p2 = FOCAL_ ? v3(x2_0 * F.if2, x2_1 * F.if2, 1.0) : v3(x2_0, x2_1, 1.0);
    double cost = 0.0;
    const M3 &R = F.R;
    const M3 &E = F.E;
    const double px = p1.x, py = p1.y, qx = p2.x, qy = p2.y;
    if (P.weight_sampson > 0.0) {
        const V3 Ep1 = v3(fma_(E.r0.x, px, fma_(E.r0.y, py, E.r0.z)), fma_(E.r1.x, px, fma_(E.r1.y, py, E.r1.z)),
                          fma_(E.r2.x, px, fma_(E.r2.y, py, E.r2.z)));
        const V3 Etp2 = v3(fma_(E.r0.x, qx, fma_(E.r1.x, qy, E.r2.x)), fma_(E.r0.y, qx, fma_(E.r1.y, qy, E.r2.y)),
                           fma_(E.r0.z, qx, fma_(E.r1.z, qy, E.r2.z)));
        const double C = fma_(qx, Ep1.x, fma_(qy, Ep1.y, Ep1.z));
        const double A = Ep1.x * Ep1.x + Ep1.y * Ep1.y, B = Etp2.x * Etp2.x + Etp2.y * Etp2.y;
        const double inv = lm_rsqrt(A * if2sq + B * if1sq);
        const double rs = C * inv;
        cost += robust_cost<LOSS, true>(P, loss_type, rs * rs, lp);
    }
    if (P.scale_reproj > 0.0) {
        // Z = R (a p1) + t = a s + t,  Y = R^T (b p2 - t) = b m - R^T t   (s = R p1, m = R^T p2: the forms point_eval uses)
        const V3 s = v3(fma_(R.r0.x, px, fma_(R.r0.y, py, R.r0.z)), fma_(R.r1.x, px, fma_(R.r1.y, py, R.r1.z)),
                        fma_(R.r2.x, px, fma_(R.r2.y, py, R.r2.z)));
        const V3 m = v3(fma_(R.r0.x, qx, fma_(R.r1.x, qy, R.r2.x)), fma_(R.r0.y, qx, fma_(R.r1.y, qy, R.r2.y)),
                        fma_(R.r0.z, qx, fma_(R.r1.z, qy, R.r2.z)));
        const double a = d1 + F.shift1;
        const V3 Z = v3(fma_(a, s.x, F.t.x), fma_(a, s.y, F.t.y), fma_(a, s.z, F.t.z));
        if (Z.z > 0.0) {
            const double iz = lm_rcp(Z.z);
            const double r0 = f2 * (Z.x * iz) - x2_0, r1 = f2 * (Z.y * iz) - x2_1;
            cost += robust_cost<LOSS, false>(P, loss_type, P.scale_reproj * (r0 * r0 + r1 * r1), lp);
        }
        const double b = F.scale * (d2 + F.shift2);
        const V3 Y = v3(fma_(b, m.x, -F.Rt.x), fma_(b, m.y, -F.Rt.y), fma_(b, m.z, -F.Rt.z));
        if (Y.z > 0.0) {
            const double iz = lm_rcp(Y.z);
            const double r0 = f1 * (Y.x * iz) - x1_0, r1 = f1 * (Y.y * iz) - x1_1;
            cost += robust_cost<LOSS, false>(P, loss_type, P.scale_reproj * (r0 * r0 + r1 * r1), lp);
        }
    }
    return cost;
}

// J^T J / J^T r contribution of one correspondence.  Derivatives are written out per parameter
// (cross products with unit vectors expanded by hand) and each residual row only touches its
// structurally non-zero columns:
//   Sampson          : w, t            (+ f | f1, f2)
//   reprojection 1->2: w, t, shift1    (+ f | f1, f2)         (no scale, no shift2)
//   reprojection 2->1: w, t, scale, shift2 (+ f | f1, f2)     (no shift1)
// point_eval returns the cost contribution of the same correspondence as well (the value point_cost
// computes), so one pass over the data serves both the accept test of the trial step and — when it is
// accepted, the usual case — the normal equations of the next iteration.
// FP64 flops of one correspondence in one LM pass, counted from the formulas below (FMA = 2, mul / add / compare = 1,
// rcp = 1, rsqrt = 2; structural zeros and the calibrated variants' literal unit focals not counted):
//   residuals + cost (always)          : LM_FLOPS[v][0]
//   Sampson row, Jacobian + J^T J      : LM_FLOPS[v][1]   (6 | 6 | 7 | 8 columns)
//   reprojection 1->2, both rows       : LM_FLOPS[v][2]   (6 | 7 | 7 | 8 columns, of which each row skips one t column)
//   reprojection 2->1, both rows       : LM_FLOPS[v][3]   (7 | 8 | 8 | 9 columns)
// (v = RP_CALIB, RP_CALIB_SHIFT, RP_SHARED, RP_VARYING; derivation in DESIGN.md §5).  `rows` counts the accumulated
// rows of the three kinds in three 21-bit fields; the LM kernel turns the counts into the bench's lm_flops.
constexpr int LM_FLOPS[4][4] = {{104, 146, 131, 182}, {104, 146, 162, 222}, {112, 201, 183, 244}, {112, 220, 217, 286}};

template <int VARIANT, int NP, int LOSS = -1>
RP_HD double point_eval(const LMFrame &F, const LMParams &P, double x1_0, double x1_1, double x2_0,
                        double x2_1, double d1, double d2, NormalEq<NP> &N, unsigned long long &rows, LogProd &lp) {
    constexpr bool FOCAL = (VARIANT == RP_SHARED || VARIANT == RP_VARYING);
    const int loss_type = LOSS >= 0 ? LOSS : P.loss_type;
    // calibrated variants carry f1 = f2 = 1: literal ones let the compiler drop the multiplications (and the
    // six registers that would hold them)
    const double f1 = FOCAL ? F.f1 : 1.0, f2 = FOCAL ? F.f2 : 1.0;
    const double if1sq = FOCAL ? F.if1sq : 1.0, if2sq = FOCAL ? F.if2sq : 1.0;
    constexpr int CF2 = (VARIANT == RP_SHARED) ? 7 : 8;  // column of f2 (== f column when shared)
    constexpr unsigned M_POSE = 0x3Fu;                    // w (0-2), t (3-5)
    constexpr unsigned M_FOC = VARIANT == RP_SHARED ? 0x80u : (VARIANT == RP_VARYING ? 0x180u : 0u);
    constexpr unsigned M_S = M_POSE | M_FOC;
    constexpr unsigned M_12 = M_POSE | M_FOC | (VARIANT == RP_CALIB_SHIFT ? 0x80u : 0u);
    constexpr unsigned M_21 = M_POSE | 0x40u | M_FOC | (VARIANT == RP_CALIB_SHIFT ? 0x100u : 0u);
    const double px = FOCAL ? x1_0 * F.if1 : x1_0, py = FOCAL ? x1_1 * F.if1 : x1_1;  // p1 = (px, py, 1)
    const double qx = FOCAL ? x2_0 * F.if2 : x2_0, qy = FOCAL ? x2_1 * F.if2 : x2_1;  // p2 = (qx, qy, 1)
    const M3 &R = F.R;
    const M3 &E = F.E;
    double J[NP];
    double cost = 0.0;
    // s = R p1 and m = R^T p2 serve all three residual blocks: Z = R (a p1) + t = a s + t, Y = R^T (b p2 - t) = b m - R^T t,
    // the translation columns of the Sampson row, the shift1 column (= s) and the scale / shift2 columns (along m).
    // Three-term sums are written as nested FMAs: `a*b + c*d + e` contracts to MUL + FMA + ADD, and the FP64 pipe's issue
    // rate is what bounds this kernel.
    const V3 s = v3(fma_(R.r0.x, px, fma_(R.r0.y, py, R.r0.z)), fma_(R.r1.x, px, fma_(R.r1.y, py, R.r1.z)),
                    fma_(R.r2.x, px, fma_(R.r2.y, py, R.r2.z)));
    const V3 m = v3(fma_(R.r0.x, qx, fma_(R.r1.x, qy, R.r2.x)), fma_(R.r0.y, qx, fma_(R.r1.y, qy, R.r2.y)),
                    fma_(R.r0.z, qx, fma_(R.r1.z, qy, R.r2.z)));

    // ---- Sampson row ----
    if (P.weight_sampson > 0.0) {
        const V3 Ep1 = v3(fma_(E.r0.x, px, fma_(E.r0.y, py, E.r0.z)), fma_(E.r1.x, px, fma_(E.r1.y, py, E.r1.z)),
                          fma_(E.r2.x, px, fma_(E.r2.y, py, E.r2.z)));
        const V3 Etp2 = v3(fma_(E.r0.x, qx, fma_(E.r1.x, qy, E.r2.x)), fma_(E.r0.y, qx, fma_(E.r1.y, qy, E.r2.y)),
                           fma_(E.r0.z, qx, fma_(E.r1.z, qy, E.r2.z)));
        const double C = fma_(qx, Ep1.x, fma_(qy, Ep1.y, Ep1.z));
        const double A = Ep1.x * Ep1.x + Ep1.y * Ep1.y, B = Etp2.x * Etp2.x + Etp2.y * Etp2.y;
        const double inv = lm_rsqrt(A * if2sq + B * if1sq);
        const double rs = C * inv;
        cost += robust_cost<LOSS, true>(P, loss_type, rs * rs, lp);
        // the reference scales the Sampson residual and its Jacobian row by weight_sampson, so the normal equations
        // carry weight_sampson^2 although the cost carries weight_sampson (verified on the binary; invisible at 1)
        // ... and the focal accumulators evaluate the robust weight at weight_sampson * r^2, the calibrated one at r^2
        const double w = P.weight_sampson * P.weight_sampson *
                         robust_weight<LOSS>(P, loss_type, FOCAL ? P.weight_sampson * (rs * rs) : rs * rs);
        if (w != 0.0) {
#pragma unroll
            for (int i = 0; i < NP; ++i) J[i] = 0.0;
            // The row is inv * J' with J'_i = dC_i - c2 * D_i (c2 = C inv^2, D_i = half the derivative of the
            // denominator): J' is accumulated with the weight w inv^2 against the residual rs / inv = C, which is the same
            // J^T J and J^T r with one multiplication less per column (the FP64 pipe is what bounds this kernel).
            const double c2 = rs * inv;
            const double a2 = if2sq, a1 = if1sq;
            // rotation: dE = E [e_i]x ;  d(Ep1) = E (e_i x p1),  d(E^T p2) = -(e_i x E^T p2)
            {
                const double dx = py * E.r0.z - E.r0.y, dy = py * E.r1.z - E.r1.y;
                const double dC = py * Etp2.z - Etp2.y;
                J[0] = dC - c2 * ((Ep1.x * dx + Ep1.y * dy) * a2 + (Etp2.y * Etp2.z) * a1);
            }
            {
                const double dx = E.r0.x - px * E.r0.z, dy = E.r1.x - px * E.r1.z;
                const double dC = Etp2.x - px * Etp2.z;
                J[1] = dC - c2 * ((Ep1.x * dx + Ep1.y * dy) * a2 - (Etp2.x * Etp2.z) * a1);
            }
            {
                const double dx = px * E.r0.y - py * E.r0.x, dy = px * E.r1.y - py * E.r1.x;
                const double dC = px * Etp2.y - py * Etp2.x;
                J[2] = dC - c2 * ((Ep1.x * dx + Ep1.y * dy) * a2);
            }
            // translation: dE = [e_i]x R ;  d(Ep1) = e_i x (R p1) = e_i x s,  d(E^T p2) = -R^T (e_i x p2)
            {
                // e_0 x s = (0, -s.z, s.y);  e_0 x p2 = (0, -1, qy) -> d(E^T p2) = row1(R) - qy row2(R)
                const double tx = R.r1.x - qy * R.r2.x, ty = R.r1.y - qy * R.r2.y;
                const double dC = s.y - qy * s.z;
                J[3] = dC - c2 * ((-Ep1.y * s.z) * a2 + (Etp2.x * tx + Etp2.y * ty) * a1);
            }
            {
                // e_1 x s = (s.z, 0, -s.x);  e_1 x p2 = (1, 0, -qx) -> d(E^T p2) = qx row2(R) - row0(R)
                const double tx = qx * R.r2.x - R.r0.x, ty = qx * R.r2.y - R.r0.y;
                const double dC = qx * s.z - s.x;
                J[4] = dC - c2 * ((Ep1.x * s.z) * a2 + (Etp2.x * tx + Etp2.y * ty) * a1);
            }
            {
                // e_2 x s = (-s.y, s.x, 0);  e_2 x p2 = (-qy, qx, 0) -> d(E^T p2) = qy row0(R) - qx row1(R)
                const double tx = qy * R.r0.x - qx * R.r1.x, ty = qy * R.r0.y - qx * R.r1.y;
                const double dC = qy * s.x - qx * s.y;
                J[5] = dC - c2 * ((Ep1.y * s.x - Ep1.x * s.y) * a2 + (Etp2.x * tx + Etp2.y * ty) * a1);
            }
            if (FOCAL) {
                // p1 = (x1/f1, 1): dp1/df1 = -(px, py, 0)/f1 ; den = A/f2^2 + B/f1^2
                const double dpx = -px * F.if1, dpy = -py * F.if1, dqx = -qx * F.if2, dqy = -qy * F.if2;
                const double e1x = E.r0.x * dpx + E.r0.y * dpy, e1y = E.r1.x * dpx + E.r1.y * dpy;
                const double e2x = E.r0.x * dqx + E.r1.x * dqy, e2y = E.r0.y * dqx + E.r1.y * dqy;
                const double j1 = (Etp2.x * dpx + Etp2.y * dpy) -
                                  c2 * ((Ep1.x * e1x + Ep1.y * e1y) * a2 - B * a1 * F.if1);
                const double j2 = (Ep1.x * dqx + Ep1.y * dqy) -
                                  c2 * ((Etp2.x * e2x + Etp2.y * e2y) * a1 - A * a2 * F.if2);
                if (VARIANT == RP_SHARED) J[7] = j1 + j2;
                else { J[7] = j1; J[CF2] = j2; }
            }
            N.template add_row<M_S>(w * (inv * inv), J, C);
            rows += 1ull;
        }
    }
    if (!(P.scale_reproj > 0.0)) return cost;

    // The reprojection rows are g * J' with g = f / z: J' is accumulated with the weight w g^2 against the residual
    // r / g = r z / f (again one multiplication less per column than scaling every entry by g first).
    // ---- reprojection 1 -> 2 : Z = R (a p1) + t ----
    {
        const double a = d1 + F.shift1;
        const V3 Z = v3(fma_(a, s.x, F.t.x), fma_(a, s.y, F.t.y), fma_(a, s.z, F.t.z));
        if (Z.z > 0.0) {
            const double iz = lm_rcp(Z.z);
            const double u0 = Z.x * iz, u1 = Z.y * iz;
            const double r0 = f2 * u0 - x2_0, r1 = f2 * u1 - x2_1;
            cost += robust_cost<LOSS, false>(P, loss_type, P.scale_reproj * (r0 * r0 + r1 * r1), lp);
            const double w = P.scale_reproj * robust_weight<LOSS>(P, loss_type, P.scale_reproj * (r0 * r0 + r1 * r1));
            if (w != 0.0) {
                const double g = f2 * iz;
                const double zg = FOCAL ? Z.z * F.if2 : Z.z;   // 1 / g
                double J0[NP], J1[NP];
#pragma unroll
                for (int i = 0; i < NP; ++i) { J0[i] = 0.0; J1[i] = 0.0; }
                // dZ/dw_i = R (e_i x P) = a R (e_i x p1):  a (py c2 - c1),  a (c0 - px c2),  a (px c1 - py c0)  (c_j columns of R)
                {
                    const double dx = py * R.r0.z - R.r0.y, dy = py * R.r1.z - R.r1.y, dz = py * R.r2.z - R.r2.y;
                    J0[0] = a * (dx - u0 * dz); J1[0] = a * (dy - u1 * dz);
                }
                {
                    const double dx = R.r0.x - px * R.r0.z, dy = R.r1.x - px * R.r1.z, dz = R.r2.x - px * R.r2.z;
                    J0[1] = a * (dx - u0 * dz); J1[1] = a * (dy - u1 * dz);
                }
                {
                    const double dx = px * R.r0.y - py * R.r0.x, dy = px * R.r1.y - py * R.r1.x, dz = px * R.r2.y - py * R.r2.x;
                    J0[2] = a * (dx - u0 * dz); J1[2] = a * (dy - u1 * dz);
                }
                // dZ/dt = I
                J0[3] = 1.0; J0[5] = -u0;
                J1[4] = 1.0; J1[5] = -u1;
                if (VARIANT == RP_CALIB_SHIFT) {
                    // dZ/dshift1 = R p1 = s
                    J0[7] = s.x - u0 * s.z; J1[7] = s.y - u1 * s.z;
                }
                if (FOCAL) {
                    // dZ/df1 = R (-a px/f1, -a py/f1, 0) ; d(pi)/df2 = (u0, u1) = g (Z.x, Z.y) / f2^2... kept as (u0, u1) / g
                    const double ex = -(a * px) * F.if1, ey = -(a * py) * F.if1;
                    const double dx = R.r0.x * ex + R.r0.y * ey, dy = R.r1.x * ex + R.r1.y * ey, dz = R.r2.x * ex + R.r2.y * ey;
                    J0[7] = dx - u0 * dz; J1[7] = dy - u1 * dz;
                    J0[CF2] += Z.x * F.if2; J1[CF2] += Z.y * F.if2;
                }
                // dZ/dt = I: the x row has no t_y column, the y row no t_x column (structural zeros skipped)
                const double sw = w * (g * g);
                N.template add_row<(M_12 & ~0x10u)>(sw, J0, r0 * zg);
                N.template add_row<(M_12 & ~0x08u)>(sw, J1, r1 * zg);
                rows += 1ull << 21;
            }
        }
    }
    // ---- reprojection 2 -> 1 : Y = R^T (b p2 - t) ----
    {
        const double bb = d2 + F.shift2;
        const double b = F.scale * bb;
        const V3 Y = v3(fma_(b, m.x, -F.Rt.x), fma_(b, m.y, -F.Rt.y), fma_(b, m.z, -F.Rt.z));
        if (Y.z > 0.0) {
            const double iz = lm_rcp(Y.z);
            const double u0 = Y.x * iz, u1 = Y.y * iz;
            const double r0 = f1 * u0 - x1_0, r1 = f1 * u1 - x1_1;
            cost += robust_cost<LOSS, false>(P, loss_type, P.scale_reproj * (r0 * r0 + r1 * r1), lp);
            const double w = P.scale_reproj * robust_weight<LOSS>(P, loss_type, P.scale_reproj * (r0 * r0 + r1 * r1));
            if (w != 0.0) {
                const double g = f1 * iz;
                const double zg = FOCAL ? Y.z * F.if1 : Y.z;   // 1 / g
                double J0[NP], J1[NP];
#pragma unroll
                for (int i = 0; i < NP; ++i) { J0[i] = 0.0; J1[i] = 0.0; }
                // dY/dw_i = Y x e_i:  (0, Yz, -Yy), (-Yz, 0, Yx), (Yy, -Yx, 0)
                J0[0] = u0 * Y.y;            J1[0] = Y.z + u1 * Y.y;
                J0[1] = -Y.z - u0 * Y.x;     J1[1] = -u1 * Y.x;
                J0[2] = Y.y;                 J1[2] = -Y.x;
                // dY/dt_i = -row_i(R)
                J0[3] = u0 * R.r0.z - R.r0.x; J1[3] = u1 * R.r0.z - R.r0.y;
                J0[4] = u0 * R.r1.z - R.r1.x; J1[4] = u1 * R.r1.z - R.r1.y;
                J0[5] = u0 * R.r2.z - R.r2.x; J1[5] = u1 * R.r2.z - R.r2.y;
                // dY/dscale = R^T ((d2+v) p2),  dY/dshift2 = R^T (scale p2): both along m = R^T p2
                const double m0 = m.x - u0 * m.z, m1 = m.y - u1 * m.z;
                J0[6] = bb * m0; J1[6] = bb * m1;
                if (VARIANT == RP_CALIB_SHIFT) { J0[8] = F.scale * m0; J1[8] = F.scale * m1; }
                if (FOCAL) {
                    // dY/df2 = R^T (-b qx/f2, -b qy/f2, 0) ; d(pi1)/df1 = (u0, u1), i.e. (Y.x, Y.y) / f1 in units of g
                    const double ex = -b * qx * F.if2, ey = -b * qy * F.if2;
                    const double dx = R.r0.x * ex + R.r1.x * ey, dy = R.r0.y * ex + R.r1.y * ey, dz = R.r0.z * ex + R.r1.z * ey;
                    J0[CF2] += dx - u0 * dz; J1[CF2] += dy - u1 * dz;
                    J0[7] += Y.x * F.if1; J1[7] += Y.y * F.if1;
                }
                const double sw = w * (g * g);
                N.template add_row<M_21>(sw, J0, r0 * zg);
                N.template add_row<M_21>(sw, J1, r1 * zg);
                rows += 1ull << 42;
            }
        }
    }
    return cost;
}

template <int VARIANT, int NP>
RP_HD void point_accumulate(const LMFrame &F, const LMParams &P, double x1_0, double x1_1, double x2_0,
                            double x2_1, double d1, double d2, NormalEq<NP> &N) {
    unsigned long long rows = 0;
    LogProd lp;
    lp.init();
    (void)point_eval<VARIANT, NP>(F, P, x1_0, x1_1, x2_0, x2_1, d1, d2, N, rows, lp);
}

// parameter update of lm_impl's problem.step(): R <- R exp([dw]x), everything else additive
template <int VARIANT>
RP_HD Model model_step(const Model &m, const double *dp) {
    Model o = m;
    o.q = quat_mul(m.q, quat_exp(v3(dp[0], dp[1], dp[2])));
    o.t = v3(m.t.x + dp[3], m.t.y + dp[4], m.t.z + dp[5]);
    o.scale = m.scale + dp[6];
    if (VARIANT == RP_CALIB_SHIFT) { o.shift1 = m.shift1 + dp[7]; o.shift2 = m.shift2 + dp[8]; }
    if (VARIANT == RP_SHARED) { o.f1 = m.f1 + dp[7]; o.f2 = o.f1; }
    if (VARIANT == RP_VARYING) { o.f1 = m.f1 + dp[7]; o.f2 = m.f2 + dp[8]; }
    return o;
}

// (J^T J + lambda I) x = b by Cholesky on the packed lower triangle (Eigen's
// selfadjointView<Lower>().llt().solve()); a non-PD matrix propagates NaN like Eigen does.
template <int NP>
RP_HD void llt_solve(const double *A, double lambda, const double *b, double *x) {
    // one sqrt and one reciprocal per column; the triangular solves multiply by the reciprocals
    // (the serial part of an LM iteration: keep the slow FP64 ops off its critical path)
    double L[NP * (NP + 1) / 2], inv[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) {
        double s = A[j * (j + 1) / 2 + j] + lambda;
#pragma unroll
        for (int k = 0; k < j; ++k) s -= L[j * (j + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
        const double d = sqrt(s);
        L[j * (j + 1) / 2 + j] = d;
        inv[j] = 1.0 / d;
#pragma unroll
        for (int i = j + 1; i < NP; ++i) {
            double v = A[i * (i + 1) / 2 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) v -= L[i * (i + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
            L[i * (i + 1) / 2 + j] = v * inv[j];
        }
    }
    double y[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        double v = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) v -= L[i * (i + 1) / 2 + k] * y[k];
        y[i] = v * inv[i];
    }
#pragma unroll
    for (int i = NP - 1; i >= 0; --i) {
        double v = y[i];
#pragma unroll
        for (int k = i + 1; k < NP; ++k) v -= L[k * (k + 1) / 2 + i] * x[k];
        x[i] = v * inv[i];
    }
}

}  // namespace rp
