// rp_tc.cuh — tensor-core tier of the minimal-model scoring (sm_100a: tcgen05.mma + TMEM + TMA).
//
// What it computes.  score_models() (so@0x22ebc0) looks at a minimal model only when it has more inliers
// or a lower MSAC score than every earlier one, so a model with provably MANY certain outliers can be
// dropped unseen (DESIGN.md §5).  For one (model, correspondence) the Sampson test of
// compute_sampson_msac_score (so@0x4f61d0 / so@0x4f65d0) is  r2 = C^2 / den < thr^2  with
//     C   = x2^T E x1                       = sum_j E_j  phi_j(p)      (9 monomials of the point)
//     den = |E x1|_{01}^2 + |E^T x2|_{01}^2 = sum_k G_k(E) psi_k(p)    (11 monomials of the point)
// i.e. two contractions [models x K] . [K x points]: a GEMM with a threshold epilogue.  This kernel runs
// them on the 5th-generation tensor cores:
//     Cs = 2^s C~                                    4 x tcgen05.mma kind::tf32 (hi/lo split, see below)
//     Ts = -2^2s [(1+a) g (den~ + d_den) + (1+1/a) eps^2]   2 x tcgen05.mma kind::tf32
//     certain outlier  <=>  Cs*Cs + Ts > 0           one FFMA.SAT per point-score out of TMEM
// and counts the certain outliers of every model.  It is a FILTER, never the score: a point is counted
// only if the FP64 reference test is certainly false, so  out <= N - inlier_count  and
// thr^2 * out <= score  hold rigorously (error model below); survivors go on to the FP32 bound kernel
// and the exact FP64 kernel (rp_kernels.cuh).
//
// Precision.  TF32 keeps 11 significand bits, far too few for C (the threshold sits at ~1e-3 |E|), so
// both operands of C are split  v = hi + lo,  hi = tf32(v), lo = tf32(v - hi)  and the three products
// hi*hi + lo*hi + hi*lo are accumulated (the products of TF32 numbers are exact in the FP32 accumulator):
//     |2^-s Cs - C| <= eps_tc = 64 u Emax (M + thr m),   u = 2^-24
// (input roundings 4u, dropped lo*lo and the two split residuals 3*2^-22 = 12u, four FP32 accumulation steps <= 8u even
// with truncation: 24u, so 2.7x slack; measured on B200 by tools/tc_probe.cu: max 1.6u; M, m, Emax as in rp_score.cuh).  den only scales the threshold, so single TF32 suffices:
//     |den~ - den| <= d_den = 2^-7 Emax^2 m^2    (two 2^-11 roundings per term on sum|G_k psi_k| <= 4 Emax^2 m^2,
//                                                 accumulation, 2x slack)
// and with (x+y)^2 <= (1+a) x^2 + (1+1/a) y^2, a = 1/32:
//     Cs^2 + Ts > 0  =>  C~^2 > (1+a) g (den + 0) + (1+1/a) eps^2  =>  (|C~| - eps)^2 > g den  =>  r2 > thr^2 (1+1e-6).
// tests/test_gpu_tc.py measures the actual errors against FP64 and checks out <= N - exact count on random
// and adversarial models.
//
// Layout / schedule (one CTA per SM, persistent, 512 threads):
//   B operand  per-point feature rows, 32 floats = 128 B, written once per pair by tc_features_kernel, fetched 64 rows
//              at a time by TMA (cp.async.bulk.tensor, SWIZZLE_128B) into a 6-stage ring; one more, constant, slice
//              (0,0,0,0,1,1,0,0) per row sits in shared memory for the whole kernel                       [warp 0]
//   A operand  256 models per work item (2 M-tiles).  A does not change over the ~32 point tiles of an item, so the
//              builder warps compute the rows from the 96-byte models (E, G(E), hi/lo split, constants) and write them
//              ONCE per item straight into TENSOR MEMORY (tcgen05.st, thread = row = TMEM lane, double buffered); the
//              MMAs take A from there.  (With A in shared memory every MMA re-read 4 KB of A next to 2 KB of B for
//              128 x 64 x 8 MACs: measured 86 cycles per MMA, tensor pipe at 17 %.)                       [warps 12-15]
//   MMA        one elected thread issues 6 tcgen05.mma per (64-point tile, M-tile) into one of three accumulator
//              slots (Cs | Ts, 128 columns); TMEM map: 3 x 128 accumulator + 2 x 2 x 32 A columns = 512   [warp 1]
//   epilogue   group m = the four warps of M-tile m, thread = model (TMEM lane), tcgen05.ld 16 columns at a time,
//              FFMA.SAT + FADD; two MMA groups of slack to drain a slot                                    [warps 4-11]
// Per (model, point): 48 tensor-core MACs, 8 B of TMEM read, ~2 issue slots.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include "rp_types.cuh"

namespace rp {
namespace tc {

constexpr int MT = 2;                        // M-tiles (128 models) per work item
constexpr int TILE_MODELS = 128 * MT;
constexpr int FEAT = 32;                     // floats per point feature row (128 B)
constexpr double A_SPLIT = 1.0 / 32.0;                // a of (x+y)^2 <= (1+a) x^2 + (1+1/a) y^2
constexpr double EPS_UNITS = 64.0;                    // eps_tc = EPS_UNITS u Emax (M + thr m)

// ---- TF32 rounding (round to nearest, ties away: cvt.rna.tf32.f32) ---------------------------------
RP_HD float tf32_round(float v) {
#if defined(__CUDA_ARCH__)
    unsigned r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
#else
    unsigned b;
    memcpy(&b, &v, 4);
    if ((b & 0x7f800000u) != 0x7f800000u) b = (b + 0x1000u) & 0xffffe000u;
    float o;
    memcpy(&o, &b, 4);
    return o;
#endif
}

// ---- per-point feature row (B operand) ---------------------------------------------------------------
// slice 0: tf32(phi_0..7)   slice 1: tf32(phi - slice 0)   slice 2: tf32(psi_0..7)   slice 3: (x2x, x2y, 1, 0, 0, 0, 0, 0)
// (+ the constant slice K = (0, 0, 0, 0, 1, 1, 0, 0), the same for every point: kept once in shared memory)
//   phi = (x2x x1x, x2x x1y, x2x, x2y x1x, x2y x1y, x2y, x1x, x1y)            <-> E00 E01 E02 E10 E11 E12 E20 E21 (E22: const)
//   psi = (x1x^2, x1x x1y, x1y^2, x1x, x1y, x2x^2, x2x x2y, x2y^2 | x2x, x2y | 1)
RP_HD void feature_row(float x1x, float x1y, float x2x, float x2y, float *row /*32*/) {
    const float phi[8] = {x2x * x1x, x2x * x1y, x2x, x2y * x1x, x2y * x1y, x2y, x1x, x1y};
    const float psi[8] = {x1x * x1x, x1x * x1y, x1y * x1y, x1x, x1y, x2x * x2x, x2x * x2y, x2y * x2y};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float hi = tf32_round(phi[j]);
        row[j] = hi;
        row[8 + j] = tf32_round(phi[j] - hi);
        row[16 + j] = tf32_round(psi[j]);
    }
    row[24] = tf32_round(x2x); row[25] = tf32_round(x2y); row[26] = 1.0f;
    row[27] = row[28] = row[29] = row[30] = row[31] = 0.0f;
}

// ---- per-model operand row (A operand): 4 slices of 8 floats ---------------------------------------------
//   a0 = tf32(2^s E_j)   a1 = tf32(2^s E_j - a0)                                      . slice 0 / 1 / 0 of B  -> Cs
//   a2 = tf32(-2^2s (1+a) g G_0..7)                                                    . slice 2               -> Ts
//   a3 = (G_8', G_9', const, 0 | E22 hi, E22 lo, 0, 0)   . slice 3 (x2x, x2y, 1, 0 | 0...) -> Ts,  . slice K -> Cs
// A model whose parameters leave the range the error model covers gets the zero row (no point is ever counted:
// the model simply survives this tier); a model with a non-finite E / F — the minimal solvers return NaN models
// now and then — has r2 = NaN for every correspondence in the reference, i.e. no inliers and score N thr^2:
// its row is (0, ..., const = +2^100), which counts EVERY point.
RP_HD void model_row(const M3 &E, double thr, double Mmax, double mmax, float *r0 /*32: a0 a1 a2 a3*/) {
#pragma unroll
    for (int i = 0; i < 32; ++i) r0[i] = 0.f;
    const double e[9] = {E.r0.x, E.r0.y, E.r0.z, E.r1.x, E.r1.y, E.r1.z, E.r2.x, E.r2.y, E.r2.z};
    double emax = 0.0;
    bool finite = true;
#pragma unroll
    for (int i = 0; i < 9; ++i) { emax = fmax(emax, fabs(e[i])); finite = finite && (e[i] - e[i] == 0.0); }
    if (!finite) { r0[24 + 2] = 1.2676506002282294e30f; return; }   // 2^100
    const bool sane = emax > 1e-3 && emax < 1e3 && thr > 1e-6 && thr < 1.0 && Mmax < 1e3 && mmax < 1e3;
    if (!sane) return;
    const double u = 5.9604644775390625e-08;  // 2^-24
    const double eps = EPS_UNITS * u * emax * (Mmax + thr * mmax) * 1.0001;
    const double g = thr * thr * (1.0 + 1e-5);
    const double dden = 0.0078125 * emax * emax * mmax * mmax;   // 2^-7 Emax^2 m^2
    // Per-model power-of-two scaling: Cs = 2^s C~, Ts = 2^2s T~ with 2^2s (1+1/a) eps^2 >= 2^48.  Then |Ts| >= 2^47, and
    // whenever Cs^2 + Ts > 0 we have |Cs| > 2^23.5: both FP32 numbers are integers, so the exact value of Cs^2 + Ts is
    // an integer and FFMA.SAT returns exactly 0 or 1 — the per-model sums are exact counts (N < 2^24).
    // Ranges: Cs^2 <= 2^2s Emax^2 M^2 and |Ts| <= 2^2s 1.04 g (4 Emax^2 m^2 + ...) stay below 2^48 * 2^28 (sane ranges above).
    int ex;
    (void)frexp((1.0 + 1.0 / A_SPLIT) * eps * eps, &ex);     // value in [2^(ex-1), 2^ex)
    const int sc = (48 - (ex - 1) + 1) / 2;                    // 2 sc >= 48 - (ex - 1)
    const double cs = ldexp(1.0, sc), ts = ldexp(1.0, 2 * sc);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float v = (float)(e[j] * cs);
        const float hi = tf32_round(v);
        r0[j] = hi;
        r0[8 + j] = tf32_round(v - hi);
    }
    {
        const float v = (float)(e[8] * cs);
        const float hi = tf32_round(v);
        r0[24 + 4] = hi;
        r0[24 + 5] = tf32_round(v - hi);
    }
    const double G[11] = {e[0] * e[0] + e[3] * e[3], 2.0 * (e[0] * e[1] + e[3] * e[4]), e[1] * e[1] + e[4] * e[4],
                          2.0 * (e[0] * e[2] + e[3] * e[5]), 2.0 * (e[1] * e[2] + e[4] * e[5]),
                          e[0] * e[0] + e[1] * e[1], 2.0 * (e[0] * e[3] + e[1] * e[4]), e[3] * e[3] + e[4] * e[4],
                          2.0 * (e[0] * e[6] + e[1] * e[7]), 2.0 * (e[3] * e[6] + e[4] * e[7]),
                          e[2] * e[2] + e[5] * e[5] + e[6] * e[6] + e[7] * e[7]};
    const double k = -ts * (1.0 + A_SPLIT) * g;
#pragma unroll
    for (int j = 0; j < 8; ++j) r0[16 + j] = tf32_round((float)(k * G[j]));
    r0[24] = tf32_round((float)(k * G[8]));
    r0[25] = tf32_round((float)(k * G[9]));
    // the constant: pushed away from zero by 2^-9 before rounding (more negative = fewer certain outliers = conservative)
    const double kc = (k * (G[10] + dden) - ts * (1.0 + 1.0 / A_SPLIT) * eps * eps) * (1.0 + 0.001953125);
    r0[26] = tf32_round((float)kc);
}

// ---- PTX wrappers ------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
RP_D uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
RP_D void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
RP_D void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
RP_D void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
RP_D bool mbar_try(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a barrier that never completes (a protocol bug) traps instead of hanging the GPU.
RP_D void mbar_wait(uint64_t *bar, uint32_t parity) {
    for (unsigned spins = 0; !mbar_try(bar, parity); ++spins)
        if (spins > (1u << 28)) __trap();
}
RP_D void tma_load_2d(void *smem_dst, const CUtensorMap *tmap, int c0, int c1, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
RP_D void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
RP_D void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
RP_D void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
RP_D void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
RP_D void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
RP_D void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
RP_D void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
RP_D void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr) : "memory");
}
RP_D void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// one lane of a CONVERGED warp (the tensor-core and TMA instructions take uniform-register operands: issued from a
// `lane == 0` branch the compiler wraps each of them in a waterfall loop; under elect.sync it does not)
RP_D bool elect_one() {
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
RP_D unsigned long long pack2f(float lo, float hi) { unsigned long long r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
RP_D void unpack2f(unsigned long long v, float &lo, float &hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
RP_D unsigned long long add2(unsigned long long a, unsigned long long b) { unsigned long long d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
RP_D float fma_sat(float a, float b, float c) {
    float d;
    asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 version bit set): rows of 128 B, 8-row
// groups 1024 B apart; a K slice of 8 TF32 (32 B) inside the 128-byte span is selected by the start address
RP_D uint64_t desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// ---- feature kernel ------------------------------------------------------------------------------------------
// one thread per correspondence: pts32 (float4) -> 128-byte feature row
__global__ void tc_features_kernel(long long n, const float4 *pts32, float4 *feat) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts32[i];
    float row[32];
    feature_row(p.x, p.y, p.z, p.w, row);
    float4 *o = feat + i * 8;
#pragma unroll
    for (int c = 0; c < 8; ++c) o[c] = make_float4(row[4 * c], row[4 * c + 1], row[4 * c + 2], row[4 * c + 3]);
}

// ---- the tier ---------------------------------------------------------------------------------------------------
struct TcArgs {
    int n_pairs, nseg;
    const PairParams *pairs;
    const int *seg_count;        // [n_pairs * nseg] models per (pair, segment)
    const int *item_prefix;      // [n_pairs + 1] work items (TILE_MODELS models of one pair) before pair p
    const int *n_items;
    const Model *models;         // slots: (pair * nseg + seg) * 4 * SEG + i
    int *out;                    // slots: certain outliers (<= N - inlier count; == N for a model with a non-finite E / F)
    int pose;                    // 1: E = [t]x R,  0: F = diag(1,1,f2) E diag(1,1,f1)
    unsigned long long *evaluated;  // optional: point-scores evaluated
    float *debug;                // optional: raw (Cs, Ts) of work item 0, [TILE_MODELS][2][debug_cols]
    int debug_cols;
    // Two passes over the correspondences (abandonment at the granularity of this tier): pass 0 counts over the first
    // tc_split(n) correspondences of every model, the caller drops what already has enough certain outliers, pass 1
    // counts the remaining correspondences for the survivors only (`list`) and adds to `out`.
    int two_pass;                // 0: one pass over all correspondences; else two passes split at split[pair]
    const int *split;            // per pair: first correspondence of pass 1 (tc_split_kernel), a multiple of the point tile or n
    int first;                   // without a list: the pair's models start at position `first` of its first segment
    int pass;                    // 0 / 1
    const int *list;             // pass 1: pair-relative slots of the models to process, [n_pairs][list_stride]
    const int *list_cnt;         //         [n_pairs]
    int list_stride;
};

// Certain outliers after which a model can neither exceed the best inlier count B0 nor undercut the best score S0 of the
// pair's exactly scored head (the abandonment threshold of the FP32 bound kernel, shared by every tier)
RP_HD int need_outliers(int n, double sq_thr, int B0, double S0) {
#if defined(__CUDA_ARCH__)
    const float thr2_lo = __double2float_rd(sq_thr);
#else
    const float thr2_lo = (float)(sq_thr * (1.0 - 1e-7));
#endif
    const double need_d = fmax((double)(n - B0), S0 < 1e300 ? ceil(S0 / ((double)thr2_lo * (1.0 - 2e-4))) : 4.0e9);
    return need_d > 2.0e9 ? 0x7fffffff : (need_d < 1.0 ? 1 : (int)need_d);
}

// First correspondence of pass 1 (a multiple of the point tile; n itself = no second pass), adaptive: a hopeless model
// collects ~0.97 certain outliers per correspondence, so it can be dropped after need / 0.95 of them; the split sits at
// 115 % of `need` (profiles/r02_tc_adapt_sweep.txt: 105 / 115 / 125 % and a fixed half, r02_tc_split_sweep.txt: fixed
// shares); pairs whose threshold sits beyond 85 % of their correspondences (many outliers, a weak head) are not worth a
// second pass.  Any choice gives the same results — only the amount of work changes.
RP_HD int tc_split(int n, int need) {
    if (n < 4 * 64 || need > n) return n;
    const long long s = ((long long)need * 115 / 100 + 1 + 63) / 64 * 64;
    return s >= (long long)n * 85 / 100 ? n : (int)s;
}

// Per pair, once per chunk: the split of the two passes (the kernel's three warp roles only read it; evaluating
// need_outliers' FP64 division per work item inside them cost 2-4 ms per 10 000 pairs).
__global__ void tc_split_kernel(int n_pairs, const PairParams *pairs, const int *B0, const double *S0, int *split) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const PairParams pp = pairs[p];
    split[p] = tc_split(pp.n, need_outliers(pp.n, pp.sq_thr, B0[p], S0[p]));
}

// ---- the kernel -------------------------------------------------------------------------------------------------
constexpr int NT = 64;                                       // points per accumulator tile (MMA N)
constexpr int A_COLS = 32;                                   // a0 a1 a2 a3, 8 TMEM columns each
constexpr int SLOTS = 3;                                     // accumulator slots (one M-tile x one point tile: Cs | Ts)
constexpr int TMEM_A = SLOTS * 2 * NT;                       // first A column: 384
constexpr int B_STAGE_BYTES = NT * 128;
constexpr int B_STAGES = 6;
constexpr int KSLICE_BYTES = NT * 32;                        // constant slice, SWIZZLE_NONE K-major: 8-row groups of 256 B
constexpr int EPI_WARP0 = 4, BUILD_WARP0 = EPI_WARP0 + 4 * MT, THREADS = 32 * (BUILD_WARP0 + 4);
constexpr int SMEM_BYTES = 1024 + B_STAGES * B_STAGE_BYTES + KSLICE_BYTES + 256;
// kind::tf32, FP32 accumulate, A and B K-major, M = 128, N = NT
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NT >> 3) << 17) | ((128u >> 4) << 24);
static_assert(TMEM_A + 2 * MT * A_COLS == 512, "accumulator slots + A buffers fill the tensor memory exactly");

// K-major SWIZZLE_NONE descriptor of the constant slice: core matrices (8 rows x 16 B) 128 B apart along K, 8-row groups
// 256 B apart
RP_D uint64_t desc_kslice(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | (8ull << 16) | (16ull << 32) | (1ull << 46);
}
RP_D void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
RP_D void tmem_st8(uint32_t taddr, const float *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
                   "r"(__float_as_uint(v[7])) : "memory");
}
RP_D void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
RP_D void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}

// MODE 0: the tier.  Probe modes (tools/tc_probe.cu): 1 = epilogue loads the accumulators but skips the arithmetic,
// 2 = epilogue neither loads nor computes (TMA + MMA pipeline alone).
template <int MODE>
__global__ void __launch_bounds__(THREADS, 1) tc_count_kernel(const __grid_constant__ CUtensorMap tmap, TcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *sB = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // [B_STAGES][NT x 128 B]
    uint8_t *sK = sB + B_STAGES * B_STAGE_BYTES;                                   // constant slice
    uint64_t *bars = (uint64_t *)(sK + KSLICE_BYTES);
    uint64_t *b_full = bars, *b_empty = bars + B_STAGES, *a_full = bars + 2 * B_STAGES, *a_empty = a_full + 2,
             *slot_full = a_empty + 2, *slot_empty = slot_full + SLOTS;
    uint32_t *tmem_base_s = (uint32_t *)(slot_empty + SLOTS);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < B_STAGES; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&a_full[i], 4); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < SLOTS; ++i) { mbar_init(&slot_full[i], 1); mbar_init(&slot_empty[i], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_base_s, 512);
    // the constant slice (0,0,0,0 | 1,1,0,0) per row: row r, 16-byte chunk c at (r / 8) * 256 + c * 128 + (r % 8) * 16
    for (int i = tid; i < NT * 2; i += THREADS) {
        const int r = i >> 1, c = i & 1;
        *(float4 *)(sK + (r >> 3) * 256 + c * 128 + (r & 7) * 16) = c ? make_float4(1.f, 1.f, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_s;
    const uint32_t tmem_a = tmem_base + (uint32_t)TMEM_A;
    const int n_items = *a.n_items;

    auto pair_of = [&](int item) {
        int lo = 0, hi = a.n_pairs;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (a.item_prefix[mid] <= item) lo = mid; else hi = mid;
        }
        return lo;
    };

    // correspondences [p0, p1) of this pass, as point tiles [t0, t1)
    auto tile_range = [&](int pair, const PairParams &pp, int &t0, int &t1, int &p1) {
        const int sp = a.two_pass ? a.split[pair] : pp.n;
        const int p0 = a.pass ? sp : 0;
        p1 = a.pass ? pp.n : sp;
        t0 = p0 / NT;
        t1 = p1 > p0 ? (p1 + NT - 1) / NT : t0;
    };
    // pair-relative slot of logical model j of the pair (or -1)
    auto slot_of = [&](int pair, int j) -> int {
        if (a.list) return j < a.list_cnt[pair] ? a.list[(size_t)pair * a.list_stride + j] : -1;
        const int *segc = a.seg_count + (size_t)pair * a.nseg;
        j += min(a.first, segc[0]);
        for (int seg = 0; seg < a.nseg; ++seg) {
            const int c = segc[seg];
            if (j < c) return seg * (4 * SEG) + j;
            j -= c;
        }
        return -1;
    };

    if (warp == 0) {
        // ===== TMA producer =====
        int st = 0;
        uint32_t ph = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int pair = pair_of(item);
            const PairParams pp = a.pairs[pair];
            int t0, t1, p1;
            tile_range(pair, pp, t0, t1, p1);
            for (int t = t0; t < t1; ++t) {
                mbar_wait(&b_empty[st], ph ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(&b_full[st], B_STAGE_BYTES);
                    tma_load_2d(sB + st * B_STAGE_BYTES, &tmap, 0, (int)(pp.off + (long long)t * NT), &b_full[st]);
                }
                __syncwarp();
                if (++st == B_STAGES) { st = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: per point tile one group of 6 MMAs per M-tile, each group into its own accumulator slot =====
        int st = 0, k = 0;
        uint32_t ph = 0;
        unsigned seq = 0;   // running (point tile, M-tile) index: slot = seq % SLOTS
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++k) {
            const int pair = pair_of(item);
            const PairParams pp = a.pairs[pair];
            int t0, t1, p1;
            tile_range(pair, pp, t0, t1, p1);
            const int ab = k & 1;
            mbar_wait(&a_full[ab], (k >> 1) & 1);
            tc_fence_after();
            if (t1 == t0 && elect_one()) umma_commit(&a_empty[ab]);   // nothing to do for this item: hand the A buffer back
            __syncwarp();
            for (int t = t0; t < t1; ++t) {
                mbar_wait(&b_full[st], ph);
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const unsigned slot = (seq + m) % SLOTS;
                    mbar_wait(&slot_empty[slot], (((seq + m) / SLOTS) & 1) ^ 1);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t b_base = smem_u32(sB + st * B_STAGE_BYTES);
                        const uint64_t b0 = desc_sw128(b_base), b1 = desc_sw128(b_base + 32), b2 = desc_sw128(b_base + 64),
                                       b3 = desc_sw128(b_base + 96), bK = desc_kslice(smem_u32(sK));
                        const uint32_t ar = tmem_a + (uint32_t)((ab * MT + m) * A_COLS);
                        const uint32_t dC = tmem_base + slot * (2 * NT), dT = dC + NT;
                        umma_tf32_ts(dC, ar, b0, IDESC, 0);        // E_hi . phi_hi
                        umma_tf32_ts(dC, ar + 8, b0, IDESC, 1);    // E_lo . phi_hi
                        umma_tf32_ts(dC, ar, b1, IDESC, 1);        // E_hi . phi_lo
                        umma_tf32_ts(dC, ar + 24, bK, IDESC, 1);   // E22 (hi, lo) . (1, 1)            [constant slice]
                        umma_tf32_ts(dT, ar + 16, b2, IDESC, 0);   // G_0..7 . psi_0..7
                        umma_tf32_ts(dT, ar + 24, b3, IDESC, 1);   // G_8, G_9, const . (x2x, x2y, 1)
                        umma_commit(&slot_full[slot]);
                        if (m == MT - 1) {
                            umma_commit(&b_empty[st]);
                            if (t == t1 - 1) umma_commit(&a_empty[ab]);
                        }
                    }
                    __syncwarp();
                }
                seq += MT;
                if (++st == B_STAGES) { st = 0; ph ^= 1; }
            }
        }
    } else if (warp >= EPI_WARP0 && warp < BUILD_WARP0) {
        // ===== epilogue: group m = the four warps of M-tile m, thread = model =====
        const int m = (warp - EPI_WARP0) / 4, q = warp & 3;
        const int row = m * 128 + q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        unsigned seq = (unsigned)m;
        unsigned long long evaluated = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int pair = pair_of(item);
            const PairParams pp = a.pairs[pair];
            int t0, t1, n;   // n = end of this pass's correspondence range
            tile_range(pair, pp, t0, t1, n);
            float acc0 = 0.f;
            unsigned long long accA = 0ull, accB = 0ull;   // packed FP32 pairs
            for (int t = t0; t < t1; ++t, seq += MT) {
                const unsigned slot = seq % SLOTS;
                mbar_wait(&slot_full[slot], (seq / SLOTS) & 1);
                tc_fence_after();
                const uint32_t cC = lane_addr + slot * (2 * NT), cT = cC + NT;
                const int nv = min(NT, n - t * NT);
                if (MODE != 2) {
#pragma unroll
                    for (int h = 0; h < NT; h += 32) {
                        uint32_t c[32], tt[32];
                        tmem_ld32(cC + h, c);
                        tmem_ld32(cT + h, tt);
                        tmem_ld_wait();
                        if (a.debug && item == 0) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const int col = t * NT + h + j;
                                if (col < a.debug_cols) {
                                    a.debug[((size_t)row * 2 + 0) * a.debug_cols + col] = __uint_as_float(c[j]);
                                    a.debug[((size_t)row * 2 + 1) * a.debug_cols + col] = __uint_as_float(tt[j]);
                                }
                            }
                        }
                        if (MODE == 1) {
                            acc0 += __uint_as_float(c[0] ^ c[31]) + __uint_as_float(tt[0] ^ tt[31]);
                        } else if (nv >= h + 32) {
                            // 1 FFMA.SAT per point-score + 1 packed FADD2 per two; four independent accumulation chains
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const float s0 = fma_sat(__uint_as_float(c[j]), __uint_as_float(c[j]), __uint_as_float(tt[j]));
                                const float s1 = fma_sat(__uint_as_float(c[j + 1]), __uint_as_float(c[j + 1]), __uint_as_float(tt[j + 1]));
                                const float s2 = fma_sat(__uint_as_float(c[j + 2]), __uint_as_float(c[j + 2]), __uint_as_float(tt[j + 2]));
                                const float s3 = fma_sat(__uint_as_float(c[j + 3]), __uint_as_float(c[j + 3]), __uint_as_float(tt[j + 3]));
                                accA = add2(accA, pack2f(s0, s1));
                                accB = add2(accB, pack2f(s2, s3));
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (h + j < nv) acc0 += fma_sat(__uint_as_float(c[j]), __uint_as_float(c[j]), __uint_as_float(tt[j]));
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&slot_empty[slot]);
            }
            const int rel = slot_of(pair, (item - a.item_prefix[pair]) * TILE_MODELS + row);
            if (rel >= 0) {
                float a0, a1, b0, b1;
                unpack2f(accA, a0, a1);
                unpack2f(accB, b0, b1);
                // every addend is exactly 0 or 1 (model_row's scaling), so the FP32 sums are exact counts
                const int cnt = (int)(acc0 + a0 + a1 + b0 + b1);
                int *o = a.out + ((size_t)pair * a.nseg) * (size_t)(4 * SEG) + rel;
                *o = a.pass ? *o + cnt : cnt;
                evaluated += (unsigned long long)(t1 > t0 ? n - t0 * NT : 0);
            }
        }
        if (a.evaluated) {
            for (int o = 16; o > 0; o >>= 1) evaluated += __shfl_xor_sync(0xffffffffu, evaluated, o);
            if (lane == 0 && evaluated) atomicAdd(a.evaluated, evaluated);
        }
    } else if (warp >= BUILD_WARP0) {
        // ===== A builder: four warps = the 128 TMEM lanes; thread = row, MT rows per work item, written with tcgen05.st =====
        const int q = warp & 3;
        const uint32_t lane_addr = tmem_a + ((uint32_t)(q * 32) << 16);
        int k = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++k) {
            const int pair = pair_of(item);
            const PairParams pp = a.pairs[pair];
            const int ab = k & 1;
            mbar_wait(&a_empty[ab], ((k >> 1) & 1) ^ 1);
            tc_fence_after();
            const int j0 = (item - a.item_prefix[pair]) * TILE_MODELS;
#pragma unroll 1
            for (int m = 0; m < MT; ++m) {
                const int slot = slot_of(pair, j0 + m * 128 + q * 32 + lane);
                float r0[32];
                if (slot >= 0) {
                    const Model mdl = a.models[((size_t)pair * a.nseg) * (size_t)(4 * SEG) + slot];
                    const M3 E = a.pose ? essential_from_motion(mdl.q, mdl.t) : fundamental_from_model(mdl);
                    model_row(E, pp.thr, pp.Mmax, pp.mmax, r0);
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) r0[i] = 0.f;
                }
                const uint32_t ta = lane_addr + (uint32_t)((ab * MT + m) * A_COLS);
                tmem_st8(ta, r0);
                tmem_st8(ta + 8, r0 + 8);
                tmem_st8(ta + 16, r0 + 16);
                tmem_st8(ta + 24, r0 + 24);
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&a_full[ab]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}
#endif  // __CUDACC__

}  // namespace tc
}  // namespace rp
