// rp_kernels.cuh — CUDA kernels of the batched RePoseD LO-RANSAC (sm_100a).
//
// Pipeline per chunk of image pairs (SURVEY.md §3.2 restated as a parallel schedule, §7 step 4):
//   prepare  -> normalised points (FP64 + FP32 copies), unit bearings, per-pair thresholds
//   sample   -> RandomSampler::generate_sample for every iteration (warp per pair, speculative)
//   solve    -> minimal solvers, one thread per RANSAC iteration, ordered per-segment compaction
//   score    -> hypotheses x correspondences MSAC (the dominant kernel)
//   scan     -> sequential-semantics prefix scan: which minimal models trigger LO / become best
//   lm       -> batched Levenberg-Marquardt (LO, final LO, final refinement), block per problem
//   merge    -> replay of score_models()/ransac() bookkeeping in trigger order
// HBM layout: every per-hypothesis array is indexed by a "slot"; the minimal models of
// (pair p, iteration segment s) own slots [(p*nseg+s)*4*SEG, +count) in iteration order.
#pragma once
#include <cuda_runtime.h>
#include "rp_types.cuh"
#include "rp_solvers.cuh"
#include "rp_score.cuh"
#include "rp_lm_kernel.cuh"
#include "rp_tc.cuh"
#include "rp_order.cuh"

namespace rp {

// ---------------------------------------------------------------------------------------------
// prepare: P1/P2 pre-processing (estimate_monodepth_relative_pose so@0x224170: Camera::unproject,
// threshold scaling by 0.5(1/f1+1/f2); focal variants so@0x223300/0x223a40: normalize_points
// so@0x4f6ae0 with a SEQUENTIAL sum in index order, thresholds / loss_scale divided by it).
// One warp per pair.
struct PrepareArgs {
    int variant;
    int n_pairs;
    const long long *offsets;  // [n_pairs+1], relative to the chunk
    const double *x1, *x2;     // [N,2] pixels
    const double *cams;        // [n_pairs,8] or null
    double max_epipolar_error, max_reproj_error, loss_scale;
    Pt64 *pts64;
    float4 *pts32;
    float *pts32p;  // pair-interleaved copy for the packed-FP32 bound kernel: per two correspondences (a,b)
                    // [x1x_a,x1x_b, x1y_a,x1y_b, x2x_a,x2x_b, x2y_a,x2y_b]
    Bear *bear;
    PairParams *pairs;
};

// writes one correspondence into the pair-interleaved layout
RP_D void store_interleaved(float *pts32p, long long pbase, int k, float x1x, float x1y, float x2x, float x2y) {
    float *q = pts32p + (pbase + (k >> 1)) * 8 + (k & 1);
    q[0] = x1x; q[2] = x1y; q[4] = x2x; q[6] = x2y;
}

__global__ void prepare_kernel(PrepareArgs a) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.n_pairs) return;
    const long long off = a.offsets[warp];
    const int n = (int)(a.offsets[warp + 1] - off);
    const bool pose = a.variant == RP_CALIB || a.variant == RP_CALIB_SHIFT;
    PairParams pp;
    pp.off = off;
    pp.n = n;
    pp.valid = n >= 3;
    pp.nscale = 1.0;
    pp.pbase = (off + warp + 1) >> 1;  // b_{p+1} - b_p >= ceil(n_p / 2)
    if ((n & 1) && lane == 0) store_interleaved(a.pts32p, pp.pbase, n, 0.f, 0.f, 0.f, 0.f);  // padding half
    double Mmax = 0.0, mmax = 0.0;
    if (pose) {
        const double *c = a.cams + 8 * (long long)warp;
        const double fx1 = c[0], fy1 = c[1], cx1 = c[2], cy1 = c[3], fx2 = c[4], fy2 = c[5], cx2 = c[6], cy2 = c[7];
        const double fo1 = 0.5 * (fx1 + fy1), fo2 = 0.5 * (fx2 + fy2);
        const double k = 0.5 * (1.0 / fo1 + 1.0 / fo2);
        pp.thr = a.max_epipolar_error * k;
        const double rep = a.max_reproj_error * k;
        pp.scale_reproj = rep > 0.0 ? (pp.thr * pp.thr) / (rep * rep) : 0.0;
        pp.lo_loss_scale = pp.thr;
        pp.final_loss_scale = 0.5 * pp.thr;  // user loss_scale is overwritten for this variant
        for (int k0 = lane; k0 < n; k0 += 32) {
            const long long g = off + k0;
            Pt64 p;
            p.x1_0 = (a.x1[2 * g] - cx1) / fx1;
            p.x1_1 = (a.x1[2 * g + 1] - cy1) / fy1;
            p.x2_0 = (a.x2[2 * g] - cx2) / fx2;
            p.x2_1 = (a.x2[2 * g + 1] - cy2) / fy2;
            a.pts64[g] = p;
            a.pts32[g] = make_float4((float)p.x1_0, (float)p.x1_1, (float)p.x2_0, (float)p.x2_1);
            store_interleaved(a.pts32p, pp.pbase, k0, (float)p.x1_0, (float)p.x1_1, (float)p.x2_0, (float)p.x2_1);
            const V3 b1 = bearing(p.x1_0, p.x1_1), b2 = bearing(p.x2_0, p.x2_1);
            Bear b;
            b.b1x = b1.x; b.b1y = b1.y; b.b1z = b1.z; b.b2x = b2.x; b.b2y = b2.y; b.b2z = b2.z;
            a.bear[g] = b;
            const double m1 = fabs(p.x1_0) + fabs(p.x1_1) + 1.0, m2 = fabs(p.x2_0) + fabs(p.x2_1) + 1.0;
            Mmax = fmax(Mmax, m1 * m2);
            mmax = fmax(mmax, fmax(m1, m2));
        }
    } else {
        // sequential sum s += |x1_k|; s += |x2_k| in index order: lanes compute the norms of 32
        // correspondences at a time, lane 0 adds them in order
        double s = 0.0;
        for (int base = 0; base < n; base += 32) {
            const int k0 = base + lane;
            double n1 = 0.0, n2 = 0.0;
            if (k0 < n) {
                const long long g = off + k0;
                const double ax = a.x1[2 * g], ay = a.x1[2 * g + 1], bx = a.x2[2 * g], by = a.x2[2 * g + 1];
                n1 = sqrt(ax * ax + ay * ay);
                n2 = sqrt(bx * bx + by * by);
            }
            const int cntv = min(32, n - base);
            for (int l = 0; l < cntv; ++l) {
                const double v1 = __shfl_sync(0xffffffffu, n1, l);
                const double v2 = __shfl_sync(0xffffffffu, n2, l);
                s += v1;
                s += v2;
            }
        }
        const double nscale = s / (sqrt(2.0) * (double)n);
        pp.nscale = nscale;
        pp.thr = a.max_epipolar_error / nscale;
        const double rep = a.max_reproj_error / nscale;
        pp.scale_reproj = rep > 0.0 ? (pp.thr * pp.thr) / (rep * rep) : 0.0;
        // VaryingFocalMonodepthPoseEstimator::refine_model so@0x4fb0a0 leaves loss_scale at the
        // BundleOptions default 1.0; the shared-focal estimator so@0x4fad60 uses the threshold
        pp.lo_loss_scale = a.variant == RP_VARYING ? 1.0 : pp.thr;
        pp.final_loss_scale = a.loss_scale / nscale;
        for (int k0 = lane; k0 < n; k0 += 32) {
            const long long g = off + k0;
            Pt64 p;
            p.x1_0 = a.x1[2 * g] / nscale;
            p.x1_1 = a.x1[2 * g + 1] / nscale;
            p.x2_0 = a.x2[2 * g] / nscale;
            p.x2_1 = a.x2[2 * g + 1] / nscale;
            a.pts64[g] = p;
            a.pts32[g] = make_float4((float)p.x1_0, (float)p.x1_1, (float)p.x2_0, (float)p.x2_1);
            store_interleaved(a.pts32p, pp.pbase, k0, (float)p.x1_0, (float)p.x1_1, (float)p.x2_0, (float)p.x2_1);
            const double m1 = fabs(p.x1_0) + fabs(p.x1_1) + 1.0, m2 = fabs(p.x2_0) + fabs(p.x2_1) + 1.0;
            Mmax = fmax(Mmax, m1 * m2);
            mmax = fmax(mmax, fmax(m1, m2));
        }
    }
    Mmax = warp_max(Mmax);
    mmax = warp_max(mmax);
    if (lane == 0) {
        pp.sq_thr = pp.thr * pp.thr;
        pp.Mmax = Mmax * 1.000001;  // cover the FP32 rounding of the inputs themselves
        pp.mmax = mmax * 1.000001;
        a.pairs[warp] = pp;
    }
}

// ---------------------------------------------------------------------------------------------
// sample: R2 (RandomSampler::generate_sample so@0x4f8970 -> draw_sample so@0x4f87f0 -> random_int
// so@0x4f87a0).  SplitMix64 is counter based, but the rejection of duplicate indices makes the
// number of draws per sample data dependent.  A warp speculates 32 iterations at 3 draws each;
// the first lane that sees a duplicate replays its sample sequentially and re-bases the rest.
RP_D uint32_t splitmix_int(uint64_t state_after_increment) {
    uint64_t z = state_after_increment;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    z = z ^ (z >> 31);
    return (uint32_t)z;
}
RP_D uint32_t draw_index(uint64_t &state, uint64_t n) {
    state += 0x9e3779b97f4a7c15ULL;
    const int32_t v = (int32_t)splitmix_int(state);
    return (uint32_t)((uint64_t)(int64_t)v % n);  // (size_t)(int64)ret % N as the reference does
}

__global__ void sample_kernel(int n_pairs, int iters, const PairParams *pairs, uint64_t seed, int *samples) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_pairs) return;
    const PairParams pp = pairs[warp];
    if (!pp.valid) return;
    const uint64_t n = (uint64_t)pp.n;
    const uint64_t G = 0x9e3779b97f4a7c15ULL;
    int *out = samples + (size_t)warp * iters * 3;
    uint64_t base = seed;
    for (int it0 = 0; it0 < iters; it0 += 32) {
        const int group = min(32, iters - it0);
        int done = 0;
        while (done < group) {
            uint64_t st = base + 3ULL * G * (uint64_t)(lane >= done ? lane - done : 0);
            const uint64_t st0 = st;
            const uint32_t i0 = draw_index(st, n), i1 = draw_index(st, n), i2 = draw_index(st, n);
            const bool active = lane >= done && lane < group;
            const bool dup = active && (i1 == i0 || i2 == i0 || i2 == i1);
            const unsigned m = __ballot_sync(0xffffffffu, dup);
            const int first = m ? (__ffs(m) - 1) : group;
            if (active && lane < first) {
                int *o = out + (size_t)(it0 + lane) * 3;
                o[0] = (int)i0; o[1] = (int)i1; o[2] = (int)i2;
            }
            if (first < group) {
                uint64_t s2 = st0;
                if (lane == first) {
                    uint32_t s[3];
                    for (int i = 0; i < 3; ++i) {
                        bool ok = false;
                        while (!ok) {
                            s[i] = draw_index(s2, n);
                            ok = true;
                            for (int j = 0; j < i; ++j) if (s[i] == s[j]) ok = false;
                        }
                    }
                    int *o = out + (size_t)(it0 + lane) * 3;
                    o[0] = (int)s[0]; o[1] = (int)s[1]; o[2] = (int)s[2];
                }
                base = __shfl_sync(0xffffffffu, s2, first);
                done = first + 1;
            } else {
                base = base + 3ULL * G * (uint64_t)(group - done);
                done = group;
            }
        }
    }
}

// PROSAC branch of the same sampler (generate_sample so@0x4f8970 with use_prosac, growth table of
// initialize_prosac so@0x4f8a20).  Iteration j (sample_k = j+1 on entry) is a PROSAC draw while
// j+1 < max_prosac: two distinct indices out of the first subset_sz-1 points plus the point subset_sz-1;
// afterwards the uniform 3-draw.  subset_sz does not depend on the random numbers: it grows by one
// whenever sample_k passes growth[subset_sz-1], and growth[] is a running sum that only ever has to be
// advanced by one entry at a time, so no table is stored: every lane of the warp tracks
// (subset_sz, T_n, growth[subset_sz-1]) through the 32 iterations of a step and keeps the value of its own
// iteration.  The random state is then speculated exactly as in sample_kernel (2 draws per PROSAC
// iteration, 3 per uniform one) with a sequential replay of the first lane that hits a duplicate.
struct ProsacState {
    unsigned long long subset_sz;   // current subset size (>= 3)
    unsigned long long gidx;        // index n for which gval == growth[n] (recurrence advanced so far)
    unsigned long long gval;        // growth[gidx] ("T_n_prime")
    double T_n;
};

RP_D void prosac_init(ProsacState &ps, unsigned long long num_data, unsigned long long max_prosac) {
    double T_n = (double)max_prosac;
    for (unsigned long long i = 0; i < 3; ++i) T_n *= (double)(3 - i) / (double)(num_data - i);
    ps.subset_sz = 3; ps.gidx = 2; ps.gval = 1; ps.T_n = T_n;
}
// state update at the end of a PROSAC generate_sample call; k = sample_k after its increment
RP_D void prosac_advance(ProsacState &ps, unsigned long long k, unsigned long long num_data, unsigned long long max_prosac) {
    if (k < max_prosac && k > ps.gval && ps.subset_sz < num_data) {
        // subset_sz + 1 <= num_data: growth[subset_sz] is the next entry of the recurrence
        const unsigned long long n = ps.subset_sz;  // == gidx + 1 whenever n >= 3
        const double T_next = ((double)n + 1.0) * ps.T_n / (((double)n + 1.0) - 3.0);
        ps.gval = (unsigned long long)((double)ps.gval + ceil(T_next - ps.T_n));
        ps.T_n = T_next;
        ps.gidx = n;
        ps.subset_sz = n + 1;
    }
}

__global__ void sample_prosac_kernel(int n_pairs, int iters, const PairParams *pairs, uint64_t seed,
                                     unsigned long long max_prosac, int *samples) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_pairs) return;
    const PairParams pp = pairs[warp];
    if (!pp.valid) return;
    const uint64_t n = (uint64_t)pp.n;
    const uint64_t G = 0x9e3779b97f4a7c15ULL;
    int *out = samples + (size_t)warp * iters * 3;
    uint64_t base = seed;
    ProsacState ps;
    prosac_init(ps, n, max_prosac);
    for (int it0 = 0; it0 < iters; it0 += 32) {
        const int group = min(32, iters - it0);
        // PROSAC iterations of this step: j + 1 < max_prosac
        const long long np_ll = (long long)max_prosac - 1 - (long long)it0;
        const int n_prosac = (int)max(0ll, min((long long)group, np_ll));
        unsigned long long my_sz = 3;
        for (int l = 0; l < n_prosac; ++l) {
            if (l == lane) my_sz = ps.subset_sz;
            prosac_advance(ps, (unsigned long long)(it0 + l) + 2ull, n, max_prosac);
        }
        const bool prosac = lane < n_prosac;
        const uint64_t mod = prosac ? my_sz - 1 : n;
        int done = 0;
        while (done < group) {
            // draws consumed by the lanes done..lane-1 of this round
            const int lp = max(lane, done);
            const int pro_before = max(0, min(lp, n_prosac) - min(done, n_prosac));
            const uint64_t draws_before = 2ULL * (uint64_t)pro_before + 3ULL * (uint64_t)(lp - done - pro_before);
            uint64_t st = base + G * draws_before;
            const uint64_t st0 = st;
            const uint32_t i0 = draw_index(st, mod), i1 = draw_index(st, mod);
            const uint32_t i2 = prosac ? (uint32_t)(my_sz - 1) : draw_index(st, mod);
            const bool active = lane >= done && lane < group;
            const bool dup = active && (i1 == i0 || (!prosac && (i2 == i0 || i2 == i1)));
            const unsigned m = __ballot_sync(0xffffffffu, dup);
            const int first = m ? (__ffs(m) - 1) : group;
            if (active && lane < first) {
                int *o = out + (size_t)(it0 + lane) * 3;
                o[0] = (int)i0; o[1] = (int)i1; o[2] = (int)i2;
            }
            if (first < group) {
                uint64_t s2 = st0;
                if (lane == first) {
                    uint32_t s[3];
                    const int nd = prosac ? 2 : 3;
                    for (int i = 0; i < nd; ++i) {
                        bool ok = false;
                        while (!ok) {
                            s[i] = draw_index(s2, mod);
                            ok = true;
                            for (int j = 0; j < i; ++j) if (s[i] == s[j]) ok = false;
                        }
                    }
                    if (prosac) s[2] = (uint32_t)(my_sz - 1);
                    int *o = out + (size_t)(it0 + lane) * 3;
                    o[0] = (int)s[0]; o[1] = (int)s[1]; o[2] = (int)s[2];
                }
                base = __shfl_sync(0xffffffffu, s2, first);
                done = first + 1;
            } else {
                const int pro_rest = max(0, min(group, n_prosac) - min(done, n_prosac));
                base = base + G * (2ULL * (uint64_t)pro_rest + 3ULL * (uint64_t)(group - done - pro_rest));
                done = group;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// solve: one thread per RANSAC iteration, block = (segment of SEG iterations, pair).  Solutions
// are compacted in (iteration, solution) order with a block-wide exclusive scan per round.
struct SolveArgs {
    int variant, iters, nseg;
    const PairParams *pairs;
    const int *samples;
    const Pt64 *pts64;
    const double *d1, *d2;
    Model *models;   // slots
    int *hyp_iter;   // slots
    int *seg_count;  // [n_pairs*nseg]
};

template <int VARIANT>
__global__ void __launch_bounds__(SOLVE_THREADS, RP_SOLVE_MIN_BLOCKS) solve_kernel(SolveArgs a) {
    const int seg = blockIdx.x, pair = blockIdx.y;
    const PairParams pp = a.pairs[pair];
    __shared__ int warp_tot[SOLVE_THREADS / 32];
    __shared__ int running_s;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const size_t slot0 = ((size_t)pair * a.nseg + seg) * (size_t)(4 * SEG);
    if (tid == 0) running_s = 0;
    __syncthreads();
    if (!pp.valid) {
        if (tid == 0) a.seg_count[pair * a.nseg + seg] = 0;
        return;
    }
    for (int round = 0; round < SEG / SOLVE_THREADS; ++round) {
        const int it = seg * SEG + round * SOLVE_THREADS + tid;
        ModelSet ms;
        ms.n = 0;
        if (it < a.iters) {
            const int *s = a.samples + ((size_t)pair * a.iters + it) * 3;
            Triplet t;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const long long g = pp.off + s[i];
                const Pt64 p = a.pts64[g];
                t.p1[i] = v3(p.x1_0, p.x1_1, 1.0);
                t.p2[i] = v3(p.x2_0, p.x2_1, 1.0);
                t.d1[i] = a.d1[g];
                t.d2[i] = a.d2[g];
            }
            if (VARIANT == RP_CALIB) solve_calib_scale(t, ms);
            else if (VARIANT == RP_CALIB_SHIFT) solve_calib_shift(t, ms);
            else if (VARIANT == RP_SHARED) solve_shared_focal(t, ms);
            else solve_varying_focal(t, ms);
        }
        // exclusive scan of ms.n over the block, in thread (= iteration) order
        int incl = ms.n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int w = 0; w < SOLVE_THREADS / 32; ++w) {
            const int v = warp_tot[w];
            if (w < wid) wbase += v;
            total += v;
        }
        const int running = running_s;
        const size_t dst = slot0 + running + wbase + (incl - ms.n);
        if (ms.n > 0) { a.models[dst] = ms.m[0]; a.hyp_iter[dst] = it; }
        if (ms.n > 1) { a.models[dst + 1] = ms.m[1]; a.hyp_iter[dst + 1] = it; }
        if (ms.n > 2) { a.models[dst + 2] = ms.m[2]; a.hyp_iter[dst + 2] = it; }
        if (ms.n > 3) { a.models[dst + 3] = ms.m[3]; a.hyp_iter[dst + 3] = it; }
        __syncthreads();
        if (tid == 0) running_s = running + total;
        __syncthreads();
    }
    if (tid == 0) a.seg_count[pair * a.nseg + seg] = running_s;
}

// Two-phase form of solve_kernel for the solvers with 0..4 solutions per sample (P3P + scale, scale+shift,
// shared focal).  Phase A (thread per iteration): the uniform part up to the filtered candidate roots
// (solve_roots), appended IN ORDER to a shared-memory queue (block-wide exclusive scan).  Phase B (thread per
// queued root, 256 at a time, so every lane works): the per-solution part (solve_finish: polish + pose
// assembly), model written straight to its final slot (queue position = slot).  Same arithmetic as the
// one-call solvers, hence bit-identical models; the thread-per-iteration loop over the roots ran at 12.8 of
// 32 active lanes (ncu, scale+shift).  CAND = P3PCand | ShiftCand | FocalCand selects the solver.
constexpr int SOLVE_QCAP = 4 * SOLVE_THREADS + SOLVE_THREADS;  // one round of appends on top of < 256 leftovers

RP_D Triplet load_triplet(const SolveArgs &a, const PairParams &pp, int pair, int it) {
    const int *s = a.samples + ((size_t)pair * a.iters + it) * 3;
    Triplet t;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const long long g = pp.off + s[i];
        const Pt64 p = a.pts64[g];
        t.p1[i] = v3(p.x1_0, p.x1_1, 1.0);
        t.p2[i] = v3(p.x2_0, p.x2_1, 1.0);
        t.d1[i] = a.d1[g];
        t.d2[i] = a.d2[g];
    }
    return t;
}

#ifndef RP_SOLVE2_MIN_BLOCKS
#define RP_SOLVE2_MIN_BLOCKS 3   // 85 registers: scale+shift per 10k pairs 23.1 / 17.8 / 16.8 / 17.4 ms at 1 / 2 / 3 / 4 blocks per SM
#endif
template <class CAND>
__global__ void __launch_bounds__(SOLVE_THREADS, RP_SOLVE2_MIN_BLOCKS) solve2_kernel(SolveArgs a) {
    const int seg = blockIdx.x, pair = blockIdx.y;
    const PairParams pp = a.pairs[pair];
    __shared__ int warp_tot[SOLVE_THREADS / 32];
    __shared__ CAND qc[SOLVE_QCAP];
    __shared__ int qit[SOLVE_QCAP];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const size_t slot0 = ((size_t)pair * a.nseg + seg) * (size_t)(4 * SEG);
    if (!pp.valid) {
        if (tid == 0) a.seg_count[pair * a.nseg + seg] = 0;
        return;
    }
    int head = 0, tail = 0;  // queue positions == slot indices of the segment (uniform across the block)
    auto drain = [&](int upto) {  // finish the queued roots [head, upto)
        for (int q = head + tid; q < upto; q += SOLVE_THREADS) {
            const int it = qit[q % SOLVE_QCAP];
            const CAND c = qc[q % SOLVE_QCAP];
            const Triplet t = load_triplet(a, pp, pair, it);
            a.models[slot0 + q] = solve_finish(t, c);
            a.hyp_iter[slot0 + q] = it;
        }
        head = upto;
    };
    for (int round = 0; round < SEG / SOLVE_THREADS; ++round) {
        const int it = seg * SEG + round * SOLVE_THREADS + tid;
        CAND c0, c1, c2, c3;
        int n = 0;
        if (it < a.iters) n = solve_roots(load_triplet(a, pp, pair, it), c0, c1, c2, c3);
        int incl = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        __syncthreads();  // the previous drain has read its queue entries
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int w = 0; w < SOLVE_THREADS / 32; ++w) {
            const int v = warp_tot[w];
            if (w < wid) wbase += v;
            total += v;
        }
        const int pos = tail + wbase + (incl - n);
        if (n > 0) { qc[pos % SOLVE_QCAP] = c0; qit[pos % SOLVE_QCAP] = it; }
        if (n > 1) { qc[(pos + 1) % SOLVE_QCAP] = c1; qit[(pos + 1) % SOLVE_QCAP] = it; }
        if (n > 2) { qc[(pos + 2) % SOLVE_QCAP] = c2; qit[(pos + 2) % SOLVE_QCAP] = it; }
        if (n > 3) { qc[(pos + 3) % SOLVE_QCAP] = c3; qit[(pos + 3) % SOLVE_QCAP] = it; }
        tail += total;
        __syncthreads();
        // full batches only; the remainder waits for the next round (or the final drain)
        const int full = head + ((tail - head) / SOLVE_THREADS) * SOLVE_THREADS;
        if (full > head) drain(full);
    }
    drain(tail);
    if (tid == 0) a.seg_count[pair * a.nseg + seg] = tail;
}

// stage entry point helper: independent triplets, one thread each (rp_solve_batch)
__global__ void solve_problems_kernel(int variant, long long n, const double *x1h, const double *x2h,
                                      const double *d1, const double *d2, Model *models, int *counts) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Triplet t;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        t.p1[k] = v3(x1h[9 * i + 3 * k], x1h[9 * i + 3 * k + 1], x1h[9 * i + 3 * k + 2]);
        t.p2[k] = v3(x2h[9 * i + 3 * k], x2h[9 * i + 3 * k + 1], x2h[9 * i + 3 * k + 2]);
        t.d1[k] = d1[3 * i + k];
        t.d2[k] = d2[3 * i + k];
    }
    ModelSet ms;
    solve_minimal(variant, t, ms);
    counts[i] = ms.n;
    if (ms.n > 0) models[4 * i] = ms.m[0];
    if (ms.n > 1) models[4 * i + 1] = ms.m[1];
    if (ms.n > 2) models[4 * i + 2] = ms.m[2];
    if (ms.n > 3) models[4 * i + 3] = ms.m[3];
}

// ---------------------------------------------------------------------------------------------
// work items of the scoring kernel: group e (a (pair, segment), or a pair) owns grp_cnt[e] models
// at slots [e*grp_stride, …); item = HB consecutive models of one group.  Exclusive scan of
// ceil(cnt/HB) over the groups; single block.
__global__ void build_items_kernel(int n_groups, const int *grp_cnt, int *item_prefix, int *n_items,
                                   long long *n_hyp_total, int gran = HB) {
    // tiles of 1024 groups: shuffle scan inside each warp, the 32 warp totals scanned by warp 0
    __shared__ int wtot[32];
    __shared__ long long whyp[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int carry = 0;          // items before this tile (uniform)
    long long hyps = 0;     // per-thread partial of the model count
    for (int base = 0; base < n_groups; base += 1024) {
        const int e = base + threadIdx.x;
        const int c = e < n_groups ? grp_cnt[e] : 0;
        const int v = (c + gran - 1) / gran;
        hyps += c;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        __syncthreads();  // wtot of the previous tile has been read
        if (lane == 31) wtot[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            const int w = wtot[lane];
            int wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            wtot[lane] = wi - w;  // exclusive
            if (lane == 31) whyp[0] = wi;  // tile total (reuses the 64-bit scratch)
        }
        __syncthreads();
        if (e < n_groups) item_prefix[e] = carry + wtot[wid] + incl - v;
        carry += (int)whyp[0];
    }
    // model count: warp sums, then thread 0
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) hyps += __shfl_xor_sync(0xffffffffu, hyps, o);
    __syncthreads();
    if (lane == 0) whyp[wid] = hyps;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long tot = 0;
        for (int w = 0; w < 32; ++w) tot += whyp[w];
        item_prefix[n_groups] = carry;
        *n_items = carry;
        if (n_hyp_total) *n_hyp_total = tot;
    }
}

// ---------------------------------------------------------------------------------------------
// score: SC / SF / I1.  Block = one work item = up to HB models of one pair against all of the
// pair's correspondences.  Lanes are correspondences (coalesced FP32 float4 loads, PT per thread),
// the models' E / F matrices are staged in shared memory and broadcast.  Tier 0 is the FP32
// filter, tier 1 the exact FP64 test (rp_score.cuh).  Inlier counts are exact; the MSAC score is
// thr^2 (N - count) + sum of inlier r^2 with a fixed (deterministic) summation order.
struct ScoreArgs {
    int n_groups, grp_stride, grp_per_pair;
    const int *grp_cnt;
    const int *item_prefix;  // [n_groups+1]
    const int *n_items;
    const PairParams *pairs;
    const Model *models;     // slots
    const float4 *pts32;
    const Pt64 *pts64;
    const Bear *bear;
    double *score;           // slots
    int *count;              // slots
    unsigned char *mask;     // optional, per correspondence; only with one model per pair
    unsigned long long *point_scores;  // optional counter
    const int *slot_list;    // optional indirection: model i of group e lives at slot
    int list_stride;         //   e*grp_stride + slot_list[e*list_stride + i]   (survivor lists)
    int *work_counter;       // zeroed before the launch: blocks take items dynamically
};

struct HypConst {
    M3 E;      // essential (pose variants) or fundamental matrix
    Quat q;
    V3 t;
};

constexpr int QCAP = 32 + 32 * PT;  // per-warp candidate queue: < 32 left over + one full push

struct ScoreShared {
    HypConst hc[HB];
    Filter32 hf[HB];
    Cheir32 hch[HB];
    double psum[HB][SCORE_WARPS];  // per-warp partial sums of inlier r^2 (only warp w touches [.][w])
    int pcnt[HB][SCORE_WARPS];
    unsigned queue[SCORE_WARPS][QCAP];
};

// tier 1 for up to 32 queued (model, correspondence) candidates, one per lane.  The queue content
// and order of a warp are a pure function of its inputs, and the reductions below have a fixed
// shape, so the FP64 sums are reproducible run to run (no floating-point atomics).
template <bool POSE, bool MASK>
__device__ __noinline__ void score_candidates(ScoreShared &sh, const ScoreArgs &a, const PairParams &pp,
                                              unsigned entry, bool active) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int h = active ? (int)(entry >> 24) : 0;
    const int k = (int)(entry & 0xffffffu);
    bool inl = false;
    double v = 0.0;
    if (active) {
        const long long g = pp.off + k;
        const Pt64 p = a.pts64[g];
        const double r2 = sampson_r2_exact(sh.hc[h].E, p.x1_0, p.x1_1, p.x2_0, p.x2_1);
        inl = r2 < pp.sq_thr;
        if (POSE && inl) {
            const int scr = cheirality32(sh.hch[h], (float)p.x1_0, (float)p.x1_1, (float)p.x2_0, (float)p.x2_1);
            if (scr == 0) {
                const Bear b = a.bear[g];
                inl = cheirality_exact(sh.hc[h].q, sh.hc[h].t, v3(b.b1x, b.b1y, b.b1z), v3(b.b2x, b.b2y, b.b2z));
            } else {
                inl = scr > 0;
            }
        }
        if (inl) {
            v = r2;
            if (MASK) a.mask[g] = 1;
        }
    }
    const unsigned inl_mask = __ballot_sync(0xffffffffu, inl);
    if (inl_mask == 0) return;
    const int h0 = __shfl_sync(0xffffffffu, h, __ffs(inl_mask) - 1);
    if (__all_sync(0xffffffffu, !inl || h == h0)) {
        // every inlier of this batch belongs to one model: butterfly sum, one update
        v = warp_sum(v);
        if (lane == 0) {
            sh.pcnt[h0][wid] += __popc(inl_mask);
            sh.psum[h0][wid] += v;
        }
        __syncwarp();
        return;
    }
    // general case: segmented inclusive scan over runs of equal model index (lane order)
    int c = inl ? 1 : 0;
    const int h_prev = __shfl_up_sync(0xffffffffu, h, 1);
    const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || h != h_prev);
    const int run_start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double vu = __shfl_up_sync(0xffffffffu, v, o);
        const int cu = __shfl_up_sync(0xffffffffu, c, o);
        if (lane - o >= run_start) { v += vu; c += cu; }
    }
    const bool tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
    const bool do_add = tail && c > 0;
    const unsigned add_mask = __ballot_sync(0xffffffffu, do_add);
    unsigned rank = 0;
    if (do_add) rank = __popc(__match_any_sync(add_mask, h) & lt_mask);  // same model in two runs of the batch
    const unsigned max_rank = __reduce_max_sync(0xffffffffu, rank);
    for (unsigned r = 0; r <= max_rank; ++r) {
        if (do_add && rank == r) {
            sh.pcnt[h][wid] += c;
            sh.psum[h][wid] += v;
        }
        __syncwarp();
    }
}

template <bool POSE, bool MASK>
__global__ void __launch_bounds__(SCORE_THREADS) score_kernel(ScoreArgs a) {
    __shared__ ScoreShared sh;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int n_items = *a.n_items;
    unsigned *q = sh.queue[wid];
    __shared__ int item_s;
    // items differ in cost (share of candidates that reach the exact tier): blocks draw them from a counter
    for (;;) {
        __syncthreads();
        if (tid == 0) item_s = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int item = item_s;
        if (item >= n_items) break;
        // group of this item: last e with item_prefix[e] <= item
        int lo = 0, hi = a.n_groups;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (a.item_prefix[mid] <= item) lo = mid; else hi = mid;
        }
        const int e = lo;
        const int pair = e / a.grp_per_pair;
        const int h0 = (item - a.item_prefix[e]) * HB;
        const int nh = min(HB, a.grp_cnt[e] - h0);
        const size_t slot0 = (size_t)e * a.grp_stride + h0;
        const PairParams pp = a.pairs[pair];
        __syncthreads();  // previous item's shared state fully consumed
        size_t my_slot = slot0 + tid;
        if (a.slot_list && tid < nh) my_slot = (size_t)e * a.grp_stride + a.slot_list[(size_t)e * a.list_stride + h0 + tid];
        if (tid < nh) {
            const Model m = a.models[my_slot];
            HypConst c;
            c.E = POSE ? essential_from_motion(m.q, m.t) : fundamental_from_model(m);
            c.q = m.q;
            c.t = m.t;
            sh.hc[tid] = c;
            Filter32 f32 = make_filter32(c.E, pp.thr, pp.Mmax, pp.mmax);
            // non-finite E (NaN model from a minimal solver): r2 is NaN for every correspondence, i.e. no inliers
            // and score N thr^2 — exactly what the loop below leaves behind when it skips the model
            f32.pad = (isfinite(c.E.r0.x) && isfinite(c.E.r0.y) && isfinite(c.E.r0.z) && isfinite(c.E.r1.x) &&
                       isfinite(c.E.r1.y) && isfinite(c.E.r1.z) && isfinite(c.E.r2.x) && isfinite(c.E.r2.y) &&
                       isfinite(c.E.r2.z)) ? 0.f : 1.f;
            sh.hf[tid] = f32;
            if (POSE) sh.hch[tid] = make_cheir32(m.q, m.t);
        }
        for (int i = tid; i < HB * SCORE_WARPS; i += SCORE_THREADS) {
            (&sh.psum[0][0])[i] = 0.0;
            (&sh.pcnt[0][0])[i] = 0;
        }
        __syncthreads();
        const int n = pp.n;
        const int slice_pts = 32 * PT;
        const int n_slices = (n + slice_pts - 1) / slice_pts;
        int qn = 0;
        for (int sl = wid; sl < n_slices; sl += SCORE_WARPS) {
            float4 p[PT];
            bool valid[PT];
            const int kbase = sl * slice_pts + lane;
#pragma unroll
            for (int j = 0; j < PT; ++j) {
                const int k = kbase + j * 32;
                valid[j] = k < n;
                p[j] = valid[j] ? a.pts32[pp.off + k] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            for (int h = 0; h < nh; ++h) {
                const Filter32 f = sh.hf[h];
                if (f.pad != 0.f) continue;  // NaN model: nothing can be an inlier
                unsigned cand = 0;
#pragma unroll
                for (int j = 0; j < PT; ++j)
                    if (valid[j] && !certain_outlier32(f, p[j].x, p[j].y, p[j].z, p[j].w)) cand |= 1u << j;
                if (__any_sync(0xffffffffu, cand != 0)) {
                    // warp-aggregated push of (model, correspondence) candidates
#pragma unroll
                    for (int j = 0; j < PT; ++j) {
                        const bool c = (cand >> j) & 1u;
                        const unsigned m = __ballot_sync(0xffffffffu, c);
                        if (c) q[qn + __popc(m & lt_mask)] = ((unsigned)h << 24) | (unsigned)(kbase + j * 32);
                        qn += __popc(m);
                    }
                    __syncwarp();
                    while (qn >= 32) {
                        qn -= 32;
                        const unsigned entry = q[qn + lane];
                        __syncwarp();
                        score_candidates<POSE, MASK>(sh, a, pp, entry, true);
                    }
                }
            }
        }
        if (qn > 0) {
            const unsigned entry = lane < qn ? q[lane] : 0u;
            __syncwarp();
            score_candidates<POSE, MASK>(sh, a, pp, entry, lane < qn);
        }
        __syncthreads();
        if (tid < nh) {
            int c = 0;
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < SCORE_WARPS; ++w) { c += sh.pcnt[tid][w]; s += sh.psum[tid][w]; }
            a.count[my_slot] = c;
            a.score[my_slot] = s + pp.sq_thr * (double)(n - c);
        }
        if (a.point_scores && tid == 0) atomicAdd(a.point_scores, (unsigned long long)nh * (unsigned long long)n);
    }
}

// ---------------------------------------------------------------------------------------------
// bound: hypothesis-level pruning.  RANSAC only ever looks at a minimal model when it has MORE inliers
// than every earlier one or a LOWER score than every earlier one (score_models so@0x22ebc0); a model
// that provably does neither can be dropped without changing anything downstream.  After the first
// HB models of a pair have been scored exactly (B0 = their max count, S0 = their min score, both
// bounds of the running best at every later position), this kernel computes for every later model,
// from the FP32 tier alone,
//     ub = #(correspondences that are not certain outliers)            >= inlier count
//     lb = sum min(r2_lb, thr^2) over those + thr^2 * #certain outliers <= MSAC score
// with r2_lb = (|C~|-eps)_+^2 / (1.001 den~ + 1012 delta_a^2) (same error model as certain_outlier32:
// |C| >= |C~|-eps, sqrt(den) <= sqrt(den~)(1+2.1u) + delta_a, (a+b)^2 <= 1.001 a^2 + 1001 b^2).
// Only models with ub > B0 or lb < S0 go on to the exact kernel.  Lanes are correspondences, two
// slices (8 points) per lane per pass; no FP64, no queue.
struct BoundArgs {
    int n_groups, grp_stride, grp_per_pair;
    const int *grp_cnt;
    const int *item_prefix;
    const int *n_items;
    const PairParams *pairs;
    const Model *models;
    const ulonglong2 *pts32p;  // pair-interleaved FP32 correspondences (see PrepareArgs)
    int *ub;       // slots
    float *lb;     // slots
    const int *B0;     // per pair: max inlier count / min score over the exactly scored first HB models
    const double *S0;
    unsigned long long *point_scores;
    unsigned long long *evaluated;  // optional: (model, correspondence) pairs actually evaluated
    int *work_counter;              // zeroed before the launch: blocks take work items dynamically
    int head;                       // the first `head` models of a pair were scored exactly (multiple of SCORE_WARPS)
    const int *slot_list;           // optional indirection (survivors of the tensor-core tier): model i of group e lives
    int list_stride;                //   at slot e*grp_stride + slot_list[e*list_stride + i]; the head is not in the list
};

#ifndef RP_SOLVE_MIN_BLOCKS
#define RP_SOLVE_MIN_BLOCKS 1
#endif
#ifndef RP_BOUND_MIN_BLOCKS
#define RP_BOUND_MIN_BLOCKS 2
#endif
#ifndef RP_BOUND_BSG
#define RP_BOUND_BSG 2
#endif
constexpr int BSG = RP_BOUND_BSG;            // slices (of 32*PT points) per pass: 8 points per lane (measured optimum)
constexpr int BHW = HB / SCORE_WARPS;        // models per warp (each warp owns its models over ALL points)

// Packed FP32 arithmetic of sm_100a: fma.rn.f32x2 / mul.rn.f32x2 (SASS FFMA2 / FMUL2) do two FP32
// operations per lane per instruction.  Measured on B200 (tools/ffma2_bench.cu): same FLOP/s as FFMA,
// i.e. half the issue slots — exactly what an issue-bound FP32 kernel needs.  The bound kernel evaluates
// correspondences two at a time with them.
typedef unsigned long long f32x2;
RP_D f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
RP_D void unpack2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
RP_D f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
RP_D float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
RP_D f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// per-model constants of the bound kernel, every scalar duplicated into both halves of a packed register
struct alignas(16) BoundFilter {
    f32x2 e[9];   // E / F, row-major
    f32x2 g;      // thr^2 (1+1e-5)
    f32x2 kh;     // 1012 delta_a^2
    f32x2 eps;    // eps (filter disabled: +inf)
    f32x2 ng1;    // -(1.001 g): count-only test C^2 > 1.001 g den + 1001 eps^2  (see bound_eval)
    f32x2 nk;     // -(1001 eps^2) (filter disabled: -inf)
};

struct BoundShared {
    BoundFilter hf[SCORE_WARPS][BHW];  // per warp: the filters of the models of its current work unit
    float sp[SCORE_WARPS][BHW][32];  // per-lane partial lower-bound sums of the warp's models
    int outc[SCORE_WARPS][BHW];      // certain outliers collected so far by each of the warp's models
};

// one model against the 8 correspondences a lane holds (4 packed pairs).  FULL: all 256 correspondences
// of the group exist (no validity predicates).  CHEAP: count certain outliers only (the model already
// looks hopeless; its lower bound is given up, see bound_kernel).
template <bool FULL, bool CHEAP>
RP_D void bound_eval(const BoundFilter &f, const f32x2 (&X1x)[PT * BSG / 2], const f32x2 (&X1y)[PT * BSG / 2],
                     const f32x2 (&X2x)[PT * BSG / 2], const f32x2 (&X2y)[PT * BSG / 2], unsigned vmask, float thr2_lo,
                     int &c, float &s) {
    float eps, eps_hi;
    unpack2(f.eps, eps, eps_hi);
    const f32x2 k1001 = pack2(1.001f, 1.001f);
#pragma unroll
    for (int q = 0; q < PT * BSG / 2; ++q) {
        const f32x2 a0 = fma2(f.e[0], X1x[q], fma2(f.e[1], X1y[q], f.e[2]));
        const f32x2 a1 = fma2(f.e[3], X1x[q], fma2(f.e[4], X1y[q], f.e[5]));
        const f32x2 a2 = fma2(f.e[6], X1x[q], fma2(f.e[7], X1y[q], f.e[8]));
        const f32x2 b0 = fma2(f.e[0], X2x[q], fma2(f.e[3], X2y[q], f.e[6]));
        const f32x2 b1 = fma2(f.e[1], X2x[q], fma2(f.e[4], X2y[q], f.e[7]));
        const f32x2 C = fma2(X2x[q], a0, fma2(X2y[q], a1, a2));
        const f32x2 den = fma2(a0, a0, fma2(a1, a1, fma2(b0, b0, mul2(b1, b1))));
        if (CHEAP) {
            // count-only: |C| - eps > sqrt(g den)  <=  C^2 > (1+a) g den + (1+1/a) eps^2  with a = 1e-3
            // ((x+y)^2 <= (1+a) x^2 + (1+1/a) y^2), evaluated as the sign of one packed FMA chain; the
            // 1e-5 slack folded into ng1 / nk covers its two roundings.  NaN compares false: candidate.
            const f32x2 D = fma2(C, C, fma2(f.ng1, den, f.nk));
            float dd0, dd1;
            unpack2(D, dd0, dd1);
            bool cand0 = !(dd0 > 0.f), cand1 = !(dd1 > 0.f);
            if (!FULL) {
                cand0 = cand0 && ((vmask >> (2 * q)) & 1u);
                cand1 = cand1 && ((vmask >> (2 * q + 1)) & 1u);
            }
            c += (int)cand0 + (int)cand1;
            continue;
        }
        float c0, c1;
        unpack2(C, c0, c1);
        const float tt0 = fmaxf(fabsf(c0) - eps, 0.0f), tt1 = fmaxf(fabsf(c1) - eps, 0.0f);
        const f32x2 TT = pack2(tt0, tt1);
        const f32x2 T2 = mul2(TT, TT), GD = mul2(f.g, den);
        float t20, t21, gd0, gd1;
        unpack2(T2, t20, t21);
        unpack2(GD, gd0, gd1);
        bool cand0 = !(t20 > gd0), cand1 = !(t21 > gd1);
        if (!FULL) {
            cand0 = cand0 && ((vmask >> (2 * q)) & 1u);
            cand1 = cand1 && ((vmask >> (2 * q + 1)) & 1u);
        }
        c += (int)cand0 + (int)cand1;
        if (!CHEAP) {
            // r2_lb = t2 / (1.001 den + kh); kh >= 1e-29 for every enabled filter and +inf for disabled
            // ones, so the approximate reciprocal never sees a denormal (its 1-ulp error is inside the
            // 1e-4 slack of lb)
            const f32x2 DU = fma2(den, k1001, f.kh);
            float du0, du1;
            unpack2(DU, du0, du1);
            const float r0 = fminf(t20 * rcp_approx(du0), thr2_lo), r1 = fminf(t21 * rcp_approx(du1), thr2_lo);
            s += (cand0 ? r0 : 0.f) + (cand1 ? r1 : 0.f);
        }
    }
}

// Warps split the MODELS of an item (model h belongs to warp h % SCORE_WARPS) and each walks all
// correspondences of the pair in groups of 256.  A warp therefore knows, after every group, how many
// certain outliers each of its models has collected, and abandons a model as soon as
//     out >= N - B0   (final ub <= B0)   and   thr^2 * out >= S0   (final lb >= S0)
// i.e. as soon as it is certain to be pruned: bad models (the majority) stop after ~1/3 of the points.
template <bool POSE>
__global__ void __launch_bounds__(SCORE_THREADS, RP_BOUND_MIN_BLOCKS) bound_kernel(BoundArgs a) {
    __shared__ BoundShared sh;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n_items = *a.n_items;
    // Work unit = the models h = w, w+8, w+16, ... (at most BHW) of one item; units differ a lot in cost
    // (abandonment), so every WARP takes them one at a time from a global counter and nothing in this kernel
    // synchronises across warps: a warp with many good models never holds up the other seven.
    for (;;) {
        int unit = 0;
        if (lane == 0) unit = atomicAdd(a.work_counter, 1);
        unit = __shfl_sync(0xffffffffu, unit, 0);
        const int item = unit / SCORE_WARPS, w = unit % SCORE_WARPS;
        if (item >= n_items) break;
        int lo = 0, hi = a.n_groups;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (a.item_prefix[mid] <= item) lo = mid; else hi = mid;
        }
        const int e = lo;
        const int chunk = item - a.item_prefix[e];
        const int pair = e / a.grp_per_pair;
        const int h0 = chunk * HB;
        const int nh = min(HB, a.grp_cnt[e] - h0);
        const size_t slot0 = (size_t)e * a.grp_stride + h0;
        const PairParams pp = a.pairs[pair];
        const int my_nh = (nh - w + SCORE_WARPS - 1) / SCORE_WARPS;  // models h = w + i*SCORE_WARPS
        // the first `head` models of a pair are scored exactly: in its first item the warp skips i < i0
        const int i0 = (!a.slot_list && e % a.grp_per_pair == 0 && chunk == 0) ? a.head / SCORE_WARPS : 0;
        if (my_nh <= i0) continue;
        __syncwarp();
        bool nonfinite = false;
        // slot of the warp's i-th model (lane i keeps it for the result write)
        size_t my_slot = slot0 + w + lane * SCORE_WARPS;
        if (a.slot_list && lane < my_nh)
            my_slot = (size_t)e * a.grp_stride + a.slot_list[(size_t)e * a.list_stride + h0 + w + lane * SCORE_WARPS];
        if (lane < my_nh) {
            const Model m = a.models[my_slot];
            const M3 E = POSE ? essential_from_motion(m.q, m.t) : fundamental_from_model(m);
            // A model with a non-finite E (the minimal solvers return NaN models now and then, P3P for ~6 % of
            // its solutions) has r2 = NaN for every correspondence: the reference counts 0 inliers and sums
            // N thr^2, which can neither exceed B0 >= 0 nor undercut S0 <= N thr^2 (S0 exists: the pair has an
            // exactly scored head, checked below).  Dead on arrival.
            nonfinite = !(isfinite(E.r0.x) && isfinite(E.r0.y) && isfinite(E.r0.z) && isfinite(E.r1.x) && isfinite(E.r1.y) &&
                          isfinite(E.r1.z) && isfinite(E.r2.x) && isfinite(E.r2.y) && isfinite(E.r2.z));
            const Filter32 f = make_filter32(E, pp.thr, pp.Mmax, pp.mmax);
            // 1012 * delta_a^2 with delta_a = 16 u Emax m (the sqrt(den) term of eps)
            const double emax = fmax(fmax(fmax(fabs(E.r0.x), fabs(E.r0.y)), fmax(fabs(E.r0.z), fabs(E.r1.x))),
                                     fmax(fmax(fabs(E.r1.y), fabs(E.r1.z)), fmax(fmax(fabs(E.r2.x), fabs(E.r2.y)), fabs(E.r2.z))));
            const double da = 16.0 * 5.9604644775390625e-08 * emax * pp.mmax;
            // disabled filter (eps = +inf): kh = +inf makes every r2_lb exactly 0
            const float kh = isinf(f.eps) ? INFINITY : fmaxf((float)(1012.0 * da * da * 1.0001), 1e-29f);
            BoundFilter bf;
            bf.e[0] = pack2(f.e00, f.e00); bf.e[1] = pack2(f.e01, f.e01); bf.e[2] = pack2(f.e02, f.e02);
            bf.e[3] = pack2(f.e10, f.e10); bf.e[4] = pack2(f.e11, f.e11); bf.e[5] = pack2(f.e12, f.e12);
            bf.e[6] = pack2(f.e20, f.e20); bf.e[7] = pack2(f.e21, f.e21); bf.e[8] = pack2(f.e22, f.e22);
            bf.g = pack2(f.g, f.g); bf.kh = pack2(kh, kh); bf.eps = pack2(f.eps, f.eps);
            const float ng1 = -__double2float_ru((double)f.g * 1.001 * 1.00001);
            const float nk = isinf(f.eps) ? -INFINITY : -__double2float_ru(1001.0 * (double)f.eps * (double)f.eps * 1.00001);
            bf.ng1 = pack2(ng1, ng1); bf.nk = pack2(nk, nk);
            sh.hf[wid][lane] = bf;
        }
        __syncwarp();
        const int n = pp.n;
        const float thr2_lo = __double2float_rd(pp.sq_thr);
        // abandonment threshold on the number of certain outliers (see header comment)
        const int B0 = a.B0[pair];
        const double S0 = a.S0[pair];
        double need_d = fmax((double)(n - B0), S0 < 1e300 ? ceil(S0 / ((double)thr2_lo * (1.0 - 2e-4))) : 4.0e9);
        const int need_out = need_d > 2.0e9 ? 0x7fffffff : max((int)need_d, 1);
        unsigned alive = (my_nh >= 32 ? 0xffffffffu : ((1u << my_nh) - 1u)) & ~((1u << i0) - 1u);
        if (S0 < 1e300) alive &= ~__ballot_sync(0xffffffffu, nonfinite);
        unsigned cheap = 0;  // models that switched to count-only evaluation (their lb is void)
        int *out_cnt = sh.outc[wid];
#pragma unroll
        for (int i = 0; i < BHW; ++i) sh.sp[wid][i][lane] = 0.f;
        if (lane < BHW) out_cnt[lane] = 0;
        __syncwarp();
        const int group_pts = 32 * PT * BSG;
        const int n_pgroups = (n + group_pts - 1) / group_pts;
        unsigned long long evaluated = 0;
        for (int g = 0; g < n_pgroups && alive; ++g) {
            // lane owns the correspondence pairs (2m, 2m+1), m = g*128 + q*32 + lane: two 128-bit loads give
            // the four packed operands directly in aligned register pairs
            f32x2 X1x[PT * BSG / 2], X1y[PT * BSG / 2], X2x[PT * BSG / 2], X2y[PT * BSG / 2];
            unsigned vmask = 0;
#pragma unroll
            for (int q = 0; q < PT * BSG / 2; ++q) {
                const int m = g * (group_pts / 2) + q * 32 + lane;
                const int k0 = 2 * m, k1 = k0 + 1;
                ulonglong2 A = make_ulonglong2(0ull, 0ull), Bq = make_ulonglong2(0ull, 0ull);
                if (k0 < n) {
                    A = a.pts32p[(pp.pbase + m) * 2];
                    Bq = a.pts32p[(pp.pbase + m) * 2 + 1];
                }
                vmask |= (k0 < n ? 1u : 0u) << (2 * q) | (k1 < n ? 1u : 0u) << (2 * q + 1);
                X1x[q] = A.x; X1y[q] = A.y; X2x[q] = Bq.x; X2y[q] = Bq.y;
            }
            const int nvalid = min(group_pts, n - g * group_pts);
            const bool full = nvalid == group_pts;
            evaluated += (unsigned long long)__popc(alive) * nvalid;
            // only the models still alive (late groups: a handful of the 16)
#pragma unroll 1
            for (unsigned todo = alive; todo; todo &= todo - 1) {
                const int i = __ffs(todo) - 1;
                const BoundFilter f = sh.hf[wid][i];
                int c = 0;
                float s = 0.f;
                const bool is_cheap = (cheap >> i) & 1u;
                if (!full) bound_eval<false, false>(f, X1x, X1y, X2x, X2y, vmask, thr2_lo, c, s);
                else if (is_cheap) bound_eval<true, true>(f, X1x, X1y, X2x, X2y, vmask, thr2_lo, c, s);
                else bound_eval<true, false>(f, X1x, X1y, X2x, X2y, vmask, thr2_lo, c, s);
                if (!is_cheap) sh.sp[wid][i][lane] += s;
                const int nc = __reduce_add_sync(0xffffffffu, c);
                const int oc = out_cnt[i] + nvalid - nc;
                __syncwarp();
                if (lane == 0) out_cnt[i] = oc;
                if (oc >= need_out) alive &= ~(1u << i);  // certain to be pruned: stop here
                // more than half certain outliers so far: this model will almost surely be abandoned, stop
                // paying for its score bound (if it does stay alive it simply goes to the exact kernel)
                else if (2 * oc >= (g + 1) * group_pts) cheap |= 1u << i;
            }
        }
        // results: abandoned models can never survive the prune (ub = 0, lb = +inf)
        __syncwarp();
#pragma unroll 1
        for (int i = i0; i < my_nh; ++i) {
            const size_t slot_i = __shfl_sync(0xffffffffu, (unsigned long long)my_slot, i);
            float s = sh.sp[wid][i][lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) {
                const bool dead = !((alive >> i) & 1u);
                a.ub[slot_i] = dead ? 0 : n - out_cnt[i];
                // lb = thr^2 * (#certain outliers) + sum of candidate lower bounds; FP32 rounding of the
                // terms, the rcp and the partial sums is covered by 1e-4 relative
                const double lbv = ((double)thr2_lo * (double)out_cnt[i] + (double)s) * (1.0 - 1e-4);
                a.lb[slot_i] = dead ? INFINITY : (((cheap >> i) & 1u) ? -INFINITY : __double2float_rd(lbv));
            }
        }
        if (a.point_scores && lane == 0) atomicAdd(a.point_scores, (unsigned long long)(my_nh - i0) * (unsigned long long)n);
        if (a.evaluated && lane == 0) atomicAdd(a.evaluated, evaluated);
        __syncwarp();  // the unit's shared-memory rows are free for the next one
    }
}

// models per pair (sum of its segment counts): the tensor-core tier walks a pair's models as ONE list
__global__ void pair_total_kernel(int n_pairs, int nseg, const int *seg_count, int *pair_cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    int c = 0;
    for (int s = 0; s < nseg; ++s) c += seg_count[i * nseg + s];
    pair_cnt[i] = c;
}

// models of a pair at positions [start, limit) of its first segment (limit > 0), or from `start` of the first segment to
// the end of the pair (limit = 0)
__global__ void range_count_kernel(int n_pairs, int nseg, const int *seg_count, int start, int limit, int *pair_cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const int c0 = seg_count[i * nseg];
    if (limit > 0) { pair_cnt[i] = max(min(c0, limit) - start, 0); return; }
    int c = max(c0 - start, 0);
    for (int s = 1; s < nseg; ++s) c += seg_count[i * nseg + s];
    pair_cnt[i] = c;
}

// tc_select: what the tensor-core tier (rp_tc.cuh) decided.  out[slot] = certain outliers of the model, a rigorous
// lower bound of N - inlier_count, and thr^2 out of the score.  With (B0, S0) of the exactly scored head, a model with
//     out >= N - B0   and   thr^2 out >= S0
// can neither exceed the best inlier count nor undercut the best score: it gets (ub 0, lb +inf), which the prune
// drops.  Everything else is compacted, in sequence order, into the pair's list for the FP32 bound kernel.
// One warp per pair.
struct TcSelectArgs {
    int n_pairs, nseg, head;
    int limit;       // > 0: only positions [head, limit) of the first segment (the mid stage); 0: everything from `head` on
    const PairParams *pairs;
    const int *seg_count;
    const int *out;
    const int *B0;
    const double *S0;
    int *ub;
    float *lb;
    int *list;       // [n_pairs * nseg*4*SEG] pair-relative slots of the survivors
    int *list_cnt;   // [n_pairs]
    unsigned long long *n_selected;
};
__global__ void tc_select_kernel(TcSelectArgs a) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.n_pairs) return;
    const PairParams pp = a.pairs[warp];
    const size_t slots_pp = (size_t)a.nseg * (4 * SEG);
    const size_t pslot = (size_t)warp * slots_pp;
    const int n = pp.n;
    const int need_out = tc::need_outliers(n, pp.sq_thr, a.B0[warp], a.S0[warp]);   // same threshold as bound_kernel
    int ns = 0;
    for (int seg = 0; seg < (a.limit > 0 ? 1 : a.nseg); ++seg) {
        const int cnt = a.limit > 0 ? min(a.seg_count[warp * a.nseg + seg], a.limit) : a.seg_count[warp * a.nseg + seg];
        const int rel0 = seg * (4 * SEG);
        for (int base = (seg == 0 ? a.head : 0); base < cnt; base += 32) {
            const int h = base + lane;
            bool keep = false;
            if (h < cnt) {
                keep = a.out[pslot + rel0 + h] < need_out;
                if (!keep) { a.ub[pslot + rel0 + h] = 0; a.lb[pslot + rel0 + h] = INFINITY; }
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) a.list[pslot + ns + __popc(m & ((1u << lane) - 1u))] = rel0 + h;
            ns += __popc(m);
        }
    }
    if (lane == 0) {
        a.list_cnt[warp] = ns;
        if (a.n_selected && ns) atomicAdd(a.n_selected, (unsigned long long)ns);
    }
}

// the same decision after the second pass of the tensor-core tier, over the first pass's list (compacted in place:
// a batch of 32 entries is read before its survivors are written at or before the batch's first position)
__global__ void tc_select_list_kernel(TcSelectArgs a) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.n_pairs) return;
    const PairParams pp = a.pairs[warp];
    const size_t slots_pp = (size_t)a.nseg * (4 * SEG);
    const size_t pslot = (size_t)warp * slots_pp;
    const int n = pp.n;
    const int need_out = tc::need_outliers(n, pp.sq_thr, a.B0[warp], a.S0[warp]);
    const int cnt = a.list_cnt[warp];
    int ns = 0;
    for (int base = 0; base < cnt; base += 32) {
        const int i = base + lane;
        const int rel = i < cnt ? a.list[pslot + i] : 0;
        bool keep = false;
        if (i < cnt) {
            keep = a.out[pslot + rel] < need_out;
            if (!keep) { a.ub[pslot + rel] = 0; a.lb[pslot + rel] = INFINITY; }
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        __syncwarp();
        if (keep) a.list[pslot + ns + __popc(m & ((1u << lane) - 1u))] = rel;
        ns += __popc(m);
    }
    if (lane == 0) {
        a.list_cnt[warp] = ns;
        if (a.n_selected && ns) atomicAdd(a.n_selected, (unsigned long long)ns);
    }
}

// B0 / S0 of a pair: max count and min score over its first `first_cnt` (<= HB) models, scored exactly
__global__ void pair_bounds_kernel(int n_pairs, int nseg, const int *first_cnt, const double *score, const int *count,
                                   int *B0, double *S0) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_pairs) return;
    const size_t slot0 = (size_t)warp * nseg * (4 * SEG);
    const int cnt = first_cnt[warp];
    int b = 0;
    double s = DBL_MAX;
    for (int h = lane; h < cnt; h += 32) {
        b = max(b, count[slot0 + h]);
        const double v = score[slot0 + h];
        if (v == v) s = fmin(s, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        b = max(b, __shfl_xor_sync(0xffffffffu, b, o));
        s = fmin(s, __shfl_xor_sync(0xffffffffu, s, o));
    }
    if (lane == 0) { B0[warp] = b; S0[warp] = s; }
}

__global__ void first_count_kernel(int n_pairs, int nseg, const int *seg_count, int *first_cnt, int head) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pairs) first_cnt[i] = min(seg_count[i * nseg], head);
}

// prune: survivors (ub > B0 or lb < S0) are compacted, in order, into a per-pair slot list; everything
// else gets (count 0, score DBL_MAX), which can never trigger.  One warp per pair.
struct PruneArgs {
    int n_pairs, nseg;
    const int *seg_count;
    const int *ub;
    const float *lb;
    const int *B0;
    const double *S0;
    double *score;
    int *count;
    int *surv_list;   // [n_pairs * nseg*4*SEG] pair-relative slots
    int *surv_cnt;    // [n_pairs]
    unsigned long long *n_survivors;
    int head;   // models of segment 0 that were scored exactly (multiple of 32)
    int limit;  // > 0: only positions [head, limit) of the first segment (the mid stage); 0: everything from `head` on
};

__global__ void prune_kernel(PruneArgs a) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.n_pairs) return;
    const size_t slots_pp = (size_t)a.nseg * (4 * SEG);
    const size_t pslot = (size_t)warp * slots_pp;
    const int B0 = a.B0[warp];
    const double S0 = a.S0[warp];
    int ns = 0;
    for (int seg = 0; seg < (a.limit > 0 ? 1 : a.nseg); ++seg) {
        const int cnt = a.limit > 0 ? min(a.seg_count[warp * a.nseg + seg], a.limit) : a.seg_count[warp * a.nseg + seg];
        const int rel0 = seg * (4 * SEG);
        for (int base = (seg == 0 ? a.head : 0); base < cnt; base += 32) {
            const int h = base + lane;
            bool keep = false;
            if (h < cnt) {
                keep = a.ub[pslot + rel0 + h] > B0 || (double)a.lb[pslot + rel0 + h] < S0;
                if (!keep) { a.count[pslot + rel0 + h] = 0; a.score[pslot + rel0 + h] = DBL_MAX; }
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) a.surv_list[pslot + ns + __popc(m & ((1u << lane) - 1u))] = rel0 + h;
            ns += __popc(m);
        }
    }
    if (lane == 0) {
        a.surv_cnt[warp] = ns;
        if (a.n_survivors && ns) atomicAdd(a.n_survivors, (unsigned long long)ns);
    }
}

// Survivors are scored exactly in WAVES.  The prune above compares against (B0, S0) of the first HB models
// only, so every later model that beats the head's best survives (~200 per pair on the benchmark) although only
// the ~10 prefix records among them matter.  The survivor list is in sequence order: score its first few
// entries exactly, raise (B, S) to what they achieved, re-test the following entries' (ub, lb) against the new
// bar, and so on with growing wave sizes.  A survivor dropped by the re-test has ub <= B and lb >= S for exact
// values B, S of EARLIER models, hence can neither trigger nor move the running best: the result is unchanged
// while ~10x fewer models reach the exact kernel.  One warp per pair; the wave is compacted in place at the
// front of the pair's survivor list (entries before the cursor are already consumed).
struct WaveArgs {
    int n_pairs;
    size_t slots_pp;
    int wave_size;        // models to select per pair in this wave
    int first;            // first wave: nothing to fold into (B, S) yet
    int *surv_list;       // [n_pairs * slots_pp] pair-relative slots (in: survivors from cursor on; out: the wave at the front)
    const int *surv_cnt;  // [n_pairs] survivors of the prune
    int *cursor;          // [n_pairs] next unconsumed survivor
    int *wave_cnt;        // [n_pairs] in: size of the previous wave, out: size of this one
    const int *ub;
    const float *lb;
    int *B;               // [n_pairs] running exact bests (start: B0, S0)
    double *S;
    double *score;
    int *count;
    unsigned long long *n_exact;  // optional counter of models sent to the exact kernel
};

__global__ void wave_select_kernel(WaveArgs a) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.n_pairs) return;
    const size_t pslot = (size_t)warp * a.slots_pp;
    int B = a.B[warp];
    double S = a.S[warp];
    if (!a.first) {
        // fold the previous wave's exact results into the bar
        const int prev = a.wave_cnt[warp];
        for (int i = lane; i < prev; i += 32) {
            const size_t slot = pslot + a.surv_list[pslot + i];
            B = max(B, a.count[slot]);
            const double v = a.score[slot];
            if (v == v) S = fmin(S, v);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            B = max(B, __shfl_xor_sync(0xffffffffu, B, o));
            S = fmin(S, __shfl_xor_sync(0xffffffffu, S, o));
        }
    }
    const int ns = a.surv_cnt[warp];
    int pos = a.cursor[warp], nw = 0;
    while (pos < ns && nw < a.wave_size) {
        const int i = pos + lane;
        const bool valid = i < ns;
        const int rel = valid ? a.surv_list[pslot + i] : 0;
        const bool keep = valid && (a.ub[pslot + rel] > B || (double)a.lb[pslot + rel] < S);
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        const int rank = __popc(m & ((1u << lane) - 1u));
        const bool take = keep && nw + rank < a.wave_size;
        // the cursor stops in front of the first kept entry that does not fit into this wave
        const unsigned untaken = __ballot_sync(0xffffffffu, keep && !take);
        const int stop = untaken ? __ffs(untaken) - 1 : 32;
        if (valid && !keep && lane < stop) { a.count[pslot + rel] = 0; a.score[pslot + rel] = DBL_MAX; }
        __syncwarp();
        if (take) a.surv_list[pslot + nw + rank] = rel;   // nw + rank <= pos + lane: never ahead of the reads
        nw += __popc(m & (stop >= 32 ? 0xffffffffu : ((1u << stop) - 1u)));
        pos += stop;
        if (stop < 32) break;
    }
    if (lane == 0) {
        a.B[warp] = B;
        a.S[warp] = S;
        a.cursor[warp] = pos;
        a.wave_cnt[warp] = nw;
        if (a.n_exact && nw) atomicAdd(a.n_exact, (unsigned long long)nw);
    }
}

// ---------------------------------------------------------------------------------------------
// scan: the part of score_models() so@0x22ebc0 that does not depend on LO results.  A minimal
// model "triggers" when it has more inliers than every earlier minimal model or a lower MSAC
// score than every earlier one (running max / running min, strict).  One warp per pair walks the
// pair's slots in order and emits the triggering slots.
constexpr int PAIR_FLAG_OVERFLOW = 1;   // more trigger events than the list holds: outputs of the pair are void
constexpr int PAIR_FLAG_NEED_MORE = 2;  // early termination: neither stopped nor at max_iterations within the generated iterations

struct ScanArgs {
    int n_pairs, nseg;
    const int *seg_count;
    const double *score;
    const int *count;
    int *events;      // [n_pairs*ev_cap] slot of each trigger, in order
    int *n_events;    // [n_pairs]
    int ev_cap;       // capacity of a pair's event list (EV; larger when an overflowing pair is re-run)
    int *pair_flags;  // [n_pairs] PAIR_FLAG_OVERFLOW is set for a pair with more triggers than ev_cap
    int *any_flag;    // scalar: some pair was flagged
};

__global__ void scan_kernel(ScanArgs a) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.n_pairs) return;
    long long best_cnt = 0;  // best_minimal_inlier_count starts at 0
    double best_score = DBL_MAX;
    int nev = 0;
    for (int seg = 0; seg < a.nseg; ++seg) {
        const int e = warp * a.nseg + seg;
        const int cnt = a.seg_count[e];
        const size_t slot0 = (size_t)e * (4 * SEG);
        for (int base = 0; base < cnt; base += 32) {
            const int h = base + lane;
            const bool v = h < cnt;
            const long long c = v ? (long long)a.count[slot0 + h] : -1;
            double s = v ? a.score[slot0 + h] : DBL_MAX;
            if (s != s) s = DBL_MAX;  // NaN scores never compare "less" in the reference either
            // exclusive running max / min within the warp
            long long cmax = c;
            double smin = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long c2 = __shfl_up_sync(0xffffffffu, cmax, o);
                const double s2 = __shfl_up_sync(0xffffffffu, smin, o);
                if (lane >= o) { cmax = max(cmax, c2); smin = fmin(smin, s2); }
            }
            long long cprev = __shfl_up_sync(0xffffffffu, cmax, 1);
            double sprev = __shfl_up_sync(0xffffffffu, smin, 1);
            if (lane == 0) { cprev = best_cnt; sprev = best_score; }
            else { cprev = max(cprev, best_cnt); sprev = fmin(sprev, best_score); }
            const bool trig = v && (c > cprev || s < sprev);
            const unsigned m = __ballot_sync(0xffffffffu, trig);
            if (trig) {
                const int pos = nev + __popc(m & ((1u << lane) - 1));
                if (pos < a.ev_cap) a.events[(size_t)warp * a.ev_cap + pos] = (int)(slot0 + h - (size_t)warp * a.nseg * (4 * SEG));
            }
            nev += __popc(m);
            best_cnt = max(best_cnt, __shfl_sync(0xffffffffu, cmax, 31));
            best_score = fmin(best_score, __shfl_sync(0xffffffffu, smin, 31));
        }
    }
    if (lane == 0) {
        a.n_events[warp] = min(nev, a.ev_cap);
        a.pair_flags[warp] = nev > a.ev_cap ? PAIR_FLAG_OVERFLOW : 0;
        if (nev > a.ev_cap) *a.any_flag = 1;
    }
}

// LO problem list: the LO of an iteration starts from the LAST triggering model of that
// iteration (models[best_model_ind], so@0x22ed60).  Thread per pair.
struct LoPrepArgs {
    int n_pairs, nseg;
    const int *events, *n_events;
    const int *hyp_iter;
    const Model *models;
    int ev_cap;
    Model *lo_models;   // [n_pairs*ev_cap]
    int *lo_of_event;   // [n_pairs*ev_cap] index of the LO problem started by this event or -1
    int *lo_count;      // [n_pairs]
    int *prob_list;     // compact list of lo_models indices
    int *n_prob;
};

__global__ void lo_prepare_kernel(LoPrepArgs a) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= a.n_pairs) return;
    const size_t pslot = (size_t)pair * a.nseg * (4 * SEG);
    const int nev = a.n_events[pair];
    const size_t eb = (size_t)pair * a.ev_cap;
    int nlo = 0;
    for (int i = 0; i < nev; ++i) {
        const int ev = a.events[eb + i];
        const int it = a.hyp_iter[pslot + ev];
        const bool last = (i + 1 == nev) || a.hyp_iter[pslot + a.events[eb + i + 1]] != it;
        if (last) {
            a.lo_models[eb + nlo] = a.models[pslot + ev];
            a.lo_of_event[eb + i] = nlo;
            ++nlo;
        } else {
            a.lo_of_event[eb + i] = -1;
        }
    }
    a.lo_count[pair] = nlo;
    if (nlo) {
        const int p0 = atomicAdd(a.n_prob, nlo);
        for (int j = 0; j < nlo; ++j) a.prob_list[p0 + j] = pair * a.ev_cap + j;
    }
}

// ---------------------------------------------------------------------------------------------
// merge: replay of score_models() / ransac() bookkeeping (so@0x22ebc0, so@0x22f030) over the
// trigger events in order: a triggering minimal model becomes the best model if its score beats
// stats.model_score; after the last trigger of an iteration the LO result is compared (strict <).
struct MergeArgs {
    int n_pairs, nseg, iters;  // iters = iterations actually generated for this chunk
    long long min_iterations, max_iterations;
    double dyn_num_trials_mult, log_prob_missing;
    const PairParams *pairs;
    const int *events, *n_events, *lo_of_event;
    const int *hyp_iter;
    const double *score;     // minimal slots
    const int *count;
    const Model *models;
    int ev_cap;
    const double *lo_score;  // [n_pairs*ev_cap]
    const int *lo_count_inl;
    const Model *lo_models;
    const int *lo_count;     // number of LO problems per pair
    Model *best;             // [n_pairs]
    rp_stats *stats;         // [n_pairs]
    Model *final_start;      // [n_pairs] copy of best (start of the final LO)
    int *pair_flags;         // [n_pairs] |= PAIR_FLAG_NEED_MORE when a pair neither stopped nor reached max_iterations
    int *any_flag;
};

__global__ void merge_kernel(MergeArgs a) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= a.n_pairs) return;
    const PairParams pp = a.pairs[pair];
    rp_stats st;
    st.refinements = 0; st.iterations = 0; st.num_inliers = 0; st.inlier_ratio = 0.0; st.model_score = DBL_MAX;
    Model best = identity_model();
    if (pp.valid) {
        const size_t pslot = (size_t)pair * a.nseg * (4 * SEG);
        const int nev = a.n_events[pair];
        const size_t eb = (size_t)pair * a.ev_cap;
        // the loop of ransac<>() breaks at the first it > min_iterations with it > dynamic_max_iter;
        // dynamic_max_iter only changes after an LO, so the break point is known between events.  The test
        // runs at the top of an iteration: after an LO in iteration it_prev the loop cannot stop before
        // it_prev + 1, even when the new dynamic_max_iter is already far behind.
        double dyn_max_iter = (double)a.max_iterations;
        long long stop_it = -1, it_prev = -1;
        for (int i = 0; i < nev; ++i) {
            const int ev = a.events[eb + i];
            const long long it_e = a.hyp_iter[pslot + ev];
            const long long cand = max(max(a.min_iterations + 1, (long long)floor(dyn_max_iter) + 1), it_prev + 1);
            if (cand <= it_e) { stop_it = cand; break; }
            it_prev = it_e;
            const double s = a.score[pslot + ev];
            if (s < st.model_score) {
                st.model_score = s;
                best = a.models[pslot + ev];
                st.num_inliers = a.count[pslot + ev];
            }
            const int lo = a.lo_of_event[eb + i];
            if (lo >= 0) {
                st.refinements++;
                const double rs = a.lo_score[eb + lo];
                if (rs < st.model_score) {
                    st.model_score = rs;
                    st.num_inliers = a.lo_count_inl[eb + lo];
                    best = a.lo_models[eb + lo];
                }
                st.inlier_ratio = (double)st.num_inliers / (double)pp.n;
                if (st.inlier_ratio >= 0.9999) dyn_max_iter = (double)a.min_iterations;
                else if (st.inlier_ratio <= 0.0001) dyn_max_iter = (double)a.max_iterations;
                else {
                    const double prob_outlier = 1.0 - pow(st.inlier_ratio, 3.0);
                    dyn_max_iter = ceil(a.log_prob_missing / log(prob_outlier) * a.dyn_num_trials_mult);
                }
            }
        }
        if (stop_it < 0) {
            const long long cand = max(max(a.min_iterations + 1, (long long)floor(dyn_max_iter) + 1), it_prev + 1);
            if (cand < a.iters) stop_it = cand;                             // stopped inside what we generated
            else if (a.iters >= a.max_iterations) stop_it = a.max_iterations;  // loop ran to the end
            else if (cand == a.iters) stop_it = cand;                        // would stop exactly at the next it
            else { stop_it = a.iters; a.pair_flags[pair] |= PAIR_FLAG_NEED_MORE; *a.any_flag = 1; }
        }
        st.iterations = stop_it;
    }
    a.best[pair] = best;
    a.final_start[pair] = best;
    a.stats[pair] = st;
}

// final LO of ransac(): refinements++, accept when strictly better
struct Merge2Args {
    int n_pairs;
    const PairParams *pairs;
    const Model *refined;
    const double *ref_score;
    const int *ref_count;
    Model *best;
    rp_stats *stats;
};
__global__ void merge2_kernel(Merge2Args a) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= a.n_pairs) return;
    const PairParams pp = a.pairs[pair];
    if (!pp.valid) return;
    rp_stats st = a.stats[pair];
    st.refinements++;
    const double rs = a.ref_score[pair];
    // unlike the LO inside the loop, the final refinement of ransac<>() leaves stats.model_score alone: the
    // reported score is the one before this step (with no minimal model at all it stays DBL_MAX)
    if (rs < st.model_score) {
        st.num_inliers = a.ref_count[pair];
        a.best[pair] = a.refined[pair];
    }
    st.inlier_ratio = (double)st.num_inliers / (double)pp.n;
    a.stats[pair] = st;
}

// per-pair switch of the final refinement (stats.num_inliers > 3) and the output conversion
// (focal variants: f *= normalisation scale)
__global__ void enable_final_kernel(int n_pairs, const rp_stats *stats, int *enable) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair < n_pairs) enable[pair] = stats[pair].num_inliers > 3;
}
__global__ void finalize_kernel(int n_pairs, int variant, const PairParams *pairs, Model *best) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    if (variant == RP_SHARED || variant == RP_VARYING) {
        best[pair].f1 *= pairs[pair].nscale;
        best[pair].f2 *= pairs[pair].nscale;
    }
}

// ---------------------------------------------------------------------------------------------
// rp_refine_pairs_*: the final refinement above on caller-supplied start models and subsets.
// import: warp per pair.  |S_p| = subset bytes != 0 over the pair (all n without a subset), enable = |S_p| > 3 (the
// estimator's num_inliers > 3); work = init with f1, f2 divided by nscale for the focal variants, for every pair and not
// only the enabled ones, so that the inlier mask of a pair that is not refined is get_inliers of its start model in the
// normalised frame, as the estimator's mask is; bundle stats zeroed (the LM skips the pairs it does not refine).
__global__ void refine_import_kernel(int n_pairs, int variant, const PairParams *pairs, const unsigned char *subset,
                                     const Model *init, Model *work, int *enable, rp_bundle_stats *bstats) {
    const int pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (pair >= n_pairs) return;
    const PairParams pp = pairs[pair];
    int cnt = pp.n;
    if (subset) {
        cnt = 0;
        const unsigned char *s = subset + pp.off;
        for (int b0 = 0; b0 < pp.n; b0 += 32) cnt += __popc(__ballot_sync(0xffffffffu, b0 + lane < pp.n && s[b0 + lane]));
    }
    if (lane != 0) return;
    Model m = init[pair];
    if (variant == RP_SHARED || variant == RP_VARYING) {
        m.f1 /= pp.nscale;
        m.f2 /= pp.nscale;
    }
    work[pair] = m;
    enable[pair] = cnt > 3;
    if (bstats) bstats[pair] = rp_bundle_stats{};
}

// export: thread per pair.  A refined pair's model is the work model with f1, f2 multiplied by nscale (focal variants);
// any other pair gets init's bytes (no nscale round trip).  With `count` (the masked score of the work models), the
// pair's inlier count, 0 for pairs of fewer than 3 correspondences, which are not scored.  `out` may alias `init`.
__global__ void refine_export_kernel(int n_pairs, int variant, const PairParams *pairs, const int *enable,
                                     const Model *init, const Model *work, const int *count, Model *out,
                                     long long *num_inliers) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    const PairParams pp = pairs[pair];
    Model m;
    if (enable[pair]) {
        m = work[pair];
        if (variant == RP_SHARED || variant == RP_VARYING) {
            m.f1 *= pp.nscale;
            m.f2 *= pp.nscale;
        }
    } else {
        m = init[pair];
    }
    out[pair] = m;
    if (num_inliers) num_inliers[pair] = pp.valid ? count[pair] : 0;
}

// Re-run sub-batches (estimate_impl): pairs that overflowed their event list or need more iterations are gathered
// into a compact ragged batch, run again with larger limits, and their results scattered back.  Block per pair.
struct SubBatchArgs {
    int n_sub;
    const int *pair_idx;          // [n_sub] pair index inside the chunk
    const long long *src_off;     // [n_sub] first correspondence of the pair in the chunk
    const long long *dst_off;     // [n_sub + 1] offsets of the compact batch
    const double *x1, *x2, *d1, *d2, *cams;   // chunk inputs (cams may be null)
    double *sx1, *sx2, *sd1, *sd2, *scams;    // compact inputs
    Model *models; rp_stats *stats; unsigned char *masks;        // chunk outputs
    const Model *smodels; const rp_stats *sstats; const unsigned char *smasks;   // compact outputs
};
__global__ void gather_pairs_kernel(SubBatchArgs a) {
    const int j = blockIdx.x;
    if (j >= a.n_sub) return;
    const long long so = a.src_off[j], d0 = a.dst_off[j];
    const int n = (int)(a.dst_off[j + 1] - d0);
    for (int i = threadIdx.x; i < 2 * n; i += blockDim.x) {
        a.sx1[2 * d0 + i] = a.x1[2 * so + i];
        a.sx2[2 * d0 + i] = a.x2[2 * so + i];
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        a.sd1[d0 + i] = a.d1[so + i];
        a.sd2[d0 + i] = a.d2[so + i];
    }
    if (a.cams && threadIdx.x < 8) a.scams[8 * (size_t)j + threadIdx.x] = a.cams[8 * (size_t)a.pair_idx[j] + threadIdx.x];
}
__global__ void scatter_pairs_kernel(SubBatchArgs a) {
    const int j = blockIdx.x;
    if (j >= a.n_sub) return;
    const long long so = a.src_off[j], d0 = a.dst_off[j];
    const int n = (int)(a.dst_off[j + 1] - d0);
    for (int i = threadIdx.x; i < n; i += blockDim.x) a.masks[so + i] = a.smasks[d0 + i];
    if (threadIdx.x == 0) {
        a.models[a.pair_idx[j]] = a.smodels[j];
        a.stats[a.pair_idx[j]] = a.sstats[j];
    }
}

__global__ void fill_int_kernel(int *p, int n, int v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------------------------
// front end (SURVEY.md §8f item 2): the reference's callers look the monocular depth up at the matched
// keypoints, depth_map[(int)y, (int)x], and drop the rows whose two depths are both infinite
// (/root/reference/make_pair.py:97-106) on the host after a .cpu().numpy() round trip.  This kernel does
// the lookup, the mask and the stable compaction on the device, straight into the packed layout the
// estimator takes: T = double for rp_estimate_batch_*, T = float for rp_estimate_batch_*_f32 (the float
// inputs unchanged).  One block; rows keep their order.
// q_in / q_out (rp_gather_depths_*_quality; both null otherwise): a kept row's match quality goes to the same output
// position as its keypoints, copied as a 32-bit pattern (NaN payloads, -0 and infinities unchanged).  The keep rule
// never reads it.
template <class T>
__global__ void gather_depths_kernel(const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                                     const float *kp1, const float *kp2, const float *q_in, long long n, T *x1, T *x2,
                                     T *d1, T *d2, float *q_out, long long *n_out) {
    __shared__ int warp_tot[32];
    __shared__ long long running;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) running = 0;
    __syncthreads();
    for (long long base = 0; base < n; base += blockDim.x) {
        const long long i = base + tid;
        bool keep = false;
        float ax = 0, ay = 0, bx = 0, by = 0, da = 0, db = 0;
        if (i < n) {
            ax = kp1[2 * i]; ay = kp1[2 * i + 1]; bx = kp2[2 * i]; by = kp2[2 * i + 1];
            const int r1 = min(max((int)ay, 0), h1 - 1), c1 = min(max((int)ax, 0), w1 - 1);
            const int r2 = min(max((int)by, 0), h2 - 1), c2 = min(max((int)bx, 0), w2 - 1);
            da = depth1[(size_t)r1 * w1 + c1];
            db = depth2[(size_t)r2 * w2 + c2];
            keep = !(isinf(da) && isinf(db));
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warp_tot[wid] = __popc(m);
        __syncthreads();
        int wbase = 0, total = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            if (w < wid) wbase += warp_tot[w];
            total += warp_tot[w];
        }
        if (keep) {
            const long long o = running + wbase + __popc(m & ((1u << lane) - 1u));
            x1[2 * o] = ax; x1[2 * o + 1] = ay; x2[2 * o] = bx; x2[2 * o + 1] = by;
            d1[o] = da; d2[o] = db;
            if (q_out) ((unsigned *)q_out)[o] = ((const unsigned *)q_in)[i];
        }
        __syncthreads();
        if (tid == 0) running += total;
        __syncthreads();
    }
    if (tid == 0) *n_out = running;
}

// Batched form for video / many pairs (make_video.py:270-290 runs the same recipe per frame pair): depth maps of one
// size stacked [F, h, w], pair p = (frame1[p], frame2[p]) with keypoints [in_off[p], in_off[p+1]).  Pass 1: one CTA per
// pair, stable compaction of the pair's rows INTO ITS OWN INPUT RANGE of the temporary arrays + the kept count; the host
// reads the n_pairs counts once (it needs the packed offsets anyway: rp_estimate_batch_dev takes them), pass 2 moves
// every pair's block to its packed position.  T: output type, as in gather_depths_kernel.  q_in / tq / q_out: the match
// quality, carried through both passes as in gather_depths_kernel (all three null without one).
template <class T>
struct GatherBatchArgs {
    int n_pairs, h, w;
    const float *depth;            // [F, h, w]
    const int *frame1, *frame2;    // [n_pairs]
    const long long *in_off;       // [n_pairs + 1]
    const long long *out_off;      // [n_pairs + 1] (pass 2)
    const float *kp1, *kp2;        // [N, 2]
    T *tx1, *tx2, *td1, *td2;      // temporaries, capacity N
    T *x1, *x2, *d1, *d2;          // packed outputs
    int *count;                    // [n_pairs]
    const float *q_in;             // [N]
    float *tq, *q_out;             // temporary (capacity N), packed output
};
template <class T>
__global__ void gather_depths_batch_kernel(GatherBatchArgs<T> a) {
    __shared__ int warp_tot[32];
    __shared__ int running;
    const int pair = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const long long i0 = a.in_off[pair];
    const int n = (int)(a.in_off[pair + 1] - i0);
    const float *dm1 = a.depth + (size_t)a.frame1[pair] * a.h * a.w, *dm2 = a.depth + (size_t)a.frame2[pair] * a.h * a.w;
    if (tid == 0) running = 0;
    __syncthreads();
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + tid;
        bool keep = false;
        float ax = 0, ay = 0, bx = 0, by = 0, da = 0, db = 0;
        if (i < n) {
            ax = a.kp1[2 * (i0 + i)]; ay = a.kp1[2 * (i0 + i) + 1]; bx = a.kp2[2 * (i0 + i)]; by = a.kp2[2 * (i0 + i) + 1];
            const int r1 = min(max((int)ay, 0), a.h - 1), c1 = min(max((int)ax, 0), a.w - 1);
            const int r2 = min(max((int)by, 0), a.h - 1), c2 = min(max((int)bx, 0), a.w - 1);
            da = dm1[(size_t)r1 * a.w + c1];
            db = dm2[(size_t)r2 * a.w + c2];
            keep = !(isinf(da) && isinf(db));
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warp_tot[wid] = __popc(m);
        __syncthreads();
        int wbase = 0, total = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            if (w < wid) wbase += warp_tot[w];
            total += warp_tot[w];
        }
        if (keep) {
            const long long o = i0 + running + wbase + __popc(m & ((1u << lane) - 1u));
            a.tx1[2 * o] = ax; a.tx1[2 * o + 1] = ay; a.tx2[2 * o] = bx; a.tx2[2 * o + 1] = by;
            a.td1[o] = da; a.td2[o] = db;
            if (a.tq) ((unsigned *)a.tq)[o] = ((const unsigned *)a.q_in)[i0 + i];
        }
        __syncthreads();
        if (tid == 0) running += total;
        __syncthreads();
    }
    if (tid == 0) a.count[pair] = running;
}
template <class T>
__global__ void gather_depths_pack_kernel(GatherBatchArgs<T> a) {
    const int pair = blockIdx.x;
    const long long i0 = a.in_off[pair], o0 = a.out_off[pair];
    const int n = (int)(a.out_off[pair + 1] - o0);
    for (int i = threadIdx.x; i < 2 * n; i += blockDim.x) {
        a.x1[2 * o0 + i] = a.tx1[2 * i0 + i];
        a.x2[2 * o0 + i] = a.tx2[2 * i0 + i];
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        a.d1[o0 + i] = a.td1[i0 + i];
        a.d2[o0 + i] = a.td2[i0 + i];
    }
    if (a.q_out)
        for (int i = threadIdx.x; i < n; i += blockDim.x) ((unsigned *)a.q_out)[o0 + i] = ((const unsigned *)a.tq)[i0 + i];
}

// float32 inputs (rp_estimate_batch_*_f32): one chunk's x1, x2 [n,2] and d1, d2 [n] widened into the FP64 arrays every
// kernel downstream reads.  float -> double is exact, so the chunk is bit for bit what the FP64 entry points receive for
// the same values.  Grid-stride over the 6 n values of the chunk.
// With a permutation (rp_estimate_batch_*_quality, In = float or double) the same pass also gathers the chunk into its
// quality order: correspondence j of the output is correspondence perm[j] of its pair (pair_of over `offsets` - base),
// so the FP64 arrays hold each pair reordered and every kernel downstream runs unchanged on them.
template <class In>
__global__ void widen_inputs_kernel(long long n, const In *x1, const In *x2, const In *d1, const In *d2, const int *perm,
                                    const long long *offsets, long long base, int n_pairs, double *wx1, double *wx2,
                                    double *wd1, double *wd2) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (!perm) {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n; i += stride) {
            wx1[i] = (double)x1[i];
            wx2[i] = (double)x2[i];
            if (i < n) {
                wd1[i] = (double)d1[i];
                wd2[i] = (double)d2[i];
            }
        }
        return;
    }
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        const long long s = offsets[pair_of(j, offsets, base, n_pairs)] - base + perm[j];
        wx1[2 * j] = (double)x1[2 * s];
        wx1[2 * j + 1] = (double)x1[2 * s + 1];
        wx2[2 * j] = (double)x2[2 * s];
        wx2[2 * j + 1] = (double)x2[2 * s + 1];
        wd1[j] = (double)d1[s];
        wd2[j] = (double)d2[s];
    }
}

// ---------------------------------------------------------------------------------------------
// pipe micro-benchmarks (SURVEY.md §8d: the FP64 / FP32 FMA peaks are not in MEASURED_PEAKS.json)
// 16 independent FMA chains per thread, 8 blocks of 256 threads per SM: enough ILP x TLP to saturate either pipe
__global__ void fp64_pipe_kernel(double *out, int iters) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = threadIdx.x * 1e-3 + i;
    const double b = 1.0000001, c = 1e-9;
    for (int it = 0; it < iters; ++it)
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = fma(a[i], b, c);
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void fp32_pipe_kernel(float *out, int iters) {
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = threadIdx.x * 1e-3f + i;
    const float b = 1.0000001f, c = 1e-9f;
    for (int it = 0; it < iters; ++it)
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = fmaf(a[i], b, c);
    float s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace rp
