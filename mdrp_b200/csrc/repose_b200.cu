// repose_b200.cu — host orchestration + C ABI (include/repose_b200.h) of the batched RePoseD
// estimator.  Everything numeric happens in the kernels of rp_kernels.cuh; this file plans the
// chunks, owns the HBM workspace and replays the reference's call order:
//   estimate_* (so@0x224170 / 0x223300 / 0x223a40) -> ransac_* -> ransac<> -> final refinement.
// There is no host fallback: without a CUDA device rp_create fails.
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "rp_kernels.cuh"

using namespace rp;

namespace {

std::string g_create_error;

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// A device buffer that grows on demand and is freed with its owner
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T *as() const { return (T *)p; }
};

// Reserves each (buffer, bytes) in turn; stops at the first failure
cudaError_t reserve_all(std::initializer_list<std::pair<DevBuf *, size_t>> bufs) {
    for (const auto &b : bufs)
        if (const cudaError_t e = b.first->reserve(b.second)) return e;
    return cudaSuccess;
}

// device scalars living in PointBufs::scalars
struct Scalars {
    int n_items, n_lo_items, n_one_items, n_prob, n_pairs_scalar, any_flag, reserved0, n_first_items;
    int n_surv_items, bound_work, lm_work, score_work;  // *_work: counters the persistent kernels draw work from
    unsigned long long point_scores, lm_iters, n_survivors, evaluated_ps;
    long long n_hyp;
    int n_tc_items, n_tcsel_items;
    unsigned long long tc_evaluated, tc_selected, lm_flops;
};

// ---- the work arrays of a chunk, by the stage that owns them ---------------------------------------------------
// Each group's reserve states its sizes for a chunk of P pairs, N correspondences, nseg segments (slots = P nseg 4 SEG
// model slots) and ev_cap events.  bytes_per_pair and refine_bytes_per_pair below are the chunk planner's estimate of
// the same per pair.  Between calls the stage entry points borrow these buffers as scratch.

// points and pairs: prepare_kernel's output and the device scalars
struct PointBufs {
    DevBuf offs, pairs, pts64, pts32, pts32p, bear, scalars;
    cudaError_t reserve(int P, long long N) {
        const size_t n = (size_t)std::max<long long>(N, 1);
        return reserve_all({{&offs, sizeof(long long) * (P + 1)}, {&pairs, sizeof(PairParams) * P}, {&pts64, sizeof(Pt64) * n},
                            {&pts32, sizeof(float4) * n}, {&pts32p, 32 * (size_t)((N + P + 4) / 2 + 1)}, {&bear, sizeof(Bear) * n},
                            {&scalars, sizeof(Scalars)}});
    }
};
// hypotheses: samples, minimal models and their exact scores, per-segment counts and work-item prefix
struct HypBufs {
    DevBuf samples, models, hyp_iter, score, count, seg_count, item_prefix;
    cudaError_t reserve(int P, int iters, int nseg) {
        const size_t slots = (size_t)P * nseg * 4 * SEG;
        return reserve_all({{&samples, sizeof(int) * 3 * (size_t)P * std::max(iters, 1)}, {&models, sizeof(Model) * slots},
                            {&hyp_iter, sizeof(int) * slots}, {&score, sizeof(double) * slots}, {&count, sizeof(int) * slots},
                            {&seg_count, sizeof(int) * (size_t)P * nseg}, {&item_prefix, sizeof(int) * ((size_t)P * nseg + 1)}});
    }
};
// LO: the trigger events, the LO problems and their scores, the re-run flags
struct LoBufs {
    DevBuf events, n_events, lo_models, lo_of_event, lo_count, prob_list, lo_score, lo_cnt, lo_item_prefix, pair_flags;
    cudaError_t reserve(int P, int ev_cap) {
        const size_t e = (size_t)P * ev_cap;
        return reserve_all({{&events, sizeof(int) * e}, {&n_events, sizeof(int) * P}, {&lo_models, sizeof(Model) * e},
                            {&lo_of_event, sizeof(int) * e}, {&lo_count, sizeof(int) * P}, {&prob_list, sizeof(int) * e},
                            {&lo_score, sizeof(double) * e}, {&pair_flags, sizeof(int) * P}, {&lo_cnt, sizeof(int) * e},
                            {&lo_item_prefix, sizeof(int) * (P + 1)}});
    }
};
// per-pair results: the best model, the final LO's start and rescore, the one-item-per-pair list, the final
// refinement's enable flags, the stats (the merge's final_start and stats only with `merge`: the refinement has no merge)
struct ResultBufs {
    DevBuf best, final_start, final_score, final_count, ones, one_prefix, enable, stats;
    cudaError_t reserve(int P, bool merge) {
        if (merge) {
            if (const cudaError_t e = reserve_all({{&final_start, sizeof(Model) * P}, {&stats, sizeof(rp_stats) * P}})) return e;
        }
        return reserve_all({{&best, sizeof(Model) * P}, {&final_score, sizeof(double) * P}, {&final_count, sizeof(int) * P},
                            {&ones, sizeof(int) * P}, {&one_prefix, sizeof(int) * (P + 1)}, {&enable, sizeof(int) * P}});
    }
};
// prune and waves (with the FP32 bound kernel): bounds per slot, the head's bar (B0, S0), survivor lists and waves
struct PruneBufs {
    DevBuf ub, lb, first_cnt, first_prefix, B0, S0, surv_list, surv_cnt, surv_prefix, wave_cursor, wave_cnt;
    cudaError_t reserve(int P, int nseg) {
        const size_t slots = (size_t)P * nseg * 4 * SEG;
        return reserve_all({{&ub, sizeof(int) * slots}, {&lb, sizeof(float) * slots}, {&surv_list, sizeof(int) * slots},
                            {&first_cnt, sizeof(int) * P}, {&first_prefix, sizeof(int) * (P + 1)}, {&B0, sizeof(int) * P},
                            {&S0, sizeof(double) * P}, {&surv_cnt, sizeof(int) * P}, {&wave_cursor, sizeof(int) * P},
                            {&wave_cnt, sizeof(int) * P}, {&surv_prefix, sizeof(int) * (P + 1)}});
    }
};
// tensor-core tier: per-correspondence feature rows, per-model certain-outlier counts, the lists it passes on
struct TcBufs {
    DevBuf feat, out, list, list_cnt, list_prefix, pair_cnt, prefix, split;
    cudaError_t reserve(int P, long long N, int nseg) {
        const size_t slots = (size_t)P * nseg * 4 * SEG;
        return reserve_all({{&feat, 128 * (size_t)std::max<long long>(N, 1) + 128 * tc::NT}, {&out, sizeof(int) * slots},
                            {&list, sizeof(int) * slots}, {&list_cnt, sizeof(int) * P}, {&list_prefix, sizeof(int) * (P + 1)},
                            {&pair_cnt, sizeof(int) * P}, {&split, sizeof(int) * P}, {&prefix, sizeof(int) * (P + 1)}});
    }
};
// re-run sub-batch of S pairs and n correspondences (rerun_flagged): pair index and offsets, the gathered inputs, the
// sub-batch's outputs.  The batch depth gather borrows idx, src, dst and x1 … d2.
struct SubBufs {
    DevBuf idx, src, dst, x1, x2, d1, d2, cams, models, stats, mask, init;
    cudaError_t reserve(int S, size_t n, bool prior) {
        if (prior) {
            if (const cudaError_t e = init.reserve(sizeof(Model) * S)) return e;
        }
        return reserve_all({{&idx, sizeof(int) * S}, {&src, 8 * (size_t)S}, {&dst, 8 * ((size_t)S + 1)}, {&x1, 16 * n},
                            {&x2, 16 * n}, {&d1, 8 * n}, {&d2, 8 * n}, {&cams, 64 * (size_t)S}, {&models, sizeof(Model) * S},
                            {&stats, sizeof(rp_stats) * S}, {&mask, n}});
    }
};
// priors (estimator calls with init): the prior of each pair in the normalised frame and its exact count and score
struct PriorBufs {
    DevBuf model, count, score;
    cudaError_t reserve(int P) {
        return reserve_all({{&model, sizeof(Model) * P}, {&count, sizeof(int) * P}, {&score, sizeof(double) * P}});
    }
};
constexpr size_t PRIOR_BYTES_PER_PAIR = sizeof(Model) + sizeof(int) + sizeof(double);
// the remaining scratch
struct ScratchBufs {
    DevBuf order;     // quality calls: global sort scratch of pairs above RP_ORDER_SMEM_CAP
    DevBuf gather_q;  // rp_gather_depths_batch_dev*_quality: the compacted quality between the two passes (4 B per row)
    DevBuf tmp2;      // rp_refine_batch: bundle stats
};

// Device bytes per pair of an estimator chunk (the chunk planner's estimate; the reserves above are the exact sizes);
// `pair_bytes`: per-pair extras (PRIOR_BYTES_PER_PAIR with priors)
size_t bytes_per_pair(int iters, long long avg_points, int ev_cap = EV, size_t input_bytes = 0, size_t pair_bytes = 0) {
    const int nseg = std::max(1, cdiv(iters, SEG));
    const size_t slots_pp = (size_t)nseg * 4 * SEG;
    // per slot: model, hyp_iter, score, count, ub, lb, survivor list, tensor-core count + list; per correspondence:
    // FP64 / FP32 / interleaved copies, bearings, mask, 128-byte feature row, `input_bytes` of input staging
    return slots_pp * (sizeof(Model) + 4 + 8 + 4 + 12 + 8) + (size_t)iters * 12 + (size_t)ev_cap * (sizeof(Model) + 24) +
           (size_t)avg_points * (sizeof(Pt64) + 32 + sizeof(Bear) + 1 + 128 + input_bytes) + 1024 + pair_bytes;
}

// Device workspace of a refine chunk.  Per correspondence: pts64 (32 B), pts32 (16), the pair-interleaved FP32 copy
// (16), bearings (48), and the chunk's I/O: FP64 inputs (48), subset (1), inlier mask (1); the host path double-buffers
// the I/O and adds the float32 staging (24 B, double-buffered) for float32 inputs.  Per pair: PairParams, the work,
// start and output models, bundle stats, cams, and a few counters.
size_t refine_bytes_per_pair(long long avg_points, bool host_io, bool f32) {
    const size_t io_pt = 48 + 1 + 1 + (host_io && f32 ? 24 : 0);
    const size_t io_pair = 2 * sizeof(Model) + sizeof(rp_bundle_stats) + 64 + 8;
    const size_t sets = host_io ? 2 : 1;
    return (size_t)avg_points * (32 + 16 + 16 + 48 + sets * io_pt) + sizeof(PairParams) + sizeof(Model) + 32 +
           sets * io_pair + 64;
}

// One double-buffer set of the chunk pipeline (stage_inputs / run_chunks): a chunk's inputs on their way in and its
// outputs on their way out.  rp_ctx keeps two; on the host path chunk c uses set c & 1, the device path uses set 0 for
// what it widens or orders, and the stage entry points borrow set 0's buffers as scratch.
struct StageSet {
    DevBuf x1, x2, d1, d2, cams;          // the chunk's FP64 inputs
    DevBuf sx1, sx2, sd1, sd2;            // host path: the chunk as uploaded (input type) when it is widened or ordered
    DevBuf qual, offs, perm, ksort;       // quality calls: quality, the chunk's offsets and order, masks in the ordered layout
    DevBuf init, subset;                  // refinement: start models, subset
    DevBuf models, stats, mask, ninl;     // output staging: models, stats or bundle stats, mask, num_inliers
    // upload [h2d_begin, h2d_end), widening / ordering [h2d_end, in_ready), kernels done, read-back [d2h_begin, d2h_end)
    cudaEvent_t h2d_begin = nullptr, h2d_end = nullptr, in_ready = nullptr, done = nullptr, d2h_begin = nullptr,
                d2h_end = nullptr;
    void create_events() {
        for (cudaEvent_t *e : {&h2d_begin, &h2d_end, &in_ready, &done, &d2h_begin, &d2h_end}) cudaEventCreate(e);
    }
    void destroy_events() {
        for (cudaEvent_t e : {h2d_begin, h2d_end, in_ready, done, d2h_begin, d2h_end}) cudaEventDestroy(e);
    }
};

// The minimal-model scoring: the exact head is HB models per pair; with the tensor-core tier a short head of
// HEAD_SMALL models is followed by one mid stage over positions [HEAD_SMALL, MID_END) of the pair's first segment
// (profiles/r02_head_sweep.txt, r02_mid_stage_sweep.txt)
constexpr int HEAD_SMALL = 32, MID_END = 256;

// run_chunk: [0..8] stage boundaries, [9] start of the bulk cascade, [10] bound kernel done, [11] tensor-core tier done;
// [12], [13]: an interval of their own (the mask scatter of quality calls, rp_measure_pipes); [14] start of the prior
// stage (calls with priors: it ends at [1])
constexpr int N_EVENTS = 15;

}  // namespace

struct rp_ctx {
    int device = 0;
    int sms = 148;
    std::string err;
    int64_t launches = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of chunk c+1 / D2H of chunk c-1 overlap the kernels of chunk c
    PointBufs pt;
    HypBufs hyp;
    LoBufs lo;
    ResultBufs res;
    PruneBufs prn;
    TcBufs tcb;
    SubBufs sub;
    PriorBufs pri;
    ScratchBufs scratch;
    StageSet set[2];
    cudaEvent_t ev[N_EVENTS];
    double last_ms[16] = {0};
    double prev_h2d_ms = 0.0, prev_dev_ms = 0.0;  // upload / kernel time of the previous host-path call (lead-chunk sizing)
    int64_t last_cnt[16] = {0};  // [5] models through the exact kernel, [6] point-scores the bound kernel evaluated
    size_t workspace_budget = (size_t)80 << 30;  // HBM is 180 GB: big chunks amortise kernel tails and launches (10 000 pairs x 10 000
                                                 // iterations = one 71 GB chunk; measured 32 -> 80 GB: +3 %); capped at half of the free memory
    bool prune = true;  // hypothesis-level pruning (RP_NO_PRUNE=1 scores every minimal model exactly)
    bool waves = true;  // survivors of the prune scored in waves (RP_NO_WAVES=1: all at once)
    bool lm_warp = true;  // the LO refinements run one warp per LM problem (lm_warp_kernel) instead of one block
                          // (RP_LM_WARP=0: the block-per-problem kernel everywhere)
    bool mid = true;    // with the tensor-core tier: short head + mid stage (RP_MID_END=0: the HB-model exact head)
    bool tc = true;     // tensor-core count tier in front of the FP32 bound kernel (RP_NO_TC=1: off)
    bool tc_two_pass = true;  // that tier in two passes, split per pair by tc_split (RP_TC_ONE_PASS=1: one pass over everything)
    bool solve_generic = false;  // RP_SOLVE_GENERIC: the thread-per-iteration solve kernel for every variant (the
                                 // two-phase kernels must give bit-identical models)
    void *encode_tiled = nullptr;  // cuTensorMapEncodeTiled (driver entry point, resolved at rp_create)
    int ev_cap0 = EV;   // event-list capacity of the first pass (RP_EV_CAP: small values exercise the re-run path)
    std::vector<int32_t> pair_status;  // per pair of the last rp_estimate_batch_* call (rp_pair_status)
};

namespace {

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            char b_[512];                                                                            \
            snprintf(b_, sizeof b_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,             \
                     cudaGetErrorString(e_));                                                        \
            ctx->err = b_;                                                                           \
            return RP_ERR_CUDA;                                                                      \
        }                                                                                            \
    } while (0)

#define LAUNCHED()                                                                                   \
    do {                                                                                             \
        ctx->launches++;                                                                             \
        CK(cudaGetLastError());                                                                      \
    } while (0)

int fail(rp_ctx *ctx, int code, const char *msg) {
    if (ctx) ctx->err = msg;
    return code;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// tensor-core count tier over every minimal model of the chunk (rp_tc.cuh): feature rows [n_rows x 32 floats] through a
// SWIZZLE_128B tensor map, 64 rows per TMA box
int launch_tc(rp_ctx *ctx, const tc::TcArgs &a, float4 *feat, long long n_rows, cudaStream_t st) {
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {(cuuint64_t)tc::FEAT, (cuuint64_t)std::max<long long>(n_rows, 1)};
    const cuuint64_t gstride[1] = {(cuuint64_t)tc::FEAT * 4};
    const cuuint32_t box[2] = {(cuuint32_t)tc::FEAT, (cuuint32_t)tc::NT};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult cr = ((EncodeTiledFn)ctx->encode_tiled)(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, feat, gdim, gstride, box, estr,
                                                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
        ctx->err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)cr) + ")";
        return RP_ERR_CUDA;
    }
    tc::tc_count_kernel<0><<<ctx->sms, tc::THREADS, tc::SMEM_BYTES, st>>>(tmap, a);
    LAUNCHED();
    return RP_OK;
}

template <class K>
int occupancy_grid(rp_ctx *ctx, K kernel, int threads) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, 0) != cudaSuccess || nb < 1) nb = 1;
    return nb * ctx->sms;
}

// ---- kernel launch helpers ---------------------------------------------------------------------
int launch_score(rp_ctx *ctx, bool pose, bool mask, const ScoreArgs &args, cudaStream_t st) {
    int grid;
    ScoreArgs a = args;
    a.work_counter = &ctx->pt.scalars.as<Scalars>()->score_work;
    CK(cudaMemsetAsync(a.work_counter, 0, sizeof(int), st));
    if (pose) {
        if (mask) { grid = occupancy_grid(ctx, score_kernel<true, true>, SCORE_THREADS); score_kernel<true, true><<<grid, SCORE_THREADS, 0, st>>>(a); }
        else { grid = occupancy_grid(ctx, score_kernel<true, false>, SCORE_THREADS); score_kernel<true, false><<<grid, SCORE_THREADS, 0, st>>>(a); }
    } else {
        if (mask) { grid = occupancy_grid(ctx, score_kernel<false, true>, SCORE_THREADS); score_kernel<false, true><<<grid, SCORE_THREADS, 0, st>>>(a); }
        else { grid = occupancy_grid(ctx, score_kernel<false, false>, SCORE_THREADS); score_kernel<false, false><<<grid, SCORE_THREADS, 0, st>>>(a); }
    }
    LAUNCHED();
    return RP_OK;
}

int launch_bound(rp_ctx *ctx, bool pose, const BoundArgs &a, cudaStream_t st) {
    CK(cudaMemsetAsync(a.work_counter, 0, sizeof(int), st));   // (launched twice per chunk: mid stage and bulk)
    if (pose) bound_kernel<true><<<occupancy_grid(ctx, bound_kernel<true>, SCORE_THREADS), SCORE_THREADS, 0, st>>>(a);
    else bound_kernel<false><<<occupancy_grid(ctx, bound_kernel<false>, SCORE_THREADS), SCORE_THREADS, 0, st>>>(a);
    LAUNCHED();
    return RP_OK;
}

// (counted by hand: launch_lm_kernel launches the one LM kernel it selects)
int launch_lm(rp_ctx *ctx, int variant, const LMArgs &a, cudaStream_t st) {
    ctx->launches++;
    // problems differ in cost (1..max_iterations LM iterations): blocks draw them from a counter
    LMArgs la = a;
    la.work_counter = &ctx->pt.scalars.as<Scalars>()->lm_work;
    la.warp_kernel = ctx->lm_warp ? 1 : 0;
    la.warp_single = 0;   // the final LO (one problem per pair, no problem list) stays on the block kernel
    CK(cudaMemsetAsync(la.work_counter, 0, sizeof(int), st));
    CK((cudaError_t)launch_lm_kernel(ctx->sms, variant, la, st));
    return RP_OK;
}

__global__ void valid_ones_kernel(int n_pairs, const PairParams *pairs, int *ones) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pairs) ones[i] = pairs[i].valid ? 1 : 0;
}

// stage helper: already-normalised correspondences of ONE pair -> pts64 / pts32 / bearings + bounds
__global__ void stage_points_kernel(int n, const double *x1, const double *x2, double sq_thr, Pt64 *pts64,
                                    float4 *pts32, Bear *bear, PairParams *pair) {
    const int lane = threadIdx.x;
    double Mmax = 0.0, mmax = 0.0;
    for (int k = lane; k < n; k += 32) {
        Pt64 p;
        p.x1_0 = x1[2 * k]; p.x1_1 = x1[2 * k + 1]; p.x2_0 = x2[2 * k]; p.x2_1 = x2[2 * k + 1];
        pts64[k] = p;
        pts32[k] = make_float4((float)p.x1_0, (float)p.x1_1, (float)p.x2_0, (float)p.x2_1);
        const V3 b1 = bearing(p.x1_0, p.x1_1), b2 = bearing(p.x2_0, p.x2_1);
        Bear b;
        b.b1x = b1.x; b.b1y = b1.y; b.b1z = b1.z; b.b2x = b2.x; b.b2y = b2.y; b.b2z = b2.z;
        bear[k] = b;
        const double m1 = fabs(p.x1_0) + fabs(p.x1_1) + 1.0, m2 = fabs(p.x2_0) + fabs(p.x2_1) + 1.0;
        Mmax = fmax(Mmax, m1 * m2);
        mmax = fmax(mmax, fmax(m1, m2));
    }
    Mmax = warp_max(Mmax);
    mmax = warp_max(mmax);
    if (lane == 0) {
        PairParams pp;
        pp.off = 0; pp.n = n; pp.valid = 1;
        pp.sq_thr = sq_thr;
        pp.thr = sqrt(sq_thr) * (1.0 + 1e-15);  // only feeds the (conservative) FP32 filter bound
        pp.scale_reproj = 0.0; pp.lo_loss_scale = pp.thr; pp.final_loss_scale = pp.thr; pp.nscale = 1.0;
        pp.Mmax = Mmax * 1.000001; pp.mmax = mmax * 1.000001; pp.pbase = 0;
        *pair = pp;
    }
}

// ---- one chunk of pairs, everything on device ----------------------------------------------------
// The chunk's FP64 inputs on the device (stage_inputs) and where run_chunk / refine_chunk write its results
struct ChunkIO {
    int n_pairs = 0;
    long long n_points = 0;
    const long long *h_offsets_rel = nullptr;  // host, [n_pairs+1], relative to the chunk
    const double *x1 = nullptr, *x2 = nullptr, *d1 = nullptr, *d2 = nullptr, *cams = nullptr;  // device, chunk-local
    const Model *init = nullptr;               // refinement: start models; estimator: priors (null: none) [n_pairs]
    const unsigned char *subset = nullptr;     // refinement: [n_points] or null (every correspondence)
    Model *models_out = nullptr;               // [n_pairs] (refinement: may alias init)
    rp_stats *stats_out = nullptr;             // estimator: [n_pairs]
    rp_bundle_stats *bstats_out = nullptr;     // refinement: [n_pairs] or null
    long long *num_inliers_out = nullptr;      // refinement: [n_pairs] or null
    unsigned char *masks_out = nullptr;        // [n_points]; refinement: null = no scoring (then num_inliers_out is null)
};

// First step of run_chunk and refine_chunk: the workspace both need, the Scalars (n_pairs_scalar = P) and the chunk's
// offsets, then prepare_kernel (PairParams, pts64 / pts32 / pts32p / bearings).  `ev_uploaded`, if given, is recorded
// between the uploads and the launch (run_chunk's slot [0] starts there).
int prepare_chunk(rp_ctx *ctx, int variant, const rp_options &opt, const ChunkIO &io, cudaEvent_t ev_uploaded,
                  cudaStream_t st) {
    const int P = io.n_pairs;
    PointBufs &B = ctx->pt;
    CK(B.reserve(P, io.n_points));
    Scalars h_sc;
    memset(&h_sc, 0, sizeof h_sc);
    h_sc.n_pairs_scalar = P;
    CK(cudaMemcpyAsync(B.scalars.p, &h_sc, sizeof h_sc, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B.offs.p, io.h_offsets_rel, sizeof(long long) * (P + 1), cudaMemcpyHostToDevice, st));
    if (ev_uploaded) CK(cudaEventRecord(ev_uploaded, st));
    PrepareArgs a;
    a.variant = variant; a.n_pairs = P; a.offsets = B.offs.as<long long>();
    a.x1 = io.x1; a.x2 = io.x2; a.cams = io.cams;
    a.max_epipolar_error = opt.max_epipolar_error; a.max_reproj_error = opt.max_reproj_error;
    a.loss_scale = opt.loss_scale;
    a.pts64 = B.pts64.as<Pt64>(); a.pts32 = B.pts32.as<float4>(); a.bear = B.bear.as<Bear>();
    a.pairs = B.pairs.as<PairParams>(); a.pts32p = B.pts32p.as<float>();
    prepare_kernel<<<cdiv((long long)P * 32, 256), 256, 0, st>>>(a);
    LAUNCHED();
    return RP_OK;
}

// The final refinement (run_chunk's step 8, refine_chunk): the caller's bundle options on one model per pair, on the
// correspondences of `mask` (null: all of them), for the pairs `enable` marks
LMArgs final_lm_args(rp_ctx *ctx, const rp_options &opt, const ChunkIO &io, Model *models, const unsigned char *mask,
                     const int *enable) {
    const PointBufs &B = ctx->pt;
    LMArgs la;
    memset(&la, 0, sizeof la);
    la.pairs = B.pairs.as<PairParams>(); la.pts64 = B.pts64.as<Pt64>(); la.d1 = io.d1; la.d2 = io.d2;
    la.weight_sampson = opt.weight_sampson;
    la.loss_scale_override = -1.0; la.scale_reproj_override = -1.0;
    la.prob_list = nullptr; la.n_prob = &B.scalars.as<Scalars>()->n_pairs_scalar; la.prob_per_pair = 1;
    la.models = models; la.use_final = 1; la.mask = mask; la.enable = enable;
    la.max_iterations = (int)opt.bundle_max_iterations; la.loss_type = opt.loss_type;
    la.gradient_tol = opt.gradient_tol; la.step_tol = opt.step_tol; la.initial_lambda = opt.initial_lambda;
    la.min_lambda = opt.min_lambda; la.max_lambda = opt.max_lambda;
    return la;
}

// One work item per valid pair (ones, one_prefix, n_one_items): the list pair_score_args scores over.  run_chunk builds
// it once for the final LO's rescore and its get_inliers.
int launch_pair_items(rp_ctx *ctx, int P, cudaStream_t st) {
    const ResultBufs &R = ctx->res;
    valid_ones_kernel<<<cdiv(P, 256), 256, 0, st>>>(P, ctx->pt.pairs.as<PairParams>(), R.ones.as<int>());
    LAUNCHED();
    build_items_kernel<<<1, 1024, 0, st>>>(P, R.ones.as<int>(), R.one_prefix.as<int>(),
                                           &ctx->pt.scalars.as<Scalars>()->n_one_items, nullptr);
    LAUNCHED();
    return RP_OK;
}

// score_kernel's view of the chunk's pairs and correspondences; the caller fills in the models and the work items
ScoreArgs chunk_score_args(const rp_ctx *ctx) {
    ScoreArgs s;
    memset(&s, 0, sizeof s);
    s.pairs = ctx->pt.pairs.as<PairParams>();
    s.pts32 = ctx->pt.pts32.as<float4>(); s.pts64 = ctx->pt.pts64.as<Pt64>(); s.bear = ctx->pt.bear.as<Bear>();
    return s;
}

// score_kernel over one model per pair on the launch_pair_items list; score and count per pair go to final_score /
// final_count, the mask (with the mask variant) to `mask`
ScoreArgs pair_score_args(rp_ctx *ctx, int P, const Model *models, unsigned char *mask) {
    const ResultBufs &R = ctx->res;
    ScoreArgs s = chunk_score_args(ctx);
    s.n_groups = P; s.grp_stride = 1; s.grp_per_pair = 1; s.grp_cnt = R.ones.as<int>();
    s.item_prefix = R.one_prefix.as<int>(); s.n_items = &ctx->pt.scalars.as<Scalars>()->n_one_items;
    s.models = models;
    s.score = R.final_score.as<double>(); s.count = R.final_count.as<int>(); s.mask = mask;
    return s;
}

// get_inliers: the inlier mask of `models` (one per pair) over the chunk's correspondences
int launch_get_inliers(rp_ctx *ctx, bool pose, const ChunkIO &io, const Model *models, unsigned char *mask,
                       cudaStream_t st) {
    if (io.n_points > 0) CK(cudaMemsetAsync(mask, 0, (size_t)io.n_points, st));
    return launch_score(ctx, pose, true, pair_score_args(ctx, io.n_pairs, models, mask), st);
}

// What the stages of one run_chunk call share, filled once after the reserves (rerun_flagged's nested run_chunk fills
// its own)
struct Chunk {
    const rp_options *opt;
    const ChunkIO *io;
    int variant, P, iters, nseg, ev_cap;
    bool pose, use_tc, mid;  // use_tc: the tensor-core tier (it needs the prune); mid: short head + mid stage (with that tier)
    int head;                // with the prune: models per pair scored exactly up front
    long long N;
    size_t slots_pp;
    cudaStream_t st;
    // the device arrays the stages share
    Scalars *sc;
    PairParams *pairs;
    Pt64 *pts64;
    float4 *pts32;
    Model *models;
    double *score;
    int *hyp_iter, *count, *seg_count, *item_prefix;
    // with priors (io->init): the normalised priors and their exact counts and scores; null otherwise
    Model *prior;
    int *prior_cnt;
    double *prior_score;
};

Chunk chunk_of(rp_ctx *ctx, int variant, const rp_options &opt, const ChunkIO &io, int iters, int ev_cap,
               cudaStream_t st) {
    Chunk c;
    c.opt = &opt; c.io = &io; c.variant = variant; c.pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    c.use_tc = ctx->prune && ctx->tc; c.mid = c.use_tc && ctx->mid; c.head = c.mid ? HEAD_SMALL : HB;
    c.P = io.n_pairs; c.N = io.n_points; c.iters = iters; c.nseg = std::max(1, cdiv(iters, SEG)); c.ev_cap = ev_cap;
    c.slots_pp = (size_t)c.nseg * 4 * SEG; c.st = st;
    c.sc = ctx->pt.scalars.as<Scalars>(); c.pairs = ctx->pt.pairs.as<PairParams>(); c.pts64 = ctx->pt.pts64.as<Pt64>();
    c.pts32 = ctx->pt.pts32.as<float4>();
    c.models = ctx->hyp.models.as<Model>(); c.hyp_iter = ctx->hyp.hyp_iter.as<int>(); c.score = ctx->hyp.score.as<double>();
    c.count = ctx->hyp.count.as<int>(); c.seg_count = ctx->hyp.seg_count.as<int>();
    c.item_prefix = ctx->hyp.item_prefix.as<int>();
    const bool pri = io.init != nullptr;
    c.prior = pri ? ctx->pri.model.as<Model>() : nullptr;
    c.prior_cnt = pri ? ctx->pri.count.as<int>() : nullptr;
    c.prior_score = pri ? ctx->pri.score.as<double>() : nullptr;
    return c;
}

// 1b. the prior stage (calls with priors): the priors into the normalised frame, and one exact score per pair with a
// usable prior (count, score of the prior: scan_kernel's starting point, the seed of the cascade's bars, the merge's
// first event)
int prior_stage(rp_ctx *ctx, const Chunk &c) {
    prior_import_kernel<<<cdiv(c.P, 256), 256, 0, c.st>>>(c.P, c.variant, c.pairs, c.io->init, c.prior,
                                                          ctx->res.ones.as<int>(), c.prior_cnt, c.prior_score);
    LAUNCHED();
    build_items_kernel<<<1, 1024, 0, c.st>>>(c.P, ctx->res.ones.as<int>(), ctx->res.one_prefix.as<int>(),
                                             &c.sc->n_one_items, nullptr);
    LAUNCHED();
    ScoreArgs s = pair_score_args(ctx, c.P, c.prior, nullptr);
    s.score = c.prior_score; s.count = c.prior_cnt;
    return launch_score(ctx, c.pose, false, s, c.st);
}

// 2. sample
int sample_stage(rp_ctx *ctx, const Chunk &c) {
    if (c.iters <= 0) return RP_OK;
    const rp_options &opt = *c.opt;
    int *samples = ctx->hyp.samples.as<int>();
    if (opt.progressive_sampling)
        sample_prosac_kernel<<<cdiv((long long)c.P * 32, 256), 256, 0, c.st>>>(
            c.P, c.iters, c.pairs, opt.seed, (unsigned long long)std::max<int64_t>(opt.max_prosac_iterations, 0), samples);
    else
        sample_kernel<<<cdiv((long long)c.P * 32, 256), 256, 0, c.st>>>(c.P, c.iters, c.pairs, opt.seed, samples);
    LAUNCHED();
    return RP_OK;
}

// 3. solve: the two-phase kernel of the variant, or with RP_SOLVE_GENERIC the thread-per-iteration kernel (the one
// RP_VARYING always runs)
int solve_stage(rp_ctx *ctx, const Chunk &c) {
    SolveArgs a;
    a.variant = c.variant; a.iters = c.iters; a.nseg = c.nseg; a.pairs = c.pairs; a.samples = ctx->hyp.samples.as<int>();
    a.pts64 = c.pts64; a.d1 = c.io->d1; a.d2 = c.io->d2; a.models = c.models; a.hyp_iter = c.hyp_iter; a.seg_count = c.seg_count;
    const dim3 grid(c.nseg, c.P);
    const bool generic = ctx->solve_generic;
    cudaStream_t st = c.st;
    switch (c.variant) {
    case RP_CALIB:
        if (generic) solve_kernel<RP_CALIB><<<grid, SOLVE_THREADS, 0, st>>>(a);
        else solve2_kernel<P3PCand><<<grid, SOLVE_THREADS, 0, st>>>(a);
        break;
    case RP_CALIB_SHIFT:
        if (generic) solve_kernel<RP_CALIB_SHIFT><<<grid, SOLVE_THREADS, 0, st>>>(a);
        else solve2_kernel<ShiftCand><<<grid, SOLVE_THREADS, 0, st>>>(a);
        break;
    case RP_SHARED:
        if (generic) solve_kernel<RP_SHARED><<<grid, SOLVE_THREADS, 0, st>>>(a);
        else solve2_kernel<FocalCand><<<grid, SOLVE_THREADS, 0, st>>>(a);
        break;
    default: solve_kernel<RP_VARYING><<<grid, SOLVE_THREADS, 0, st>>>(a); break;
    }
    LAUNCHED();
    return RP_OK;
}

// The tensor-core tier over the models at positions [start, limit) of the first segment (limit > 0) or [start, end) of
// the pair (limit = 0): pass 0 counts every model of the range against the first part of its pair's correspondences
// (with `two_pass`; all of them otherwise) and tc_select_kernel drops what already has enough certain outliers; pass 1
// counts the remaining correspondences for the models that are left and tc_select_list_kernel decides again.  The
// models it passes on are the per-pair lists (list, list_cnt, list_prefix, n_tcsel_items) of the bound kernel.
// `ev_tc`, if given, is recorded when the tier is done.
int tc_tier(rp_ctx *ctx, const Chunk &c, int start, int limit, bool two_pass, cudaEvent_t ev_tc) {
    const int P = c.P;
    cudaStream_t st = c.st;
    Scalars *sc = c.sc;
    const TcBufs &T = ctx->tcb;
    const PruneBufs &W = ctx->prn;
    range_count_kernel<<<cdiv(P, 256), 256, 0, st>>>(P, c.nseg, c.seg_count, start, limit, T.pair_cnt.as<int>());
    LAUNCHED();
    build_items_kernel<<<1, 1024, 0, st>>>(P, T.pair_cnt.as<int>(), T.prefix.as<int>(), &sc->n_tc_items, nullptr, tc::TILE_MODELS);
    LAUNCHED();
    tc::TcArgs ta;
    memset(&ta, 0, sizeof ta);
    ta.n_pairs = P; ta.nseg = c.nseg; ta.pairs = c.pairs; ta.seg_count = c.seg_count; ta.item_prefix = T.prefix.as<int>();
    ta.n_items = &sc->n_tc_items; ta.models = c.models; ta.out = T.out.as<int>(); ta.pose = c.pose ? 1 : 0;
    ta.evaluated = &sc->tc_evaluated; ta.first = start;
    ta.two_pass = two_pass ? 1 : 0; ta.pass = 0; ta.split = T.split.as<int>();
    if (two_pass) {
        tc::tc_split_kernel<<<cdiv(P, 256), 256, 0, st>>>(P, c.pairs, W.B0.as<int>(), W.S0.as<double>(), T.split.as<int>());
        LAUNCHED();
    }
    int rc = launch_tc(ctx, ta, T.feat.as<float4>(), c.N, st);
    if (rc) return rc;
    TcSelectArgs sel;
    sel.n_pairs = P; sel.nseg = c.nseg; sel.head = start; sel.limit = limit; sel.pairs = c.pairs; sel.seg_count = c.seg_count;
    sel.out = T.out.as<int>(); sel.B0 = W.B0.as<int>(); sel.S0 = W.S0.as<double>(); sel.ub = W.ub.as<int>();
    sel.lb = W.lb.as<float>(); sel.list = T.list.as<int>(); sel.list_cnt = T.list_cnt.as<int>();
    sel.n_selected = two_pass ? nullptr : &sc->tc_selected;
    tc_select_kernel<<<cdiv((long long)P * 32, 256), 256, 0, st>>>(sel);
    LAUNCHED();
    if (two_pass) {
        build_items_kernel<<<1, 1024, 0, st>>>(P, T.list_cnt.as<int>(), T.prefix.as<int>(), &sc->n_tc_items, nullptr, tc::TILE_MODELS);
        LAUNCHED();
        ta.pass = 1; ta.first = 0; ta.list = T.list.as<int>(); ta.list_cnt = T.list_cnt.as<int>(); ta.list_stride = (int)c.slots_pp;
        rc = launch_tc(ctx, ta, T.feat.as<float4>(), c.N, st);
        if (rc) return rc;
        sel.n_selected = &sc->tc_selected;
        tc_select_list_kernel<<<cdiv((long long)P * 32, 256), 256, 0, st>>>(sel);
        LAUNCHED();
    }
    if (ev_tc) CK(cudaEventRecord(ev_tc, st));
    build_items_kernel<<<1, 1024, 0, st>>>(P, T.list_cnt.as<int>(), T.list_prefix.as<int>(), &sc->n_tcsel_items, nullptr);
    LAUNCHED();
    return RP_OK;
}

// The survivors of the prune scored exactly, all at once (RP_NO_WAVES=1: the check that the waves change nothing).
// `fold`: a later stage follows, so these exact results are folded into (B0, S0).
int score_survivors_at_once(rp_ctx *ctx, const Chunk &c, ScoreArgs sv, WaveArgs wa, bool fold) {
    build_items_kernel<<<1, 1024, 0, c.st>>>(c.P, wa.surv_cnt, ctx->prn.surv_prefix.as<int>(), &c.sc->n_surv_items, nullptr);
    LAUNCHED();
    sv.grp_cnt = wa.surv_cnt;
    int rc = launch_score(ctx, c.pose, false, sv, c.st);
    if (rc) return rc;
    if (fold) {
        CK(cudaMemsetAsync(wa.cursor, 0, sizeof(int) * c.P, c.st));
        CK(cudaMemcpyAsync(wa.wave_cnt, wa.surv_cnt, sizeof(int) * c.P, cudaMemcpyDeviceToDevice, c.st));
        wa.wave_size = 0; wa.first = 0; wa.n_exact = nullptr;
        wave_select_kernel<<<cdiv((long long)c.P * 32, 256), 256, 0, c.st>>>(wa);
        LAUNCHED();
    }
    return RP_OK;
}

// The survivors of the prune scored exactly in waves of growing size, each raising the bar for the next
// (wave_select_kernel).  `fold`: a later stage follows, so the last wave's exact results are folded into (B0, S0).
int score_survivors_in_waves(rp_ctx *ctx, const Chunk &c, ScoreArgs sv, WaveArgs wa, bool fold) {
    CK(cudaMemsetAsync(wa.cursor, 0, sizeof(int) * c.P, c.st));
    static const int WAVES[] = {8, 16, 32, 64, 0x7fffffff};
    for (int k = 0; k < 5; ++k) {
        wa.wave_size = WAVES[k]; wa.first = k == 0;
        wave_select_kernel<<<cdiv((long long)c.P * 32, 256), 256, 0, c.st>>>(wa);
        LAUNCHED();
        build_items_kernel<<<1, 1024, 0, c.st>>>(c.P, wa.wave_cnt, ctx->prn.surv_prefix.as<int>(), &c.sc->n_surv_items, nullptr);
        LAUNCHED();
        sv.grp_cnt = wa.wave_cnt;
        int rc = launch_score(ctx, c.pose, false, sv, c.st);
        if (rc) return rc;
    }
    if (fold) {
        wa.wave_size = 0; wa.first = 0; wa.n_exact = nullptr;
        wave_select_kernel<<<cdiv((long long)c.P * 32, 256), 256, 0, c.st>>>(wa);
        LAUNCHED();
    }
    return RP_OK;
}

// 4b / 4c for the models at positions [start, limit) of the first segment (limit > 0: the mid stage) or [start, end) of
// the pair (limit = 0: the bulk): tensor-core tier (with the tier on), FP32 bound kernel over what that tier could not
// drop, prune, exact scoring of the survivors.  (B0, S0) are raised in place.  `ev_bound`, if given, is recorded when
// the bound kernel is done.
int cascade(rp_ctx *ctx, const Chunk &c, int start, int limit, bool two_pass, cudaEvent_t ev_tc, cudaEvent_t ev_bound) {
    const int P = c.P;
    const int stride = (int)c.slots_pp;
    cudaStream_t st = c.st;
    Scalars *sc = c.sc;
    const PruneBufs &W = ctx->prn;
    const TcBufs &T = ctx->tcb;
    BoundArgs ba;
    ba.n_groups = P * c.nseg; ba.grp_stride = 4 * SEG; ba.grp_per_pair = c.nseg; ba.grp_cnt = c.seg_count;
    ba.item_prefix = c.item_prefix; ba.n_items = &sc->n_items; ba.pairs = c.pairs; ba.models = c.models;
    ba.pts32p = ctx->pt.pts32p.as<ulonglong2>();
    ba.ub = W.ub.as<int>(); ba.lb = W.lb.as<float>(); ba.point_scores = &sc->point_scores;
    ba.B0 = W.B0.as<int>(); ba.S0 = W.S0.as<double>();
    ba.evaluated = &sc->evaluated_ps;
    ba.work_counter = &sc->bound_work; ba.head = start;
    ba.slot_list = nullptr; ba.list_stride = 0;
    int rc;
    if (c.use_tc) {
        if ((rc = tc_tier(ctx, c, start, limit, two_pass, ev_tc))) return rc;
        ba.n_groups = P; ba.grp_stride = stride; ba.grp_per_pair = 1; ba.grp_cnt = T.list_cnt.as<int>();
        ba.item_prefix = T.list_prefix.as<int>(); ba.n_items = &sc->n_tcsel_items;
        ba.slot_list = T.list.as<int>(); ba.list_stride = stride;
    }
    if ((rc = launch_bound(ctx, c.pose, ba, st))) return rc;
    if (ev_bound) CK(cudaEventRecord(ev_bound, st));
    // prune, then score the survivors exactly
    PruneArgs pa;
    pa.n_pairs = P; pa.nseg = c.nseg; pa.seg_count = c.seg_count; pa.ub = ba.ub; pa.lb = ba.lb;
    pa.B0 = ba.B0; pa.S0 = ba.S0; pa.score = c.score; pa.count = c.count; pa.head = start; pa.limit = limit;
    pa.surv_list = W.surv_list.as<int>(); pa.surv_cnt = W.surv_cnt.as<int>();
    pa.n_survivors = ctx->waves ? nullptr : &sc->n_survivors;
    prune_kernel<<<cdiv((long long)P * 32, 256), 256, 0, st>>>(pa);
    LAUNCHED();
    ScoreArgs sv = chunk_score_args(ctx);
    sv.n_groups = P; sv.grp_stride = stride; sv.grp_per_pair = 1; sv.models = c.models; sv.score = c.score; sv.count = c.count;
    sv.item_prefix = W.surv_prefix.as<int>(); sv.n_items = &sc->n_surv_items;
    sv.slot_list = pa.surv_list; sv.list_stride = stride;
    WaveArgs wa;
    wa.n_pairs = P; wa.slots_pp = c.slots_pp; wa.surv_list = pa.surv_list; wa.surv_cnt = pa.surv_cnt;
    wa.cursor = W.wave_cursor.as<int>(); wa.wave_cnt = W.wave_cnt.as<int>(); wa.ub = ba.ub; wa.lb = ba.lb;
    wa.B = W.B0.as<int>(); wa.S = W.S0.as<double>(); wa.score = c.score; wa.count = c.count;
    wa.n_exact = &sc->n_survivors;
    return ctx->waves ? score_survivors_in_waves(ctx, c, sv, wa, limit != 0)
                      : score_survivors_at_once(ctx, c, sv, wa, limit != 0);
}

// 4. score the minimal models: all of them exactly (RP_NO_PRUNE=1), or the first c.head models of every pair exactly
// -> (B0, S0), then with the mid stage the models at positions [HEAD_SMALL, MID_END) of the pair's first segment
// through the same cascade as the bulk (one tensor-core pass, FP32 bound, prune, exact waves) against the short head's
// bar, which leaves (B0, S0) = the exact best of everything before MID_END for the bulk at a fraction of the cost of
// scoring a long head exactly; then the bulk.  ev[9] starts the bulk, ev[10] marks its bound kernel done, ev[11] its
// tensor-core tier.
int score_minimal(rp_ctx *ctx, const Chunk &c) {
    const int P = c.P;
    cudaStream_t st = c.st;
    Scalars *sc = c.sc;
    build_items_kernel<<<1, 1024, 0, st>>>(P * c.nseg, c.seg_count, c.item_prefix, &sc->n_items, &sc->n_hyp);
    LAUNCHED();
    ScoreArgs sa = chunk_score_args(ctx);
    sa.models = c.models; sa.score = c.score; sa.count = c.count; sa.point_scores = &sc->point_scores;
    if (!ctx->prune) {
        sa.n_groups = P * c.nseg; sa.grp_stride = 4 * SEG; sa.grp_per_pair = c.nseg; sa.grp_cnt = c.seg_count;
        sa.item_prefix = c.item_prefix; sa.n_items = &sc->n_items;
        return launch_score(ctx, c.pose, false, sa, st);
    }
    // 4a. the exact head
    const PruneBufs &W = ctx->prn;
    int *first_cnt = W.first_cnt.as<int>();
    first_count_kernel<<<cdiv(P, 256), 256, 0, st>>>(P, c.nseg, c.seg_count, first_cnt, c.head);
    LAUNCHED();
    build_items_kernel<<<1, 1024, 0, st>>>(P, first_cnt, W.first_prefix.as<int>(), &sc->n_first_items, nullptr);
    LAUNCHED();
    sa.n_groups = P; sa.grp_stride = (int)c.slots_pp; sa.grp_per_pair = 1; sa.grp_cnt = first_cnt;
    sa.item_prefix = W.first_prefix.as<int>(); sa.n_items = &sc->n_first_items;
    int rc = launch_score(ctx, c.pose, false, sa, st);
    if (rc) return rc;
    pair_bounds_kernel<<<cdiv((long long)P * 32, 256), 256, 0, st>>>(P, c.nseg, first_cnt, c.score, c.count,
                                                                   W.B0.as<int>(), W.S0.as<double>(), c.prior_cnt,
                                                                   c.prior_score);
    LAUNCHED();
    // 4b. the mid stage, 4c. the bulk
    if (c.mid && (rc = cascade(ctx, c, HEAD_SMALL, MID_END, false, nullptr, nullptr))) return rc;
    CK(cudaEventRecord(ctx->ev[9], st));
    return cascade(ctx, c, c.mid ? MID_END : c.head, 0, ctx->tc_two_pass, c.use_tc ? ctx->ev[11] : nullptr, ctx->ev[10]);
}

// 5. scan for the trigger events, and the LO problem list
int scan_stage(rp_ctx *ctx, const Chunk &c) {
    const LoBufs &L = ctx->lo;
    ScanArgs a;
    a.n_pairs = c.P; a.nseg = c.nseg; a.seg_count = c.seg_count; a.score = c.score; a.count = c.count;
    a.events = L.events.as<int>(); a.n_events = L.n_events.as<int>(); a.ev_cap = c.ev_cap;
    a.pair_flags = L.pair_flags.as<int>(); a.any_flag = &c.sc->any_flag;
    a.prior_cnt = c.prior_cnt; a.prior_score = c.prior_score;
    scan_kernel<<<cdiv((long long)c.P * 32, 256), 256, 0, c.st>>>(a);
    LAUNCHED();
    LoPrepArgs l;
    l.n_pairs = c.P; l.nseg = c.nseg; l.events = a.events; l.n_events = a.n_events; l.hyp_iter = c.hyp_iter; l.ev_cap = c.ev_cap;
    l.models = c.models; l.lo_models = L.lo_models.as<Model>(); l.lo_of_event = L.lo_of_event.as<int>();
    l.lo_count = L.lo_count.as<int>(); l.prob_list = L.prob_list.as<int>(); l.n_prob = &c.sc->n_prob; l.prior = c.prior;
    lo_prepare_kernel<<<cdiv(c.P, 128), 128, 0, c.st>>>(l);
    LAUNCHED();
    return RP_OK;
}

// The LM settings of the LO refinements (the trigger LOs and the final LO)
LMArgs lo_lm_args(const Chunk &c) {
    LMArgs la;
    memset(&la, 0, sizeof la);
    la.pairs = c.pairs; la.pts64 = c.pts64; la.d1 = c.io->d1; la.d2 = c.io->d2;
    la.weight_sampson = c.opt->weight_sampson; la.gradient_tol = 1e-10; la.step_tol = 1e-8;
    la.initial_lambda = 1e-3; la.min_lambda = 1e-10; la.max_lambda = 1e10;
    la.loss_scale_override = -1.0; la.scale_reproj_override = -1.0;
    la.lm_iters = &c.sc->lm_iters;
    la.lm_flops = &c.sc->lm_flops;
    return la;
}

// 6. LO refinement of every trigger (independent problems)
int lo_stage(rp_ctx *ctx, const Chunk &c) {
    LMArgs la = lo_lm_args(c);
    la.prob_list = ctx->lo.prob_list.as<int>(); la.n_prob = &c.sc->n_prob; la.prob_per_pair = c.ev_cap;
    la.models = ctx->lo.lo_models.as<Model>();
    return launch_lm(ctx, c.variant, la, c.st);
}

// 7. score the LO results and merge them into the pair's record; the final LO from the best model, its rescore
// (accepted when strictly better); get_inliers of the RANSAC model (the mask the reference returns in `info`)
int merge_stage(rp_ctx *ctx, const Chunk &c) {
    const int P = c.P;
    cudaStream_t st = c.st;
    Scalars *sc = c.sc;
    const LoBufs &L = ctx->lo;
    const ResultBufs &R = ctx->res;
    build_items_kernel<<<1, 1024, 0, st>>>(P, L.lo_count.as<int>(), L.lo_item_prefix.as<int>(), &sc->n_lo_items, nullptr);
    LAUNCHED();
    ScoreArgs s = chunk_score_args(ctx);
    s.n_groups = P; s.grp_stride = c.ev_cap; s.grp_per_pair = 1; s.grp_cnt = L.lo_count.as<int>();
    s.item_prefix = L.lo_item_prefix.as<int>(); s.n_items = &sc->n_lo_items; s.models = L.lo_models.as<Model>();
    s.score = L.lo_score.as<double>(); s.count = L.lo_cnt.as<int>();
    int rc = launch_score(ctx, c.pose, false, s, st);
    if (rc) return rc;
    const rp_options &opt = *c.opt;
    MergeArgs m;
    m.n_pairs = P; m.nseg = c.nseg; m.iters = c.iters; m.pairs = c.pairs; m.events = L.events.as<int>();
    m.min_iterations = opt.min_iterations; m.max_iterations = opt.max_iterations;
    m.dyn_num_trials_mult = opt.dyn_num_trials_mult; m.log_prob_missing = log(1.0 - opt.success_prob);
    m.hyp_iter = c.hyp_iter; m.ev_cap = c.ev_cap; m.pair_flags = L.pair_flags.as<int>(); m.any_flag = &sc->any_flag;
    m.n_events = L.n_events.as<int>(); m.lo_of_event = L.lo_of_event.as<int>(); m.score = c.score; m.count = c.count;
    m.models = c.models; m.lo_score = L.lo_score.as<double>(); m.lo_count_inl = L.lo_cnt.as<int>();
    m.lo_models = L.lo_models.as<Model>(); m.lo_count = L.lo_count.as<int>();
    m.best = R.best.as<Model>(); m.stats = R.stats.as<rp_stats>(); m.final_start = R.final_start.as<Model>();
    m.prior = c.prior; m.prior_score = c.prior_score; m.prior_cnt = c.prior_cnt;
    merge_kernel<<<cdiv(P, 128), 128, 0, st>>>(m);
    LAUNCHED();
    // final LO from the best model, rescore, accept when strictly better
    LMArgs la = lo_lm_args(c);
    la.prob_list = nullptr; la.n_prob = &sc->n_pairs_scalar; la.prob_per_pair = 1;
    la.models = R.final_start.as<Model>();
    if ((rc = launch_lm(ctx, c.variant, la, st))) return rc;
    if ((rc = launch_pair_items(ctx, P, st))) return rc;
    if ((rc = launch_score(ctx, c.pose, false, pair_score_args(ctx, P, R.final_start.as<Model>(), nullptr), st))) return rc;
    Merge2Args m2;
    m2.n_pairs = P; m2.pairs = c.pairs; m2.refined = R.final_start.as<Model>(); m2.ref_score = R.final_score.as<double>();
    m2.ref_count = R.final_count.as<int>(); m2.best = R.best.as<Model>(); m2.stats = R.stats.as<rp_stats>();
    merge2_kernel<<<cdiv(P, 128), 128, 0, st>>>(m2);
    LAUNCHED();
    return launch_get_inliers(ctx, c.pose, *c.io, R.best.as<Model>(), c.io->masks_out, st);
}

// 8. final refinement on the inliers with the user's bundle options (if num_inliers > 3); the chunk's models and stats out
int final_stage(rp_ctx *ctx, const Chunk &c) {
    const ResultBufs &R = ctx->res;
    enable_final_kernel<<<cdiv(c.P, 256), 256, 0, c.st>>>(c.P, R.stats.as<rp_stats>(), R.enable.as<int>());
    LAUNCHED();
    LMArgs lf = final_lm_args(ctx, *c.opt, *c.io, R.best.as<Model>(), c.io->masks_out, R.enable.as<int>());
    lf.lm_iters = &c.sc->lm_iters;
    lf.lm_flops = &c.sc->lm_flops;
    int rc = launch_lm(ctx, c.variant, lf, c.st);
    if (rc) return rc;
    finalize_kernel<<<cdiv(c.P, 256), 256, 0, c.st>>>(c.P, c.variant, c.pairs, R.best.as<Model>());
    LAUNCHED();
    CK(cudaMemcpyAsync(c.io->models_out, R.best.p, sizeof(Model) * c.P, cudaMemcpyDeviceToDevice, c.st));
    CK(cudaMemcpyAsync(c.io->stats_out, R.stats.p, sizeof(rp_stats) * c.P, cudaMemcpyDeviceToDevice, c.st));
    return RP_OK;
}

// Waits for the chunk's kernels, adds its stage times (rp_last_timing) and counters, and returns its pairs' flags
int read_back(rp_ctx *ctx, const Chunk &c, std::vector<int> &flags) {
    cudaEvent_t *ev = ctx->ev;
    Scalars h_sc;
    CK(cudaMemcpyAsync(&h_sc, c.sc, sizeof h_sc, cudaMemcpyDeviceToHost, c.st));
    CK(cudaStreamSynchronize(c.st));
    const bool pri = c.prior != nullptr;
    for (int i = 0; i < 8; ++i) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ev[i], i == 0 && pri ? ev[14] : ev[i + 1]));
        ctx->last_ms[i] += ms;
    }
    if (pri) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ev[14], ev[1]));
        ctx->last_ms[15] += ms;
    }
    {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ev[0], ev[8]));
        ctx->last_ms[8] += ms;
    }
    ctx->last_cnt[0] += h_sc.n_hyp;
    ctx->last_cnt[1] += (int64_t)h_sc.point_scores;
    ctx->last_cnt[2] += h_sc.n_prob + c.P;
    ctx->last_cnt[3] += (int64_t)h_sc.lm_iters;
    ctx->last_cnt[4] += 1;
    ctx->last_cnt[6] += (int64_t)h_sc.evaluated_ps;
    if (ctx->prune) {
        float msb = 0.f;
        CK(cudaEventElapsedTime(&msb, c.use_tc ? ev[11] : ev[9], ev[10]));
        ctx->last_ms[11] += msb;
        if (c.use_tc) {
            CK(cudaEventElapsedTime(&msb, ev[9], ev[11]));
            ctx->last_ms[12] += msb;
        }
    }
    ctx->last_cnt[8] += (int64_t)h_sc.tc_evaluated;
    ctx->last_cnt[9] += (int64_t)h_sc.tc_selected;
    ctx->last_cnt[10] += (int64_t)h_sc.lm_flops;
    // models through the exact kernel: the survivors and the exact head
    ctx->last_cnt[5] += ctx->prune ? (int64_t)h_sc.n_survivors + std::min<int64_t>(h_sc.n_hyp, (int64_t)c.P * c.head) : h_sc.n_hyp;
    ctx->last_cnt[7] = HB;
    flags.assign((size_t)c.P, 0);
    if (h_sc.any_flag) {
        CK(cudaMemcpyAsync(flags.data(), ctx->lo.pair_flags.p, sizeof(int) * (size_t)c.P, cudaMemcpyDeviceToHost, c.st));
        CK(cudaStreamSynchronize(c.st));
    }
    return RP_OK;
}

// One pass over a chunk.  `flags` (host, [n_pairs]) receives PAIR_FLAG_* per pair: a flagged pair's outputs are void and
// the caller runs it again with a larger `ev_cap` / more iterations (estimate_impl).
int run_chunk(rp_ctx *ctx, int variant, const rp_options &opt, const ChunkIO &io, int iters, int ev_cap,
              std::vector<int> &flags, cudaStream_t st) {
    const int P = io.n_pairs;
    const int nseg = std::max(1, cdiv(iters, SEG));
    CK(ctx->hyp.reserve(P, iters, nseg));
    CK(ctx->lo.reserve(P, ev_cap));
    CK(ctx->res.reserve(P, true));
    if (ctx->prune) CK(ctx->prn.reserve(P, nseg));
    if (ctx->prune && ctx->tc) CK(ctx->tcb.reserve(P, io.n_points, nseg));
    if (io.init) CK(ctx->pri.reserve(P));
    cudaEvent_t *ev = ctx->ev;
    // 1. prepare, and the tensor-core tier's feature rows
    int rc = prepare_chunk(ctx, variant, opt, io, ev[0], st);
    if (rc) return rc;
    const Chunk c = chunk_of(ctx, variant, opt, io, iters, ev_cap, st);
    if (c.use_tc && c.N > 0) {
        tc::tc_features_kernel<<<cdiv(c.N, 256), 256, 0, st>>>(c.N, c.pts32, ctx->tcb.feat.as<float4>());
        LAUNCHED();
    }
    if (c.prior) {
        CK(cudaEventRecord(ev[14], st));
        if ((rc = prior_stage(ctx, c))) return rc;
    }
    CK(cudaEventRecord(ev[1], st));
    if ((rc = sample_stage(ctx, c))) return rc;
    CK(cudaEventRecord(ev[2], st));
    if ((rc = solve_stage(ctx, c))) return rc;
    CK(cudaEventRecord(ev[3], st));
    if ((rc = score_minimal(ctx, c))) return rc;
    CK(cudaEventRecord(ev[4], st));
    if ((rc = scan_stage(ctx, c))) return rc;
    CK(cudaEventRecord(ev[5], st));
    if ((rc = lo_stage(ctx, c))) return rc;
    CK(cudaEventRecord(ev[6], st));
    if ((rc = merge_stage(ctx, c))) return rc;
    CK(cudaEventRecord(ev[7], st));
    if ((rc = final_stage(ctx, c))) return rc;
    CK(cudaEventRecord(ev[8], st));
    return read_back(ctx, c, flags);
}

// widens a float32 chunk into the FP64 input arrays (no-op for an empty chunk); with `perm` (quality calls, float or
// double inputs) it gathers the chunk into its quality order in the same pass (pairs: [offsets[p] - base, ...))
template <class In>
int launch_widen(rp_ctx *ctx, long long n, const In *x1, const In *x2, const In *d1, const In *d2, double *wx1,
                 double *wx2, double *wd1, double *wd2, cudaStream_t st, const int *perm = nullptr,
                 const long long *offsets = nullptr, long long base = 0, int n_pairs = 0) {
    if (n <= 0) return RP_OK;
    const int grid = std::min<long long>(cdiv(perm ? n : 2 * n, 256), 16LL * ctx->sms);
    widen_inputs_kernel<In><<<grid, 256, 0, st>>>(n, x1, x2, d1, d2, perm, offsets, base, n_pairs, wx1, wx2, wd1, wd2);
    LAUNCHED();
    return RP_OK;
}

// quality order of the P pairs of a chunk of n correspondences: `h_offsets` (host) and `d_offsets` (device) are the
// same P+1 offsets, pair p owning [offsets[p] - base, offsets[p+1] - base) of `quality` and `perm` (no-op for n = 0).
// The dynamic shared memory is sized to the largest pair up to RP_ORDER_SMEM_CAP; larger pairs use the global sort scratch.
int launch_order(rp_ctx *ctx, int P, long long n, const int64_t *h_offsets, const long long *d_offsets, long long base,
                 const float *quality, int *perm, cudaStream_t st) {
    if (n <= 0) return RP_OK;
    long long max_n = 0;
    for (int p = 0; p < P; ++p) max_n = std::max<long long>(max_n, h_offsets[p + 1] - h_offsets[p]);
    OrderArgs a;
    a.offsets = d_offsets; a.base = base; a.quality = quality; a.perm = perm;
    a.smem_cap = (int)std::min<long long>(max_n, ORDER_SMEM_CAP);
    a.gkeys = nullptr; a.gidx = nullptr;
    if (max_n > ORDER_SMEM_CAP) {
        CK(ctx->scratch.order.reserve(12 * (size_t)n));
        a.gkeys = ctx->scratch.order.as<unsigned>();
        a.gidx = (int *)(a.gkeys + 2 * n);
    }
    order_by_quality_kernel<<<P, ORDER_THREADS, (size_t)ORDER_SMEM_PER_POINT * a.smem_cap, st>>>(a);
    LAUNCHED();
    return RP_OK;
}

// masks of a chunk in the ordered layout -> the caller's order (no-op for an empty chunk)
int launch_scatter_masks(rp_ctx *ctx, int P, long long n, const long long *d_offsets, long long base, const int *perm,
                         const unsigned char *sorted, unsigned char *out, cudaStream_t st) {
    if (n <= 0) return RP_OK;
    scatter_masks_kernel<<<(int)std::min<long long>(cdiv(n, 256), 16LL * ctx->sms), 256, 0, st>>>(n, P, d_offsets, base, perm,
                                                                                                  sorted, out);
    LAUNCHED();
    return RP_OK;
}

// Pairs of a chunk whose first pass was flagged — more trigger events than the list holds, or (early termination) more
// iterations needed than were generated — are gathered into compact sub-batches and run again on their own with the
// limits raised (iterations x4 up to max_iterations, event capacity x8), until no flag is left.  Everybody else's
// results are untouched; what a hard pair costs is bounded by ~1.33x what the reference spends on that pair.  A
// sub-batch that cannot be run (out of device memory) marks its pairs RP_PAIR_FAILED instead of failing the call.
int rerun_flagged(rp_ctx *ctx, int variant, const rp_options &opt, const ChunkIO &io, const long long *rel,
                  const std::vector<int> &flags0, int iters0, int64_t p0, cudaStream_t st) {
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    std::vector<int> todo;
    for (int i = 0; i < io.n_pairs; ++i)
        if (flags0[(size_t)i]) todo.push_back(i);
    int iters = iters0, ev_cap = ctx->ev_cap0;
    std::vector<int> flags_of((size_t)io.n_pairs, 0);
    for (int i : todo) flags_of[(size_t)i] = flags0[(size_t)i];
    while (!todo.empty()) {
        bool any_more = false, any_ovf = false;
        for (int i : todo) {
            any_more |= (flags_of[(size_t)i] & PAIR_FLAG_NEED_MORE) != 0;
            any_ovf |= (flags_of[(size_t)i] & PAIR_FLAG_OVERFLOW) != 0;
            ctx->pair_status[(size_t)(p0 + i)] |= ((flags_of[(size_t)i] & PAIR_FLAG_NEED_MORE) ? RP_PAIR_CONTINUED : 0) |
                                                  ((flags_of[(size_t)i] & PAIR_FLAG_OVERFLOW) ? RP_PAIR_EVENTS_RERUN : 0);
        }
        if (any_more) iters = (int)std::min<int64_t>(opt.max_iterations, (int64_t)iters * 4);
        const int slots_pp = std::max(1, cdiv(iters, SEG)) * 4 * SEG;
        if (any_ovf) ev_cap = (int)std::min<int64_t>((int64_t)ev_cap * 8, slots_pp);
        std::vector<int> next;
        size_t pos = 0;
        while (pos < todo.size()) {
            // sub-batch [pos, end): as many pairs as the workspace budget holds at these limits
            size_t end = pos;
            size_t bytes = 0;
            long long npts = 0;
            while (end < todo.size()) {
                const long long n = rel[(size_t)todo[end] + 1] - rel[(size_t)todo[end]];
                const size_t b = bytes_per_pair(iters, n, ev_cap, 0, io.init ? PRIOR_BYTES_PER_PAIR : 0);
                if (end > pos && bytes + b > ctx->workspace_budget) break;
                bytes += b;
                npts += n;
                ++end;
            }
            const int S = (int)(end - pos);
            std::vector<int> idx((size_t)S);
            std::vector<long long> src((size_t)S), dst((size_t)S + 1, 0);
            for (int j = 0; j < S; ++j) {
                idx[(size_t)j] = todo[pos + j];
                src[(size_t)j] = rel[(size_t)idx[(size_t)j]];
                dst[(size_t)j + 1] = dst[(size_t)j] + (rel[(size_t)idx[(size_t)j] + 1] - rel[(size_t)idx[(size_t)j]]);
            }
            const size_t nn = (size_t)std::max<long long>(npts, 1);
            int rc = RP_OK;
            std::vector<int> flags;
            do {  // single pass; `break` = this sub-batch failed
                SubBufs &B = ctx->sub;
                if (B.reserve(S, nn, io.init != nullptr)) {
                    rc = RP_ERR_CUDA;
                    break;
                }
                CK(cudaMemcpyAsync(B.idx.p, idx.data(), sizeof(int) * S, cudaMemcpyHostToDevice, st));
                CK(cudaMemcpyAsync(B.src.p, src.data(), 8 * (size_t)S, cudaMemcpyHostToDevice, st));
                CK(cudaMemcpyAsync(B.dst.p, dst.data(), 8 * ((size_t)S + 1), cudaMemcpyHostToDevice, st));
                SubBatchArgs g;
                g.n_sub = S; g.pair_idx = B.idx.as<int>(); g.src_off = B.src.as<long long>();
                g.dst_off = B.dst.as<long long>();
                g.x1 = io.x1; g.x2 = io.x2; g.d1 = io.d1; g.d2 = io.d2; g.cams = pose ? io.cams : nullptr;
                g.sx1 = B.x1.as<double>(); g.sx2 = B.x2.as<double>(); g.sd1 = B.d1.as<double>();
                g.sd2 = B.d2.as<double>(); g.scams = B.cams.as<double>();
                g.models = io.models_out; g.stats = io.stats_out; g.masks = io.masks_out;
                g.smodels = B.models.as<Model>(); g.sstats = B.stats.as<rp_stats>();
                g.smasks = B.mask.as<unsigned char>();
                g.init = io.init; g.sinit = io.init ? B.init.as<Model>() : nullptr;
                gather_pairs_kernel<<<S, 256, 0, st>>>(g);
                LAUNCHED();
                CK(cudaStreamSynchronize(st));  // idx / src / dst are stack-lifetime host buffers
                ChunkIO sub;
                sub.n_pairs = S; sub.n_points = npts; sub.h_offsets_rel = dst.data();
                sub.x1 = g.sx1; sub.x2 = g.sx2; sub.d1 = g.sd1; sub.d2 = g.sd2; sub.cams = pose ? g.scams : nullptr;
                sub.models_out = B.models.as<Model>(); sub.stats_out = B.stats.as<rp_stats>();
                sub.masks_out = B.mask.as<unsigned char>();
                sub.init = g.sinit;
                rc = run_chunk(ctx, variant, opt, sub, iters, ev_cap, flags, st);
                if (rc) break;
                scatter_pairs_kernel<<<S, 256, 0, st>>>(g);
                LAUNCHED();
                CK(cudaStreamSynchronize(st));
            } while (false);
            if (rc) {
                // isolate the failure: these pairs keep their (void) first-pass outputs and are reported; a failed
                // allocation leaves the CUDA context usable
                (void)cudaGetLastError();
                for (int j = 0; j < S; ++j) ctx->pair_status[(size_t)(p0 + idx[(size_t)j])] = RP_PAIR_FAILED;
            } else {
                for (int j = 0; j < S; ++j) {
                    int f = flags[(size_t)j];
                    if (iters >= opt.max_iterations) f &= ~PAIR_FLAG_NEED_MORE;  // cannot happen: the merge stops at max_iterations
                    flags_of[(size_t)idx[(size_t)j]] = f;
                    if (f) next.push_back(idx[(size_t)j]);
                }
            }
            pos = end;
        }
        todo.swap(next);
    }
    return RP_OK;
}

// Checks and set-up shared by estimate_impl and refine_impl (RP_CALIB with estimate_shift runs as RP_CALIB_SHIFT)
int begin_batch(rp_ctx *ctx, int &variant, int64_t n_pairs, const int64_t *offsets, const double *cams,
                const rp_options *opt_in, rp_options &opt) {
    if (!ctx) return RP_ERR_INVALID;
    if (variant < 0 || variant > 3) return fail(ctx, RP_ERR_INVALID, "unknown variant");
    if (n_pairs < 0 || !offsets || !opt_in) return fail(ctx, RP_ERR_INVALID, "null or negative argument");
    if (opt_in->max_iterations < 0 || opt_in->max_iterations > (1 << 24))
        return fail(ctx, RP_ERR_INVALID, "max_iterations out of range");
    for (int64_t p = 0; p < n_pairs; ++p)
        if (offsets[p + 1] < offsets[p] || offsets[p + 1] - offsets[p] >= (1 << 24))
            return fail(ctx, RP_ERR_INVALID, "offsets must be non-decreasing, at most 2^24-1 correspondences per pair");
    CK(cudaSetDevice(ctx->device));
    opt = *opt_in;
    if (variant == RP_CALIB && opt.estimate_shift) variant = RP_CALIB_SHIFT;
    if (variant == RP_CALIB_SHIFT) opt.estimate_shift = 1;
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    if (pose && !cams && n_pairs > 0) return fail(ctx, RP_ERR_INVALID, "calibrated variants need cams");
    return RP_OK;
}

// Chunk boundaries of a batch: at most as many pairs per chunk as the workspace budget holds at `bpp` bytes per pair
// (and 32 768), the remainder split evenly (no tiny last chunk).  On the host path, batches of 1024 pairs or more are
// split so that uploads hide behind kernels, by one of two policies:
//   lead = true (the estimator): a small first chunk goes ahead so that the kernels start early and every later upload
//     hides behind the previous chunk's kernels.  With U = upload time (+ widening or ordering) and C = kernel time of
//     the whole batch, the exposed time f U + max(0, (1-f) U - f C) is smallest at f = U / (U + C); U / C is taken
//     from the previous host call on this context (1/8 of the batch before there is one).
//   lead = false (the refinement): at least four chunks, so that three uploads hide behind kernels.
// Only timing depends on the boundaries, never results.
std::vector<int64_t> plan_chunks(const rp_ctx *ctx, int64_t n_pairs, size_t bpp, bool host_io, bool lead) {
    int64_t chunk = (int64_t)std::max<size_t>(1, ctx->workspace_budget / bpp);
    chunk = std::min<int64_t>(chunk, 32768);
    int64_t first = 0;
    if (host_io && n_pairs >= 1024) {
        if (!lead) {
            chunk = std::min<int64_t>(chunk, (n_pairs + 3) / 4);
        } else {
            double f = 0.125;
            if (ctx->prev_h2d_ms > 0.0 && ctx->prev_dev_ms > 0.0) f = ctx->prev_h2d_ms / (ctx->prev_h2d_ms + ctx->prev_dev_ms);
            f = std::min(1.0 / 3.0, std::max(1.0 / 32.0, f));
            first = std::min<int64_t>(std::min<int64_t>(n_pairs, chunk), std::max<int64_t>(256, (int64_t)(f * (double)n_pairs)));
        }
    }
    std::vector<int64_t> bounds(1, 0);
    if (first > 0) bounds.push_back(first);
    const int64_t rest = n_pairs - first;
    const int64_t k = (rest + chunk - 1) / chunk;
    for (int64_t i = 1; i <= k; ++i) bounds.push_back(first + (rest * i) / k);
    return bounds;
}

// A batch's inputs as the caller passed them: host memory on the host path, device memory on the device path (offsets
// are host memory either way)
template <class In>
struct BatchIn {
    const int64_t *offsets;
    const In *x1, *x2, *d1, *d2;
    const double *cams;       // null for the focal variants
    const float *quality;     // quality calls: each chunk is ordered pair by pair
    const rp_model *init;     // refinement: start models, subset (null: every correspondence)
    const uint8_t *subset;
    bool host_io;
};

// Where the kernels write one output of a chunk, `n` elements from element `at` of the batch: the caller's array on the
// device path, set buffer `staging` on the host path (read back by the download of run_chunks), null when the caller
// did not ask for the output
template <class T>
cudaError_t chunk_out(bool host_io, DevBuf &staging, T *caller, int64_t at, size_t n, T *&out) {
    out = caller && !host_io ? caller + at : nullptr;
    if (!caller || !host_io) return cudaSuccess;
    const cudaError_t e = staging.reserve(sizeof(T) * n);
    out = staging.as<T>();
    return e;
}

// Puts the inputs of the pairs [p0, p1) where the kernels read them and points io's inputs there.  The kernels read
// FP64; float32 inputs are widened first, and quality calls sort each pair (order_by_quality_kernel) and gather it in
// that order with the permuting widen_inputs_kernel.
//   Host path, on the copy stream into set s: the upload (into the input-type staging when the chunk is widened or
//   ordered), the widening or ordering, then s.in_ready.
//   Device path, on the compute stream `st`: FP64 inputs without quality are read where they are; otherwise they are
//   widened, or ordered, into set s.
// [s.h2d_begin, s.h2d_end) is the host path's upload (rp_last_timing [9]), [s.h2d_end, s.in_ready) the widening or
// ordering ([13] / [14]).
template <class In>
int stage_inputs(rp_ctx *ctx, const BatchIn<In> &b, int64_t p0, int64_t p1, StageSet &s, cudaStream_t st, ChunkIO &io) {
    constexpr bool f32 = std::is_same<In, float>::value;
    const bool ordered = b.quality != nullptr, widen = f32 || ordered;
    const int P = (int)(p1 - p0);
    const long long o0 = b.offsets[p0], N = b.offsets[p1] - o0;
    const size_t nn = (size_t)std::max<long long>(N, 1);
    // what the kernels or the widening read: the caller's arrays, or on the host path their upload
    const In *x1 = b.x1 + 2 * o0, *x2 = b.x2 + 2 * o0, *d1 = b.d1 + o0, *d2 = b.d2 + o0;
    const float *quality = ordered ? b.quality + o0 : nullptr;
    io.cams = b.cams ? b.cams + 8 * p0 : nullptr;
    io.init = b.init ? (const Model *)b.init + p0 : nullptr;
    io.subset = b.subset ? b.subset + o0 : nullptr;
    if (!b.host_io && !widen) {
        // (In = double here: float32 inputs are always widened)
        io.x1 = (const double *)x1; io.x2 = (const double *)x2; io.d1 = (const double *)d1; io.d2 = (const double *)d2;
        return RP_OK;
    }
    const cudaStream_t ws = b.host_io ? ctx->copy_stream : st;
    CK(s.x1.reserve(16 * nn)); CK(s.x2.reserve(16 * nn));
    CK(s.d1.reserve(8 * nn)); CK(s.d2.reserve(8 * nn));
    if (ordered) {
        CK(s.perm.reserve(4 * nn)); CK(s.ksort.reserve(nn)); CK(s.offs.reserve(8 * ((size_t)P + 1)));
    }
    if (b.host_io) {
        constexpr size_t E = sizeof(In);
        DevBuf &ux1 = widen ? s.sx1 : s.x1, &ux2 = widen ? s.sx2 : s.x2, &ud1 = widen ? s.sd1 : s.d1,
               &ud2 = widen ? s.sd2 : s.d2;
        CK(ux1.reserve(2 * E * nn)); CK(ux2.reserve(2 * E * nn));
        CK(ud1.reserve(E * nn)); CK(ud2.reserve(E * nn));
        CK(s.cams.reserve(64 * (size_t)P));
        CK(cudaEventRecord(s.h2d_begin, ws));
        CK(cudaMemcpyAsync(ux1.p, x1, 2 * E * (size_t)N, cudaMemcpyHostToDevice, ws));
        CK(cudaMemcpyAsync(ux2.p, x2, 2 * E * (size_t)N, cudaMemcpyHostToDevice, ws));
        CK(cudaMemcpyAsync(ud1.p, d1, E * (size_t)N, cudaMemcpyHostToDevice, ws));
        CK(cudaMemcpyAsync(ud2.p, d2, E * (size_t)N, cudaMemcpyHostToDevice, ws));
        if (io.cams) {
            CK(cudaMemcpyAsync(s.cams.p, io.cams, 64 * (size_t)P, cudaMemcpyHostToDevice, ws));
            io.cams = s.cams.as<double>();
        }
        if (ordered) {
            CK(s.qual.reserve(4 * nn));
            CK(cudaMemcpyAsync(s.qual.p, quality, 4 * (size_t)N, cudaMemcpyHostToDevice, ws));
            CK(cudaMemcpyAsync(s.offs.p, b.offsets + p0, 8 * ((size_t)P + 1), cudaMemcpyHostToDevice, ws));
            quality = s.qual.as<float>();
        }
        if (io.init) {
            CK(s.init.reserve(sizeof(Model) * P));
            CK(cudaMemcpyAsync(s.init.p, io.init, sizeof(Model) * P, cudaMemcpyHostToDevice, ws));
            io.init = s.init.as<Model>();
        }
        if (io.subset) {
            CK(s.subset.reserve(nn));
            CK(cudaMemcpyAsync(s.subset.p, io.subset, (size_t)N, cudaMemcpyHostToDevice, ws));
            io.subset = s.subset.as<unsigned char>();
        }
        x1 = ux1.as<In>(); x2 = ux2.as<In>(); d1 = ud1.as<In>(); d2 = ud2.as<In>();
    }
    CK(cudaEventRecord(s.h2d_end, ws));
    if (ordered) {
        if (!b.host_io) CK(cudaMemcpyAsync(s.offs.p, b.offsets + p0, 8 * ((size_t)P + 1), cudaMemcpyHostToDevice, ws));
        int rc = launch_order(ctx, P, N, b.offsets + p0, s.offs.as<long long>(), o0, quality, s.perm.as<int>(), ws);
        if (rc) return rc;
    }
    if (widen) {
        int rc = launch_widen(ctx, N, x1, x2, d1, d2, s.x1.as<double>(), s.x2.as<double>(), s.d1.as<double>(),
                              s.d2.as<double>(), ws, ordered ? s.perm.as<int>() : nullptr,
                              ordered ? s.offs.as<long long>() : nullptr, o0, P);
        if (rc) return rc;
    }
    CK(cudaEventRecord(s.in_ready, ws));
    io.x1 = s.x1.as<double>(); io.x2 = s.x2.as<double>(); io.d1 = s.d1.as<double>(); io.d2 = s.d2.as<double>();
    return RP_OK;
}

// The chunk pipeline of estimate_impl and refine_impl.  For each chunk c, in this order:
//   host path: make the compute stream wait for chunk c's in_ready; device path: stage_inputs of chunk c on the
//     compute stream;
//   work(c, set, io) enqueues chunk c's kernels on the compute stream;
//   host path: record set.done on the compute stream, make the copy stream wait for it, and download(c, io, copy
//     stream) reads chunk c's outputs back between set.d2h_begin and set.d2h_end.
// On the host path the upload of chunk c+1 into the other staging set (stage_inputs on the copy stream) is enqueued
// next to chunk c's work, so that it overlaps chunk c's kernels, and chunk c's read-back overlaps chunk c+1's kernels.
// Where depends on what may block the host: with `work_waits` the work returns only after chunk c's kernels have
// finished (run_chunk synchronises), so the upload goes before it; otherwise it goes after the work, because an upload
// from pageable host memory waits for the copy stream, and chunk c's kernels must already be enqueued by then.  Either
// way the copy stream runs upload c+1 before read-back c.  The rule that makes this safe: the copy stream must not
// write a set before the kernels that last read it have finished.  Chunk c+2's upload into set c & 1 follows chunk c's
// read-back on the copy stream, which waits for chunk c's `done` event.  At the end the host synchronises the copy
// stream (host path) or the compute stream (device path).
template <class In, class Work, class Download>
int run_chunks(rp_ctx *ctx, const BatchIn<In> &b, const std::vector<int64_t> &bounds, cudaStream_t st, bool work_waits,
               Work work, Download download) {
    cudaStream_t cs = ctx->copy_stream;
    const int64_t n_chunks = (int64_t)bounds.size() - 1;
    ChunkIO io[2];
    std::vector<long long> rel;
    int rc = b.host_io ? stage_inputs(ctx, b, bounds[0], bounds[1], ctx->set[0], st, io[0]) : RP_OK;
    if (rc) return rc;
    for (int64_t c = 0; c < n_chunks; ++c) {
        StageSet &s = ctx->set[b.host_io ? c & 1 : 0];
        ChunkIO &cur = io[c & 1];
        auto upload_next = [&]() {
            return b.host_io && c + 1 < n_chunks
                       ? stage_inputs(ctx, b, bounds[c + 1], bounds[c + 2], ctx->set[(c + 1) & 1], st, io[(c + 1) & 1])
                       : RP_OK;
        };
        if (work_waits && (rc = upload_next())) return rc;
        if (b.host_io) {
            CK(cudaStreamWaitEvent(st, s.in_ready, 0));
        } else {
            rc = stage_inputs(ctx, b, bounds[c], bounds[c + 1], s, st, cur);
            if (rc) return rc;
        }
        const int64_t p0 = bounds[c];
        cur.n_pairs = (int)(bounds[c + 1] - p0);
        cur.n_points = b.offsets[bounds[c + 1]] - b.offsets[p0];
        rel.resize((size_t)cur.n_pairs + 1);
        for (int i = 0; i <= cur.n_pairs; ++i) rel[(size_t)i] = b.offsets[p0 + i] - b.offsets[p0];
        cur.h_offsets_rel = rel.data();
        rc = work(c, s, cur);
        if (rc) return rc;
        if (!work_waits && (rc = upload_next())) return rc;
        if (b.host_io) {
            CK(cudaEventRecord(s.done, st));
            CK(cudaStreamWaitEvent(cs, s.done, 0));
            CK(cudaEventRecord(s.d2h_begin, cs));
            rc = download(c, cur, cs);
            if (rc) return rc;
            CK(cudaEventRecord(s.d2h_end, cs));
        }
    }
    CK(cudaStreamSynchronize(b.host_io ? cs : st));
    return RP_OK;
}

// rp_estimate_batch_*: run_chunks with run_chunk and rerun_flagged as the work of a chunk.  In = double: the FP64 entry
// points; In = float: the _f32 ones (24 B per correspondence uploaded instead of 48, then widened); quality != null: the
// _quality ones, whose chunks run_chunk and rerun_flagged see in the quality order and whose masks they write in that
// order, which scatter_masks_kernel writes back in the caller's order.  Either way every kernel after stage_inputs
// reads the same FP64 chunk arrays as the FP64 entry points.  init != null: the _init ones, one prior per pair (host
// memory on the host path, uploaded with the chunk's inputs; device memory on the device path).
template <class In>
int estimate_impl(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const In *x1,
                  const In *x2, const In *d1, const In *d2, const float *quality, const double *cams,
                  const rp_options *opt_in, const rp_model *init, rp_model *models, rp_stats *stats, uint8_t *masks,
                  bool host_io, cudaStream_t st) {
    constexpr bool f32 = std::is_same<In, float>::value;
    const bool ordered = quality != nullptr;
    const bool staged = f32 || ordered;   // the chunk is widened or ordered before its kernels
    rp_options opt;
    int rc = begin_batch(ctx, variant, n_pairs, offsets, cams, opt_in, opt);
    if (rc) return rc;
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    memset(ctx->last_ms, 0, sizeof ctx->last_ms);
    memset(ctx->last_cnt, 0, sizeof ctx->last_cnt);
    ctx->pair_status.assign((size_t)n_pairs, RP_PAIR_OK);
    if (n_pairs == 0) return RP_OK;
    const long long Ntot = offsets[n_pairs] - offsets[0];
    // Early termination (min_iterations < max_iterations): the reference stops at the first it > min_iterations with
    // it > dynamic_max_iter.  The first pass generates min_iterations + 1 iterations for every pair and the merge
    // kernel replays the stop rule exactly; only the pairs that would have kept going are run again, on their own,
    // with 4x more iterations (same seed => same prefix), see rerun_flagged above.
    const int iters0 = opt.min_iterations < opt.max_iterations
                           ? (int)std::min<int64_t>(opt.max_iterations, opt.min_iterations + 1)
                           : (int)opt.max_iterations;
    // float32 inputs: two 24-byte staging sets (host path) or the 48-byte widened copy (device path) per correspondence.
    // Quality calls: two staging sets of the inputs, quality, order and ordered-layout mask (host path), or the 48-byte
    // gathered copy, the order and the ordered-layout mask (device path).
    size_t in_bytes = f32 ? 48 : 0;
    if (ordered) in_bytes = host_io ? 2 * (6 * sizeof(In) + 4 + 4 + 1) : 48 + 4 + 1;
    const std::vector<int64_t> bounds = plan_chunks(
        ctx, n_pairs, bytes_per_pair(iters0, Ntot / n_pairs + 1, ctx->ev_cap0, in_bytes, init ? PRIOR_BYTES_PER_PAIR : 0),
        host_io, true);
    const BatchIn<In> b = {offsets, x1, x2, d1, d2, pose ? cams : nullptr, quality, init, nullptr, host_io};
    double stage_per_point0 = 0.0;  // host path: widening / ordering time of chunk 0 per correspondence (ms)
    auto work = [&](int64_t c, StageSet &s, ChunkIO &io) -> int {
        const int64_t p0 = bounds[c];
        const int P = io.n_pairs;
        const long long o0 = offsets[p0], N = io.n_points;
        CK(chunk_out(host_io, s.models, (Model *)models, p0, P, io.models_out));
        CK(chunk_out(host_io, s.stats, stats, p0, P, io.stats_out));
        CK(chunk_out(host_io, s.mask, masks, o0, (size_t)std::max<long long>(N, 1), io.masks_out));
        // quality calls: where the masks go in the caller's order
        unsigned char *masks_caller = io.masks_out;
        if (ordered) io.masks_out = s.ksort.as<unsigned char>();
        std::vector<int> flags;
        int rc2 = run_chunk(ctx, variant, opt, io, iters0, ctx->ev_cap0, flags, st);
        if (rc2) return rc2;
        const long long *rel = io.h_offsets_rel;
        for (int i = 0; i < P; ++i) ctx->pair_status[(size_t)(p0 + i)] = rel[i + 1] - rel[i] < 3 ? RP_PAIR_DEGENERATE : RP_PAIR_OK;
        rc2 = rerun_flagged(ctx, variant, opt, io, rel, flags, iters0, p0, st);
        if (rc2) return rc2;
        float ms = 0.f;
        if (ordered) {
            // the re-runs wrote into the ordered-layout masks too: now they go back to the caller's order.  The host
            // waits for this one small kernel so that its time can be read.
            cudaEvent_t scatter_begin = ctx->ev[12], scatter_end = ctx->ev[13];
            CK(cudaEventRecord(scatter_begin, st));
            rc2 = launch_scatter_masks(ctx, P, N, s.offs.as<long long>(), o0, s.perm.as<int>(), io.masks_out, masks_caller, st);
            if (rc2) return rc2;
            CK(cudaEventRecord(scatter_end, st));
            CK(cudaEventSynchronize(scatter_end));
            if (cudaEventElapsedTime(&ms, scatter_begin, scatter_end) == cudaSuccess) ctx->last_ms[14] += ms;
            io.masks_out = masks_caller;
        }
        // (run_chunk returned after synchronising the compute stream, which waited for s.in_ready)
        if (host_io && cudaEventElapsedTime(&ms, s.h2d_begin, s.h2d_end) == cudaSuccess) ctx->last_ms[9] += ms;
        if (staged && cudaEventElapsedTime(&ms, s.h2d_end, s.in_ready) == cudaSuccess) {
            // on the host path the widening / ordering of chunks c >= 1 runs while chunk c-1's kernels hold the SMs, so
            // its interval includes waiting for them; chunk 0's is that work alone (nothing of this call runs yet) and
            // sizes the next lead chunk
            ctx->last_ms[ordered ? 14 : 13] += ms;
            if (c == 0 && N > 0) stage_per_point0 = ms / (double)N;
        }
        return RP_OK;
    };
    auto download = [&](int64_t c, const ChunkIO &io, cudaStream_t cs) -> int {
        const int64_t p0 = bounds[c];
        CK(cudaMemcpyAsync(models + p0, io.models_out, sizeof(Model) * io.n_pairs, cudaMemcpyDeviceToHost, cs));
        CK(cudaMemcpyAsync(stats + p0, io.stats_out, sizeof(rp_stats) * io.n_pairs, cudaMemcpyDeviceToHost, cs));
        if (io.n_points > 0) CK(cudaMemcpyAsync(masks + offsets[p0], io.masks_out, (size_t)io.n_points, cudaMemcpyDeviceToHost, cs));
        return RP_OK;
    };
    rc = run_chunks(ctx, b, bounds, st, true, work, download);
    if (rc) return rc;
    if (host_io) {
        ctx->prev_h2d_ms = ctx->last_ms[9] + stage_per_point0 * (double)Ntot;   // + widening / ordering of the batch, 0 with FP64 inputs
        ctx->prev_dev_ms = ctx->last_ms[8];
        for (int par = 0; par < 2 && par + 1 < (int)bounds.size(); ++par) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ctx->set[par].d2h_begin, ctx->set[par].d2h_end) == cudaSuccess) ctx->last_ms[10] += ms;
        }
    }
    for (int32_t v : ctx->pair_status)
        if (v < 0) return fail(ctx, RP_ERR_PARTIAL, "some pairs could not be finished (rp_pair_status); all other outputs are valid");
    return RP_OK;
}

// ---- rp_refine_pairs_*: the estimator's final refinement on caller-supplied start models --------------------------
// One chunk, everything on `st`, no synchronisation: prepare_chunk, refine_import_kernel, the final refinement
// (final_lm_args) on the work models, the one-item-per-pair list and get_inliers on the refined work models,
// refine_export_kernel (last, because it also turns get_inliers' counts into num_inliers).  These are run_chunk's
// launches on the same inputs, which is why the refinement returns the estimator's bytes.
int refine_chunk(rp_ctx *ctx, int variant, const rp_options &opt, const ChunkIO &io, cudaStream_t st) {
    const int P = io.n_pairs;
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    CK(ctx->res.reserve(P, false));
    int rc = prepare_chunk(ctx, variant, opt, io, nullptr, st);
    if (rc) return rc;
    PairParams *pairs = ctx->pt.pairs.as<PairParams>();
    Model *work = ctx->res.best.as<Model>();
    int *enable = ctx->res.enable.as<int>();
    refine_import_kernel<<<cdiv((long long)P * 32, 256), 256, 0, st>>>(P, variant, pairs, io.subset, io.init, work, enable,
                                                                      io.bstats_out);
    LAUNCHED();
    LMArgs la = final_lm_args(ctx, opt, io, work, io.subset, enable);
    la.stats = io.bstats_out;
    rc = launch_lm(ctx, variant, la, st);
    if (rc) return rc;
    if (io.masks_out) {
        rc = launch_pair_items(ctx, P, st);
        if (rc) return rc;
        rc = launch_get_inliers(ctx, pose, io, work, io.masks_out, st);
        if (rc) return rc;
    }
    refine_export_kernel<<<cdiv(P, 256), 256, 0, st>>>(P, variant, pairs, enable, io.init, work, ctx->res.final_count.as<int>(),
                                                       io.models_out, io.num_inliers_out);
    LAUNCHED();
    return RP_OK;
}

// rp_refine_pairs_{host,dev}[_f32]: run_chunks with refine_chunk as the work of a chunk.  In = float: the float32
// inputs are widened into the FP64 chunk arrays first, so every kernel after that runs on the bytes the FP64 entry
// points see.  Neither rp_pair_status nor rp_last_timing changes.
template <class In>
int refine_impl(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const In *x1, const In *x2,
                const In *d1, const In *d2, const double *cams, const rp_options *opt_in, const rp_model *init,
                const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats, int64_t *num_inliers, uint8_t *inliers,
                bool host_io, cudaStream_t st) {
    constexpr bool f32 = std::is_same<In, float>::value;
    if (!ctx) return RP_ERR_INVALID;
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2)) return fail(ctx, RP_ERR_INVALID, "null data pointer");
    if (n_pairs > 0 && (!init || !models)) return fail(ctx, RP_ERR_INVALID, "null init / models");
    rp_options opt;
    int rc = begin_batch(ctx, variant, n_pairs, offsets, cams, opt_in, opt);
    if (rc) return rc;
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    if (n_pairs == 0) return RP_OK;
    const long long Ntot = offsets[n_pairs] - offsets[0];
    const std::vector<int64_t> bounds =
        plan_chunks(ctx, n_pairs, refine_bytes_per_pair(Ntot / n_pairs + 1, host_io, f32), host_io, false);
    const BatchIn<In> b = {offsets, x1, x2, d1, d2, pose ? cams : nullptr, nullptr, init, subset, host_io};
    auto work = [&](int64_t c, StageSet &s, ChunkIO &io) -> int {
        const int64_t p0 = bounds[c];
        const int P = io.n_pairs;
        const size_t nn = (size_t)std::max<long long>(io.n_points, 1);
        CK(chunk_out(host_io, s.models, (Model *)models, p0, P, io.models_out));
        CK(chunk_out(host_io, s.stats, bstats, p0, P, io.bstats_out));
        CK(chunk_out(host_io, s.ninl, (long long *)num_inliers, p0, P, io.num_inliers_out));
        CK(chunk_out(host_io, s.mask, inliers, offsets[p0], nn, io.masks_out));
        if (num_inliers && !inliers) {
            // num_inliers alone: the mask goes to scratch
            CK(s.mask.reserve(nn));
            io.masks_out = s.mask.as<unsigned char>();
        }
        return refine_chunk(ctx, variant, opt, io, st);
    };
    auto download = [&](int64_t c, const ChunkIO &io, cudaStream_t cs) -> int {
        const int64_t p0 = bounds[c];
        const int P = io.n_pairs;
        CK(cudaMemcpyAsync(models + p0, io.models_out, sizeof(Model) * P, cudaMemcpyDeviceToHost, cs));
        if (bstats) CK(cudaMemcpyAsync(bstats + p0, io.bstats_out, sizeof(rp_bundle_stats) * P, cudaMemcpyDeviceToHost, cs));
        if (num_inliers) CK(cudaMemcpyAsync(num_inliers + p0, io.num_inliers_out, sizeof(long long) * P, cudaMemcpyDeviceToHost, cs));
        if (inliers && io.n_points > 0) CK(cudaMemcpyAsync(inliers + offsets[p0], io.masks_out, (size_t)io.n_points, cudaMemcpyDeviceToHost, cs));
        return RP_OK;
    };
    return run_chunks(ctx, b, bounds, st, false, work, download);
}

}  // namespace

// ================================================================================================
extern "C" {

int rp_create(int device, rp_ctx **out) {
    if (!out) return RP_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
        return RP_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) {
        g_create_error = "device index out of range";
        return RP_ERR_INVALID;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10) {
        g_create_error = "device is not sm_100-class (this library only ships sm_100a code)";
        return RP_ERR_NO_DEVICE;
    }
    rp_ctx *ctx = new rp_ctx();
    ctx->device = device;
    ctx->sms = prop.multiProcessorCount;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
        g_create_error = "cudaSetDevice / stream creation failed";
        delete ctx;
        return RP_ERR_CUDA;
    }
    for (auto &ev : ctx->ev) cudaEventCreate(&ev);
    for (auto &s : ctx->set) s.create_events();
    if (const char *np = getenv("RP_NO_PRUNE")) ctx->prune = !(np[0] == '1');
    if (const char *nw = getenv("RP_NO_WAVES")) ctx->waves = !(nw[0] == '1');
    if (const char *lw = getenv("RP_LM_WARP")) ctx->lm_warp = atoi(lw) != 0;
    if (const char *me = getenv("RP_MID_END")) ctx->mid = atoi(me) != 0;
    if (const char *nt = getenv("RP_NO_TC")) ctx->tc = !(nt[0] == '1');
    if (const char *op = getenv("RP_TC_ONE_PASS")) { if (op[0] == '1') ctx->tc_two_pass = false; }
    ctx->solve_generic = getenv("RP_SOLVE_GENERIC") != nullptr;
    if (const char *ec = getenv("RP_EV_CAP")) { const int v = atoi(ec); if (v >= 1 && v <= EV) ctx->ev_cap0 = v; }
    {
        cudaDriverEntryPointQueryResult qres;
        void *fn = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
            qres != cudaDriverEntryPointSuccess ||
            cudaFuncSetAttribute(tc::tc_count_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES) != cudaSuccess ||
            cudaFuncSetAttribute(order_by_quality_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 ORDER_SMEM_PER_POINT * ORDER_SMEM_CAP) != cudaSuccess) {
            g_create_error = "tensor-map entry point / shared-memory opt-in unavailable (driver too old for sm_100a TMA?)";
            rp_destroy(ctx);
            return RP_ERR_CUDA;
        }
        ctx->encode_tiled = fn;
    }
    if (const char *gb = getenv("RP_WORKSPACE_GB")) {
        const double v = atof(gb);
        if (v > 0.01) ctx->workspace_budget = (size_t)(v * (double)((size_t)1 << 30));
    }
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) ctx->workspace_budget = std::min(ctx->workspace_budget, free_b / 2);
    *out = ctx;
    return RP_OK;
}

void rp_destroy(rp_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (auto &s : ctx->set) s.destroy_events();
    for (auto &ev : ctx->ev) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;   // frees the workspace
}

const char *rp_last_error(const rp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int64_t rp_launch_count(const rp_ctx *ctx) { return ctx ? ctx->launches : 0; }

void rp_default_options(rp_options *o) {
    if (!o) return;
    memset(o, 0, sizeof *o);
    o->max_iterations = 100000; o->min_iterations = 1000; o->dyn_num_trials_mult = 3.0; o->success_prob = 0.9999;
    o->max_reproj_error = 12.0; o->max_epipolar_error = 1.0; o->seed = 0; o->estimate_shift = 0; o->weight_sampson = 1.0;
    o->progressive_sampling = 0; o->max_prosac_iterations = 100000;
    o->bundle_max_iterations = 100; o->loss_type = RP_LOSS_CAUCHY; o->loss_scale = 1.0; o->gradient_tol = 1e-10;
    o->step_tol = 1e-8; o->initial_lambda = 1e-3; o->min_lambda = 1e-10; o->max_lambda = 1e10;
}

int rp_estimate_batch_host(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                           const double *x2, const double *d1, const double *d2, const double *cams,
                           const rp_options *opt, rp_model *models, rp_stats *stats, uint8_t *masks) {
    if (!ctx) return RP_ERR_INVALID;
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2 || !models || !stats || !masks))
        return fail(ctx, RP_ERR_INVALID, "null data pointer");
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, nullptr, cams, opt, nullptr, models, stats, masks, true,
                         ctx->stream);
}

int rp_estimate_batch_dev(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                          const double *x2, const double *d1, const double *d2, const double *cams,
                          const rp_options *opt, rp_model *models, rp_stats *stats, uint8_t *masks, void *stream) {
    if (!ctx) return RP_ERR_INVALID;
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2 || !models || !stats || !masks))
        return fail(ctx, RP_ERR_INVALID, "null data pointer");
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, nullptr, cams, opt, nullptr, models, stats, masks, false,
                         stream ? (cudaStream_t)stream : ctx->stream);
}

int rp_estimate_batch_host_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                               const float *x2, const float *d1, const float *d2, const double *cams,
                               const rp_options *opt, rp_model *models, rp_stats *stats, uint8_t *masks) {
    if (!ctx) return RP_ERR_INVALID;
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2 || !models || !stats || !masks))
        return fail(ctx, RP_ERR_INVALID, "null data pointer");
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, nullptr, cams, opt, nullptr, models, stats, masks, true,
                         ctx->stream);
}

int rp_estimate_batch_dev_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                              const float *x2, const float *d1, const float *d2, const double *cams,
                              const rp_options *opt, rp_model *models, rp_stats *stats, uint8_t *masks, void *stream) {
    if (!ctx) return RP_ERR_INVALID;
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2 || !models || !stats || !masks))
        return fail(ctx, RP_ERR_INVALID, "null data pointer");
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, nullptr, cams, opt, nullptr, models, stats, masks, false,
                         stream ? (cudaStream_t)stream : ctx->stream);
}

// quality calls: the twins' checks, and a quality array for a non-empty batch
#define RP_QUALITY_CHECKS()                                                                          \
    if (!ctx) return RP_ERR_INVALID;                                                                 \
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2 || !models || !stats || !masks))                     \
        return fail(ctx, RP_ERR_INVALID, "null data pointer");                                       \
    if (n_pairs > 0 && !quality) return fail(ctx, RP_ERR_INVALID, "null quality")

int rp_estimate_batch_host_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                                   const double *x2, const double *d1, const double *d2, const float *quality,
                                   const double *cams, const rp_options *opt, rp_model *models, rp_stats *stats,
                                   uint8_t *masks) {
    RP_QUALITY_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, nullptr, models, stats, masks, true,
                         ctx->stream);
}

int rp_estimate_batch_dev_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                                  const double *x2, const double *d1, const double *d2, const float *quality,
                                  const double *cams, const rp_options *opt, rp_model *models, rp_stats *stats,
                                  uint8_t *masks, void *stream) {
    RP_QUALITY_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, nullptr, models, stats, masks, false,
                         stream ? (cudaStream_t)stream : ctx->stream);
}

int rp_estimate_batch_host_f32_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                                       const float *x2, const float *d1, const float *d2, const float *quality,
                                       const double *cams, const rp_options *opt, rp_model *models, rp_stats *stats,
                                       uint8_t *masks) {
    RP_QUALITY_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, nullptr, models, stats, masks, true,
                         ctx->stream);
}

int rp_estimate_batch_dev_f32_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                                      const float *x2, const float *d1, const float *d2, const float *quality,
                                      const double *cams, const rp_options *opt, rp_model *models, rp_stats *stats,
                                      uint8_t *masks, void *stream) {
    RP_QUALITY_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, nullptr, models, stats, masks, false,
                         stream ? (cudaStream_t)stream : ctx->stream);
}

// prior calls: the _quality twins' checks with quality nullable, and an init array for a non-empty batch
#define RP_INIT_CHECKS()                                                                             \
    if (!ctx) return RP_ERR_INVALID;                                                                 \
    if (n_pairs > 0 && (!x1 || !x2 || !d1 || !d2 || !models || !stats || !masks))                     \
        return fail(ctx, RP_ERR_INVALID, "null data pointer");                                       \
    if (n_pairs > 0 && !init) return fail(ctx, RP_ERR_INVALID, "null init")

int rp_estimate_batch_host_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                                const double *x2, const double *d1, const double *d2, const float *quality,
                                const double *cams, const rp_options *opt, const rp_model *init, rp_model *models,
                                rp_stats *stats, uint8_t *masks) {
    RP_INIT_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, init, models, stats, masks,
                         true, ctx->stream);
}

int rp_estimate_batch_dev_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                               const double *x2, const double *d1, const double *d2, const float *quality,
                               const double *cams, const rp_options *opt, const rp_model *init, rp_model *models,
                               rp_stats *stats, uint8_t *masks, void *stream) {
    RP_INIT_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, init, models, stats, masks,
                         false, stream ? (cudaStream_t)stream : ctx->stream);
}

int rp_estimate_batch_host_f32_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                                    const float *x2, const float *d1, const float *d2, const float *quality,
                                    const double *cams, const rp_options *opt, const rp_model *init, rp_model *models,
                                    rp_stats *stats, uint8_t *masks) {
    RP_INIT_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, init, models, stats, masks,
                         true, ctx->stream);
}

int rp_estimate_batch_dev_f32_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                                   const float *x2, const float *d1, const float *d2, const float *quality,
                                   const double *cams, const rp_options *opt, const rp_model *init, rp_model *models,
                                   rp_stats *stats, uint8_t *masks, void *stream) {
    RP_INIT_CHECKS();
    return estimate_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, quality, cams, opt, init, models, stats, masks,
                         false, stream ? (cudaStream_t)stream : ctx->stream);
}

int rp_refine_pairs_host(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                         const double *x2, const double *d1, const double *d2, const double *cams, const rp_options *opt,
                         const rp_model *init, const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                         int64_t *num_inliers, uint8_t *inliers) {
    return refine_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, cams, opt, init, subset, models, bstats, num_inliers,
                       inliers, true, ctx ? ctx->stream : nullptr);
}

int rp_refine_pairs_dev(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const double *x1,
                        const double *x2, const double *d1, const double *d2, const double *cams, const rp_options *opt,
                        const rp_model *init, const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                        int64_t *num_inliers, uint8_t *inliers, void *stream) {
    return refine_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, cams, opt, init, subset, models, bstats, num_inliers,
                       inliers, false, stream ? (cudaStream_t)stream : ctx ? ctx->stream : nullptr);
}

int rp_refine_pairs_host_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                             const float *x2, const float *d1, const float *d2, const double *cams, const rp_options *opt,
                             const rp_model *init, const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                             int64_t *num_inliers, uint8_t *inliers) {
    return refine_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, cams, opt, init, subset, models, bstats, num_inliers,
                       inliers, true, ctx ? ctx->stream : nullptr);
}

int rp_refine_pairs_dev_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets, const float *x1,
                            const float *x2, const float *d1, const float *d2, const double *cams, const rp_options *opt,
                            const rp_model *init, const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                            int64_t *num_inliers, uint8_t *inliers, void *stream) {
    return refine_impl(ctx, variant, n_pairs, offsets, x1, x2, d1, d2, cams, opt, init, subset, models, bstats, num_inliers,
                       inliers, false, stream ? (cudaStream_t)stream : ctx ? ctx->stream : nullptr);
}

int rp_pair_status(const rp_ctx *ctx, int64_t n_pairs, int32_t *status) {
    if (!ctx || n_pairs < 0 || (n_pairs > 0 && !status)) return RP_ERR_INVALID;
    for (int64_t i = 0; i < n_pairs; ++i) status[i] = (size_t)i < ctx->pair_status.size() ? ctx->pair_status[(size_t)i] : RP_PAIR_FAILED;
    return RP_OK;
}

int rp_last_timing(const rp_ctx *ctx, double *ms16, int64_t *counters16) {
    if (!ctx) return RP_ERR_INVALID;
    if (ms16) memcpy(ms16, ctx->last_ms, sizeof ctx->last_ms);
    if (counters16) memcpy(counters16, ctx->last_cnt, sizeof ctx->last_cnt);
    return RP_OK;
}

// ---- stage entry points -----------------------------------------------------------------------
int rp_sample_batch(rp_ctx *ctx, int64_t n, uint64_t seed, int64_t iters, int32_t *samples) {
    return rp_sample_batch_prosac(ctx, n, seed, iters, 0, 0, samples);
}

int rp_sample_batch_prosac(rp_ctx *ctx, int64_t n, uint64_t seed, int64_t iters, int32_t progressive_sampling,
                           int64_t max_prosac_iterations, int32_t *samples) {
    if (!ctx || !samples || n < 3 || iters < 0 || max_prosac_iterations < 0) return fail(ctx, RP_ERR_INVALID, "bad argument");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    CK(ctx->pt.pairs.reserve(sizeof(PairParams)));
    CK(ctx->hyp.samples.reserve(sizeof(int) * 3 * (size_t)std::max<int64_t>(iters, 1)));
    PairParams pp;
    memset(&pp, 0, sizeof pp);
    pp.n = (int)n; pp.valid = 1;
    CK(cudaMemcpyAsync(ctx->pt.pairs.p, &pp, sizeof pp, cudaMemcpyHostToDevice, st));
    if (iters > 0) {
        if (progressive_sampling)
            sample_prosac_kernel<<<1, 32, 0, st>>>(1, (int)iters, ctx->pt.pairs.as<PairParams>(), seed,
                                                   (unsigned long long)max_prosac_iterations, ctx->hyp.samples.as<int>());
        else
            sample_kernel<<<1, 32, 0, st>>>(1, (int)iters, ctx->pt.pairs.as<PairParams>(), seed, ctx->hyp.samples.as<int>());
        LAUNCHED();
        CK(cudaMemcpyAsync(samples, ctx->hyp.samples.p, sizeof(int) * 3 * (size_t)iters, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return RP_OK;
}

int rp_order_by_quality(rp_ctx *ctx, int64_t n_pairs, const int64_t *offsets, const float *quality, int32_t *perm) {
    if (!ctx || n_pairs < 0 || n_pairs > INT32_MAX || !offsets) return fail(ctx, RP_ERR_INVALID, "bad argument");
    for (int64_t p = 0; p < n_pairs; ++p)
        if (offsets[p + 1] < offsets[p] || offsets[p + 1] - offsets[p] >= (1 << 24))
            return fail(ctx, RP_ERR_INVALID, "offsets must be non-decreasing, at most 2^24-1 correspondences per pair");
    const long long N = offsets[n_pairs] - offsets[0];
    if (N > 0 && (!quality || !perm)) return fail(ctx, RP_ERR_INVALID, "bad argument");
    if (N == 0) return RP_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StageSet &s0 = ctx->set[0];  // the chunk pipeline's set 0, free between calls
    const int P = (int)n_pairs;
    CK(s0.qual.reserve(4 * (size_t)N)); CK(s0.perm.reserve(4 * (size_t)N));
    CK(s0.offs.reserve(8 * ((size_t)P + 1)));
    CK(cudaMemcpyAsync(s0.qual.p, quality + offsets[0], 4 * (size_t)N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s0.offs.p, offsets, 8 * ((size_t)P + 1), cudaMemcpyHostToDevice, st));
    int rc = launch_order(ctx, P, N, offsets, s0.offs.as<long long>(), offsets[0], s0.qual.as<float>(),
                          s0.perm.as<int>(), st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(perm + offsets[0], s0.perm.p, 4 * (size_t)N, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return RP_OK;
}

int rp_solve_batch(rp_ctx *ctx, int variant, int64_t n, const double *x1h, const double *x2h, const double *d1,
                   const double *d2, rp_model *models, int32_t *counts) {
    if (!ctx || variant < 0 || variant > 3 || n < 0 || (n > 0 && (!x1h || !x2h || !d1 || !d2 || !models || !counts)))
        return fail(ctx, RP_ERR_INVALID, "bad argument");
    if (n == 0) return RP_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StageSet &s0 = ctx->set[0];  // the chunk pipeline's set 0, free between calls
    CK(s0.x1.reserve(72 * (size_t)n)); CK(s0.x2.reserve(72 * (size_t)n));
    CK(s0.d1.reserve(24 * (size_t)n)); CK(s0.d2.reserve(24 * (size_t)n));
    CK(ctx->hyp.models.reserve(sizeof(Model) * 4 * (size_t)n)); CK(ctx->hyp.count.reserve(sizeof(int) * (size_t)n));
    CK(cudaMemcpyAsync(s0.x1.p, x1h, 72 * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s0.x2.p, x2h, 72 * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s0.d1.p, d1, 24 * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s0.d2.p, d2, 24 * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(ctx->hyp.models.p, 0, sizeof(Model) * 4 * (size_t)n, st));
    solve_problems_kernel<<<cdiv(n, 128), 128, 0, st>>>(variant, n, s0.x1.as<double>(), s0.x2.as<double>(),
                                                       s0.d1.as<double>(), s0.d2.as<double>(),
                                                       ctx->hyp.models.as<Model>(), ctx->hyp.count.as<int>());
    LAUNCHED();
    CK(cudaMemcpyAsync(models, ctx->hyp.models.p, sizeof(Model) * 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(counts, ctx->hyp.count.p, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return RP_OK;
}

static int stage_pair(rp_ctx *ctx, int64_t n_points, const double *x1, const double *x2, double sq_thr, cudaStream_t st) {
    StageSet &s0 = ctx->set[0];  // the chunk pipeline's set 0, free between calls
    const size_t nn = (size_t)std::max<int64_t>(n_points, 1);
    CK(ctx->pt.pairs.reserve(sizeof(PairParams)));
    CK(ctx->pt.pts64.reserve(sizeof(Pt64) * nn)); CK(ctx->pt.pts32.reserve(sizeof(float4) * nn)); CK(ctx->pt.bear.reserve(sizeof(Bear) * nn));
    CK(s0.x1.reserve(16 * nn)); CK(s0.x2.reserve(16 * nn));
    CK(cudaMemcpyAsync(s0.x1.p, x1, 16 * (size_t)n_points, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s0.x2.p, x2, 16 * (size_t)n_points, cudaMemcpyHostToDevice, st));
    stage_points_kernel<<<1, 32, 0, st>>>((int)n_points, s0.x1.as<double>(), s0.x2.as<double>(), sq_thr,
                                         ctx->pt.pts64.as<Pt64>(), ctx->pt.pts32.as<float4>(), ctx->pt.bear.as<Bear>(),
                                         ctx->pt.pairs.as<PairParams>());
    LAUNCHED();
    return RP_OK;
}

int rp_score_batch(rp_ctx *ctx, int variant, int64_t n_models, const rp_model *models, int64_t n_points,
                   const double *x1, const double *x2, double sq_threshold, double *scores, int64_t *counts,
                   uint8_t *masks) {
    if (!ctx || variant < 0 || variant > 3 || n_models < 0 || n_points < 0 ||
        (n_models > 0 && (!models || !scores || !counts)) || (n_points > 0 && (!x1 || !x2)))
        return fail(ctx, RP_ERR_INVALID, "bad argument");
    if (n_models == 0) return RP_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StageSet &s0 = ctx->set[0];  // the chunk pipeline's set 0, free between calls
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    int rc = stage_pair(ctx, n_points, x1, x2, sq_threshold, st);
    if (rc) return rc;
    CK(ctx->hyp.models.reserve(sizeof(Model) * (size_t)n_models));
    CK(ctx->hyp.score.reserve(sizeof(double) * (size_t)n_models)); CK(ctx->hyp.count.reserve(sizeof(int) * (size_t)n_models));
    CK(ctx->hyp.seg_count.reserve(sizeof(int) * 2)); CK(ctx->hyp.item_prefix.reserve(sizeof(int) * 4)); CK(ctx->pt.scalars.reserve(sizeof(Scalars)));
    Scalars *sc = ctx->pt.scalars.as<Scalars>();
    CK(cudaMemsetAsync(sc, 0, sizeof(Scalars), st));
    CK(cudaMemcpyAsync(ctx->hyp.models.p, models, sizeof(Model) * (size_t)n_models, cudaMemcpyHostToDevice, st));
    const int cnt = (int)n_models;
    CK(cudaMemcpyAsync(ctx->hyp.seg_count.p, &cnt, sizeof(int), cudaMemcpyHostToDevice, st));
    build_items_kernel<<<1, 1024, 0, st>>>(1, ctx->hyp.seg_count.as<int>(), ctx->hyp.item_prefix.as<int>(), &sc->n_items, nullptr);
    LAUNCHED();
    ScoreArgs a;
    a.n_groups = 1; a.grp_stride = 0; a.grp_per_pair = 1; a.grp_cnt = ctx->hyp.seg_count.as<int>();
    a.item_prefix = ctx->hyp.item_prefix.as<int>(); a.n_items = &sc->n_items; a.pairs = ctx->pt.pairs.as<PairParams>();
    a.models = ctx->hyp.models.as<Model>(); a.pts32 = ctx->pt.pts32.as<float4>(); a.pts64 = ctx->pt.pts64.as<Pt64>();
    a.bear = ctx->pt.bear.as<Bear>(); a.score = ctx->hyp.score.as<double>(); a.count = ctx->hyp.count.as<int>();
    a.mask = nullptr; a.point_scores = nullptr; a.slot_list = nullptr; a.list_stride = 0;
    rc = launch_score(ctx, pose, false, a, st);
    if (rc) return rc;
    std::vector<int> h_cnt((size_t)n_models);
    CK(cudaMemcpyAsync(scores, ctx->hyp.score.p, sizeof(double) * (size_t)n_models, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h_cnt.data(), ctx->hyp.count.p, sizeof(int) * (size_t)n_models, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < n_models; ++i) counts[i] = h_cnt[(size_t)i];
    if (masks && n_points > 0) {
        // I1 get_inliers: one launch per model with the mask variant of the same kernel
        CK(s0.mask.reserve((size_t)n_points)); CK(s0.models.reserve(sizeof(double))); CK(s0.stats.reserve(sizeof(int)));
        const int one = 1;
        CK(cudaMemcpyAsync(ctx->hyp.seg_count.p, &one, sizeof(int), cudaMemcpyHostToDevice, st));
        build_items_kernel<<<1, 1024, 0, st>>>(1, ctx->hyp.seg_count.as<int>(), ctx->hyp.item_prefix.as<int>(), &sc->n_items, nullptr);
        LAUNCHED();
        for (int64_t i = 0; i < n_models; ++i) {
            CK(cudaMemsetAsync(s0.mask.p, 0, (size_t)n_points, st));
            ScoreArgs m = a;
            m.models = ctx->hyp.models.as<Model>() + i; m.score = s0.models.as<double>(); m.count = s0.stats.as<int>();
            m.mask = s0.mask.as<unsigned char>();
            rc = launch_score(ctx, pose, true, m, st);
            if (rc) return rc;
            CK(cudaMemcpyAsync(masks + i * n_points, s0.mask.p, (size_t)n_points, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaStreamSynchronize(st));
    }
    return RP_OK;
}

int rp_tc_count_batch(rp_ctx *ctx, int variant, int64_t n_models, const rp_model *models, int64_t n_points,
                      const double *x1, const double *x2, double sq_threshold, int64_t *certain_outliers) {
    if (!ctx || variant < 0 || variant > 3 || n_models < 0 || n_points < 0 || n_models > 4 * SEG ||
        (n_models > 0 && (!models || !certain_outliers)) || (n_points > 0 && (!x1 || !x2)))
        return fail(ctx, RP_ERR_INVALID, "bad argument (at most 4096 models per call)");
    if (n_models == 0) return RP_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const bool pose = variant == RP_CALIB || variant == RP_CALIB_SHIFT;
    int rc = stage_pair(ctx, n_points, x1, x2, sq_threshold, st);
    if (rc) return rc;
    const size_t nn = (size_t)std::max<int64_t>(n_points, 1);
    CK(ctx->tcb.feat.reserve(128 * nn + 128 * tc::NT));
    CK(ctx->hyp.models.reserve(sizeof(Model) * 4 * SEG)); CK(ctx->tcb.out.reserve(sizeof(int) * 4 * SEG));
    CK(ctx->hyp.seg_count.reserve(sizeof(int) * 2)); CK(ctx->tcb.prefix.reserve(sizeof(int) * 4)); CK(ctx->pt.scalars.reserve(sizeof(Scalars)));
    Scalars *sc = ctx->pt.scalars.as<Scalars>();
    CK(cudaMemsetAsync(sc, 0, sizeof(Scalars), st));
    CK(cudaMemcpyAsync(ctx->hyp.models.p, models, sizeof(Model) * (size_t)n_models, cudaMemcpyHostToDevice, st));
    const int cnt = (int)n_models;
    CK(cudaMemcpyAsync(ctx->hyp.seg_count.p, &cnt, sizeof(int), cudaMemcpyHostToDevice, st));
    if (n_points > 0) {
        tc::tc_features_kernel<<<cdiv(n_points, 256), 256, 0, st>>>(n_points, ctx->pt.pts32.as<float4>(), ctx->tcb.feat.as<float4>());
        LAUNCHED();
    }
    build_items_kernel<<<1, 1024, 0, st>>>(1, ctx->hyp.seg_count.as<int>(), ctx->tcb.prefix.as<int>(), &sc->n_tc_items, nullptr, tc::TILE_MODELS);
    LAUNCHED();
    tc::TcArgs ta;
    memset(&ta, 0, sizeof ta);
    ta.n_pairs = 1; ta.nseg = 1; ta.pairs = ctx->pt.pairs.as<PairParams>(); ta.seg_count = ctx->hyp.seg_count.as<int>();
    ta.item_prefix = ctx->tcb.prefix.as<int>(); ta.n_items = &sc->n_tc_items; ta.models = ctx->hyp.models.as<Model>();
    ta.out = ctx->tcb.out.as<int>(); ta.pose = pose ? 1 : 0;
    rc = launch_tc(ctx, ta, ctx->tcb.feat.as<float4>(), n_points, st);
    if (rc) return rc;
    std::vector<int> h((size_t)n_models);
    CK(cudaMemcpyAsync(h.data(), ctx->tcb.out.p, sizeof(int) * (size_t)n_models, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < n_models; ++i) certain_outliers[i] = h[(size_t)i];
    return RP_OK;
}

int rp_refine_batch(rp_ctx *ctx, int variant, int64_t n_models, rp_model *models, int64_t n_points, const double *x1,
                    const double *x2, const double *d1, const double *d2, const uint8_t *mask, double scale_reproj,
                    double weight_sampson, const rp_bundle_options *opt, rp_bundle_stats *stats) {
    if (!ctx || variant < 0 || variant > 3 || n_models < 0 || n_points < 0 || !opt ||
        (n_models > 0 && !models) || (n_points > 0 && (!x1 || !x2 || !d1 || !d2)))
        return fail(ctx, RP_ERR_INVALID, "bad argument");
    if (n_models == 0) return RP_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StageSet &s0 = ctx->set[0];  // the chunk pipeline's set 0, free between calls
    int rc = stage_pair(ctx, n_points, x1, x2, 1.0, st);
    if (rc) return rc;
    const size_t nn = (size_t)std::max<int64_t>(n_points, 1);
    CK(s0.d1.reserve(8 * nn)); CK(s0.d2.reserve(8 * nn)); CK(s0.mask.reserve(nn));
    CK(ctx->hyp.models.reserve(sizeof(Model) * (size_t)n_models)); CK(ctx->pt.scalars.reserve(sizeof(Scalars)));
    CK(ctx->scratch.tmp2.reserve(sizeof(rp_bundle_stats) * (size_t)n_models));
    CK(cudaMemcpyAsync(s0.d1.p, d1, 8 * (size_t)n_points, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s0.d2.p, d2, 8 * (size_t)n_points, cudaMemcpyHostToDevice, st));
    if (mask) CK(cudaMemcpyAsync(s0.mask.p, mask, (size_t)n_points, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->hyp.models.p, models, sizeof(Model) * (size_t)n_models, cudaMemcpyHostToDevice, st));
    Scalars h;
    memset(&h, 0, sizeof h);
    h.n_prob = (int)n_models;
    Scalars *sc = ctx->pt.scalars.as<Scalars>();
    CK(cudaMemcpyAsync(sc, &h, sizeof h, cudaMemcpyHostToDevice, st));
    LMArgs la;
    memset(&la, 0, sizeof la);
    la.prob_list = nullptr; la.n_prob = &sc->n_prob; la.prob_per_pair = 1 << 30;  // every problem -> pair 0
    la.pairs = ctx->pt.pairs.as<PairParams>(); la.pts64 = ctx->pt.pts64.as<Pt64>();
    la.d1 = s0.d1.as<double>(); la.d2 = s0.d2.as<double>();
    la.mask = mask ? s0.mask.as<unsigned char>() : nullptr; la.enable = nullptr;
    la.models = ctx->hyp.models.as<Model>(); la.use_final = 1;
    la.max_iterations = (int)opt->max_iterations; la.loss_type = opt->loss_type;
    la.weight_sampson = weight_sampson; la.gradient_tol = opt->gradient_tol; la.step_tol = opt->step_tol;
    la.initial_lambda = opt->initial_lambda; la.min_lambda = opt->min_lambda; la.max_lambda = opt->max_lambda;
    la.loss_scale_override = opt->loss_scale; la.scale_reproj_override = scale_reproj;
    la.stats = ctx->scratch.tmp2.as<rp_bundle_stats>(); la.lm_iters = nullptr;
    rc = launch_lm(ctx, variant, la, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(models, ctx->hyp.models.p, sizeof(Model) * (size_t)n_models, cudaMemcpyDeviceToHost, st));
    if (stats) CK(cudaMemcpyAsync(stats, ctx->scratch.tmp2.p, sizeof(rp_bundle_stats) * (size_t)n_models, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return RP_OK;
}

}  // extern "C"

namespace {

// rp_gather_depths_dev[_f32][_quality]: T is the output type; with_q: the _quality entry points (quality / quality_out)
template <class T>
int gather_depths_impl(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                       const float *kp1, const float *kp2, const float *quality, int64_t n, T *x1, T *x2, T *d1, T *d2,
                       float *quality_out, int64_t *n_out, void *stream, bool with_q) {
    if (!ctx || n < 0 || !n_out || h1 <= 0 || w1 <= 0 || h2 <= 0 || w2 <= 0 ||
        (n > 0 && (!depth1 || !depth2 || !kp1 || !kp2 || !x1 || !x2 || !d1 || !d2)))
        return fail(ctx, RP_ERR_INVALID, "bad argument");
    if (with_q && n > 0 && (!quality || !quality_out)) return fail(ctx, RP_ERR_INVALID, "null quality / quality_out");
    *n_out = 0;
    if (n == 0) return RP_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    CK(ctx->pt.scalars.reserve(sizeof(Scalars)));
    long long *d_n = (long long *)ctx->pt.scalars.p;
    gather_depths_kernel<T><<<1, 1024, 0, st>>>(depth1, h1, w1, depth2, h2, w2, kp1, kp2, quality, (long long)n,
                                                x1, x2, d1, d2, quality_out, d_n);
    LAUNCHED();
    long long h_n = 0;
    CK(cudaMemcpyAsync(&h_n, d_n, sizeof h_n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *n_out = h_n;
    return RP_OK;
}

// rp_gather_depths_batch_dev[_f32][_quality]: T is the output type; with_q as above
template <class T>
int gather_depths_batch_impl(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps, int n_frames,
                             int h, int w, const int32_t *frame1, const int32_t *frame2, const float *kp1, const float *kp2,
                             const float *quality, T *x1, T *x2, T *d1, T *d2, float *quality_out, int64_t *out_offsets,
                             void *stream, bool with_q) {
    if (!ctx || n_pairs < 0 || !in_offsets || !out_offsets || h <= 0 || w <= 0 || n_frames <= 0 ||
        (n_pairs > 0 && (!depth_maps || !frame1 || !frame2)))
        return fail(ctx, RP_ERR_INVALID, "bad argument");
    out_offsets[0] = 0;
    if (n_pairs == 0) return RP_OK;
    const long long N = in_offsets[n_pairs] - in_offsets[0];
    for (int64_t p = 0; p < n_pairs; ++p) {
        if (in_offsets[p + 1] < in_offsets[p] || frame1[p] < 0 || frame1[p] >= n_frames || frame2[p] < 0 || frame2[p] >= n_frames)
            return fail(ctx, RP_ERR_INVALID, "offsets must be non-decreasing and frame indices inside [0, n_frames)");
    }
    if (N > 0 && (!kp1 || !kp2 || !x1 || !x2 || !d1 || !d2)) return fail(ctx, RP_ERR_INVALID, "null data pointer");
    if (with_q && N > 0 && (!quality || !quality_out)) return fail(ctx, RP_ERR_INVALID, "null quality / quality_out");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    const size_t nn = (size_t)std::max<long long>(N, 1);
    CK(ctx->sub.x1.reserve(16 * nn)); CK(ctx->sub.x2.reserve(16 * nn)); CK(ctx->sub.d1.reserve(8 * nn)); CK(ctx->sub.d2.reserve(8 * nn));
    if (with_q) CK(ctx->scratch.gather_q.reserve(4 * nn));
    CK(ctx->sub.src.reserve(8 * ((size_t)n_pairs + 1))); CK(ctx->sub.dst.reserve(8 * ((size_t)n_pairs + 1)));
    CK(ctx->sub.idx.reserve(sizeof(int) * 3 * (size_t)n_pairs));
    std::vector<long long> rel((size_t)n_pairs + 1);
    for (int64_t p = 0; p <= n_pairs; ++p) rel[(size_t)p] = in_offsets[p] - in_offsets[0];
    int *d_f1 = ctx->sub.idx.as<int>(), *d_f2 = d_f1 + n_pairs, *d_cnt = d_f2 + n_pairs;
    CK(cudaMemcpyAsync(ctx->sub.src.p, rel.data(), 8 * ((size_t)n_pairs + 1), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_f1, frame1, sizeof(int) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_f2, frame2, sizeof(int) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));
    GatherBatchArgs<T> g;
    g.n_pairs = (int)n_pairs; g.h = h; g.w = w; g.depth = depth_maps; g.frame1 = d_f1; g.frame2 = d_f2;
    g.in_off = ctx->sub.src.as<long long>(); g.out_off = ctx->sub.dst.as<long long>();
    g.kp1 = kp1; g.kp2 = kp2;
    g.tx1 = ctx->sub.x1.as<T>(); g.tx2 = ctx->sub.x2.as<T>(); g.td1 = ctx->sub.d1.as<T>(); g.td2 = ctx->sub.d2.as<T>();
    g.x1 = x1; g.x2 = x2; g.d1 = d1; g.d2 = d2; g.count = d_cnt;
    g.q_in = quality; g.tq = with_q ? ctx->scratch.gather_q.as<float>() : nullptr; g.q_out = quality_out;
    gather_depths_batch_kernel<T><<<(unsigned)n_pairs, 256, 0, st>>>(g);
    LAUNCHED();
    std::vector<int> cnt((size_t)n_pairs);
    CK(cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(int) * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));   // the one synchronisation of the batch: the caller needs the packed offsets
    std::vector<long long> out((size_t)n_pairs + 1, 0);
    for (int64_t p = 0; p < n_pairs; ++p) out[(size_t)p + 1] = out[(size_t)p] + cnt[(size_t)p];
    for (int64_t p = 0; p <= n_pairs; ++p) out_offsets[p] = out[(size_t)p];
    CK(cudaMemcpyAsync(ctx->sub.dst.p, out.data(), 8 * ((size_t)n_pairs + 1), cudaMemcpyHostToDevice, st));
    gather_depths_pack_kernel<T><<<(unsigned)n_pairs, 256, 0, st>>>(g);
    LAUNCHED();
    CK(cudaStreamSynchronize(st));   // `out` is a stack-lifetime host buffer
    return RP_OK;
}

}  // namespace

extern "C" {

int rp_gather_depths_dev(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                         const float *kp1, const float *kp2, int64_t n, double *x1, double *x2, double *d1, double *d2,
                         int64_t *n_out, void *stream) {
    return gather_depths_impl(ctx, depth1, h1, w1, depth2, h2, w2, kp1, kp2, nullptr, n, x1, x2, d1, d2, nullptr, n_out,
                              stream, false);
}

int rp_gather_depths_dev_f32(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                             const float *kp1, const float *kp2, int64_t n, float *x1, float *x2, float *d1, float *d2,
                             int64_t *n_out, void *stream) {
    return gather_depths_impl(ctx, depth1, h1, w1, depth2, h2, w2, kp1, kp2, nullptr, n, x1, x2, d1, d2, nullptr, n_out,
                              stream, false);
}

int rp_gather_depths_batch_dev(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps, int n_frames,
                               int h, int w, const int32_t *frame1, const int32_t *frame2, const float *kp1, const float *kp2,
                               double *x1, double *x2, double *d1, double *d2, int64_t *out_offsets, void *stream) {
    return gather_depths_batch_impl(ctx, n_pairs, in_offsets, depth_maps, n_frames, h, w, frame1, frame2, kp1, kp2, nullptr,
                                    x1, x2, d1, d2, nullptr, out_offsets, stream, false);
}

int rp_gather_depths_batch_dev_f32(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps,
                                   int n_frames, int h, int w, const int32_t *frame1, const int32_t *frame2, const float *kp1,
                                   const float *kp2, float *x1, float *x2, float *d1, float *d2, int64_t *out_offsets,
                                   void *stream) {
    return gather_depths_batch_impl(ctx, n_pairs, in_offsets, depth_maps, n_frames, h, w, frame1, frame2, kp1, kp2, nullptr,
                                    x1, x2, d1, d2, nullptr, out_offsets, stream, false);
}

int rp_gather_depths_dev_quality(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                                 const float *kp1, const float *kp2, const float *quality, int64_t n, double *x1, double *x2,
                                 double *d1, double *d2, float *quality_out, int64_t *n_out, void *stream) {
    return gather_depths_impl(ctx, depth1, h1, w1, depth2, h2, w2, kp1, kp2, quality, n, x1, x2, d1, d2, quality_out, n_out,
                              stream, true);
}

int rp_gather_depths_dev_f32_quality(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                                     const float *kp1, const float *kp2, const float *quality, int64_t n, float *x1,
                                     float *x2, float *d1, float *d2, float *quality_out, int64_t *n_out, void *stream) {
    return gather_depths_impl(ctx, depth1, h1, w1, depth2, h2, w2, kp1, kp2, quality, n, x1, x2, d1, d2, quality_out, n_out,
                              stream, true);
}

int rp_gather_depths_batch_dev_quality(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps,
                                       int n_frames, int h, int w, const int32_t *frame1, const int32_t *frame2,
                                       const float *kp1, const float *kp2, const float *quality, double *x1, double *x2,
                                       double *d1, double *d2, float *quality_out, int64_t *out_offsets, void *stream) {
    return gather_depths_batch_impl(ctx, n_pairs, in_offsets, depth_maps, n_frames, h, w, frame1, frame2, kp1, kp2, quality,
                                    x1, x2, d1, d2, quality_out, out_offsets, stream, true);
}

int rp_gather_depths_batch_dev_f32_quality(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps,
                                           int n_frames, int h, int w, const int32_t *frame1, const int32_t *frame2,
                                           const float *kp1, const float *kp2, const float *quality, float *x1, float *x2,
                                           float *d1, float *d2, float *quality_out, int64_t *out_offsets, void *stream) {
    return gather_depths_batch_impl(ctx, n_pairs, in_offsets, depth_maps, n_frames, h, w, frame1, frame2, kp1, kp2, quality,
                                    x1, x2, d1, d2, quality_out, out_offsets, stream, true);
}

int rp_measure_pipes(rp_ctx *ctx, double *fp64_tflops, double *fp32_tflops) {
    if (!ctx) return RP_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StageSet &s0 = ctx->set[0];  // the chunk pipeline's set 0, free between calls
    const int blocks = ctx->sms * 8, threads = 256, iters = 1 << 13;
    CK(s0.models.reserve(sizeof(double) * (size_t)blocks * threads));
    cudaEvent_t e0 = ctx->ev[9], e1 = ctx->ev[10];
    for (int pass = 0; pass < 2; ++pass) {
        double best = 0.0;
        for (int rep = 0; rep < 4; ++rep) {
            CK(cudaEventRecord(e0, st));
            if (pass == 0) fp64_pipe_kernel<<<blocks, threads, 0, st>>>(s0.models.as<double>(), iters);
            else fp32_pipe_kernel<<<blocks, threads, 0, st>>>(s0.models.as<float>(), iters);
            LAUNCHED();
            CK(cudaEventRecord(e1, st));
            CK(cudaStreamSynchronize(st));
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            const double flops = 2.0 * 16.0 * (double)iters * (double)blocks * threads;
            if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
        }
        if (pass == 0 && fp64_tflops) *fp64_tflops = best;
        if (pass == 1 && fp32_tflops) *fp32_tflops = best;
    }
    return RP_OK;
}

}  // extern "C"
