// rp_order.cuh — ordering of a ragged batch by per-correspondence match quality (rp_estimate_batch_*_quality,
// rp_order_by_quality).  PROSAC draws its samples from a growing prefix of each pair's correspondences, so it needs them
// sorted by decreasing quality; these kernels compute that order on the device:
//   order_by_quality_kernel  one CTA per pair: stable LSD radix sort of the pair's 32-bit order keys -> perm (pair-local)
//   scatter_masks_kernel     the chunk's inlier masks, computed in the ordered layout, back to the caller's order
// The gather of the inputs into the ordered layout is widen_inputs_kernel (rp_kernels.cuh) with a permutation.
#pragma once
#include <cuda_runtime.h>
#include "rp_types.cuh"

namespace rp {

constexpr int ORDER_THREADS = 256;                  // one thread per radix digit in the prefix step
constexpr int ORDER_WARPS = ORDER_THREADS / 32;
constexpr int ORDER_SMEM_CAP = RP_ORDER_SMEM_CAP;   // pairs up to this size sort in shared memory (16 B per correspondence)
constexpr int ORDER_SMEM_PER_POINT = 16;            // two key buffers and two index buffers

// 32-bit key whose ascending order is the order the estimator wants: quality descending, with NaN as -inf and -0 as +0.
// Ties are left to the sort, which is stable: equal keys keep ascending original index.
__device__ __forceinline__ unsigned order_key(float q) {
    unsigned b = isnan(q) ? 0xff800000u : __float_as_uint(q);   // -inf
    if (b == 0x80000000u) b = 0u;                               // -0 -> +0
    b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);             // ascending float order as unsigned order
    return ~b;                                                  // descending
}

// pair of correspondence j of a chunk: the last p with offsets[p] - base <= j.  Pairs are non-empty around j, because
// offsets are non-decreasing and j < offsets[n_pairs] - base.
__device__ __forceinline__ int pair_of(long long j, const long long *offsets, long long base, int n_pairs) {
    int lo = 0, hi = n_pairs - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (offsets[mid] - base <= j) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

struct OrderArgs {
    const long long *offsets;  // [n_pairs + 1]; pair p owns [offsets[p] - base, offsets[p+1] - base) of the chunk
    long long base;
    const float *quality;      // [N] chunk-local
    int *perm;                 // [N] chunk-local: perm[o + j] = index inside the pair of the j-th best correspondence
    int smem_cap;              // pairs of at most this many correspondences sort in dynamic shared memory
    unsigned *gkeys;           // [2N] scratch of the pairs above smem_cap (null when the chunk has none)
    int *gidx;                 // [N]  scratch of the pairs above smem_cap
};

// One CTA per pair, four 8-bit LSD passes.  Every warp owns a contiguous segment of the pair; a pass counts the digits
// per (warp, digit), turns the counts into start positions (digit-major, then warp), and each warp scatters its segment
// in order, ranking equal digits within 32 elements with __match_any_sync.  That keeps every pass stable.  A pass in which
// every key has the same digit is the identity and is skipped.  Pairs above smem_cap run the same code on global
// scratch: rare, and slower.
__global__ void __launch_bounds__(ORDER_THREADS) order_by_quality_kernel(OrderArgs a) {
    static_assert(ORDER_THREADS == 256, "the prefix step gives every thread one of the 256 digits");
    extern __shared__ unsigned order_smem[];
    __shared__ int pos[ORDER_WARPS * 256];   // per (warp, digit): count, then next output position
    __shared__ int warp_tot[ORDER_WARPS];
    __shared__ int identity;
    const int pair = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const long long o = a.offsets[pair] - a.base;
    const int n = (int)(a.offsets[pair + 1] - a.offsets[pair]);
    int *out = a.perm + o;
    if (n <= 1) {
        if (n == 1 && tid == 0) out[0] = 0;
        return;
    }
    unsigned *k0, *k1;
    int *i0, *i1;
    if (n <= a.smem_cap) {
        k0 = order_smem; k1 = k0 + a.smem_cap;
        i0 = (int *)(k1 + a.smem_cap); i1 = i0 + a.smem_cap;
    } else {
        k0 = a.gkeys + 2 * o; k1 = k0 + n;
        i0 = a.gidx + o; i1 = out;
    }
    for (int j = tid; j < n; j += ORDER_THREADS) {
        k0[j] = order_key(a.quality[o + j]);
        i0[j] = j;
    }
    const int seg = (n + ORDER_WARPS - 1) / ORDER_WARPS;
    const int lo = min(n, w * seg), hi = min(n, lo + seg);
    int *wpos = pos + w * 256;
    for (int shift = 0; shift < 32; shift += 8) {
        for (int d = tid; d < ORDER_WARPS * 256; d += ORDER_THREADS) pos[d] = 0;
        if (tid == 0) identity = 0;
        __syncthreads();
        for (int b = lo; b < hi; b += 32) {
            const int j = b + lane;
            const unsigned d = j < hi ? (k0[j] >> shift) & 255u : 256u + lane;
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            if (j < hi && lane == __ffs(peers) - 1) wpos[d] += __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        // thread tid owns digit tid: exclusive prefix over the warps, then over the digits
        int tot = 0;
        for (int v = 0; v < ORDER_WARPS; ++v) {
            const int c = pos[v * 256 + tid];
            pos[v * 256 + tid] = tot;
            tot += c;
        }
        if (tot == n) identity = 1;
        int incl = tot;
        for (int s = 1; s < 32; s <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, s);
            if (lane >= s) incl += t;
        }
        if (lane == 31) warp_tot[w] = incl;
        __syncthreads();
        int excl = incl - tot;
        for (int v = 0; v < w; ++v) excl += warp_tot[v];
        for (int v = 0; v < ORDER_WARPS; ++v) pos[v * 256 + tid] += excl;
        __syncthreads();
        const bool skip = identity != 0;
        if (!skip) {
            for (int b = lo; b < hi; b += 32) {
                const int j = b + lane;
                const bool in = j < hi;
                const unsigned key = in ? k0[j] : 0u;
                const unsigned d = in ? (key >> shift) & 255u : 256u + lane;
                const unsigned peers = __match_any_sync(0xffffffffu, d);
                if (in) {
                    const int p = wpos[d] + __popc(peers & ((1u << lane) - 1u));
                    k1[p] = key;
                    i1[p] = i0[j];
                }
                __syncwarp();
                if (in && lane == __ffs(peers) - 1) wpos[d] += __popc(peers);
                __syncwarp();
            }
        }
        __syncthreads();
        if (!skip) {
            unsigned *tk = k0; k0 = k1; k1 = tk;
            int *ti = i0; i0 = i1; i1 = ti;
        }
    }
    if (i0 != out)
        for (int j = tid; j < n; j += ORDER_THREADS) out[j] = i0[j];
}

// The chunk's masks, computed in the ordered layout (`sorted`), written in the caller's order:
// out[o + perm[o + j]] = sorted[o + j] for the pair starting at o.  Grid-stride over the n correspondences of the chunk.
__global__ void scatter_masks_kernel(long long n, int n_pairs, const long long *offsets, long long base, const int *perm,
                                     const unsigned char *sorted, unsigned char *out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        const int p = pair_of(j, offsets, base, n_pairs);
        out[offsets[p] - base + perm[j]] = sorted[j];
    }
}

}  // namespace rp
