// lmcheck.cu — test harness of the LM kernels (tests/test_gpu_lm_reference.py).
//
// The LO configuration of the LM kernels (use_final = 0: lm_warp_kernel and the block kernel with the TRUNCATED
// loss) is only launched from inside the estimator, so no product entry point reaches it.  This file is built
// together with the product's own mdrp_b200/csrc/repose_lm.cu into tests/lmcheck/liblmcheck.so and exposes one
// call that fills every LMArgs field from the caller and runs rp::launch_lm_kernel once.
#include "../../mdrp_b200/csrc/rp_lm_kernel.cuh"

#include <string.h>

using namespace rp;

namespace {

struct Dev {
    void *p = nullptr;
    ~Dev() { if (p) cudaFree(p); }
};

}  // namespace

// Pair p owns the correspondences off[p] .. off[p] + n[p] - 1 of pts ([n_points, 4]: x1_0, x1_1, x2_0, x2_1), d1 and d2.
// models ([n_models], rp_model) and stats ([n_models], rp_bundle_stats) are uploaded, updated in place by the kernel
// for the problems it runs, and copied back whole, so untouched entries return as the caller wrote them.
// iopt: use_final, warp_kernel, warp_single, max_iterations, loss_type, prob_per_pair
// dopt: weight_sampson, gradient_tol, step_tol, initial_lambda, min_lambda, max_lambda, loss_scale_override,
//       scale_reproj_override
// mask, enable and prob_list may be null.  Returns the first CUDA error (0 on success).
extern "C" __attribute__((visibility("default"))) int lmc_run(
    int variant, int n_pairs, const long long *off, const int *n, const int *valid, const double *scale_reproj,
    const double *lo_loss_scale, const double *final_loss_scale, long long n_points, const double *pts,
    const double *d1, const double *d2, const unsigned char *mask, const int *enable, int n_prob, const int *prob_list,
    int n_models, rp_model *models, rp_bundle_stats *stats, const int *iopt, const double *dopt) {
    cudaError_t err = cudaSuccess;
    auto ck = [&](cudaError_t e) { if (err == cudaSuccess) err = e; };
    int dev = 0, sms = 0;
    ck(cudaGetDevice(&dev));
    ck(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t np = (size_t)(n_points > 0 ? n_points : 1);

    PairParams *hp = new PairParams[n_pairs > 0 ? n_pairs : 1];
    memset(hp, 0, sizeof(PairParams) * (size_t)(n_pairs > 0 ? n_pairs : 1));
    for (int p = 0; p < n_pairs; ++p) {
        hp[p].off = off[p]; hp[p].n = n[p]; hp[p].valid = valid[p];
        hp[p].scale_reproj = scale_reproj[p]; hp[p].lo_loss_scale = lo_loss_scale[p];
        hp[p].final_loss_scale = final_loss_scale[p];
    }
    Dev d_pairs, d_pts, d_d1, d_d2, d_mask, d_enable, d_list, d_nprob, d_models, d_stats, d_work;
    ck(cudaMalloc(&d_pairs.p, sizeof(PairParams) * (size_t)(n_pairs > 0 ? n_pairs : 1)));
    ck(cudaMalloc(&d_pts.p, sizeof(Pt64) * np));
    ck(cudaMalloc(&d_d1.p, 8 * np));
    ck(cudaMalloc(&d_d2.p, 8 * np));
    if (mask) ck(cudaMalloc(&d_mask.p, np));
    if (enable) ck(cudaMalloc(&d_enable.p, sizeof(int) * (size_t)n_pairs));
    if (prob_list) ck(cudaMalloc(&d_list.p, sizeof(int) * (size_t)(n_prob > 0 ? n_prob : 1)));
    ck(cudaMalloc(&d_nprob.p, sizeof(int)));
    ck(cudaMalloc(&d_models.p, sizeof(rp_model) * (size_t)(n_models > 0 ? n_models : 1)));
    ck(cudaMalloc(&d_stats.p, sizeof(rp_bundle_stats) * (size_t)(n_models > 0 ? n_models : 1)));
    ck(cudaMalloc(&d_work.p, sizeof(int)));
    if (err == cudaSuccess) {
        ck(cudaMemcpy(d_pairs.p, hp, sizeof(PairParams) * (size_t)n_pairs, cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_pts.p, pts, sizeof(Pt64) * (size_t)n_points, cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_d1.p, d1, 8 * (size_t)n_points, cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_d2.p, d2, 8 * (size_t)n_points, cudaMemcpyHostToDevice));
        if (mask) ck(cudaMemcpy(d_mask.p, mask, (size_t)n_points, cudaMemcpyHostToDevice));
        if (enable) ck(cudaMemcpy(d_enable.p, enable, sizeof(int) * (size_t)n_pairs, cudaMemcpyHostToDevice));
        if (prob_list) ck(cudaMemcpy(d_list.p, prob_list, sizeof(int) * (size_t)n_prob, cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_nprob.p, &n_prob, sizeof(int), cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_models.p, models, sizeof(rp_model) * (size_t)n_models, cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_stats.p, stats, sizeof(rp_bundle_stats) * (size_t)n_models, cudaMemcpyHostToDevice));
        ck(cudaMemset(d_work.p, 0, sizeof(int)));
    }
    if (err == cudaSuccess) {
        LMArgs a;
        memset(&a, 0, sizeof a);
        a.prob_list = (const int *)d_list.p; a.n_prob = (const int *)d_nprob.p; a.prob_per_pair = iopt[5];
        a.pairs = (const PairParams *)d_pairs.p; a.pts64 = (const Pt64 *)d_pts.p;
        a.d1 = (const double *)d_d1.p; a.d2 = (const double *)d_d2.p;
        a.mask = (const unsigned char *)d_mask.p; a.enable = (const int *)d_enable.p;
        a.models = (Model *)d_models.p;
        a.use_final = iopt[0]; a.warp_kernel = iopt[1]; a.warp_single = iopt[2];
        a.max_iterations = iopt[3]; a.loss_type = iopt[4];
        a.weight_sampson = dopt[0]; a.gradient_tol = dopt[1]; a.step_tol = dopt[2];
        a.initial_lambda = dopt[3]; a.min_lambda = dopt[4]; a.max_lambda = dopt[5];
        a.loss_scale_override = dopt[6]; a.scale_reproj_override = dopt[7];
        a.stats = (rp_bundle_stats *)d_stats.p; a.lm_iters = nullptr; a.lm_flops = nullptr;
        a.work_counter = (int *)d_work.p;
        ck((cudaError_t)launch_lm_kernel(sms, variant, a, 0));
        ck(cudaDeviceSynchronize());
    }
    if (err == cudaSuccess) {
        ck(cudaMemcpy(models, d_models.p, sizeof(rp_model) * (size_t)n_models, cudaMemcpyDeviceToHost));
        ck(cudaMemcpy(stats, d_stats.p, sizeof(rp_bundle_stats) * (size_t)n_models, cudaMemcpyDeviceToHost));
    }
    delete[] hp;
    return (int)err;
}
