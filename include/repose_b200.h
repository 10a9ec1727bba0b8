/*
 * repose_b200.h — C ABI of the B200-native batched RePoseD relative-pose estimator.
 *
 * This is the drop-in boundary for the hot path behind
 *   poselib.estimate_monodepth_relative_pose                 (whl:_core.pyi:446-475, so@0x224170)
 *   poselib.estimate_monodepth_shared_focal_relative_pose    (whl:_core.pyi:477-488, so@0x223300)
 *   poselib.estimate_monodepth_varying_focal_relative_pose   (whl:_core.pyi:490-501, so@0x223a40)
 * of PoseLib 2.0.5 + PR #152 as used by kocurvik/mdrp (/root/reference/make_pair.py:111,
 * make_video.py:284, README.md:86-96).  The reference binds these through pybind11 one
 * pair per call; this library takes a ragged BATCH of pairs per call (a single pair is a
 * batch of one).  Plain pointers and sizes only; no exceptions cross the boundary: every
 * function returns 0 on success or a negative rp_status, and rp_last_error() explains.
 *
 * There is no CPU execution path: every entry point needs a CUDA device (sm_100a).
 */
#ifndef REPOSE_B200_H
#define REPOSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RP_API __attribute__((visibility("default")))

typedef struct rp_ctx rp_ctx;

enum rp_status {
    RP_OK = 0,
    RP_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, unknown variant) */
    RP_ERR_CUDA = -2,      /* CUDA runtime error; text in rp_last_error */
    RP_ERR_NO_DEVICE = -3, /* no CUDA device / wrong architecture */
    RP_ERR_OVERFLOW = -4,  /* an internal fixed-capacity list overflowed (no longer returned by the estimators: see rp_pair_status) */
    RP_ERR_PARTIAL = -5    /* the call finished, but some pairs could not be (rp_pair_status < 0); all other outputs are valid */
};

/* per-pair status of the last rp_estimate_batch_* call (rp_pair_status).  Non-negative values are informational. */
enum rp_pair_state {
    RP_PAIR_OK = 0,
    RP_PAIR_DEGENERATE = 1,    /* fewer than 3 correspondences: identity model, iterations 0 (as the reference) */
    RP_PAIR_EVENTS_RERUN = 2,  /* bit: the pair had more LO triggers than the first pass keeps and was run again on its own */
    RP_PAIR_CONTINUED = 4,     /* bit: early termination needed more than min_iterations + 1 iterations; run again on its own */
    RP_PAIR_FAILED = -1        /* the pair's re-run could not be done (device memory); its outputs are void */
};

/* estimator variants (which minimal solver / Jacobian accumulator is used) */
enum rp_variant {
    RP_CALIB = 0,       /* calibrated, scale only:   P3P + scale (generate_models so@0x4fe090), 7 params */
    RP_CALIB_SHIFT = 1, /* calibrated, scale+shifts: relpose_monodepth_3pt so@0x155ca0, 9 params        */
    RP_SHARED = 2,      /* shared unknown focal:     relpose_monodepth_3pt_shared_focal so@0x18fdf0, 8   */
    RP_VARYING = 3      /* two unknown focals:       relpose_monodepth_3pt_varying_focal so@0x19bcd0, 9  */
};

/* BundleOptions.loss_type (SURVEY.md Appendix A.2) */
enum rp_loss {
    RP_LOSS_TRIVIAL = 0, RP_LOSS_TRUNCATED = 1, RP_LOSS_HUBER = 2, RP_LOSS_CAUCHY = 3,
    RP_LOSS_TRUNCATED_CAUCHY = 4
};

/* MonoDepthTwoViewGeometry / MonoDepthImagePair (whl:_core.pyi:171-204): 12 doubles.
 * X2 = scale*(d2+shift2)*K2^-1 x2 = R(q)*(d1+shift1)*K1^-1 x1 + t ; q is w-first.
 * f1,f2 are 1 for the calibrated variants. */
typedef struct {
    double q[4];
    double t[3];
    double scale, shift1, shift2;
    double f1, f2;
} rp_model;

/* RansacStats (SURVEY.md §8a row R1) */
typedef struct {
    int64_t refinements, iterations, num_inliers;
    double inlier_ratio, model_score;
} rp_stats;

/* RansacOptions + BundleOptions (whl:METADATA:71-107), the keys the monodepth path reads */
typedef struct {
    int64_t max_iterations, min_iterations;
    double dyn_num_trials_mult, success_prob;
    double max_reproj_error, max_epipolar_error;
    uint64_t seed;
    int32_t estimate_shift; /* monodepth_estimate_shift (calibrated variants) */
    int32_t progressive_sampling; /* PROSAC sampling: correspondences sorted by decreasing quality */
    double weight_sampson;  /* monodepth_weight_sampson */
    /* final refinement (bundle_opt) */
    int64_t bundle_max_iterations;
    int32_t loss_type;
    int32_t reserved1;
    double loss_scale, gradient_tol, step_tol, initial_lambda, min_lambda, max_lambda;
    int64_t max_prosac_iterations; /* RansacOptions::max_prosac_iterations (default 100000) */
} rp_options;

/* LM options for the stage entry point rp_refine_batch (BundleOptions) */
typedef struct {
    int64_t max_iterations;
    int32_t loss_type;
    int32_t reserved;
    double loss_scale, gradient_tol, step_tol, initial_lambda, min_lambda, max_lambda;
} rp_bundle_options;

/* BundleStats */
typedef struct {
    int64_t iterations;
    double initial_cost, cost, lambda;
    int64_t invalid_steps;
    double step_norm, grad_norm;
} rp_bundle_stats;

/* ---- lifetime ------------------------------------------------------------------ */
RP_API int rp_create(int device, rp_ctx **out);
RP_API void rp_destroy(rp_ctx *ctx);
RP_API const char *rp_last_error(const rp_ctx *ctx); /* ctx may be NULL: last creation error */
RP_API void rp_default_options(rp_options *opt);     /* PoseLib defaults (RansacOptions(), BundleOptions()) */
/* number of kernels this library launched on ctx since creation (bench "gpu_launches") */
RP_API int64_t rp_launch_count(const rp_ctx *ctx);

/* ---- the hot path: batched estimators -------------------------------------------
 * n_pairs image pairs, pair p owning correspondences [offsets[p], offsets[p+1]).
 * x1,x2: [offsets[n_pairs], 2] pixel coordinates (row-major), d1,d2: [offsets[n_pairs]].
 * variant RP_CALIB / RP_CALIB_SHIFT (replaces estimate_monodepth_relative_pose):
 *     cams: [n_pairs, 8] = (fx1, fy1, cx1, cy1, fx2, fy2, cx2, cy2) pinhole intrinsics;
 *     opt->estimate_shift selects RP_CALIB_SHIFT when variant is RP_CALIB.
 * variant RP_SHARED / RP_VARYING (replace the two focal estimators): x already
 *     principal-point-centred, cams ignored (may be NULL).
 * Outputs: models [n_pairs], stats [n_pairs], masks [offsets[n_pairs]] (0/1 bytes, the
 * `inliers` list of the reference's info dict).
 * _host: all pointers are HOST memory (pinned or pageable); copies are inside the call.
 * _dev : x1,x2,d1,d2,cams,models,stats,masks are DEVICE memory on ctx's device (inputs already
 *        resident in HBM); `offsets` and `opt` stay HOST memory (the host plans the chunks from
 *        them); `stream` is a cudaStream_t (NULL = default stream); the call returns after the
 *        stream has finished. */
RP_API int rp_estimate_batch_host(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                  const double *x1, const double *x2, const double *d1, const double *d2,
                                  const double *cams, const rp_options *opt, rp_model *models,
                                  rp_stats *stats, uint8_t *masks);
RP_API int rp_estimate_batch_dev(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                 const double *x1, const double *x2, const double *d1, const double *d2,
                                 const double *cams, const rp_options *opt, rp_model *models,
                                 rp_stats *stats, uint8_t *masks, void *stream);

/* The same two estimators for float32 keypoints and depths, the type matchers and depth networks produce: x1, x2, d1, d2
 * are `const float *` with the layout above; cams, offsets, options and outputs are as above, and so are the argument
 * checks and error codes.  The inputs are widened to FP64 on the device (float -> double is exact) and everything after
 * that is the FP64 path, so the outputs are byte for byte those of rp_estimate_batch_host / _dev on the same values
 * converted to double.  _host uploads 24 B per correspondence instead of 48 (double-buffered float staging, widened on
 * the copy stream); _dev reads the caller's float arrays and needs 48 B per correspondence of the current chunk for the
 * widened copy instead of an FP64 copy of the whole batch.  rp_last_timing slot [13] reports the widening time. */
RP_API int rp_estimate_batch_host_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                      const float *x1, const float *x2, const float *d1, const float *d2,
                                      const double *cams, const rp_options *opt, rp_model *models,
                                      rp_stats *stats, uint8_t *masks);
RP_API int rp_estimate_batch_dev_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                     const float *x1, const float *x2, const float *d1, const float *d2,
                                     const double *cams, const rp_options *opt, rp_model *models,
                                     rp_stats *stats, uint8_t *masks, void *stream);

/* The four estimators with one float32 match quality per correspondence (LightGlue score, RoMa certainty, ...):
 * quality [offsets[n_pairs]], HOST memory for _host and DEVICE memory for _dev, inserted after d2 in the twin's argument
 * list.  They order each pair on the device so that PROSAC (opt->progressive_sampling) sees its correspondences from
 * best to worst, and they are defined by that order:
 *   - the outputs (models, stats, masks, rp_pair_status) are, as bytes, those of the twin called with every pair's
 *     correspondences reordered by (quality descending, original index ascending);
 *   - the ordering key is the float32 quality with NaN taken as -inf and -0 as +0;
 *   - masks come back in the CALLER's order: masks[o + perm[j]] = (mask of the reordered pair)[o + j].
 * opt->progressive_sampling is honoured as given (0: uniform sampling on the reordered pairs).  Results depend only on a
 * pair's data, its quality and opt->seed, never on the batch around it or on the chunking.  A null quality with
 * n_pairs > 0 is RP_ERR_INVALID; every other check and error code is the twin's.  rp_last_timing slot [14] reports the
 * ordering (sort, permuting gather, mask scatter). */
RP_API int rp_estimate_batch_host_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                          const double *x1, const double *x2, const double *d1, const double *d2,
                                          const float *quality, const double *cams, const rp_options *opt,
                                          rp_model *models, rp_stats *stats, uint8_t *masks);
RP_API int rp_estimate_batch_dev_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                         const double *x1, const double *x2, const double *d1, const double *d2,
                                         const float *quality, const double *cams, const rp_options *opt,
                                         rp_model *models, rp_stats *stats, uint8_t *masks, void *stream);
RP_API int rp_estimate_batch_host_f32_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                              const float *x1, const float *x2, const float *d1, const float *d2,
                                              const float *quality, const double *cams, const rp_options *opt,
                                              rp_model *models, rp_stats *stats, uint8_t *masks);
RP_API int rp_estimate_batch_dev_f32_quality(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                             const float *x1, const float *x2, const float *d1, const float *d2,
                                             const float *quality, const double *cams, const rp_options *opt,
                                             rp_model *models, rp_stats *stats, uint8_t *masks, void *stream);

/* ---- estimation from a prior ----------------------------------------------------
 * The estimator with one prior model per pair (a tracker's previous pose, another method's estimate): the _quality
 * twin's arguments with quality NULLABLE (NULL: the plain twin), plus init [n_pairs] inserted after opt, HOST memory for
 * _host and DEVICE memory for _dev, in the layout and frame of the models the estimator returns (focal variants: f1, f2
 * in pixels).  For each pair, RANSAC runs as the twin's except that before its first iteration the prior is scored
 * (MSAC, as a minimal model is) and, as a minimal model that beats every earlier one, locally optimised by the in-loop LO;
 * the best model, stats.model_score / num_inliers / inlier_ratio and the dynamic iteration limit are updated exactly as
 * after an in-loop LO, and stats.refinements counts that LO.  Then come the sampled iterations (stats.iterations counts
 * only those), the final LO, the final refinement and the mask, unchanged.  So:
 *   - stats.model_score <= min(score(prior), score(LO(prior))): the result is never worse than the locally optimised
 *     prior, and RANSAC still samples, so a wrong prior is recovered from;
 *   - opt->max_iterations = 0 returns the LO of the prior, then the final LO and the final refinement (refinements 2);
 *   - a prior with a non-finite field the variant reads (q, t, scale, shift1, shift2; f1, f2 for the focal variants)
 *     means "no prior" for that pair: NaN rows leave pairs without a prior, and such a pair's bytes are the twin's;
 *   - pairs of fewer than 3 correspondences keep the degenerate result (identity, iterations 0).
 * The calibrated variants use q, t, scale, shift1, shift2 as given (RP_CALIB holds the shifts, as its LO does); the
 * focal variants divide f1, f2 by the pair's normalisation scale, as the estimator's own frame is.  Results depend only
 * on a pair's data, its prior, its quality and opt, never on the batch around it or on the chunking; the float32 entry
 * points return the FP64 bytes.  A null init with n_pairs > 0 is RP_ERR_INVALID; every other check and error code is
 * the twin's, and so is rp_pair_status.  rp_last_timing slot [15] reports the prior stage. */
RP_API int rp_estimate_batch_host_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                       const double *x1, const double *x2, const double *d1, const double *d2,
                                       const float *quality, const double *cams, const rp_options *opt,
                                       const rp_model *init, rp_model *models, rp_stats *stats, uint8_t *masks);
RP_API int rp_estimate_batch_dev_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                      const double *x1, const double *x2, const double *d1, const double *d2,
                                      const float *quality, const double *cams, const rp_options *opt,
                                      const rp_model *init, rp_model *models, rp_stats *stats, uint8_t *masks,
                                      void *stream);
RP_API int rp_estimate_batch_host_f32_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                           const float *x1, const float *x2, const float *d1, const float *d2,
                                           const float *quality, const double *cams, const rp_options *opt,
                                           const rp_model *init, rp_model *models, rp_stats *stats, uint8_t *masks);
RP_API int rp_estimate_batch_dev_f32_init(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                          const float *x1, const float *x2, const float *d1, const float *d2,
                                          const float *quality, const double *cams, const rp_options *opt,
                                          const rp_model *init, rp_model *models, rp_stats *stats, uint8_t *masks,
                                          void *stream);

/* ---- refinement of caller-supplied models ----------------------------------------
 * What the estimator does after RANSAC, on start models the caller supplies (the previous frame pair's poses of a
 * tracker, another method's poses, an estimate to re-refine with other bundle options).  Pair p owns the
 * correspondences [offsets[p], offsets[p+1]) and starts from init[p]; subset (optional, [offsets[n_pairs]] bytes) selects
 * S_p = {correspondences with subset != 0}, a null subset means every correspondence.  For every pair the call:
 *   1. runs the P1/P2 pre-processing over ALL the pair's correspondences, as the estimator does: unprojected (calibrated)
 *      or normalised (focal variants) points, thr, scale_reproj and the final loss scale (calibrated: 0.5 * thr, the
 *      user's loss_scale ignored; focal: loss_scale / nscale);
 *   2. if |S_p| > 3: divides the focal variants' f1, f2 by nscale, runs the final refinement with the bundle fields of
 *      opt and opt->weight_sampson on S_p only, and multiplies f1, f2 by nscale again;
 *   3. RP_CALIB refines 7 parameters and holds shift1 / shift2 at their input values; RP_CALIB with opt->estimate_shift,
 *      or RP_CALIB_SHIFT, refines 9.  The focal variants hold the shifts too; the calibrated variants neither read nor
 *      change f1 / f2;
 *   4. a pair that is not refined (|S_p| <= 3, including pairs of fewer than 3 correspondences) returns init[p] byte for
 *      byte (no nscale round trip) and all-zero bundle stats;
 *   5. num_inliers / inliers (optional; both are computed when either is non-null): the refined model's get_inliers mask
 *      at the estimator's thr over all the pair's correspondences (Sampson + cheirality for the calibrated variants,
 *      Sampson only for the focal ones) and its count; all-zero and 0 for pairs of fewer than 3 correspondences.
 * A pair's results depend only on its own data, init[p], S_p and opt, never on the batch around it or on the chunking.
 * The float32 entry points return the FP64 entry points' bytes for the same values.  The calls change neither
 * rp_pair_status nor rp_last_timing, which keep describing the last estimate call.
 * Layouts of offsets, x1..d2 and cams are the estimator's; cams is ignored by the focal variants (may be NULL).
 * offsets and opt are HOST memory; for _host everything else is HOST memory, for _dev DEVICE memory, and _dev returns
 * after `stream` has finished.  bstats, num_inliers and inliers may be NULL; models may alias init.  Argument checks and
 * error codes are the estimator's, plus RP_ERR_INVALID for a null init or models with n_pairs > 0. */
RP_API int rp_refine_pairs_host(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                const double *x1, const double *x2, const double *d1, const double *d2,
                                const double *cams, const rp_options *opt, const rp_model *init,
                                const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                                int64_t *num_inliers, uint8_t *inliers);
RP_API int rp_refine_pairs_dev(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                               const double *x1, const double *x2, const double *d1, const double *d2,
                               const double *cams, const rp_options *opt, const rp_model *init,
                               const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                               int64_t *num_inliers, uint8_t *inliers, void *stream);
RP_API int rp_refine_pairs_host_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                    const float *x1, const float *x2, const float *d1, const float *d2,
                                    const double *cams, const rp_options *opt, const rp_model *init,
                                    const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                                    int64_t *num_inliers, uint8_t *inliers);
RP_API int rp_refine_pairs_dev_f32(rp_ctx *ctx, int variant, int64_t n_pairs, const int64_t *offsets,
                                   const float *x1, const float *x2, const float *d1, const float *d2,
                                   const double *cams, const rp_options *opt, const rp_model *init,
                                   const uint8_t *subset, rp_model *models, rp_bundle_stats *bstats,
                                   int64_t *num_inliers, uint8_t *inliers, void *stream);

/* ---- stage entry points (parity tests; all pointers HOST memory) -----------------
 * Each mirrors one exported stage of the reference binary (SURVEY.md §8a). */

/* R2: RandomSampler::generate_sample so@0x4f8970 — `iters` consecutive 3-samples out of n
 * points from `seed`; samples: [iters,3] int32. */
RP_API int rp_sample_batch(rp_ctx *ctx, int64_t n, uint64_t seed, int64_t iters, int32_t *samples);
/* the same with the sampler's PROSAC branch (initialize_prosac so@0x4f8a20): progressive_sampling != 0
 * draws from a growing prefix of the (quality-sorted) points for the first max_prosac_iterations-1 samples */
RP_API int rp_sample_batch_prosac(rp_ctx *ctx, int64_t n, uint64_t seed, int64_t iters, int32_t progressive_sampling,
                                  int64_t max_prosac_iterations, int32_t *samples);

/* The ordering step of the rp_estimate_batch_*_quality entry points on its own (no counterpart in the reference).  Pair p
 * owns [offsets[p], offsets[p+1]) of quality and perm (offsets non-decreasing, at most 2^24-1 correspondences per pair);
 * perm[offsets[p] + j] (int32, pair-local) is the index of the pair's j-th correspondence in (quality descending,
 * index ascending) order, with NaN taken as -inf and -0 as +0.  Pairs of up to RP_ORDER_SMEM_CAP correspondences are
 * sorted in shared memory, larger ones in global scratch (slower). */
#define RP_ORDER_SMEM_CAP 12288
RP_API int rp_order_by_quality(rp_ctx *ctx, int64_t n_pairs, const int64_t *offsets, const float *quality, int32_t *perm);

/* S1-S4: minimal solvers on n_problems independent triplets.  x1h,x2h: [n,3,3] homogeneous
 * (x,y,1) points, d1,d2: [n,3].  models: [n,4], counts: [n] (solutions per problem). */
RP_API int rp_solve_batch(rp_ctx *ctx, int variant, int64_t n_problems, const double *x1h, const double *x2h,
                          const double *d1, const double *d2, rp_model *models, int32_t *counts);

/* SC/SF/I1: compute_sampson_msac_score so@0x4f61d0 / so@0x4f65d0 for n_models models against
 * ONE pair's n_points normalised correspondences x1,x2: [n_points,2].  RP_CALIB*: pose scorer
 * (Sampson + cheirality); RP_SHARED/RP_VARYING: F = diag(1,1,f2) E diag(1,1,f1), Sampson only.
 * scores,counts: [n_models]; masks (optional, may be NULL): [n_models, n_points] get_inliers bytes. */
RP_API int rp_score_batch(rp_ctx *ctx, int variant, int64_t n_models, const rp_model *models, int64_t n_points,
                          const double *x1, const double *x2, double sq_threshold, double *scores,
                          int64_t *counts, uint8_t *masks);

/* L2: refine_monodepth_relpose so@0x261030 (+ shared so@0x2592e0, varying so@0x260fa0) for
 * n_models start models against ONE pair's correspondences (all points, uniform weights;
 * `mask` optional [n_points] selects a subset, as the final refinement does). */
RP_API int rp_refine_batch(rp_ctx *ctx, int variant, int64_t n_models, rp_model *models, int64_t n_points,
                           const double *x1, const double *x2, const double *d1, const double *d2,
                           const uint8_t *mask, double scale_reproj, double weight_sampson,
                           const rp_bundle_options *opt, rp_bundle_stats *stats);

/* ---- device-resident front end (SURVEY.md §8f item 2) --------------------------------------
 * What the reference's callers do on the host between the networks and the estimator
 * (/root/reference/make_pair.py:97-106): depth lookup at the matched keypoints,
 * depth_map[(int)y, (int)x], and removal of the rows whose two depths are both infinite.
 * All pointers are DEVICE memory: depth maps [h,w] float32, keypoints [n,2] float32 (x,y) as the
 * matcher produces them; outputs are the packed FP64 arrays rp_estimate_batch_dev takes
 * (capacity n rows), *n_out (host) the number of rows kept, order preserved.  Coordinates outside
 * the map are clamped to its border. */
RP_API int rp_gather_depths_dev(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                                const float *kp1, const float *kp2, int64_t n, double *x1, double *x2, double *d1,
                                double *d2, int64_t *n_out, void *stream);

/* The same recipe for a whole batch of pairs in one call (the reference's video demo runs it per frame pair,
 * /root/reference/make_video.py:270-290): depth maps of one size stacked [n_frames, h, w] (DEVICE), pair p reads frames
 * frame1[p] / frame2[p] (HOST index arrays) and owns the keypoint rows [in_offsets[p], in_offsets[p+1]) of kp1 / kp2
 * (DEVICE [N,2] float32; in_offsets HOST).  One CTA per pair compacts its rows; the call synchronises ONCE to return
 * out_offsets (HOST, [n_pairs+1]) — the packed offsets rp_estimate_batch_dev needs — and leaves x1, x2, d1, d2 (DEVICE,
 * capacity N rows) packed accordingly. */
RP_API int rp_gather_depths_batch_dev(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps,
                                      int n_frames, int h, int w, const int32_t *frame1, const int32_t *frame2,
                                      const float *kp1, const float *kp2, double *x1, double *x2, double *d1, double *d2,
                                      int64_t *out_offsets, void *stream);

/* The two gathers with float32 outputs x1, x2, d1, d2 (otherwise identical): what rp_estimate_batch_dev_f32 takes, so
 * that the chain matcher -> gather -> estimate never holds an FP64 copy of its inputs. */
RP_API int rp_gather_depths_dev_f32(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2, int w2,
                                    const float *kp1, const float *kp2, int64_t n, float *x1, float *x2, float *d1,
                                    float *d2, int64_t *n_out, void *stream);
RP_API int rp_gather_depths_batch_dev_f32(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets, const float *depth_maps,
                                          int n_frames, int h, int w, const int32_t *frame1, const int32_t *frame2,
                                          const float *kp1, const float *kp2, float *x1, float *x2, float *d1, float *d2,
                                          int64_t *out_offsets, void *stream);

/* The four gathers carrying one float32 match quality per keypoint row (LightGlue score, RoMa certainty, ...), so that the
 * quality of the rows they keep arrives packed next to them for rp_estimate_batch_dev[_f32]_quality: quality (DEVICE,
 * one value per input row) inserted after kp2 in the twin's argument list, quality_out (DEVICE, capacity as d1) after d2.
 * They are defined against their twin:
 *   - x1, x2, d1, d2 and *n_out / out_offsets are byte for byte the twin's for the same inputs;
 *   - quality_out is quality[keep], where keep is the twin's keep rule: input order, packed at the same offsets.  Each
 *     value is copied as its 32-bit pattern (NaN payloads, -0 and infinities unchanged); the keep rule never reads it.
 * For a non-empty input a null quality or quality_out is RP_ERR_INVALID; every other check and error code is the twin's,
 * and an empty input returns RP_OK with nothing written.  They synchronise as often as the twin (the batch: twice). */
RP_API int rp_gather_depths_dev_quality(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2,
                                        int w2, const float *kp1, const float *kp2, const float *quality, int64_t n,
                                        double *x1, double *x2, double *d1, double *d2, float *quality_out,
                                        int64_t *n_out, void *stream);
RP_API int rp_gather_depths_dev_f32_quality(rp_ctx *ctx, const float *depth1, int h1, int w1, const float *depth2, int h2,
                                            int w2, const float *kp1, const float *kp2, const float *quality, int64_t n,
                                            float *x1, float *x2, float *d1, float *d2, float *quality_out,
                                            int64_t *n_out, void *stream);
RP_API int rp_gather_depths_batch_dev_quality(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets,
                                              const float *depth_maps, int n_frames, int h, int w, const int32_t *frame1,
                                              const int32_t *frame2, const float *kp1, const float *kp2,
                                              const float *quality, double *x1, double *x2, double *d1, double *d2,
                                              float *quality_out, int64_t *out_offsets, void *stream);
RP_API int rp_gather_depths_batch_dev_f32_quality(rp_ctx *ctx, int64_t n_pairs, const int64_t *in_offsets,
                                                  const float *depth_maps, int n_frames, int h, int w,
                                                  const int32_t *frame1, const int32_t *frame2, const float *kp1,
                                                  const float *kp2, const float *quality, float *x1, float *x2, float *d1,
                                                  float *d2, float *quality_out, int64_t *out_offsets, void *stream);

/* ---- measurement helpers ---------------------------------------------------------
 * Pipe micro-benchmarks for the roofline denominators SURVEY.md §8d asks for (the driver's
 * MEASURED_PEAKS.json has only HBM and bf16): sustained FP64 and FP32 FMA throughput of
 * this device, in TFLOP/s (2 flops per FMA). */
RP_API int rp_measure_pipes(rp_ctx *ctx, double *fp64_tflops, double *fp32_tflops);

/* Stage entry point of the tensor-core tier (mdrp_b200/csrc/rp_tc.cuh; no counterpart in the reference: it only decides
 * which minimal models compute_sampson_msac_score so@0x4f61d0 / so@0x4f65d0 has to see at all).  For every model:
 * the number of correspondences that are CERTAIN outliers of the Sampson test r2 < sq_threshold, a rigorous lower
 * bound of N - inlier_count (== N for a model with a non-finite E / F).  x1 / x2 as in rp_score_batch; at most 4096
 * models per call. */
RP_API int rp_tc_count_batch(rp_ctx *ctx, int variant, int64_t n_models, const rp_model *models, int64_t n_points,
                             const double *x1, const double *x2, double sq_threshold, int64_t *certain_outliers);

/* status[p] (enum rp_pair_state) of every pair of the last rp_estimate_batch_* call on ctx.  One hard pair never fails
 * or slows down the rest of its batch: it is finished on its own and flagged here. */
RP_API int rp_pair_status(const rp_ctx *ctx, int64_t n_pairs, int32_t *status);

/* per-stage device time of the last rp_estimate_batch_* call on ctx, milliseconds (summed over chunks):
 * [0] prepare, [1] sample, [2] solve, [3] score(minimal: exact head + bound + prune + exact survivors),
 * [4] scan, [5] LO refine, [6] LO score+merge+final LO, [7] final refine, [8] total device, [9] H2D,
 * [10] D2H, [11] FP32 bound kernel alone, [12] tensor-core count tier alone, [13] widening of float32 inputs to FP64
 * (rp_estimate_batch_*_f32; 0 otherwise).  On the host path the widening runs on the copy stream after the H2D of [9],
 * and for every chunk but the first it overlaps the previous chunk's kernels, so [13] there also counts the time the
 * widening waits for SMs those kernels hold; the device path's [13] is the widening alone.  [14] ordering of a
 * rp_estimate_batch_*_quality call: sort, permuting gather (which also widens float32 inputs, so [13] is 0 for these
 * calls) and mask scatter; 0 for every other call.  On the host path the sort and gather run on the copy stream after
 * the H2D of [9], so [14] there carries the same caveat as [13].  [15] the prior stage of a rp_estimate_batch_*_init call
 * (import and exact scoring of the priors; its LO runs with the others in [5]), 0 for every other call.
 * counters: [0] minimal models generated, [1] point-scores the FP32 bound kernel resolved (models x correspondences),
 * [2] LM problems, [3] LM iterations, [4] chunks (= launches of each pipeline kernel), [5] minimal models
 * that needed the exact scorer, [6] point-scores the FP32 bound kernel actually evaluated (before abandoning),
 * [7] exact head size, [8] point-scores the tensor-core tier evaluated, [9] minimal models that tier passed on to the
 * FP32 bound kernel, [10] FP64 flops of the LM kernels (device counter), [11..15] reserved */
RP_API int rp_last_timing(const rp_ctx *ctx, double *ms16, int64_t *counters16);

#ifdef __cplusplus
}
#endif
#endif /* REPOSE_B200_H */
