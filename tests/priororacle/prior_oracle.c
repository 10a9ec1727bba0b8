/*
 * prior_oracle.c — the oracle's RANSAC and estimator started from a prior (TEST INFRASTRUCTURE ONLY).
 *
 * PoseLib 2.0.5 has no prior option, so this file defines what rp_estimate_batch_*_init computes, as twins of
 * ro_ransac / ro_estimate (oracle/repose_oracle.c, included unchanged so that every step is the oracle's own code):
 * before the first iteration score_models runs on the one-model list {prior}, with the in-loop LO when the prior
 * triggers, which a finite prior always does; the prior is not an iteration.  A NULL prior, or one with a non-finite
 * field the variant reads, gives ro_ransac's / ro_estimate's bytes (tests/test_prior_host.py checks that).
 * Built by tests/prior_oracle.py with the oracle's flags (-ffp-contract=off).
 */
#include "../../oracle/repose_oracle.c"

/* The in-loop LO's bookkeeping after a refinement: the refined model replaces the best one when its score is
 * strictly lower, then inlier_ratio and the dynamic iteration limit follow the best model. */
static void lo_update(const estimator *e, const ro_model *refined, ro_ransac_stats *stats, ro_model *best,
                      double *dyn_max_iter, double log_prob_missing) {
    size_t cnt = 0;
    const ro_ransac_opt *opt = e->opt;
    double rs = est_score(e, refined, &cnt);
    if (rs < stats->model_score) {
        stats->model_score = rs;
        stats->num_inliers = (int64_t)cnt;
        *best = *refined;
    }
    stats->inlier_ratio = (double)stats->num_inliers / (double)e->n;
    if (stats->inlier_ratio >= 0.9999) *dyn_max_iter = (double)opt->min_iterations;
    else if (stats->inlier_ratio <= 0.0001) *dyn_max_iter = (double)opt->max_iterations;
    else {
        const double prob_outlier = 1.0 - pow(stats->inlier_ratio, 3.0);
        *dyn_max_iter = ceil(log_prob_missing / log(prob_outlier) * opt->dyn_num_trials_mult);
    }
}

/* A prior model "means no prior" when a field the variant reads is not finite (the calibrated variants do not read
 * f1 / f2). */
static int prior_usable(int variant, const ro_model *m) {
    const double *v = (const double *)m;
    const int nf = variant == RO_CALIB || variant == RO_CALIB_SHIFT ? 10 : 12;
    for (int i = 0; i < nf; ++i)
        if (!isfinite(v[i])) return 0;
    return 1;
}

/* ro_ransac from a prior: before the first iteration score_models runs on the one-model list {prior} (in the
 * normalised frame the points are in), with the in-loop LO when it triggers, which a finite prior always does.  The
 * prior is not an iteration.  NULL, or a prior with a non-finite field the variant reads, is ro_ransac. */
RO_API void ro_ransac_prior(int variant, const double *x1, const double *x2, const double *d1, const double *d2,
                            size_t n, const ro_ransac_opt *opt, const ro_model *prior, ro_model *best,
                            ro_ransac_stats *stats, char *inliers) {
    estimator e;
    e.variant = variant; e.n = n; e.x1 = x1; e.x2 = x2; e.d1 = d1; e.d2 = d2; e.opt = opt;
    e.sq_thr = opt->max_epipolar_error * opt->max_epipolar_error;
    e.scale_reproj = opt->max_reproj_error > 0.0
                         ? (opt->max_epipolar_error * opt->max_epipolar_error) /
                               (opt->max_reproj_error * opt->max_reproj_error)
                         : 0.0;
    e.lo.max_iterations = 25; e.lo.loss_type = RO_LOSS_TRUNCATED;
    /* VaryingFocalMonodepthPoseEstimator::refine_model so@0x4fb0a0 never copies the threshold into its
     * BundleOptions: loss_scale stays at the struct default 1.0 (so@0x5232a0); the calibrated (so@0x4fa550)
     * and shared-focal (so@0x4fad60) estimators use opt.max_epipolar_error.  Reproduced as is. */
    e.lo.loss_scale = variant == RO_VARYING ? 1.0 : opt->max_epipolar_error;
    e.lo.gradient_tol = 1e-10; e.lo.step_tol = 1e-8; e.lo.initial_lambda = 1e-3;
    e.lo.min_lambda = 1e-10; e.lo.max_lambda = 1e10;

    model_init(best);
    stats->refinements = 0; stats->iterations = 0; stats->num_inliers = 0;
    stats->inlier_ratio = 0.0; stats->model_score = DBL_MAX;
    if (inliers) memset(inliers, 0, n);
    if (n < 3) return;
    ro_sampler_init(&e.sampler, n, 3, opt->seed, opt->progressive_sampling, (size_t)opt->max_prosac_iterations);

    size_t best_minimal_inliers = 0;
    double best_minimal_score = DBL_MAX;
    double dyn_max_iter = (double)opt->max_iterations;
    const double log_prob_missing = log(1.0 - opt->success_prob);
    ro_model models[8];
    size_t cnt = 0;
    if (prior && prior_usable(variant, prior)) {
        const double score = est_score(&e, prior, &cnt);
        if (cnt > best_minimal_inliers || score < best_minimal_score) {
            if (cnt > best_minimal_inliers) best_minimal_inliers = cnt;
            if (score < best_minimal_score) best_minimal_score = score;
            if (score < stats->model_score) {
                stats->model_score = score;
                *best = *prior;
                stats->num_inliers = (int64_t)cnt;
            }
            ro_model refined = *prior;
            est_refine(&e, &refined);
            stats->refinements++;
            lo_update(&e, &refined, stats, best, &dyn_max_iter, log_prob_missing);
        }
    }
    for (stats->iterations = 0; stats->iterations < opt->max_iterations; stats->iterations++) {
        if (stats->iterations > opt->min_iterations && (double)stats->iterations > dyn_max_iter) break;
        int nm = est_generate(&e, models);
        int best_idx = -1;
        for (int i = 0; i < nm; ++i) {
            double score = est_score(&e, &models[i], &cnt);
            int more = cnt > best_minimal_inliers;
            int better = score < best_minimal_score;
            if (more || better) {
                if (more) best_minimal_inliers = cnt;
                if (better) best_minimal_score = score;
                best_idx = i;
                if (score < stats->model_score) {
                    stats->model_score = score;
                    *best = models[i];
                    stats->num_inliers = (int64_t)cnt;
                }
            }
        }
        if (best_idx == -1) continue;
        ro_model refined = models[best_idx];
        est_refine(&e, &refined);
        stats->refinements++;
        lo_update(&e, &refined, stats, best, &dyn_max_iter, log_prob_missing);
    }
    /* final refinement: unlike the LO inside the loop it does NOT write stats.model_score (the reported score is
     * the one before this step) — seen on the binary: with no minimal model at all model_score stays DBL_MAX
     * while num_inliers / the model are taken from the refined identity, and one-iteration runs report the
     * pre-refinement score. */
    ro_model refined = *best;
    est_refine(&e, &refined);
    stats->refinements++;
    double rs = est_score(&e, &refined, &cnt);
    if (rs < stats->model_score) {
        stats->num_inliers = (int64_t)cnt;
        *best = refined;
    }
    stats->inlier_ratio = (double)stats->num_inliers / (double)n;
    free(e.sampler.growth);
    if (inliers) {
        if (variant == RO_CALIB || variant == RO_CALIB_SHIFT)
            ro_get_inliers_pose(best->q, best->t, x1, x2, n, e.sq_thr, inliers);
        else {
            double F[9];
            ro_fundamental_from_model(best, F);
            ro_get_inliers_F(F, x1, x2, n, e.sq_thr, inliers);
        }
    }
}


RO_API void ro_estimate_prior(int variant, const double *x1, const double *x2, const double *d1, const double *d2,
                              size_t n, const double *cam1, const double *cam2, const ro_ransac_opt *ropt,
                              const ro_bundle_opt *bopt, const ro_model *prior, ro_model *best,
                              ro_ransac_stats *stats, char *inliers) {
    double *a = (double *)malloc(sizeof(double) * (4 * n + 4));
    double *b = a + 2 * n;
    ro_ransac_opt ro = *ropt;
    ro_bundle_opt bo = *bopt;
    double nscale = 1.0;
    if (variant == RO_CALIB || variant == RO_CALIB_SHIFT) {
        for (size_t k = 0; k < n; ++k) {
            a[2 * k] = (x1[2 * k] - cam1[2]) / cam1[0];
            a[2 * k + 1] = (x1[2 * k + 1] - cam1[3]) / cam1[1];
            b[2 * k] = (x2[2 * k] - cam2[2]) / cam2[0];
            b[2 * k + 1] = (x2[2 * k + 1] - cam2[3]) / cam2[1];
        }
        const double fo1 = 0.5 * (cam1[0] + cam1[1]), fo2 = 0.5 * (cam2[0] + cam2[1]);
        const double k = 0.5 * (1.0 / fo1 + 1.0 / fo2);
        ro.max_epipolar_error = ropt->max_epipolar_error * k;
        ro.max_reproj_error = ropt->max_reproj_error * k;
        bo.loss_scale = 0.5 * ro.max_epipolar_error;
    } else {
        /* normalize_points so@0x4f6ae0: shared scale, no centroid */
        double s = 0.0;
        for (size_t k = 0; k < n; ++k) {
            s += sqrt(x1[2 * k] * x1[2 * k] + x1[2 * k + 1] * x1[2 * k + 1]);
            s += sqrt(x2[2 * k] * x2[2 * k] + x2[2 * k + 1] * x2[2 * k + 1]);
        }
        nscale = s / (sqrt(2.0) * (double)n);
        for (size_t k = 0; k < 2 * n; ++k) { a[k] = x1[k] / nscale; b[k] = x2[k] / nscale; }
        ro.max_epipolar_error = ropt->max_epipolar_error / nscale;
        ro.max_reproj_error = ropt->max_reproj_error / nscale;
        bo.loss_scale = bopt->loss_scale / nscale;
    }
    /* the prior in the normalised frame: the focal variants' f1, f2 divided by nscale, the rest as given */
    ro_model p0;
    if (prior) {
        p0 = *prior;
        if (variant == RO_SHARED || variant == RO_VARYING) { p0.f1 /= nscale; p0.f2 /= nscale; }
    }
    ro_ransac_prior(variant, a, b, d1, d2, n, &ro, prior ? &p0 : NULL, best, stats, inliers);
    if (stats->num_inliers > 3) {
        size_t m = 0;
        double *ia = (double *)malloc(sizeof(double) * (6 * n));
        double *ib = ia + 2 * n, *id1 = ia + 4 * n, *id2 = ia + 5 * n;
        for (size_t k = 0; k < n; ++k)
            if (inliers[k]) {
                ia[2 * m] = a[2 * k]; ia[2 * m + 1] = a[2 * k + 1];
                ib[2 * m] = b[2 * k]; ib[2 * m + 1] = b[2 * k + 1];
                id1[m] = d1[k]; id2[m] = d2[k];
                ++m;
            }
        const double sr = ro.max_reproj_error > 0.0
                              ? (ro.max_epipolar_error * ro.max_epipolar_error) /
                                    (ro.max_reproj_error * ro.max_reproj_error)
                              : 0.0;
        ro_refine(variant, ia, ib, id1, id2, m, best, sr, ropt->weight_sampson, &bo, NULL);
        free(ia);
    }
    if (variant == RO_SHARED || variant == RO_VARYING) {
        best->f1 *= nscale;
        best->f2 *= nscale;
    }
    free(a);
}

