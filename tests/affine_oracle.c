/*
 * affine_oracle.c — CPU restatement of cv::estimateAffine2D(method=RANSAC) as built in cv2 4.13.0 (calib3d/src/ptsetreg.cpp:
 * RANSACPointSetRegistrator::run with Affine2DEstimatorCallback, then LMSolver with Affine2DRefineCallback).  TEST
 * INFRASTRUCTURE ONLY, pinned to cv2 through tests/golden/golden_affine.npz.  It is built on the pinned pieces the CPU
 * oracle exports (oracle/cvoracle.h): the cv::RNG step, checkSubset (for three points: collinearity of both triples only),
 * RANSACUpdateNumIters and the 6-parameter LM refine.  Build with -ffp-contract=off (no FMA anywhere).
 */
#include "../oracle/cvoracle.h"
#include <stdlib.h>
#include <string.h>

/* Affine2DEstimatorCallback::runKernel: the closed-form fit of the first three correspondences, fp64 (never "no model") */
void aff_run_kernel(const float* from, const float* to, double M[6])
{
    double x1 = from[0], y1 = from[1], x2 = from[2], y2 = from[3], x3 = from[4], y3 = from[5];
    double X1 = to[0], Y1 = to[1], X2 = to[2], Y2 = to[3], X3 = to[4], Y3 = to[5];
    double d = 1. / (x1 * (y2 - y3) + x2 * (y3 - y1) + x3 * (y1 - y2));
    M[0] = d * (X1 * (y2 - y3) + X2 * (y3 - y1) + X3 * (y1 - y2));
    M[1] = d * (X1 * (x3 - x2) + X2 * (x1 - x3) + X3 * (x2 - x1));
    M[2] = d * (X1 * (x2 * y3 - x3 * y2) + X2 * (x3 * y1 - x1 * y3) + X3 * (x1 * y2 - x2 * y1));
    M[3] = d * (Y1 * (y2 - y3) + Y2 * (y3 - y1) + Y3 * (y1 - y2));
    M[4] = d * (Y1 * (x3 - x2) + Y2 * (x1 - x3) + Y3 * (x2 - x1));
    M[5] = d * (Y1 * (x2 * y3 - x3 * y2) + Y2 * (x3 * y1 - x1 * y3) + Y3 * (x1 * y2 - x2 * y1));
}

/* computeError: F = (float)M, a = F0 x + F1 y + F2 - X, b likewise, err = a a + b b, fp32 */
static void aff_compute_error(const float* src, const float* dst, int n, const double M[6], float* err)
{
    float F[6];
    for (int i = 0; i < 6; i++) F[i] = (float)M[i];
    for (int i = 0; i < n; i++) {
        float x = src[2 * i], y = src[2 * i + 1];
        float a = F[0] * x + F[1] * y + F[2] - dst[2 * i];
        float b = F[3] * x + F[4] * y + F[5] - dst[2 * i + 1];
        err[i] = a * a + b * b;
    }
}

/* getSubset with modelPoints = 3: distinct draws (redraw on a duplicate), checkSubset, up to max_attempts attempts */
static int aff_get_subset(const float* src, const float* dst, int n, uint64_t* rng, int max_attempts, float* ms1,
                          float* ms2, int64_t* draws)
{
    int idx[3];
    for (int it = 0; it < max_attempts; it++) {
        for (int i = 0; i < 3; i++) {
            int v, dup;
            do {
                v = (int)(cvo_rng_next(rng) % (uint32_t)n);
                (*draws)++;
                dup = 0;
                for (int k = 0; k < i; k++) dup |= idx[k] == v;
            } while (dup);
            idx[i] = v;
            ms1[2 * i] = src[2 * v]; ms1[2 * i + 1] = src[2 * v + 1];
            ms2[2 * i] = dst[2 * v]; ms2[2 * i + 1] = dst[2 * v + 1];
        }
        if (cvo_check_subset(ms1, ms2, 3)) return 1;
    }
    return 0;
}

/* cv::estimateAffine2D(src, dst, inliers, RANSAC, thr, max_iters, conf, refine_iters).  Returns 1 when a model was found
 * (M6 = the 2x3 matrix row-major), 0 when cv2 returns an empty matrix (M6 and mask zero), -1 for n = 0 (cv2 fails an
 * assertion).  The mask is the RANSAC-stage mask: the refine moves M, not the mask.  n = 3 returns the closed-form fit
 * with mask 1,1,1 and no refine (cv2 4.13.0 leaves that M unrefined).  M_ransac: the RANSAC-stage model; info: as for
 * cvo_ransac_stage (iterations run, best iteration and count, draws, LM return value, inliers refined). */
int aff_estimate(const float* src, const float* dst, int n, double thr, double conf, int max_iters, int refine_iters,
                 double M6[6], uint8_t* mask, double M_ransac[6], cvo_ransac_info* info)
{
    memset(info, 0, sizeof *info);
    info->best_iter = -1;
    memset(M6, 0, 6 * sizeof(double));
    memset(M_ransac, 0, 6 * sizeof(double));
    if (n <= 0) return -1;
    int niters = max_iters > 1 ? max_iters : 1;
    info->niters_final = niters;
    if (n < 3) { memset(mask, 0, n); return 0; }
    if (n == 3) {
        aff_run_kernel(src, dst, M6);
        memcpy(M_ransac, M6, 6 * sizeof(double));
        memset(mask, 1, 3);
        info->best_count = 3;
        return 1;
    }
    uint64_t rng = (uint64_t)-1;
    const float t = (float)(thr * thr);
    float* err = (float*)malloc(sizeof(float) * n);
    uint8_t* cur = (uint8_t*)malloc(n);
    int max_good = 0, iter;
    for (iter = 0; iter < niters; iter++) {
        float ms1[6], ms2[6];
        double M[6];
        if (!aff_get_subset(src, dst, n, &rng, 10000, ms1, ms2, &info->draws)) break;   /* iter == 0: no model */
        aff_run_kernel(ms1, ms2, M);
        aff_compute_error(src, dst, n, M, err);
        int good = 0;
        for (int i = 0; i < n; i++) { cur[i] = (uint8_t)(err[i] <= t); good += cur[i]; }
        if (good > (max_good > 2 ? max_good : 2)) {            /* good > MAX(maxGoodCount, modelPoints - 1) */
            memcpy(mask, cur, n);
            memcpy(M_ransac, M, sizeof M);
            max_good = good;
            info->best_iter = iter;
            niters = cvo_update_num_iters(conf, (double)(n - good) / n, 3, niters);
        }
    }
    info->iters_run = iter;
    info->niters_final = niters;
    info->best_count = max_good;
    free(err); free(cur);
    if (max_good <= 0) {
        memset(mask, 0, n);
        return 0;
    }
    memcpy(M6, M_ransac, 6 * sizeof(double));
    /* the refine runs on the inliers compressed in their original order */
    float* s1 = (float*)malloc(sizeof(float) * 2 * n);
    float* d1 = (float*)malloc(sizeof(float) * 2 * n);
    int np = 0;
    for (int i = 0; i < n; i++)
        if (mask[i]) {
            s1[2 * np] = src[2 * i]; s1[2 * np + 1] = src[2 * i + 1];
            d1[2 * np] = dst[2 * i]; d1[2 * np + 1] = dst[2 * i + 1];
            np++;
        }
    info->n_refit = np;
    if (refine_iters > 0 && np > 0) info->lm_iters = cvo_lm_refine_affine(s1, d1, np, M6, refine_iters);
    free(s1); free(d1);
    return 1;
}
