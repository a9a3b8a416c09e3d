/*
 * affine_partial_oracle.c — CPU restatement of cv::estimateAffinePartial2D(method=RANSAC) as built in cv2 4.13.0
 * (calib3d/src/ptsetreg.cpp: RANSACPointSetRegistrator::run with AffinePartial2DEstimatorCallback, then LMSolver with
 * AffinePartial2DRefineCallback).  TEST INFRASTRUCTURE ONLY, pinned to cv2 through tests/golden/golden_affine_partial.npz.
 * It is built on the pinned pieces the CPU oracle exports (oracle/cvoracle.h): the cv::RNG step, RANSACUpdateNumIters and
 * solve / invert(DECOMP_EIG).  LMSolverImpl::run and the summation orders it needs (cv::norm, cv::gemm, mulTransposed,
 * Mat::dot) are static inside the oracle, so they are restated here for four parameters, in the same order; the oracle
 * and the estimateAffine2D restatement stay as they were pinned.  Build with -ffp-contract=off (no FMA anywhere).
 */
#include "../oracle/cvoracle.h"
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* AffinePartial2DEstimatorCallback::runKernel: the closed-form similarity through the first two correspondences, fp64,
 * in OpenCV's operand order (never "no model": coincident source points give NaN) */
static void affp_run_kernel(const float* from, const float* to, double M[6])
{
    double x1 = from[0], y1 = from[1], x2 = from[2], y2 = from[3];
    double X1 = to[0], Y1 = to[1], X2 = to[2], Y2 = to[3];
    double d = 1. / ((x1 - x2) * (x1 - x2) + (y1 - y2) * (y1 - y2));
    double S0 = d * ((X1 - X2) * (x1 - x2) + (Y1 - Y2) * (y1 - y2));
    double S1 = d * ((Y1 - Y2) * (x1 - x2) - (X1 - X2) * (y1 - y2));
    double S2 = d * ((Y1 - Y2) * (x1 * y2 - x2 * y1) - (X1 * y2 - X2 * y1) * (y1 - y2) - (X1 * x2 - X2 * x1) * (x1 - x2));
    double S3 = d * (-(X1 - X2) * (x1 * y2 - x2 * y1) - (Y1 * x2 - Y2 * x1) * (x1 - x2) - (Y1 * y2 - Y2 * y1) * (y1 - y2));
    M[0] = S0; M[1] = -S1; M[2] = S2;
    M[3] = S1; M[4] = S0; M[5] = S3;
}

/* computeError (inherited from Affine2DEstimatorCallback): F = (float)M, a = F0 x + F1 y + F2 - X, b likewise, a a + b b */
static void affp_compute_error(const float* src, const float* dst, int n, const double M[6], float* err)
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

/* getSubset with modelPoints = 2: two distinct draws (redraw on a duplicate).  checkSubset is inherited from
 * Affine2DEstimatorCallback (haveCollinearPoints on both subsets), which tests no triple for two points: every attempt
 * passes, so the 10000-attempt limit is never reached. */
static void affp_get_subset(const float* src, const float* dst, int n, uint64_t* rng, float* ms1, float* ms2,
                            int64_t* draws)
{
    int idx[2];
    for (int i = 0; i < 2; i++) {
        int v, dup;
        do {
            v = (int)(cvo_rng_next(rng) % (uint32_t)n);
            (*draws)++;
            dup = i > 0 && idx[0] == v;
        } while (dup);
        idx[i] = v;
        ms1[2 * i] = src[2 * v]; ms1[2 * i + 1] = src[2 * v + 1];
        ms2[2 * i] = dst[2 * v]; ms2[2 * i + 1] = dst[2 * v + 1];
    }
}

/* ---- LMSolverImpl::run for AffinePartial2DRefineCallback (the orders of lm_run in oracle/cvoracle.c) ---------------- */
/* AffinePartial2DRefineCallback::compute: h = (a, b, tx, ty); rows (X, -Y, 1, 0) and (Y, X, 0, 1) */
static void affp_refine_compute(const float* M, const float* m, int n, const double* h, double* r, double* J)
{
    for (int i = 0; i < n; i++) {
        double Mx = M[2 * i], My = M[2 * i + 1];
        double xi = h[0] * Mx - h[1] * My + h[2];
        double yi = h[1] * Mx + h[0] * My + h[3];
        r[2 * i] = xi - m[2 * i];
        r[2 * i + 1] = yi - m[2 * i + 1];
        if (J) {
            double* Jp = J + 8 * i;
            Jp[0] = Mx; Jp[1] = -My; Jp[2] = 1.; Jp[3] = 0.;
            Jp[4] = My; Jp[5] = Mx; Jp[6] = 0.; Jp[7] = 1.;
        }
    }
}
/* cv::norm(r, NORM_L2SQR) for CV_64F (AVX2 dispatch): 4 lanes x 4 FMA accumulators over blocks of 16, then groups of 4
 * with separate multiply and in-order adds, then a scalar FMA tail */
static double norm_l2sqr(const double* a, int n)
{
    double acc[4][4];
    memset(acc, 0, sizeof acc);
    int j = 0;
    for (; j <= n - 16; j += 16)
        for (int k = 0; k < 4; k++)
            for (int l = 0; l < 4; l++) {
                double v = a[j + 4 * k + l];
                acc[k][l] = fma(v, v, acc[k][l]);
            }
    double r[4];
    for (int l = 0; l < 4; l++) r[l] = ((acc[0][l] + acc[1][l]) + acc[2][l]) + acc[3][l];
    double s = (r[0] + r[1]) + (r[2] + r[3]);
    s = 0.0 + s;
    for (; j <= n - 4; j += 4)
        for (int q = 0; q < 4; q++) s = s + a[j + q] * a[j + q];
    for (; j < n; j++) s = fma(a[j], a[j], s);
    return s;
}
/* cv::gemm inner product below 100 rows: 4 interleaved accumulators, ((s0+s1)+s2)+s3 */
static double dot4acc(const double* a, int sa, const double* b, int sb, int n)
{
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
    int k = 0;
    for (; k <= n - 4; k += 4) {
        s0 += a[(k) * sa] * b[(k) * sb];
        s1 += a[(k + 1) * sa] * b[(k + 1) * sb];
        s2 += a[(k + 2) * sa] * b[(k + 2) * sb];
        s3 += a[(k + 3) * sa] * b[(k + 3) * sb];
    }
    for (; k < n; k++) s0 += a[k * sa] * b[k * sb];
    return ((s0 + s1) + s2) + s3;
}
/* cv::Mat::dot generic path: unrolled by 4 */
static double dot_unrolled(const double* a, const double* b, int n)
{
    double r = 0;
    int i = 0;
    for (; i <= n - 4; i += 4)
        r += ((a[i] * b[i] + a[i + 1] * b[i + 1]) + a[i + 2] * b[i + 2]) + a[i + 3] * b[i + 3];
    for (; i < n; i++) r += a[i] * b[i];
    return r;
}
static double norm_inf(const double* r, int n)
{
    double s = 0;
    for (int i = 0; i < n; i++) { double a = fabs(r[i]); if (a > s) s = a; }
    return s;
}
/* A = J^T J (mulTransposed: sequential over rows), v = J^T r (gemm; sequential from 100 rows on, not pinned there) */
static void normal_eqs4(const double* J, const double* r, int rows, double* A, double* v)
{
    for (int i = 0; i < 4; i++) {
        for (int j = i; j < 4; j++) {
            double s = 0;
            for (int k = 0; k < rows; k++) s += J[k * 4 + i] * J[k * 4 + j];
            A[i * 4 + j] = s;
        }
        if (rows < 100) {
            v[i] = dot4acc(J + i, 4, r, 1, rows);
        } else {
            double s = 0;
            for (int k = 0; k < rows; k++) s += J[k * 4 + i] * r[k];
            v[i] = s;
        }
    }
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < i; j++) A[i * 4 + j] = A[j * 4 + i];
}
/* LMSolverImpl::run (Balda's LMFsolve schedule), eps = FLT_EPSILON, on (a, b, tx, ty) = x */
static int affp_lm_refine(const float* M, const float* m, int n, double x[4], int max_iters)
{
    const int rows = 2 * n;
    const double epsx = FLT_EPSILON, epsf = FLT_EPSILON;
    double xd[4], A[16], Ap[16], v[4], d[4], D[4], temp_d[4];
    double* r = (double*)malloc(sizeof(double) * rows);
    double* rd = (double*)malloc(sizeof(double) * rows);
    double* J = (double*)malloc(sizeof(double) * rows * 4);
    int i, iter = 0;

    affp_refine_compute(M, m, n, x, r, J);
    double S = norm_l2sqr(r, rows);
    normal_eqs4(J, r, rows, A, v);
    for (i = 0; i < 4; i++) D[i] = A[i * 4 + i];

    const double Rlo = 0.25, Rhi = 0.75;
    double lambda = 1, lc = 0.75;
    for (;;) {
        memcpy(Ap, A, sizeof A);
        for (i = 0; i < 4; i++) Ap[i * 4 + i] += lambda * D[i];
        cvo_solve_eig(Ap, v, d, 4);
        for (i = 0; i < 4; i++) xd[i] = x[i] - d[i];
        affp_refine_compute(M, m, n, xd, rd, NULL);
        double Sd = norm_l2sqr(rd, rows);
        for (i = 0; i < 4; i++) {                           /* temp_d = -A*d + 2*v ; dS = d . temp_d */
            double s = dot4acc(A + i * 4, 1, d, 1, 4);
            temp_d[i] = -1 * s + 2 * v[i];
        }
        double dS = dot_unrolled(d, temp_d, 4);
        double R = (S - Sd) / (fabs(dS) > DBL_EPSILON ? dS : 1);
        if (R > Rhi) {
            lambda *= 0.5;
            if (lambda < lc) lambda = 0;
        } else if (R < Rlo) {
            double t = dot_unrolled(d, v, 4);
            double nu = (Sd - S) / (fabs(t) > DBL_EPSILON ? t : 1) + 2;
            nu = nu > 2. ? nu : 2.;
            nu = nu < 10. ? nu : 10.;
            if (lambda == 0) {
                cvo_invert_eig(A, Ap, 4);
                double maxval = DBL_EPSILON;
                for (i = 0; i < 4; i++) {
                    double a = fabs(Ap[i * 4 + i]);
                    if (a > maxval) maxval = a;
                }
                lambda = lc = 1. / maxval;
                nu *= 0.5;
            }
            lambda *= nu;
        }
        if (Sd < S) {
            S = Sd;
            memcpy(x, xd, sizeof xd);
            affp_refine_compute(M, m, n, x, r, J);
            normal_eqs4(J, r, rows, A, v);
        }
        iter++;
        int proceed = iter < max_iters && norm_inf(d, 4) >= epsx && norm_inf(r, rows) >= epsf;
        if (!proceed) break;
    }
    free(r); free(rd); free(J);
    return iter == max_iters ? -iter : iter;
}

/* cv::estimateAffinePartial2D(src, dst, inliers, RANSAC, thr, max_iters, conf, refine_iters).  Returns 1 when a model
 * was found (M6 = the 2x3 matrix row-major), 0 when cv2 returns an empty matrix (M6 and mask zero), -1 for n = 0 (cv2
 * fails an assertion).  The mask is the RANSAC-stage mask: the refine moves M, not the mask.  n = 2 returns the closed
 * form with mask 1,1 and no refine (NaN when the source points coincide); n = 1 returns no model.  The refine runs on
 * (a, b, tx, ty) = (M00, M10, M02, M12) and rebuilds M as [a, -b, tx; b, a, ty].  M_ransac: the RANSAC-stage model;
 * info: as for cvo_ransac_stage (iterations run, best iteration and count, draws, LM return value, inliers refined). */
int affp_estimate(const float* src, const float* dst, int n, double thr, double conf, int max_iters, int refine_iters,
                  double M6[6], uint8_t* mask, double M_ransac[6], cvo_ransac_info* info)
{
    memset(info, 0, sizeof *info);
    info->best_iter = -1;
    memset(M6, 0, 6 * sizeof(double));
    memset(M_ransac, 0, 6 * sizeof(double));
    if (n <= 0) return -1;
    int niters = max_iters > 1 ? max_iters : 1;
    info->niters_final = niters;
    if (n < 2) { memset(mask, 0, n); return 0; }
    if (n == 2) {
        affp_run_kernel(src, dst, M6);
        memcpy(M_ransac, M6, 6 * sizeof(double));
        memset(mask, 1, 2);
        info->best_count = 2;
        return 1;
    }
    uint64_t rng = (uint64_t)-1;
    const float t = (float)(thr * thr);
    float* err = (float*)malloc(sizeof(float) * n);
    uint8_t* cur = (uint8_t*)malloc(n);
    int max_good = 0, iter;
    for (iter = 0; iter < niters; iter++) {
        float ms1[4], ms2[4];
        double M[6];
        affp_get_subset(src, dst, n, &rng, ms1, ms2, &info->draws);
        affp_run_kernel(ms1, ms2, M);
        affp_compute_error(src, dst, n, M, err);
        int good = 0;
        for (int i = 0; i < n; i++) { cur[i] = (uint8_t)(err[i] <= t); good += cur[i]; }
        if (good > (max_good > 1 ? max_good : 1)) {            /* good > MAX(maxGoodCount, modelPoints - 1) */
            memcpy(mask, cur, n);
            memcpy(M_ransac, M, sizeof M);
            max_good = good;
            info->best_iter = iter;
            niters = cvo_update_num_iters(conf, (double)(n - good) / n, 2, niters);
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
    if (refine_iters > 0 && np > 0) {
        double p4[4] = { M6[0], M6[3], M6[2], M6[5] };
        info->lm_iters = affp_lm_refine(s1, d1, np, p4, refine_iters);
        M6[0] = M6[4] = p4[0];
        M6[1] = -p4[1];
        M6[2] = p4[2];
        M6[3] = p4[1];
        M6[5] = p4[3];
    }
    free(s1); free(d1);
    return 1;
}
