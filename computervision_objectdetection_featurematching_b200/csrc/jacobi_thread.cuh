// jacobi_thread.cuh — one thread per 4-point hypothesis: the throughput form of HomographyEstimatorCallback::
// runKernel (normalised DLT + cv::eigen's Jacobi, SURVEY App. B.5 / D.2) for rounds that fill the chip.
//
// jacobi_warp.cuh spends ~360 warp instructions per rotation (90 per matrix with four matrices per warp), most of
// them the rotation's scalar chain replicated across lanes.  Here a thread owns a matrix, so a warp retires 32
// rotations with one pass of the rotation loop: 771 SASS instructions (tools/jacobi_sass_digest.py; ~220 of them are
// the five divisions and two square roots of the c/s chain).  What made the generic serial routine
// (homography_math.cuh, jacobi<9,S>) slow is removed: indR/indC live in two registers as packed nibbles (no local
// memory), every loop has static bounds with predicated bodies (no divergence inside a rotation), the two lines of a
// rotation come from a table of element indices (jt_lines) and need no predicate on any load or store, the refreshed
// row/column maxima are taken from the values the rotation has just produced (no re-reads), and the pivot search is a
// tournament that keeps the serial rule "first maximum wins".  The matrix state is 126 doubles per thread (strict
// upper triangle of A, V, W) plus one spare slot that stays 0, in shared memory, element-major (element e of thread t
// at e*S + t), so divergent element indices never conflict.
// Every element sees exactly the arithmetic of the serial code (same operands, same order, no FMA): results are
// bit-identical to jacobi<9> on finite input.  (With NaN in the matrix the pivot choice may differ, as in
// jacobi_warp.cuh.)  Compiles for the host too (tests/hostmath).
#pragma once
#include "homography_math.cuh"

namespace cvg {

constexpr int JT_A = 0;                 // 36 doubles: A[i][j], i < j, at JT_A + tri(i, j)
constexpr int JT_V = 36;                // 81 doubles: V row-major
constexpr int JT_W = 117;               //  9 doubles
constexpr int JT_SPARE = 126;            //  1 double, always 0: the diagonal of jt_lines
constexpr int JT_DOUBLES = 127;

// first element of row i in the packed strict upper triangle: 0, 8, 15, 21, 26, 30, 33, 35
CVG_HD constexpr int jt_off(int i) { return i * (17 - i) / 2; }
// OFFM(i) = jt_off(i) - i - 1: tri(i, j) = OFFM(i) + j for i < j
CVG_HD constexpr int jt_offm(int i) { return jt_off(i) - i - 1; }
CVG_HD int jt_offm_dyn(int i) { return i * (17 - i) / 2 - i - 1; }

// Line x of A: jt_lines.e[x][i] = the element index of A(x, i) = A(i, x) for i != x, JT_SPARE for i == x.  A rotation
// reads its two lines from this table instead of choosing between the row and the column form per element.  The table
// sits in global memory (432 B, served by L1): lanes of a warp index it with different x, which __constant__ serialises.
struct alignas(16) JtLines { int e[9][12]; };
CVG_HD constexpr JtLines jt_make_lines()
{
    JtLines t{};
    for (int x = 0; x < 9; x++)
        for (int i = 0; i < 9; i++)
            t.e[x][i] = i == x ? JT_SPARE : JT_A + (i < x ? jt_offm(i) + x : jt_offm(x) + i);
    return t;
}
#if defined(__CUDACC__)
__device__ const JtLines jt_lines_dev = jt_make_lines();
#endif
constexpr JtLines jt_lines_host = jt_make_lines();

CVG_HD void jt_line(int x, int (&e)[9])
{
#if defined(__CUDA_ARCH__)
    const int4* q = reinterpret_cast<const int4*>(jt_lines_dev.e[x]);
    const int4 a = __ldg(q), b = __ldg(q + 1);
    e[0] = a.x; e[1] = a.y; e[2] = a.z; e[3] = a.w; e[4] = b.x; e[5] = b.y; e[6] = b.z; e[7] = b.w;
    e[8] = __ldg(&jt_lines_dev.e[x][8]);
#else
    for (int i = 0; i < 9; i++) e[i] = jt_lines_host.e[x][i];
#endif
}

CVG_HD int jt_nib(uint32_t r, int i) { return (int)((r >> (4 * i)) & 15u); }
CVG_HD uint32_t jt_set(uint32_t r, int i, int v) { return (r & ~(15u << (4 * i))) | ((uint32_t)v << (4 * i)); }

// cv_hypot without the data-dependent branch (lanes of a warp hold different matrices): the same operations on
// the same operands as cv_hypot, selected instead of branched
CVG_HD double jt_hypot(double a, double b)
{
    a = fabs(a); b = fabs(b);
    const bool agb = a > b;
    const double hi = agb ? a : b, lo = agb ? b : a;
    if (!(hi > 0)) return 0;                      // a <= b and b == 0 (or NaN input, as cv_hypot)
    const double q = lo / hi;
    return hi * sqrt(1 + q * q);
}

// (val, key) tournament step on magnitudes: the right entry wins only when strictly larger — "first maximum wins"
#define CVG_JT_PICK(va, ka, vb, kb) do { if (fabs(va) < fabs(vb)) { (va) = (vb); (ka) = (kb); } } while (0)

// HomographyEstimatorCallback::runKernel for one 4-point sample, by one thread.  m: this thread's JT_DOUBLES
// elements with stride S.  `live` = the thread has a sample.  Returns false for "no model".  `any_active` must
// return whether any thread of the warp still iterates (device: a warp vote; host: the flag itself).
template <int S, class Vote>
CVG_HD bool run_kernel4_thread(const float* ms1, const float* ms2, double* H, double* m, bool live, Vote any_active)
{
    double cMx = 0, cMy = 0, cmx = 0, cmy = 0, sMx = 0, sMy = 0, smx = 0, smy = 0;
    #pragma unroll
    for (int i = 0; i < 4; i++) { cmx += ms2[2 * i]; cmy += ms2[2 * i + 1]; cMx += ms1[2 * i]; cMy += ms1[2 * i + 1]; }
    cmx /= 4; cmy /= 4; cMx /= 4; cMy /= 4;
    #pragma unroll
    for (int i = 0; i < 4; i++) {
        smx += fabs(ms2[2 * i] - cmx); smy += fabs(ms2[2 * i + 1] - cmy);
        sMx += fabs(ms1[2 * i] - cMx); sMy += fabs(ms1[2 * i + 1] - cMy);
    }
    const bool ok = live && !(fabs(smx) < DBL_EPSILON || fabs(smy) < DBL_EPSILON ||
                              fabs(sMx) < DBL_EPSILON || fabs(sMy) < DBL_EPSILON);
    uint32_t R = 0, C = 0;              // indR[i] at nibble i (i = 0..7); indC[i] at nibble i-1 (i = 1..8)
    if (ok) {
        smx = 4 / smx; smy = 4 / smy; sMx = 4 / sMx; sMy = 4 / sMy;
        // ---- LtL = sum over the four points of Lx Lx^T + Ly Ly^T, sequential over points (upper triangle) ----
        double Lx[4][9], Ly[4][9];
        #pragma unroll
        for (int i = 0; i < 4; i++) {
            const double x = (ms2[2 * i] - cmx) * smx, y = (ms2[2 * i + 1] - cmy) * smy;
            const double X = (ms1[2 * i] - cMx) * sMx, Y = (ms1[2 * i + 1] - cMy) * sMy;
            Lx[i][0] = X; Lx[i][1] = Y; Lx[i][2] = 1; Lx[i][3] = 0; Lx[i][4] = 0; Lx[i][5] = 0;
            Lx[i][6] = -x * X; Lx[i][7] = -x * Y; Lx[i][8] = -x;
            Ly[i][0] = 0; Ly[i][1] = 0; Ly[i][2] = 0; Ly[i][3] = X; Ly[i][4] = Y; Ly[i][5] = 1;
            Ly[i][6] = -y * X; Ly[i][7] = -y * Y; Ly[i][8] = -y;
        }
        #pragma unroll
        for (int j = 0; j < 9; j++) {
            #pragma unroll
            for (int k = j; k < 9; k++) {
                double s = 0;
                #pragma unroll
                for (int i = 0; i < 4; i++) s += Lx[i][j] * Lx[i][k] + Ly[i][j] * Ly[i][k];
                if (k == j) m[(JT_W + j) * S] = s;
                else m[(JT_A + jt_off(j) + (k - j - 1)) * S] = s;
            }
        }
        #pragma unroll
        for (int e = 0; e < 81; e++) m[(JT_V + e) * S] = (e / 9 == e % 9) ? 1.0 : 0.0;
        m[JT_SPARE * S] = 0;
        // ---- initial indR / indC (first maximum wins) ----
        #pragma unroll
        for (int k = 0; k < 8; k++) {
            int mi = k + 1; double mv = fabs(m[(JT_A + jt_off(k)) * S]);
            #pragma unroll
            for (int i = k + 2; i < 9; i++) {
                const double val = fabs(m[(JT_A + jt_off(k) + (i - k - 1)) * S]);
                if (mv < val) { mv = val; mi = i; }
            }
            R |= (uint32_t)mi << (4 * k);
        }
        #pragma unroll
        for (int k = 1; k < 9; k++) {
            int mi = 0; double mv = fabs(m[(JT_A + jt_off(0) + (k - 1)) * S]);
            #pragma unroll
            for (int i = 1; i < k; i++) {
                const double val = fabs(m[(JT_A + jt_off(i) + (k - i - 1)) * S]);
                if (mv < val) { mv = val; mi = i; }
            }
            C |= (uint32_t)mi << (4 * (k - 1));
        }
    }
    // ---- rotations ----
    bool done = !ok;
    for (int iters = 0; iters < 9 * 9 * 30; iters++) {
        int k = 0, l = 1;
        double p = 0, *pp = m;
        if (!done) {
            // pivot candidates in the serial scan order: rows 0..7 (k = i, l = indR[i]), then columns 1..8; signed,
            // so that the winner is the pivot p itself
            double v[16]; int key[16];
            #pragma unroll
            for (int i = 0; i < 8; i++) {
                v[i] = m[(JT_A + jt_offm(i) + jt_nib(R, i)) * S];
                key[i] = i;
            }
            #pragma unroll
            for (int i = 1; i < 9; i++) {
                const int ci = jt_nib(C, i - 1);
                v[7 + i] = m[(JT_A + jt_offm_dyn(ci) + i) * S];
                key[7 + i] = 7 + i;
            }
            #pragma unroll
            for (int w = 1; w < 16; w <<= 1)
                #pragma unroll
                for (int i = 0; i < 16; i += 2 * w) CVG_JT_PICK(v[i], key[i], v[i + w], key[i + w]);
            const int kk = key[0];
            if (kk < 8) { k = kk; l = jt_nib(R, kk); }
            else        { l = kk - 7; k = jt_nib(C, kk - 8); }
            pp = m + (JT_A + jt_offm_dyn(k) + l) * S;
            p = v[0];
            if (fabs(p) <= DBL_EPSILON) done = true;
        }
        if (!any_active(!done)) break;
        if (!done) {
            const double wk = m[(JT_W + k) * S], wl = m[(JT_W + l) * S];
            const double y = (wl - wk) * 0.5;
            double t = fabs(y) + jt_hypot(p, y);
            double s = jt_hypot(p, t);
            const double c = t / s;
            s = p / s; t = (p / t) * p;
            if (y < 0) { s = -s; t = -t; }
            // A: element pairs (line of k, line of l) for every index i.  The pairs at i == k and i == l are
            // (spare, A[k][l]) and (A[k][l], spare): both slots hold 0 and c > 0, so they rotate to +0 and stay 0 — the
            // serial code's A[k][l] = 0 — with no predicate on any load or store.  Every load comes before every store:
            // the compiler cannot tell these dynamic addresses apart and would keep a load after an earlier store.
            int ek[9], el[9];
            jt_line(k, ek);
            jt_line(l, el);
            *pp = 0;
            m[(JT_W + k) * S] = wk - t;
            m[(JT_W + l) * S] = wl + t;
            double a0[9], b0[9];
            #pragma unroll
            for (int i = 0; i < 9; i++) { a0[i] = m[ek[i] * S]; b0[i] = m[el[i] * S]; }
            // refreshed maxima, serial scans in ascending i: column of idx (i < idx), then row of idx (i > idx).  The
            // scans keep the signed value and compare magnitudes (the |.| folds into the compare).  A column scan starts
            // at its first element, i = 0 (unused when idx == 0).  A row scan starts at (0, idx + 1) instead of at its
            // first element, which is equivalent under "strictly larger wins" and lets it take i == idx, whose value is
            // 0.  A[k][l] = 0 belongs to row k and to column l, as in the serial code.  Static bounds: k <= 7, l >= 1.
            double na[9], nb[9];
            #pragma unroll
            for (int i = 0; i < 9; i++) {
                na[i] = a0[i] * c - b0[i] * s; nb[i] = a0[i] * s + b0[i] * c;
                m[ek[i] * S] = na[i];
                m[el[i] * S] = nb[i];
            }
            double mvCk = na[0], mvRk = 0, mvCl = nb[0], mvRl = 0;
            int mCk = 0, mRk = k + 1, mCl = 0, mRl = l + 1;
            #pragma unroll
            for (int i = 1; i < 9; i++) {
                const bool ck = i < k, cl = i < l;
                const bool tCk = i < 7 && ck && fabs(mvCk) < fabs(na[i]);
                const bool tRk = !ck && fabs(mvRk) < fabs(na[i]);
                const bool tCl = cl && fabs(mvCl) < fabs(nb[i]);
                const bool tRl = i > 1 && !cl && fabs(mvRl) < fabs(nb[i]);
                mvCk = tCk ? na[i] : mvCk; mCk = tCk ? i : mCk;
                mvRk = tRk ? na[i] : mvRk; mRk = tRk ? i : mRk;
                mvCl = tCl ? nb[i] : mvCl; mCl = tCl ? i : mCl;
                mvRl = tRl ? nb[i] : mvRl; mRl = tRl ? i : mRl;
            }
            {
                double* const vk = m + (JT_V + 9 * k) * S;
                double* const vl = m + (JT_V + 9 * l) * S;
                #pragma unroll
                for (int i = 0; i < 9; i++) {
                    const double a0 = vk[i * S], b0 = vl[i * S];
                    vk[i * S] = a0 * c - b0 * s;
                    vl[i * S] = a0 * s + b0 * c;
                }
            }
            if (k < 8) R = jt_set(R, k, mRk);
            if (l < 8) R = jt_set(R, l, mRl);
            if (k > 0) C = jt_set(C, k - 1, mCk);
            C = jt_set(C, l - 1, mCl);             // l >= 1
        }
    }
    if (!ok) return false;
    // ---- the eigenvector of the smallest eigenvalue: row of V that the descending selection sort puts last ----
    double w[9]; int id[9];
    #pragma unroll
    for (int i = 0; i < 9; i++) { w[i] = m[(JT_W + i) * S]; id[i] = i; }
    #pragma unroll
    for (int k = 0; k < 8; k++) {
        double wm = w[k]; int im = id[k], pos = k;
        #pragma unroll
        for (int i = k + 1; i < 9; i++)
            if (wm < w[i]) { wm = w[i]; im = id[i]; pos = i; }
        // swap (w[pos], id[pos]) <-> (w[k], id[k])
        #pragma unroll
        for (int i = k + 1; i < 9; i++)
            if (i == pos) { w[i] = w[k]; id[i] = id[k]; }
        w[k] = wm; id[k] = im;
    }
    const int row = id[8];
    double Vl[9];
    #pragma unroll
    for (int i = 0; i < 9; i++) Vl[i] = m[(JT_V + 9 * row + i) * S];
    const double invHnorm[9] = { 1. / smx, 0, cmx, 0, 1. / smy, cmy, 0, 0, 1 };
    const double Hnorm2[9] = { sMx, 0, -cMx * sMx, 0, sMy, -cMy * sMy, 0, 0, 1 };
    double Htemp[9], H0[9];
    mat3mul(invHnorm, Vl, Htemp);
    mat3mul(Htemp, Hnorm2, H0);
    const double sc = 1. / H0[8];
    #pragma unroll
    for (int i = 0; i < 9; i++) H[i] = H0[i] * sc;
    return true;
}

}  // namespace cvg
