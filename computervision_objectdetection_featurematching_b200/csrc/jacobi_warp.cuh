// jacobi_warp.cuh — warp-cooperative, bit-exact equivalents of the 9x9 routines in homography_math.cuh.
//
// cv::eigen's Jacobi (SURVEY App. D.2) is a serial chain of ~135 rotations per 9x9 matrix; a single
// thread spends ~6000 cycles per rotation on dependent shared-memory accesses.  Here one warp runs one
// matrix: the 16 element-pairs of a rotation are rotated one per lane, the pivot search and the four
// indR/indC refreshes run redundantly in every lane as register tournaments over broadcast loads, and
// the rotation's scalar chain (two hypot, three divisions) is the only serial part.  Every element sees
// exactly the arithmetic of the serial code (same operands, same
// order, no FMA), and every argmax keeps the serial rule "first maximum wins", so results are
// bit-identical to jacobi<9>.  All 32 lanes must call; A, W, V live in warp-private shared memory.
// (Matrices containing NaN may pick different pivots than the serial scan; finite data cannot.)
#pragma once
#include "homography_math.cuh"

namespace cvg {

__device__ __forceinline__ double shfl_d(double v, int src)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_sync(0xffffffffu, lo, src);
    hi = __shfl_sync(0xffffffffu, hi, src);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_xor_d(double v, int m)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_xor_sync(0xffffffffu, lo, m);
    hi = __shfl_xor_sync(0xffffffffu, hi, m);
    return __hiloint2double(hi, lo);
}

// (Measured and rejected, against the earlier 16-lane shuffle argmax of the pivot: two redux.sync integer maxima over the
// hi / lo words of the non-negative doubles plus a ballot instead of the shuffle rounds — verify stage 2.65 -> 3.14 ms per
// 64 pairs, real dataset 365 -> 399 ms.)

// One step of a "first maximum wins" tournament: (v1, i1) comes later in the serial scan order than (v0, i0) and wins only
// if it is strictly larger, as `if (mv < val)` does.  A tree of these over candidates in scan order picks the serial scan's
// answer (for finite values).
__device__ __forceinline__ void later_wins_if_larger(double& v0, int& i0, double v1, int i1)
{
    const bool take = v0 < v1;
    v0 = take ? v1 : v0;
    i0 = take ? i1 : i0;
}

// Serial row scan of jacobi<9> (indR[idx], idx < 8): argmax of |A[idx][i]| over i = idx+1 .. 8, first maximum wins.  Reads
// all of row idx (in bounds for any idx <= 8) and disqualifies i <= idx with -1, which loses to every real candidate.
__device__ __forceinline__ int row_argmax9(const double* A, int idx)
{
    double v[8]; int m[8];
    #pragma unroll
    for (int i = 1; i < 9; i++) { const double a = fabs(A[9 * idx + i]); v[i - 1] = i > idx ? a : -1.0; m[i - 1] = i; }
    #pragma unroll
    for (int w = 1; w < 8; w *= 2)
        #pragma unroll
        for (int q = 0; q < 8; q += 2 * w) later_wins_if_larger(v[q], m[q], v[q + w], m[q + w]);
    return m[0];
}

// Serial column scan of jacobi<9> (indC[idx], idx >= 1): argmax of |A[i][idx]| over i = 0 .. idx-1, first maximum wins.
// The disqualified i >= idx come last in the order, so -1 never wins there either.
__device__ __forceinline__ int col_argmax9(const double* A, int idx)
{
    double v[8]; int m[8];
    #pragma unroll
    for (int i = 0; i < 8; i++) { const double a = fabs(A[9 * i + idx]); v[i] = i < idx ? a : -1.0; m[i] = i; }
    #pragma unroll
    for (int w = 1; w < 8; w *= 2)
        #pragma unroll
        for (int q = 0; q < 8; q += 2 * w) later_wins_if_larger(v[q], m[q], v[q + w], m[q + w]);
    return m[0];
}

// cv_hypot without branches: the larger magnitude divides the smaller, as in whichever branch cv_hypot takes, so the result
// is the same double.  Both magnitudes zero: the quotient is NaN and is not selected.
__device__ __forceinline__ double cv_hypot_sel(double a, double b)
{
    a = fabs(a); b = fabs(b);
    const bool a_big = a > b;
    const double hi = a_big ? a : b, lo = a_big ? b : a;
    const double r = lo / hi;
    const double h = hi * sqrt(1 + r * r);
    return hi > 0 ? h : 0.0;
}

// A: 81 doubles (upper triangle significant, destroyed), W: 9, V: 81 — all in shared memory.
// Every lane runs the pivot search and the four refreshed scans itself, on broadcast loads of the same shared-memory
// values, so none of them waits on a shuffle: indR / indC live in every lane as nibbles (R: indR[i] at bits 4i, i < 8;
// C: indC[i] at bits 4(i-1), 1 <= i < 9), and every lane arrives at the same k, l.  The serial scans' order and their
// strict comparisons are kept, so the pivots and the bits are jacobi<9>'s.
// Returns the number of rotations.
__device__ __noinline__ int jacobi9_warp(double* A, double* W, double* V)
{
    const int lane = threadIdx.x & 31;
    const double eps = DBL_EPSILON;
    for (int e = lane; e < 81; e += 32) V[e] = (e / 9 == e % 9) ? 1.0 : 0.0;
    if (lane < 9) W[lane] = A[10 * lane];
    uint32_t R = 0, C = 0;
    #pragma unroll
    for (int i = 0; i < 8; i++) {
        R |= (uint32_t)row_argmax9(A, i) << (4 * i);
        C |= (uint32_t)col_argmax9(A, i + 1) << (4 * i);
    }
    __syncwarp();
    int iters = 0;
    for (; iters < 9 * 9 * 30; iters++) {
        // ---- pivot: candidates in the serial scan order: rows 0..7 (k=i, l=indR[i]), then columns 1..8 (k=indC[i], l=i)
        double cv[16]; int ci[16];
        #pragma unroll
        for (int i = 0; i < 8; i++) {
            cv[i] = fabs(A[9 * i + ((R >> (4 * i)) & 15)]);
            cv[8 + i] = fabs(A[9 * ((C >> (4 * i)) & 15) + (i + 1)]);
            ci[i] = i; ci[8 + i] = 8 + i;
        }
        #pragma unroll
        for (int w = 1; w < 16; w *= 2)
            #pragma unroll
            for (int q = 0; q < 16; q += 2 * w) later_wins_if_larger(cv[q], ci[q], cv[q + w], ci[q + w]);
        const int key = ci[0];
        const int k = key < 8 ? key : (int)((C >> (4 * (key - 8))) & 15);
        const int l = key < 8 ? (int)((R >> (4 * key)) & 15) : key - 7;
        const double p = A[9 * k + l];
        if (fabs(p) <= eps) break;
        const double y = (W[l] - W[k]) * 0.5;
        double t = fabs(y) + cv_hypot_sel(p, y);
        double s = cv_hypot_sel(p, t);
        const double pt = p / t;
        const double c = t / s;
        s = p / s; t = pt * p;
        if (y < 0) { s = -s; t = -t; }
        __syncwarp();
        if (lane == 0) { A[9 * k + l] = 0; W[k] -= t; W[l] += t; }
        // ---- rotations: lanes 0..8 -> A element pair of index i = lane; lanes 16..24 -> V pair of column i = lane-16
        {
            double* a = nullptr; double* b = nullptr;
            if (lane < 9) {
                const int i = lane;
                if (i < k)                { a = &A[9 * i + k]; b = &A[9 * i + l]; }
                else if (i > k && i < l)  { a = &A[9 * k + i]; b = &A[9 * i + l]; }
                else if (i > l)           { a = &A[9 * k + i]; b = &A[9 * l + i]; }
            } else if (lane >= 16 && lane < 25) {
                const int i = lane - 16;
                a = &V[9 * k + i]; b = &V[9 * l + i];
            }
            if (a) {
                const double a0 = *a, b0 = *b;
                *a = a0 * c - b0 * s;
                *b = a0 * s + b0 * c;
            }
        }
        __syncwarp();
        // ---- refresh indR[k], indR[l], indC[k], indC[l] (k < l, so k < 8 and l >= 1 always)
        {
            const uint32_t rk = row_argmax9(A, k), rl = row_argmax9(A, l);
            const uint32_t ck = col_argmax9(A, k), cl = col_argmax9(A, l);
            R = (R & ~(15u << (4 * k))) | (rk << (4 * k));
            if (l < 8) R = (R & ~(15u << (4 * l))) | (rl << (4 * l));
            if (k > 0) C = (C & ~(15u << (4 * (k - 1)))) | (ck << (4 * (k - 1)));
            C = (C & ~(15u << (4 * (l - 1)))) | (cl << (4 * (l - 1)));
        }
    }
    __syncwarp();
    // ---- selection sort, descending, rows of V follow
    for (int k = 0; k < 8; k++) {
        double val = (lane >= k && lane < 9) ? W[lane] : -INFINITY;
        int m = lane;
        // first maximum wins: `if (W[m] < W[i]) m = i` keeps the earliest of equal values
        #pragma unroll
        for (int d = 8; d > 0; d >>= 1) {
            const double ov = shfl_xor_d(val, d);
            const int om = __shfl_xor_sync(0xffffffffu, m, d);
            if (ov > val || (ov == val && om < m)) { val = ov; m = om; }
        }
        m = __shfl_sync(0xffffffffu, m, 0);
        if (m != k) {
            if (lane == 0) { const double tmp = W[m]; W[m] = W[k]; W[k] = tmp; }
            if (lane < 9) { const double tmp = V[9 * m + lane]; V[9 * m + lane] = V[9 * k + lane]; V[9 * k + lane] = tmp; }
        }
        __syncwarp();
    }
    return iters;
}

// cv::solve(A, b, x, DECOMP_EIG) for 9x9 (see solve_eig<9>): A, b read-only (any memory), x out (9, shared);
// a, v: 81-double shared scratch, w: 9-double shared scratch.  Result visible to the warp after return.  Returns the
// number of rotations.
__device__ __forceinline__ int solve_eig9_warp(const double* A, const double* b, double* x, double* a, double* v, double* w)
{
    const int lane = threadIdx.x & 31;
    for (int e = lane; e < 81; e += 32) a[e] = A[e];
    __syncwarp();
    const int rotations = jacobi9_warp(a, w, v);
    if (lane == 0) {
        double threshold = 0;
        for (int i = 0; i < 9; i++) x[i] = 0;
        for (int i = 0; i < 9; i++) threshold += w[i];
        threshold *= DBL_EPSILON * 2;
        for (int i = 0; i < 9; i++) {
            double wi = w[i];
            if (fabs(wi) <= threshold) continue;
            wi = 1 / wi;
            double s = 0;
            for (int j = 0; j < 9; j++) s += v[i * 9 + j] * b[j];
            s *= wi;
            for (int j = 0; j < 9; j++) x[j] = x[j] + s * v[i * 9 + j];
        }
    }
    __syncwarp();
    return rotations;
}

// max |diag(cv::invert(A, DECOMP_EIG))| for 9x9 (see invert_eig_max_diag<9>); result in every lane.  *rotations (if given):
// the number of rotations.
__device__ __forceinline__ double invert_eig_max_diag9_warp(const double* A, double* a, double* v, double* w,
                                                           int* rotations = nullptr)
{
    const int lane = threadIdx.x & 31;
    for (int e = lane; e < 81; e += 32) a[e] = A[e];
    __syncwarp();
    const int rot = jacobi9_warp(a, w, v);
    if (rotations) *rotations = rot;
    double maxval = DBL_EPSILON;
    if (lane == 0) {
        double dg[9];
        double threshold = 0;
        for (int i = 0; i < 9; i++) { dg[i] = 0; threshold += w[i]; }
        threshold *= DBL_EPSILON * 2;
        for (int k = 0; k < 9; k++) {
            double wi = w[k];
            if (fabs(wi) <= threshold) continue;
            wi = 1 / wi;
            for (int i = 0; i < 9; i++) {
                const double buf = v[k * 9 + i] * wi;
                dg[i] = dg[i] + v[k * 9 + i] * buf;
            }
        }
        for (int i = 0; i < 9; i++) { const double q = fabs(dg[i]); if (q > maxval) maxval = q; }
    }
    return shfl_d(maxval, 0);
}

// HomographyEstimatorCallback::runKernel for a 4-point sample, one warp (see run_kernel_seq).
// ms1/ms2: the sample (same values in every lane).  smem: >= 81+81+9+72 doubles of warp-private scratch.
// Returns false for "no model"; H (9 doubles) valid in every lane.
__device__ __forceinline__ bool run_kernel4_warp(const float* ms1, const float* ms2, double* H, double* smem)
{
    const int lane = threadIdx.x & 31;
    double* LtL = smem; double* V = smem + 81; double* W = smem + 162; double* L = smem + 171;   // L: [4][2][9]
    double cMx = 0, cMy = 0, cmx = 0, cmy = 0, sMx = 0, sMy = 0, smx = 0, smy = 0;
    #pragma unroll
    for (int i = 0; i < 4; i++) { cmx += ms2[2 * i]; cmy += ms2[2 * i + 1]; cMx += ms1[2 * i]; cMy += ms1[2 * i + 1]; }
    cmx /= 4; cmy /= 4; cMx /= 4; cMy /= 4;
    #pragma unroll
    for (int i = 0; i < 4; i++) {
        smx += fabs(ms2[2 * i] - cmx); smy += fabs(ms2[2 * i + 1] - cmy);
        sMx += fabs(ms1[2 * i] - cMx); sMy += fabs(ms1[2 * i + 1] - cMy);
    }
    if (fabs(smx) < DBL_EPSILON || fabs(smy) < DBL_EPSILON || fabs(sMx) < DBL_EPSILON || fabs(sMy) < DBL_EPSILON)
        return false;
    smx = 4 / smx; smy = 4 / smy; sMx = 4 / sMx; sMy = 4 / sMy;
    if (lane < 4) {
        const int i = lane;
        const double x = (ms2[2 * i] - cmx) * smx, y = (ms2[2 * i + 1] - cmy) * smy;
        const double X = (ms1[2 * i] - cMx) * sMx, Y = (ms1[2 * i + 1] - cMy) * sMy;
        double* Lx = L + i * 18; double* Ly = Lx + 9;
        Lx[0] = X; Lx[1] = Y; Lx[2] = 1; Lx[3] = 0; Lx[4] = 0; Lx[5] = 0; Lx[6] = -x * X; Lx[7] = -x * Y; Lx[8] = -x;
        Ly[0] = 0; Ly[1] = 0; Ly[2] = 0; Ly[3] = X; Ly[4] = Y; Ly[5] = 1; Ly[6] = -y * X; Ly[7] = -y * Y; Ly[8] = -y;
    }
    __syncwarp();
    for (int e = lane; e < 81; e += 32) {
        int j = e / 9, k = e % 9;
        if (k < j) { const int tmp = j; j = k; k = tmp; }            // completeSymm: lower = upper
        double s = 0;
        #pragma unroll
        for (int i = 0; i < 4; i++) {
            const double* Lx = L + i * 18; const double* Ly = Lx + 9;
            s += Lx[j] * Lx[k] + Ly[j] * Ly[k];
        }
        LtL[e] = s;
    }
    __syncwarp();
    jacobi9_warp(LtL, W, V);
    const double invHnorm[9] = { 1. / smx, 0, cmx, 0, 1. / smy, cmy, 0, 0, 1 };
    const double Hnorm2[9] = { sMx, 0, -cMx * sMx, 0, sMy, -cMy * sMy, 0, 0, 1 };
    double Vl[9], Htemp[9], H0[9];
    #pragma unroll
    for (int i = 0; i < 9; i++) Vl[i] = V[72 + i];
    mat3mul(invHnorm, Vl, Htemp);
    mat3mul(Htemp, Hnorm2, H0);
    const double sc = 1. / H0[8];
    #pragma unroll
    for (int i = 0; i < 9; i++) H[i] = H0[i] * sc;
    __syncwarp();
    return true;
}


// ---------------------------------------------------------------------------------------------------
// 8-lane groups: four matrices per warp share one instruction stream.  The scalar chain of a rotation
// (five divisions, two square roots — ~230 of the ~360 warp instructions of jacobi9_warp) then serves
// four matrices at once, which is what matters when the chip is full of hypotheses (issue-bound) rather
// than waiting on one matrix (latency-bound, jacobi9_warp).  Lane = 8*g + j; every group owns its A, W,
// V in shared memory.  `live` is group-uniform; groups that converged (or never had a matrix) idle
// through the remaining rotations of their warp.  Bit-identical to jacobi<9>.
__device__ __forceinline__ void g8_argmax_first(double& val, int& key)
{
    #pragma unroll
    for (int m = 4; m > 0; m >>= 1) {
        const double ov = shfl_xor_d(val, m);
        const int ok = __shfl_xor_sync(0xffffffffu, key, m);
        if (ov > val || (ov == val && ok < key)) { val = ov; key = ok; }
    }
}

__device__ __forceinline__ void g8_rot_a(double* A, int i, int k, int l, double c, double s)
{
    double* a; double* b;
    if (i < k)      { a = &A[9 * i + k]; b = &A[9 * i + l]; }
    else if (i < l) { if (i == k) return; a = &A[9 * k + i]; b = &A[9 * i + l]; }
    else            { if (i == l) return; a = &A[9 * k + i]; b = &A[9 * l + i]; }
    const double a0 = *a, b0 = *b;
    *a = a0 * c - b0 * s;
    *b = a0 * s + b0 * c;
}

__device__ __forceinline__ void g8_rot_v(double* V, int i, int k, int l, double c, double s)
{
    double* a = &V[9 * k + i]; double* b = &V[9 * l + i];
    const double a0 = *a, b0 = *b;
    *a = a0 * c - b0 * s;
    *b = a0 * s + b0 * c;
}

__device__ __noinline__ void jacobi9_g8(double* A, double* W, double* V, bool live)
{
    const int lane = threadIdx.x & 31, j = lane & 7;
    const double eps = DBL_EPSILON;
    int myR = 0, myC = 0;          // lane j holds indR[j] (rows 0..7) and indC[j+1] (columns 1..8)
    if (live) {
        for (int e = j; e < 81; e += 8) V[e] = (e / 9 == e % 9) ? 1.0 : 0.0;
        W[j] = A[10 * j];
        if (j == 0) W[8] = A[80];
        {
            int m = j + 1; double mv = fabs(A[9 * j + m]);
            for (int i = j + 2; i < 9; i++) { const double val = fabs(A[9 * j + i]); if (mv < val) { mv = val; m = i; } }
            myR = m;
        }
        {
            const int cc = j + 1; int m = 0; double mv = fabs(A[cc]);
            for (int i = 1; i < cc; i++) { const double val = fabs(A[9 * i + cc]); if (mv < val) { mv = val; m = i; } }
            myC = m;
        }
    }
    __syncwarp();
    bool done = !live;
    for (int iters = 0; iters < 9 * 9 * 30; iters++) {
        // ---- pivot: serial scan order = rows 0..7 (order index j), then columns 1..8 (order index 8 + j)
        double val = -1.0; int key = j;
        if (!done) {
            const double va = fabs(A[9 * j + myR]), vb = fabs(A[9 * myC + (j + 1)]);
            val = va;
            if (vb > va) { val = vb; key = 8 + j; }
        }
        g8_argmax_first(val, key);
        const int src = (lane & ~7) | (key & 7);
        const bool is_col = key >= 8;
        const int k = __shfl_sync(0xffffffffu, is_col ? myC : j, src);
        const int l = __shfl_sync(0xffffffffu, is_col ? j + 1 : myR, src);
        double p = 0;
        if (!done) { p = A[9 * k + l]; if (fabs(p) <= eps) done = true; }
        if (__all_sync(0xffffffffu, done)) break;
        double c = 0, s = 0, t = 0;
        if (!done) {
            const double y = (W[l] - W[k]) * 0.5;
            t = fabs(y) + cv_hypot(p, y);
            s = cv_hypot(p, t);
            c = t / s;
            s = p / s; t = (p / t) * p;
            if (y < 0) { s = -s; t = -t; }
        }
        __syncwarp();
        if (!done) {
            if (j == 0) { A[9 * k + l] = 0; W[k] -= t; W[l] += t; }
            g8_rot_a(A, j, k, l, c, s);
            g8_rot_v(V, j, k, l, c, s);
            if (j == 0) g8_rot_a(A, 8, k, l, c, s);
            if (j == 1) g8_rot_v(V, 8, k, l, c, s);
        }
        __syncwarp();
        // ---- refresh indR[k], indR[l], indC[k], indC[l]
        int r[4];
        #pragma unroll
        for (int q = 0; q < 4; q++) {
            const int idx = (q & 1) ? l : k;
            double v2 = -1.0; int cand = 99;
            if (!done) {
                if (q < 2) { const int i = idx + 1 + j; if (i < 9) { v2 = fabs(A[9 * idx + i]); cand = i; } }
                else       { const int i = j;           if (i < idx) { v2 = fabs(A[9 * i + idx]); cand = i; } }
            }
            g8_argmax_first(v2, cand);
            r[q] = cand;
        }
        if (!done) {
            if (j == k) myR = r[0];                    // k < l <= 8, so row k always has an indR
            if (j == l && l < 8) myR = r[1];
            if (k > 0 && j == k - 1) myC = r[2];
            if (j == l - 1) myC = r[3];                // l >= 1
        }
    }
    __syncwarp();
    // ---- selection sort, descending, rows of V follow
    for (int k = 0; k < 8; k++) {
        double val = -INFINITY; int m = 99;
        if (live) {
            if (j >= k) { val = W[j]; m = j; }
            if (j == 7) { const double w8 = W[8]; if (w8 > val) { val = w8; m = 8; } }
        }
        g8_argmax_first(val, m);
        if (live && m != k) {
            if (j == 0) { const double tmp = W[m]; W[m] = W[k]; W[k] = tmp; }
            { const double tmp = V[9 * m + j]; V[9 * m + j] = V[9 * k + j]; V[9 * k + j] = tmp; }
            if (j == 1) { const double tmp = V[9 * m + 8]; V[9 * m + 8] = V[9 * k + 8]; V[9 * k + 8] = tmp; }
        }
        __syncwarp();
    }
}

// runKernel for a 4-point sample by one 8-lane group (see run_kernel4_warp).  smem: this group's 243 doubles.
// Returns the group's verdict; H valid in every lane of a group that returned true.
__device__ __forceinline__ bool run_kernel4_g8(const float* ms1, const float* ms2, double* H, double* smem, bool live)
{
    const int j = threadIdx.x & 7;
    double* LtL = smem; double* V = smem + 81; double* W = smem + 162; double* L = smem + 171;   // L: [4][2][9]
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
    if (ok) {
        smx = 4 / smx; smy = 4 / smy; sMx = 4 / sMx; sMy = 4 / sMy;
        if (j < 4) {
            const int i = j;
            const double x = (ms2[2 * i] - cmx) * smx, y = (ms2[2 * i + 1] - cmy) * smy;
            const double X = (ms1[2 * i] - cMx) * sMx, Y = (ms1[2 * i + 1] - cMy) * sMy;
            double* Lx = L + i * 18; double* Ly = Lx + 9;
            Lx[0] = X; Lx[1] = Y; Lx[2] = 1; Lx[3] = 0; Lx[4] = 0; Lx[5] = 0; Lx[6] = -x * X; Lx[7] = -x * Y; Lx[8] = -x;
            Ly[0] = 0; Ly[1] = 0; Ly[2] = 0; Ly[3] = X; Ly[4] = Y; Ly[5] = 1; Ly[6] = -y * X; Ly[7] = -y * Y; Ly[8] = -y;
        }
    }
    __syncwarp();
    if (ok) {
        for (int e = j; e < 81; e += 8) {
            int a = e / 9, b = e % 9;
            if (b < a) { const int tmp = a; a = b; b = tmp; }
            double s = 0;
            #pragma unroll
            for (int i = 0; i < 4; i++) {
                const double* Lx = L + i * 18; const double* Ly = Lx + 9;
                s += Lx[a] * Lx[b] + Ly[a] * Ly[b];
            }
            LtL[e] = s;
        }
    }
    __syncwarp();
    jacobi9_g8(LtL, W, V, ok);
    if (ok) {
        const double invHnorm[9] = { 1. / smx, 0, cmx, 0, 1. / smy, cmy, 0, 0, 1 };
        const double Hnorm2[9] = { sMx, 0, -cMx * sMx, 0, sMy, -cMy * sMy, 0, 0, 1 };
        double Vl[9], Htemp[9], H0[9];
        #pragma unroll
        for (int i = 0; i < 9; i++) Vl[i] = V[72 + i];
        mat3mul(invHnorm, Vl, Htemp);
        mat3mul(Htemp, Hnorm2, H0);
        const double sc = 1. / H0[8];
        #pragma unroll
        for (int i = 0; i < 9; i++) H[i] = H0[i] * sc;
    }
    __syncwarp();
    return ok;
}

}  // namespace cvg
