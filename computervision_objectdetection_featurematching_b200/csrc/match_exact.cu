// match_exact.cu — exact fp32 match kernel (general descriptors) and the top-2 merge kernels.
//
// Reference: BFMatcher(NORM_L2).knnMatch(q, t, 2), src/TestsDetector.cpp:59-60.  This kernel
// reproduces cv::batchDistance's fp32 arithmetic bit for bit (SURVEY App. A.3): 16 partial sums
// acc[a][l] with a = (j/4)%4, l = j%4, separate multiply and add, combine ((a0+a1)+a2)+a3 per lane
// then (v0+v2)+(v1+v3), sqrtf, strict < insertion scanning train rows in ascending order (App. A.2).
// It serves calls whose descriptors are not integer-valued; integer (SIFT) data takes match_tc.cu.
#include "common.cuh"
#include <float.h>
#include <algorithm>

namespace cvg {

constexpr int EX_THREADS = 128;
constexpr int EX_TROWS = 16;          // train rows staged per smem tile

__global__ void __launch_bounds__(EX_THREADS)
match_exact_kernel(const float* __restrict__ Q, int n_query, const float* __restrict__ T,
                   const MatchUnit* __restrict__ units, Top2* __restrict__ parts,
                   const int* __restrict__ gate_flag, int gate_want)
{
    if (gate_flag && *gate_flag != gate_want) return;
    __shared__ float4 tile[EX_TROWS][DIM / 4];
    const MatchUnit u = units[blockIdx.x];
    const int qrow = u.q_row0 + threadIdx.x;
    const bool qvalid = qrow < n_query;
    float4 q[DIM / 4];
    {
        const float4* qp = reinterpret_cast<const float4*>(Q + (size_t)(qvalid ? qrow : 0) * DIM);
        #pragma unroll
        for (int j = 0; j < DIM / 4; j++) q[j] = qp[j];
    }
    int n_cols = u.n_tiles * TILE_N;
    if (n_cols > u.seg_cols - u.t_local0) n_cols = u.seg_cols - u.t_local0;
    float bd0 = FLT_MAX, bd1 = FLT_MAX;
    int bi0 = -1, bi1 = -1;
    for (int c0 = 0; c0 < n_cols; c0 += EX_TROWS) {
        const int nr = min(EX_TROWS, n_cols - c0);
        __syncthreads();
        for (int e = threadIdx.x; e < nr * (DIM / 4); e += EX_THREADS) {
            const int r = e / (DIM / 4), k = e % (DIM / 4);
            tile[r][k] = reinterpret_cast<const float4*>(T + (size_t)(u.t_row0_f32 + c0 + r) * DIM)[k];
        }
        __syncthreads();
        for (int r = 0; r < nr; r++) {
            float acc[4][4];
            #pragma unroll
            for (int a = 0; a < 4; a++)
                #pragma unroll
                for (int l = 0; l < 4; l++) acc[a][l] = 0.f;
            #pragma unroll
            for (int j4 = 0; j4 < DIM / 4; j4++) {
                const float4 t = tile[r][j4];
                const int a = j4 & 3;
                float d;
                d = __fsub_rn(q[j4].x, t.x); acc[a][0] = __fadd_rn(acc[a][0], __fmul_rn(d, d));
                d = __fsub_rn(q[j4].y, t.y); acc[a][1] = __fadd_rn(acc[a][1], __fmul_rn(d, d));
                d = __fsub_rn(q[j4].z, t.z); acc[a][2] = __fadd_rn(acc[a][2], __fmul_rn(d, d));
                d = __fsub_rn(q[j4].w, t.w); acc[a][3] = __fadd_rn(acc[a][3], __fmul_rn(d, d));
            }
            float v[4];
            #pragma unroll
            for (int l = 0; l < 4; l++)
                v[l] = __fadd_rn(__fadd_rn(__fadd_rn(acc[0][l], acc[1][l]), acc[2][l]), acc[3][l]);
            const float s = __fadd_rn(__fadd_rn(v[0], v[2]), __fadd_rn(v[1], v[3]));
            const float dist = sqrtf(s);
            const int ti = u.t_local0 + c0 + r;
            if (dist < bd1) {                 // NaN / inf / >= FLT_MAX never enter (App. A.1)
                if (dist < bd0) { bd1 = bd0; bi1 = bi0; bd0 = dist; bi0 = ti; }
                else            { bd1 = dist; bi1 = ti; }
            }
        }
    }
    Top2 out;
    out.d1 = bi0 >= 0 ? bd0 : INFINITY; out.i1 = bi0;
    out.d2 = bi1 >= 0 ? bd1 : INFINITY; out.i2 = bi1;
    parts[(size_t)u.part_slot * TILE_M + threadIdx.x] = out;
}

void launch_match_exact(const float* Q, int n_query, const float* T, const MatchUnit* units, int n_units,
                        Top2* parts, const int* gate_flag, int gate_want, cudaStream_t st)
{
    if (n_units <= 0) return;
    match_exact_kernel<<<n_units, EX_THREADS, 0, st>>>(Q, n_query, T, units, parts, gate_flag, gate_want);
}

// Cross-check form (BFMatcher(NORM_L2, crossCheck = true)) of the kernel above, for the units of build_xc_plan: the same
// distances, each row's nearest column (strict <, ascending columns), and per train column its nearest query row of the
// unit's view — the minimum over the CTA's rows of (distance bits, absolute row), non-negative floats ordering like their
// bits — merged per column with one global atomicMin per unit.  NaN and inf enter neither side.
__global__ void __launch_bounds__(EX_THREADS)
match_exact_xc_kernel(const float* __restrict__ Q, const float* __restrict__ T, const MatchUnit* __restrict__ units,
                      XcOut out, const int* __restrict__ gate_flag)
{
    if (gate_flag && *gate_flag == 0) return;                  // the tensor-core kernel serves the call
    __shared__ float4 tile[EX_TROWS][DIM / 4];
    __shared__ unsigned long long s_col[EX_TROWS];
    const MatchUnit u = units[blockIdx.x];
    const int qrow = u.q_row0 + threadIdx.x, lane = threadIdx.x & 31;
    const bool qvalid = (int)threadIdx.x < (u.pad1 & 255);
    float4 q[DIM / 4];
    {
        const float4* qp = reinterpret_cast<const float4*>(Q + (size_t)(qvalid ? qrow : u.q_row0) * DIM);
        #pragma unroll
        for (int j = 0; j < DIM / 4; j++) q[j] = qp[j];
    }
    unsigned long long* ck = out.colkey + (u.pad1 >> 8) * out.t_total + (u.t_row0_f32 - u.t_local0 - out.t_base);
    int n_cols = u.n_tiles * TILE_N;
    if (n_cols > u.seg_cols - u.t_local0) n_cols = u.seg_cols - u.t_local0;
    if (threadIdx.x < EX_TROWS) s_col[threadIdx.x] = ~0ull;
    float bd = FLT_MAX;
    int bi = -1;
    for (int c0 = 0; c0 < n_cols; c0 += EX_TROWS) {
        const int nr = min(EX_TROWS, n_cols - c0);
        __syncthreads();
        for (int e = threadIdx.x; e < nr * (DIM / 4); e += EX_THREADS) {
            const int r = e / (DIM / 4), k = e % (DIM / 4);
            tile[r][k] = reinterpret_cast<const float4*>(T + (size_t)(u.t_row0_f32 + c0 + r) * DIM)[k];
        }
        __syncthreads();
        for (int r = 0; r < nr; r++) {
            float acc[4][4];
            #pragma unroll
            for (int a = 0; a < 4; a++)
                #pragma unroll
                for (int l = 0; l < 4; l++) acc[a][l] = 0.f;
            #pragma unroll
            for (int j4 = 0; j4 < DIM / 4; j4++) {              // the order of match_exact_kernel (SURVEY App. A.3)
                const float4 t = tile[r][j4];
                const int a = j4 & 3;
                float d;
                d = __fsub_rn(q[j4].x, t.x); acc[a][0] = __fadd_rn(acc[a][0], __fmul_rn(d, d));
                d = __fsub_rn(q[j4].y, t.y); acc[a][1] = __fadd_rn(acc[a][1], __fmul_rn(d, d));
                d = __fsub_rn(q[j4].z, t.z); acc[a][2] = __fadd_rn(acc[a][2], __fmul_rn(d, d));
                d = __fsub_rn(q[j4].w, t.w); acc[a][3] = __fadd_rn(acc[a][3], __fmul_rn(d, d));
            }
            float v[4];
            #pragma unroll
            for (int l = 0; l < 4; l++)
                v[l] = __fadd_rn(__fadd_rn(__fadd_rn(acc[0][l], acc[1][l]), acc[2][l]), acc[3][l]);
            const float dist = sqrtf(__fadd_rn(__fadd_rn(v[0], v[2]), __fadd_rn(v[1], v[3])));
            const bool ok = qvalid && dist < FLT_MAX;
            if (ok && dist < bd) { bd = dist; bi = u.t_local0 + c0 + r; }
            unsigned long long key = ok ? ((unsigned long long)__float_as_uint(dist) << 32) | (unsigned int)qrow : ~0ull;
            #pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
                key = other < key ? other : key;
            }
            if (lane == 0 && key != ~0ull) atomicMin(&s_col[r], key);
        }
        __syncthreads();
        if ((int)threadIdx.x < nr) {
            const unsigned long long k = s_col[threadIdx.x];
            s_col[threadIdx.x] = ~0ull;
            if (k != ~0ull) atomicMin(&ck[u.t_local0 + c0 + threadIdx.x], k);
        }
    }
    if (bi >= 0) atomicMin(&out.rowkey[u.part_slot * out.row_stride + qrow], ((unsigned long long)__float_as_uint(bd) << 32) | (unsigned int)bi);
}

void launch_match_exact_xc(const float* Q, const float* T, const MatchUnit* units, int n_units, XcOut out,
                           const int* gate_flag, cudaStream_t st)
{
    if (n_units <= 0) return;
    match_exact_xc_kernel<<<n_units, EX_THREADS, 0, st>>>(Q, T, units, out, gate_flag);
}

// ---- merge: lexicographic (distance, train index), the order that reproduces OpenCV's tie rule ----
__device__ __forceinline__ bool lex_less(float da, int ia, float db, int ib)
{
    return da < db || (da == db && ia < ib);
}

__device__ __forceinline__ void top2_insert(float& d1, int& i1, float& d2, int& i2, float d, int i)
{
    if (i < 0) return;
    if (lex_less(d, i, d1, i1) || i1 < 0) {
        if (i1 >= 0) { d2 = d1; i2 = i1; }
        d1 = d; i1 = i;
    } else if (i2 < 0 || lex_less(d, i, d2, i2)) {
        d2 = d; i2 = i;
    }
}

__device__ __forceinline__ void top2_emit(float d1, int i1, float d2, int i2, float ratio, size_t row,
                                          int32_t* idx, float* dist, uint8_t* accept)
{
    idx[2 * row] = i1; idx[2 * row + 1] = i2;
    dist[2 * row] = i1 >= 0 ? d1 : 0.f; dist[2 * row + 1] = i2 >= 0 ? d2 : 0.f;
    if (accept) accept[row] = (i1 >= 0 && i2 >= 0 && d1 < __fmul_rn(ratio, d2)) ? 1 : 0;   // :67, App. A.4
}

// one thread per (segment, query row)
// Guard (fb_count != NULL): the tensor-core kernel orders a unit's columns by d^2, OpenCV by sqrtf(d^2).  The two orders
// agree while distinct integer d^2 keep distinct float distances, i.e. below d = 2048 (ulp(2048) = 2^-12 = 1/(2 d)); from
// there on neighbouring d^2 collapse into one float and OpenCV's tie rule (lower train index) can pick another column.
// If the row's merged second distance is below 2048 both of its columns are the global top two in either order (every
// column with d^2 >= 2^22 has a float distance >= 2048); otherwise the row is redone by the exact fallback kernels,
// which compare rounded distances like cv::batchDistance does.
__global__ void merge_kernel(const Top2* __restrict__ parts, const MergeEntry* __restrict__ dir,
                             int n_segments, int n_rowblocks, int n_query, float ratio,
                             int32_t* __restrict__ idx, float* __restrict__ dist, uint8_t* __restrict__ accept,
                             const int* __restrict__ gate_flag, int gate_skip, int* __restrict__ fb_count,
                             int2* __restrict__ fb_list)
{
    if (gate_flag && *gate_flag == gate_skip) return;          // the candidate path writes the results instead
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (int64_t)n_segments * n_query) return;
    const int seg = (int)(gid / n_query), row = (int)(gid % n_query);
    const MergeEntry e = dir[seg * n_rowblocks + row / TILE_M];
    float d1 = INFINITY, d2 = INFINITY;
    int i1 = -1, i2 = -1;
    for (int s = 0; s < e.n_slots; s++) {
        const Top2 p = parts[(size_t)(e.first_slot + s) * TILE_M + (row % TILE_M)];
        top2_insert(d1, i1, d2, i2, p.d1, p.i1);
        top2_insert(d1, i1, d2, i2, p.d2, p.i2);
    }
    if (fb_count && i2 >= 0 && d2 >= 2048.f) {
        const int slot = atomicAdd(fb_count, 1);
        fb_list[slot] = make_int2(seg, row);
        return;
    }
    top2_emit(d1, i1, d2, i2, ratio, (size_t)gid, idx, dist, accept);
}

void launch_merge(const Top2* parts, const MergeEntry* dir, int n_segments, int n_rowblocks, int n_query,
                  float ratio, int32_t* idx, float* dist, uint8_t* accept, const int* gate_flag, int gate_skip,
                  cudaStream_t st, int* fb_count, int2* fb_list)
{
    const int64_t n = (int64_t)n_segments * n_query;
    if (n <= 0) return;
    if (fb_count) cudaMemsetAsync(fb_count, 0, 4, st);
    merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(parts, dir, n_segments, n_rowblocks, n_query,
                                                              ratio, idx, dist, accept, gate_flag, gate_skip, fb_count, fb_list);
}

// ---- candidate path (non-integer descriptors): fp32 re-rank with a proof, exact fallback ------------
// cv::batchDistance's squared L2 distance of two 128-float rows, bit for bit (SURVEY App. A.3)
__device__ __forceinline__ float l2sqr_cv(const float4* __restrict__ q, const float4* __restrict__ t)
{
    float acc[4][4];
    #pragma unroll
    for (int a = 0; a < 4; a++)
        #pragma unroll
        for (int l = 0; l < 4; l++) acc[a][l] = 0.f;
    #pragma unroll 8
    for (int j4 = 0; j4 < DIM / 4; j4++) {
        const float4 x = q[j4], y = t[j4];
        const int a = j4 & 3;
        float d;
        d = __fsub_rn(x.x, y.x); acc[a][0] = __fadd_rn(acc[a][0], __fmul_rn(d, d));
        d = __fsub_rn(x.y, y.y); acc[a][1] = __fadd_rn(acc[a][1], __fmul_rn(d, d));
        d = __fsub_rn(x.z, y.z); acc[a][2] = __fadd_rn(acc[a][2], __fmul_rn(d, d));
        d = __fsub_rn(x.w, y.w); acc[a][3] = __fadd_rn(acc[a][3], __fmul_rn(d, d));
    }
    float v[4];
    #pragma unroll
    for (int l = 0; l < 4; l++)
        v[l] = __fadd_rn(__fadd_rn(__fadd_rn(acc[0][l], acc[1][l]), acc[2][l]), acc[3][l]);
    return __fadd_rn(__fadd_rn(v[0], v[2]), __fadd_rn(v[1], v[3]));
}

// One thread per (segment, query row).  The tensor-core kernel left, per unit and column part, the four columns
// with the largest APPROXIMATE value a = 2 q.t - ||t||^2 (bf16 hi/lo split operands, three products).  Here:
//   1. the records are merged into the row's four best candidates; every other column has a <= a4;
//   2. the candidates' distances are recomputed exactly as OpenCV does (fp32, its summation order) and ordered by
//      (distance, train index);
//   3. the answer is PROVEN: with eps >= |a - (2 q.t - ||t||^2)| for every column (bf16 rounding of both operands,
//      fp32 accumulation, the fp32 norms), any other column has a true squared distance >= qn - a4 - eps; if the
//      second best candidate's squared distance is below that bound (with a relative margin that also covers
//      OpenCV's own fp32 rounding and the rounding of sqrtf), no other column can enter or tie the top two.
//      Rows that cannot be proven go to the exact fallback kernel (list `fb`).
__global__ void merge4_rerank_kernel(const Top4* __restrict__ parts4, const MergeEntry* __restrict__ dir,
                                     const SegDev* __restrict__ segs, int n_segments, int n_rowblocks, int n_query,
                                     float ratio, const float* __restrict__ Q, int q_row_begin,
                                     const float* __restrict__ T, const float* __restrict__ qnorm,
                                     const int* __restrict__ tnmax_bits,
                                     int32_t* __restrict__ idx, float* __restrict__ dist, uint8_t* __restrict__ accept,
                                     int* __restrict__ fb_count, int2* __restrict__ fb_list,
                                     const int* __restrict__ gate_flag, int gate_want)
{
    if (gate_flag && *gate_flag != gate_want) return;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (int64_t)n_segments * n_query) return;
    const int seg = (int)(gid / n_query), row = (int)(gid % n_query);
    const MergeEntry e = dir[seg * n_rowblocks + row / TILE_M];
    const SegDev sd = segs[seg];
    float b[4] = { -INFINITY, -INFINITY, -INFINITY, -INFINITY };
    int ix[4] = { -1, -1, -1, -1 };
    for (int s = 0; s < e.n_slots * 4; s++) {
        const Top4 p = parts4[((size_t)e.first_slot * 4 + s) * TILE_M + (row % TILE_M)];
        #pragma unroll
        for (int k = 0; k < 4; k++) {
            const float v = p.v[k]; const int id = p.i[k];
            if (id < 0 || !(v > b[3])) continue;
            if (v > b[2]) {
                b[3] = b[2]; ix[3] = ix[2];
                if (v > b[1]) {
                    b[2] = b[1]; ix[2] = ix[1];
                    if (v > b[0]) { b[1] = b[0]; ix[1] = ix[0]; b[0] = v; ix[0] = id; }
                    else          { b[1] = v; ix[1] = id; }
                } else { b[2] = v; ix[2] = id; }
            } else { b[3] = v; ix[3] = id; }
        }
    }
    const float4* q = reinterpret_cast<const float4*>(Q + (size_t)(q_row_begin + row) * DIM);
    float d1 = INFINITY, d2 = INFINITY, s2 = INFINITY;      // s2: squared distance of the current second best
    int i1 = -1, i2 = -1;
    float s1 = INFINITY;
    bool bad = false;
    #pragma unroll
    for (int k = 0; k < 4; k++) {
        if (ix[k] < 0) continue;
        const float4* t = reinterpret_cast<const float4*>(T + (size_t)(sd.f32_row0 + ix[k]) * DIM);
        const float s = l2sqr_cv(q, t);
        const float d = sqrtf(s);
        if (!(d < FLT_MAX)) { bad = true; continue; }        // NaN / inf: let the exact kernel apply OpenCV's rule
        if (i1 < 0 || lex_less(d, ix[k], d1, i1)) { d2 = d1; i2 = i1; s2 = s1; d1 = d; i1 = ix[k]; s1 = s; }
        else if (i2 < 0 || lex_less(d, ix[k], d2, i2)) { d2 = d; i2 = ix[k]; s2 = s; }
    }
    bool proven;
    if (sd.rows <= 4) proven = !bad;                          // every column was a candidate
    else if (bad || i2 < 0 || ix[3] < 0) proven = false;
    else {
        const float qn = qnorm[q_row_begin + row];
        const float tnmax = __int_as_float(*tnmax_bits);
        // |a - exact| is bounded by: the split operands (2q = hi + lo + O(2^-18 |2q|), same for t, the lo.lo product is
        // dropped): 3 * 2^-17 ||q|| ||t||; the fp32 accumulation of 400 products, truncating adder assumed:
        // 400 * 2^-23 (2 ||q|| ||t|| + ||t||^2); the fp32 norms: 2^-17 (||q||^2 + ||t||^2).  Each doubled for slack.
        const float qt = sqrtf(qn) * sqrtf(tnmax);
        const float eps = 2.f * (2.2888184e-5f * qt + 4.7683716e-5f * (2.f * qt + tnmax) + 7.6293945e-6f * (qn + tnmax));
        const float lower = (qn - b[3]) - eps;                // squared distance of any non-candidate is >= lower
        proven = s2 < lower * (1.f - 6.103515625e-5f);        // 2^-14: OpenCV's own fp32 sum and sqrtf rounding
    }
    if (proven) {
        top2_emit(d1, i1, d2, i2, ratio, (size_t)gid, idx, dist, accept);
    } else {
        const int slot = atomicAdd(fb_count, 1);
        fb_list[slot] = make_int2(seg, row);
    }
}

// Exact top-2 of the rows the re-rank could not prove.  A work item = (unproven row, chunk of FB_CHUNK train rows),
// one CTA each, looped over a fixed grid because the number of rows is only known on the device.  (distance, index)
// pairs are packed into 64-bit keys whose unsigned order is the lexicographic order OpenCV's insertion produces
// (distances are >= 0), so the merge across chunks is an atomicMin: pass 1 finds every row's nearest column, pass 2
// the nearest one that is not it.
constexpr int FB_THREADS = 256;
constexpr int FB_CHUNK = 512;
constexpr unsigned long long FB_ABSENT = ~0ull;

__device__ __forceinline__ unsigned long long fb_key(float d, int i)
{
    return ((unsigned long long)__float_as_uint(d) << 32) | (unsigned int)i;
}

__global__ void fallback_init_kernel(const int* __restrict__ fb_count, unsigned long long* __restrict__ g1,
                                     unsigned long long* __restrict__ g2, const int* __restrict__ gate_flag, int gate_want)
{
    if (gate_flag && *gate_flag != gate_want) return;
    const int n = *fb_count;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) { g1[e] = FB_ABSENT; g2[e] = FB_ABSENT; }
}

__global__ void __launch_bounds__(FB_THREADS)
fallback_scan_kernel(const int* __restrict__ fb_count, const int2* __restrict__ fb_list, const SegDev* __restrict__ segs,
                     int chunks, const float* __restrict__ Q, int q_row_begin, const float* __restrict__ T,
                     unsigned long long* __restrict__ g1, unsigned long long* __restrict__ g2, int pass,
                     const int* __restrict__ gate_flag, int gate_want)
{
    if (gate_flag && *gate_flag != gate_want) return;
    __shared__ unsigned long long s_min[FB_THREADS / 32];
    const int n = *fb_count;
    const long long total = (long long)n * chunks;
    for (long long w = blockIdx.x; w < total; w += gridDim.x) {
        const int e = (int)(w / chunks), c = (int)(w % chunks);
        const int2 sr = fb_list[e];
        const SegDev sd = segs[sr.x];
        const int r0 = c * FB_CHUNK, r1 = min(r0 + FB_CHUNK, sd.rows);
        if (r0 >= r1) continue;                               // block-uniform
        const float4* q = reinterpret_cast<const float4*>(Q + (size_t)(q_row_begin + sr.y) * DIM);
        const unsigned long long skip = pass == 2 ? g1[e] : FB_ABSENT;
        unsigned long long best = FB_ABSENT;
        for (int r = r0 + (int)threadIdx.x; r < r1; r += FB_THREADS) {
            const float d = sqrtf(l2sqr_cv(q, reinterpret_cast<const float4*>(T + (size_t)(sd.f32_row0 + r) * DIM)));
            if (d < FLT_MAX) {                                // NaN / inf / >= FLT_MAX never enter (App. A.1)
                const unsigned long long k = fb_key(d, r);
                if (k != skip && k < best) best = k;
            }
        }
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best, o);
            if (ob < best) best = ob;
        }
        __syncthreads();                                      // s_min of the previous work item consumed
        if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            #pragma unroll
            for (int k = 1; k < FB_THREADS / 32; k++) if (s_min[k] < best) best = s_min[k];
            if (best != FB_ABSENT) atomicMin(pass == 1 ? &g1[e] : &g2[e], best);
        }
    }
}

__global__ void fallback_emit_kernel(const int* __restrict__ fb_count, const int2* __restrict__ fb_list, int n_query, float ratio,
                                     const unsigned long long* __restrict__ g1, const unsigned long long* __restrict__ g2,
                                     int32_t* __restrict__ idx, float* __restrict__ dist, uint8_t* __restrict__ accept,
                                     const int* __restrict__ gate_flag, int gate_want)
{
    if (gate_flag && *gate_flag != gate_want) return;
    const int n = *fb_count;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int2 sr = fb_list[e];
        const unsigned long long a = g1[e], b = g2[e];
        const int i1 = a == FB_ABSENT ? -1 : (int)(unsigned int)a, i2 = b == FB_ABSENT ? -1 : (int)(unsigned int)b;
        const float d1 = __uint_as_float((unsigned int)(a >> 32)), d2 = __uint_as_float((unsigned int)(b >> 32));
        top2_emit(d1, i1, d2, i2, ratio, (size_t)sr.x * n_query + sr.y, idx, dist, accept);
    }
}

void launch_merge4_rerank(const Top4* parts4, const MergeEntry* dir, const SegDev* segs, int n_segments, int n_rowblocks,
                          int n_query, int max_seg_rows, float ratio, const float* Q, int q_row_begin, const float* T,
                          const float* qnorm, const int* tnmax_bits, int32_t* idx, float* dist, uint8_t* accept, int* fb_count,
                          int2* fb_list, unsigned long long* fb_keys /*[2][n_segments * n_query]*/,
                          const int* gate_flag, int gate_want, int n_sms, cudaStream_t st)
{
    const int64_t n = (int64_t)n_segments * n_query;
    if (n <= 0) return;
    cudaMemsetAsync(fb_count, 0, 4, st);
    merge4_rerank_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(parts4, dir, segs, n_segments, n_rowblocks, n_query, ratio,
                                                                      Q, q_row_begin, T, qnorm, tnmax_bits, idx, dist, accept,
                                                                      fb_count, fb_list, gate_flag, gate_want);
    launch_fallback_exact(fb_count, fb_list, fb_keys, segs, n_segments, n_query, max_seg_rows, ratio, Q, q_row_begin, T, idx, dist,
                          accept, gate_flag, gate_want, n_sms, st);
}

// exact top-2 (cv::batchDistance arithmetic and order) of the *fb_count rows listed in fb_list: 4 launches, all empty loops
// when the list is empty
void launch_fallback_exact(const int* fb_count, const int2* fb_list, unsigned long long* fb_keys, const SegDev* segs,
                           int n_segments, int n_query, int max_seg_rows, float ratio, const float* Q, int q_row_begin,
                           const float* T, int32_t* idx, float* dist, uint8_t* accept, const int* gate_flag, int gate_want,
                           int n_sms, cudaStream_t st)
{
    const int64_t n = (int64_t)n_segments * n_query;
    if (n <= 0) return;
    unsigned long long* g1 = fb_keys; unsigned long long* g2 = fb_keys + n;
    const int chunks = (max_seg_rows + FB_CHUNK - 1) / FB_CHUNK;
    fallback_init_kernel<<<n_sms, 256, 0, st>>>(fb_count, g1, g2, gate_flag, gate_want);
    for (int pass = 1; pass <= 2; pass++)
        fallback_scan_kernel<<<n_sms * 8, FB_THREADS, 0, st>>>(fb_count, fb_list, segs, chunks, Q, q_row_begin, T, g1, g2, pass,
                                                              gate_flag, gate_want);
    fallback_emit_kernel<<<n_sms, 256, 0, st>>>(fb_count, fb_list, n_query, ratio, g1, g2, idx, dist, accept, gate_flag, gate_want);
}


// ---- cross-check: distances, the d >= 2048 guard, the mutual test -------------------------------------
constexpr unsigned long long XC_NONE = ~0ull;
constexpr uint32_t XC_GUARD_D2 = 1u << 22;                 // d = 2048: from here on distinct d^2 can share a float distance

// Tensor-core path only: the keys hold d^2.  Below 2^22 the order by (d^2, index) is cv2's order by (sqrtf(d^2), index) — every
// d^2 < 2^22 keeps its own float distance, and every larger d^2 has a distance >= 2048 — so the key becomes (distance bits,
// index).  A row or column whose best d^2 reaches 2^22 is listed for the exact scan instead: rows as (segment, absolute
// row), columns as (view slot, train row - t_base).
__global__ void xc_distance_kernel(XcOut k, int row_begin, int n_rows, int64_t n_rows_all, int64_t n_cols_all, int* __restrict__ counts,
                                   int2* __restrict__ row_list, int2* __restrict__ col_list, const int* __restrict__ gate_flag)
{
    if (gate_flag && *gate_flag != 0) return;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_rows_all + n_cols_all; e += (int64_t)gridDim.x * blockDim.x) {
        const bool is_row = e < n_rows_all;
        const int seg = is_row ? (int)(e / n_rows) : 0, row = is_row ? row_begin + (int)(e % n_rows) : 0;
        unsigned long long* p = is_row ? &k.rowkey[seg * k.row_stride + row] : &k.colkey[e - n_rows_all];
        const unsigned long long v = *p;
        if (v == XC_NONE) continue;
        const uint32_t d2 = (uint32_t)(v >> 32);
        if (d2 >= XC_GUARD_D2) {
            if (is_row) row_list[atomicAdd(&counts[0], 1)] = make_int2(seg, row);
            else { const int64_t c = e - n_rows_all; col_list[atomicAdd(&counts[1], 1)] = make_int2((int)(c / k.t_total), (int)(c % k.t_total)); }
        } else {
            *p = ((unsigned long long)__float_as_uint(sqrtf((float)d2)) << 32) | (v & 0xFFFFFFFFull);
        }
    }
}

// the exact scans' results into the key arrays (a column's scan ran over its view's rows: local row -> absolute row)
__global__ void xc_apply_kernel(XcOut k, const SegDev* __restrict__ views, const int* __restrict__ counts,
                                const int2* __restrict__ row_list, const unsigned long long* __restrict__ row_g,
                                const int2* __restrict__ col_list, const unsigned long long* __restrict__ col_g, int* __restrict__ guard_total)
{
    const int nr = counts[0], nc = counts[1];
    if (blockIdx.x == 0 && threadIdx.x == 0) *guard_total = nr + nc;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nr + nc; e += gridDim.x * blockDim.x) {
        if (e < nr) { k.rowkey[row_list[e].x * k.row_stride + row_list[e].y] = row_g[e]; continue; }
        const int2 vc = col_list[e - nr];
        const unsigned long long g = col_g[e - nr];
        k.colkey[vc.x * k.t_total + vc.y] =
            g == XC_NONE ? XC_NONE : (g & 0xFFFFFFFF00000000ull) | (unsigned int)(views[vc.x].f32_row0 + (int)(unsigned int)g);
    }
}

// row i of view slot v against segment s, nearest column j: a match iff column j's nearest row in view v is i
__global__ void xc_emit_kernel(XcOut k, int row_begin, int n_query, int n_segs, int n_views, const SegDev* __restrict__ views,
                               const SegDev* __restrict__ segs, int32_t* __restrict__ idx, float* __restrict__ dist,
                               uint8_t* __restrict__ accept)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t pv = blockIdx.y; pv < (int64_t)n_segs * n_views; pv += gridDim.y) {
        const int s = (int)(pv / n_views), v = (int)(pv % n_views);
        const SegDev vw = views[v];
        if (x >= vw.rows) continue;
        const int row = (int)vw.f32_row0 + x;
        const unsigned long long rk = k.rowkey[s * k.row_stride + row];
        int j = -1;
        float d = 0.f;
        if (rk != XC_NONE) {
            const int c = (int)(unsigned int)rk;
            if ((unsigned int)k.colkey[v * k.t_total + (segs[s].f32_row0 - k.t_base) + c] == (unsigned int)row) {
                j = c; d = __uint_as_float((unsigned int)(rk >> 32));
            }
        }
        if (accept) {
            const size_t o = (size_t)s * n_query + (row - row_begin);
            idx[2 * o] = j;
            accept[o] = j >= 0;
        } else {
            idx[row - row_begin] = j;
            dist[row - row_begin] = d;
        }
    }
}

int launch_xc_finish(const XcFinish& w, cudaStream_t st)
{
    const int nq = w.row_end - w.row_begin;
    const int64_t n_rows_all = (int64_t)w.n_segs * nq, n_cols_all = (int64_t)w.n_views * w.keys.t_total;
    if (nq <= 0 || w.n_segs <= 0) return 0;
    int launches = 0;
    if (n_cols_all > 0) {
        const int64_t n = n_rows_all + n_cols_all;
        xc_distance_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)w.n_sms * 8), 256, 0, st>>>(
            w.keys, w.row_begin, nq, n_rows_all, n_cols_all, w.guard_counts, w.row_list, w.col_list, w.gate_flag);
        // exact scans of the listed rows (over their segment's train rows) and columns (over their view's rows, roles
        // swapped); empty loops when nothing is listed
        unsigned long long* rg1 = w.row_g; unsigned long long* rg2 = w.row_g + n_rows_all;
        unsigned long long* cg1 = w.col_g; unsigned long long* cg2 = w.col_g + n_cols_all;
        fallback_init_kernel<<<w.n_sms, 256, 0, st>>>(&w.guard_counts[0], rg1, rg2, nullptr, 0);
        fallback_init_kernel<<<w.n_sms, 256, 0, st>>>(&w.guard_counts[1], cg1, cg2, nullptr, 0);
        fallback_scan_kernel<<<w.n_sms * 8, FB_THREADS, 0, st>>>(&w.guard_counts[0], w.row_list, w.segs,
                                                                 (w.max_seg_rows + FB_CHUNK - 1) / FB_CHUNK, w.Q, 0, w.T, rg1, rg2, 1, nullptr, 0);
        fallback_scan_kernel<<<w.n_sms * 8, FB_THREADS, 0, st>>>(&w.guard_counts[1], w.col_list, w.views,
                                                                 (w.max_view_rows + FB_CHUNK - 1) / FB_CHUNK, w.T, (int)w.keys.t_base, w.Q,
                                                                 cg1, cg2, 1, nullptr, 0);
        xc_apply_kernel<<<w.n_sms, 256, 0, st>>>(w.keys, w.views, w.guard_counts, w.row_list, rg1, w.col_list, cg1, w.guard_total);
        launches += 6;
    }
    // rows outside every view (models whose first view starts after row 0) keep no match
    if (w.accept) {
        cudaMemsetAsync(w.accept, 0, (size_t)n_rows_all, st);
    } else {
        cudaMemsetAsync(w.idx, 0xFF, (size_t)nq * 4, st);
        cudaMemsetAsync(w.dist, 0, (size_t)nq * 4, st);
    }
    if (w.max_view_rows <= 0 || w.n_views <= 0) return launches;
    xc_emit_kernel<<<dim3((unsigned)((w.max_view_rows + 255) / 256), (unsigned)std::min<int64_t>((int64_t)w.n_segs * w.n_views, 65535)), 256, 0, st>>>(
        w.keys, w.row_begin, nq, w.n_segs, w.n_views, w.views, w.segs, w.idx, w.dist, w.accept);
    return launches + 1;
}

// merge of n_parts partial results laid out [n_parts][n_query][2] (multi-GPU train-tile shards)
__global__ void merge_parts_kernel(const float* __restrict__ dparts, const int32_t* __restrict__ iparts,
                                   int n_parts, int n_query, float ratio, int32_t* __restrict__ idx,
                                   float* __restrict__ dist, uint8_t* __restrict__ accept)
{
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_query) return;
    float d1 = INFINITY, d2 = INFINITY;
    int i1 = -1, i2 = -1;
    for (int p = 0; p < n_parts; p++) {
        const size_t o = ((size_t)p * n_query + row) * 2;
        top2_insert(d1, i1, d2, i2, dparts[o], iparts[o]);
        top2_insert(d1, i1, d2, i2, dparts[o + 1], iparts[o + 1]);
    }
    top2_emit(d1, i1, d2, i2, ratio, (size_t)row, idx, dist, accept);
}

void launch_merge_parts(const float* dist_parts, const int32_t* idx_parts, int n_parts, int n_query, float ratio,
                        int32_t* idx, float* dist, uint8_t* accept, cudaStream_t st)
{
    if (n_query <= 0) return;
    merge_parts_kernel<<<(n_query + 255) / 256, 256, 0, st>>>(dist_parts, idx_parts, n_parts, n_query, ratio,
                                                              idx, dist, accept);
}

// final (idx,dist) arrays -> shard-exchange layout with global train indices
__global__ void shift_index_kernel(const int32_t* __restrict__ idx_in, const float* __restrict__ dist_in,
                                   int n_query, int32_t idx_base, float* __restrict__ dist, int32_t* __restrict__ idx)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * n_query) return;
    const int v = idx_in[i];
    idx[i] = v >= 0 ? v + idx_base : -1;
    dist[i] = v >= 0 ? dist_in[i] : INFINITY;
}

void launch_shift_index(const int32_t* idx_in, const float* dist_in, int n_query, int32_t idx_base,
                        float* dist, int32_t* idx, cudaStream_t st)
{
    if (n_query <= 0) return;
    shift_index_kernel<<<(2 * n_query + 255) / 256, 256, 0, st>>>(idx_in, dist_in, n_query, idx_base, dist, idx);
}

}  // namespace cvg
