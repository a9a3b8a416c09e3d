// ransac.cu — batched verify stage: cv::findHomography(src, dst, RANSAC, thr, mask) for P independent
// correspondence sets at once, plus the gates of the reference's view loop.
//
// Replaces reference src/TestsDetector.cpp:77-94 (findHomography :78, H.empty :79, countNonZero :81,
// determinant :84, inlier gather + rescale :87-94).  Semantics: cv2 4.13.0, SURVEY.md App. B / D.
//
// OpenCV's loop is serial (one RNG stream with data-dependent consumption, adaptive stop).  The
// parallel decomposition keeps its results bit for bit (App. D.5):
//   1. sample kernel   — replays cv::RNG + getSubset + checkSubset.  The raw RNG stream for the fixed
//                        per-call seed is a constant table in HBM, so the attempt starting at any draw
//                        position p can be evaluated independently; a block evaluates a window of 2048
//                        positions in parallel and recovers the chain p -> p + consumed(p) by pointer jumping.
//                        One huge round (no early stop, >= 32768 iterations) is cut into chunks walked by many CTAs
//                        (1b below: per-chunk entry -> exit maps composed in order).
//   2. solve kernel    — 4-point normalised DLT (9x9 Jacobi, fp64, no FMA), in rounds sized to one full wave.
//                        ransac_hyp_t_kernel (default): one hypothesis per thread, matrix state element-major in
//                        shared memory (jacobi_thread.cuh); it leaves the fp32 model in HBM.  Bit-identical variants
//                        for few hypotheses / A-B runs that also score: one warp per hypothesis (jacobi_warp.cuh),
//                        four per warp, and the generic serial routine (CVG_HYP_MODE = 1, 2, 3).
//   3. score kernel    — ransac_score_kernel: fp32 inlier counting of a round's models at full occupancy, the
//                        correspondences staged in shared memory, four points per reciprocal range test.
//   4. select kernel   — the sequential "good > max(best,3)" / RANSACUpdateNumIters scan, one warp per
//                        set, so the winner is the hypothesis the serial loop would have kept.
//   5. finish kernel   — winner's inlier mask, DLT refit on the inliers, 9-parameter LM (10 iterations),
//                        mask recomputed from the refined H.  Sets with <= EXACT_MAX_INLIERS inliers use
//                        OpenCV's exact summation order (bit-exact H); larger sets use block reductions.
#include "common.cuh"
#include "homography_math.cuh"
#include "jacobi_warp.cuh"
#include "jacobi_thread.cuh"
#include <stdlib.h>

namespace cvg {

constexpr int RS_THREADS = 128;
constexpr int EXACT_MAX_INLIERS = 128;
constexpr int SMEM_PTS = 1024;              // correspondences staged per shared-memory tile

// ---- draw MP distinct indices starting at table position p (getSubset's inner loop) ---------------
// `get(pos)` returns uniform(0, n) for draw position pos, i.e. rng_tab[pos] % n, or -1 past the table.
// returns the number of draws consumed, or -1 when the table would be overrun
template <int MP = 4, class Get>
__device__ __forceinline__ int draw_subset_g(const Get& get, int64_t p, int* idx)
{
    int64_t pos = p;
    #pragma unroll
    for (int i = 0; i < MP; i++) {
        for (;;) {
            const int v = get(pos++);
            if (v < 0) return -1;
            bool dup = false;
            #pragma unroll
            for (int k = 0; k < MP; k++) dup |= (k < i) && (idx[k] == v);
            if (!dup) { idx[i] = v; break; }
        }
    }
    return (int)(pos - p);
}

struct TabGet {
    const uint32_t* __restrict__ tab; int64_t len; uint32_t n;
    __device__ __forceinline__ int operator()(int64_t pos) const { return pos < len ? (int)(tab[pos] % n) : -1; }
};

__device__ __forceinline__ int draw_subset(const uint32_t* __restrict__ tab, int64_t tab_len, int64_t p,
                                           uint32_t n, int idx[4])
{
    return draw_subset_g(TabGet{ tab, tab_len, n }, p, idx);
}

// ---- 1. sample kernel ------------------------------------------------------------------------------
// A window of SW consecutive draw positions is evaluated in parallel: for every position p the attempt
// that would start there (draws consumed, checkSubset verdict).  The serial getSubset visits the chain
// p -> p + consumed(p); the nodes of that chain inside the window are found by pointer jumping
// (ceil(log2(SW/MP)) doubling rounds: an attempt of an MP-point model consumes >= MP draws, so a window holds
// <= SW/MP chain nodes), ranked by a block prefix sum, and the accepted ones become the samples of consecutive
// iterations — the same order, rejected attempts and 10000-attempt limit as the serial loop.
// MP = 4: findHomography (checkSubset: collinearity + orientation); MP = 3: estimateAffine2D (collinearity only);
// MP = 2: estimateAffinePartial2D (collinearity of two points: always accepted).
constexpr int SW = 2048;                          // measured: 512 -> 2048 halves the sampler time per draw (fewer serial windows)
constexpr int SW_ROUNDS = 9;                      // log2(SW / 4): the 4-point chunked sampler below
template <int MP> __host__ __device__ constexpr int sw_rounds() { int r = 0; while ((MP << r) < SW) r++; return r; }
static_assert(sw_rounds<4>() == SW_ROUNDS && (4 << SW_ROUNDS) == SW, "pointer-jumping rounds must cover SW / 4 chain nodes");
static_assert(sw_rounds<3>() == 10 && (3 << sw_rounds<3>()) >= SW, "pointer-jumping rounds must cover SW / 3 chain nodes");
static_assert(sw_rounds<2>() == 10 && (2 << sw_rounds<2>()) >= SW, "pointer-jumping rounds must cover SW / 2 chain nodes");
constexpr int SW_TAIL = 64;                       // draws staged beyond the window for attempts that start near its end
constexpr int SMP_THREADS = 512;                  // one window offset per thread
constexpr int SW_PER_THREAD = SW / SMP_THREADS;

// Samples are produced round by round (iterations [round_base, round_end)); the stream position and the
// running failure count persist in smp_state between rounds, and a set whose adaptive niters already
// ended before round_base is skipped.
template <int MP>
__global__ void __launch_bounds__(SMP_THREADS)
ransac_sample_kernel(RansacWork w, int round_base, int round_end, const int* __restrict__ only_if_flag)
{
    constexpr int ROUNDS = sw_rounds<MP>();
    const int set = blockIdx.x;
    if (only_if_flag && only_if_flag[set] == 0) return;          // chunked sampler handled this set
    const int n = w.counts_n[set];
    int32_t* out = w.sample_pos + (size_t)set * w.max_iters;
    if (round_base == 0) {
        if (threadIdx.x == 0) {
            w.niters_cur[set] = max(w.max_iters, 1); w.best_iter[set] = -1; w.best_count[set] = 0;
            w.n_samples[set] = 0; w.status_flags[set] = 0;
            w.smp_state[2 * set] = 0; w.smp_state[2 * set + 1] = 0;
        }
        if (n <= MP) return;                        // n < MP: nothing; n == MP: handled by finish kernel
    } else {
        // finished earlier (getSubset failure / table exhausted), or the adaptive stop is behind us
        if (n <= MP || w.smp_state[2 * set + 1] < 0 || w.n_samples[set] < round_base || round_base >= w.niters_cur[set]) return;
    }
    const float4* __restrict__ pts = w.pts + w.starts[set];
    __shared__ float4 spts[SMEM_PTS];
    __shared__ uint16_t info[SW];                   // bit 15: checkSubset ok; bits 0-14: draws consumed (0 = overrun)
    __shared__ int32_t s_draw[SW + SW_TAIL];        // uniform(0,n) of the window's draw positions (-1 past the table)
    __shared__ uint16_t jump[2][SW];
    __shared__ uint8_t reach[SW];
    __shared__ int s_wsum[SMP_THREADS / 32][2];
    __shared__ int s_last, s_first_ok, s_last_ok, s_bad;
    const bool staged = n <= SMEM_PTS;
    if (staged)
        for (int i = threadIdx.x; i < n; i += SMP_THREADS) spts[i] = pts[i];
    int64_t base = round_base == 0 ? 0 : w.smp_state[2 * set];
    int iter = round_base, attempts = round_base == 0 ? 0 : (int)w.smp_state[2 * set + 1], flags = 0;
    bool finished = false;                          // no further samples will ever come
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const TabGet slow{ w.rng_tab, w.rng_len, (uint32_t)n };
    for (;;) {
        __syncthreads();
        for (int j = threadIdx.x; j < SW + SW_TAIL; j += SMP_THREADS) {
            const int64_t pp = base + j;
            s_draw[j] = pp < w.rng_len ? (int32_t)(w.rng_tab[pp] % (uint32_t)n) : -1;
        }
        if (threadIdx.x == 0) { s_last = 0; s_first_ok = SW; s_last_ok = -1; s_bad = 0; }
        __syncthreads();
        auto get = [&](int64_t pos) -> int {
            const int64_t j = pos - base;
            return j < SW + SW_TAIL ? s_draw[j] : slow(pos);
        };
        #pragma unroll 1
        for (int k = 0; k < SW_PER_THREAD; k++) {
            const int o = k * SMP_THREADS + threadIdx.x;
            int idx[MP];
            const int cons = draw_subset_g<MP>(get, base + o, idx);
            uint16_t e = 0;
            if (cons > 0 && cons < 0x7fff) {
                float ms1[2 * MP], ms2[2 * MP];
                #pragma unroll
                for (int i = 0; i < MP; i++) {
                    const float4 q = staged ? spts[idx[i]] : pts[idx[i]];
                    ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
                }
                bool ok;
                if constexpr (MP == 4) ok = check_subset4(ms1, ms2);
                else ok = check_subset_affine<MP>(ms1, ms2);
                e = (uint16_t)(cons | (ok ? 0x8000 : 0));
            }
            info[o] = e;
            const int c = e & 0x7fff;
            jump[0][o] = (uint16_t)((c == 0 || o + c >= SW) ? SW : o + c);
            reach[o] = o == 0 ? 1 : 0;
        }
        __syncthreads();
        int cur = 0;
        #pragma unroll 1
        for (int r = 0; r < ROUNDS; r++) {            // reach = { next^i(0) : i < 2^(r+1) }
            #pragma unroll
            for (int k = 0; k < SW_PER_THREAD; k++) {
                const int o = k * SMP_THREADS + threadIdx.x;
                const int j = jump[cur][o];
                if (reach[o] && j < SW) reach[j] = 1;
                jump[cur ^ 1][o] = (uint16_t)(j < SW ? jump[cur][j] : SW);
            }
            __syncthreads();
            cur ^= 1;
        }
        // rank the chain nodes (offsets tid*4 .. tid*4+3 per thread, so ranks follow stream order)
        int n_reach = 0, n_ok = 0, mask_r = 0, mask_ok = 0;
        #pragma unroll
        for (int k = 0; k < SW_PER_THREAD; k++) {
            const int o = threadIdx.x * SW_PER_THREAD + k;
            if (reach[o]) {
                const uint16_t e = info[o];
                mask_r |= 1 << k; n_reach++;
                if ((e & 0x7fff) == 0) atomicExch(&s_bad, 1);
                if (e & 0x8000) { mask_ok |= 1 << k; n_ok++; atomicMin(&s_first_ok, o); atomicMax(&s_last_ok, o); }
                atomicMax(&s_last, o);
            }
        }
        int pre_r = n_reach, pre_ok = n_ok;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, pre_r, d), b2 = __shfl_up_sync(0xffffffffu, pre_ok, d);
            if (lane >= d) { pre_r += a; pre_ok += b2; }
        }
        if (lane == 31) { s_wsum[wid][0] = pre_r; s_wsum[wid][1] = pre_ok; }
        __syncthreads();
        int off_r = 0, off_ok = 0, tot_r = 0, tot_ok = 0;
        #pragma unroll
        for (int q = 0; q < SMP_THREADS / 32; q++) {
            if (q < wid) { off_r += s_wsum[q][0]; off_ok += s_wsum[q][1]; }
            tot_r += s_wsum[q][0]; tot_ok += s_wsum[q][1];
        }
        const int excl_r = off_r + pre_r - n_reach, excl_ok = off_ok + pre_ok - n_ok;   // exclusive ranks of this thread
        const int first_ok = s_first_ok, last_ok = s_last_ok, last = s_last;
        if (s_bad) { flags |= 1; finished = true; break; }      // RNG table exhausted
        // failures before the first accepted attempt of this window extend the running failure count
        int fails_head = 0, fails_tail = 0;
        {
            // nodes before first_ok / after last_ok: count with the same block-wide sums
            int h = 0, t = 0;
            #pragma unroll
            for (int k = 0; k < SW_PER_THREAD; k++) {
                const int o = threadIdx.x * SW_PER_THREAD + k;
                if ((mask_r >> k) & 1) { h += o < first_ok; t += o > last_ok; }
            }
            #pragma unroll
            for (int d = 16; d > 0; d >>= 1) { h += __shfl_xor_sync(0xffffffffu, h, d); t += __shfl_xor_sync(0xffffffffu, t, d); }
            __syncthreads();
            if (lane == 0) { s_wsum[wid][0] = h; s_wsum[wid][1] = t; }
            __syncthreads();
            #pragma unroll
            for (int q = 0; q < SMP_THREADS / 32; q++) { fails_head += s_wsum[q][0]; fails_tail += s_wsum[q][1]; }
        }
        if (attempts + fails_head >= 10000) { finished = true; break; }   // getSubset gave up before the next success
        // emit accepted attempts as the samples of iterations iter, iter+1, ...
        {
            int r = excl_ok;
            #pragma unroll
            for (int k = 0; k < SW_PER_THREAD; k++)
                if ((mask_ok >> k) & 1) {
                    if (iter + r < round_end) out[iter + r] = (int32_t)(base + threadIdx.x * SW_PER_THREAD + k);
                    r++;
                }
        }
        (void)excl_r; (void)tot_r;
        if (iter + tot_ok >= round_end) {
            // the round is complete inside this window: resume right after the attempt that produced its last sample
            const int need = round_end - iter;                       // >= 1 accepted attempts of this window are used
            __syncthreads();
            {
                int r = excl_ok;
                #pragma unroll
                for (int k = 0; k < SW_PER_THREAD; k++)
                    if ((mask_ok >> k) & 1) { if (r == need - 1) s_last = threadIdx.x * SW_PER_THREAD + k; r++; }
            }
            __syncthreads();
            const int lo = s_last;
            base = base + lo + (info[lo] & 0x7fff);
            attempts = 0;
            iter = round_end;
            break;
        }
        attempts = tot_ok > 0 ? fails_tail : attempts + fails_head;
        iter += tot_ok;
        base = base + last + (info[last] & 0x7fff);
        if (base + SW + SW_TAIL + 64 >= 0x7fffffffLL) { flags |= 1; finished = true; break; }
    }
    if (threadIdx.x == 0) {
        w.n_samples[set] = iter;
        if (flags) { w.status_flags[set] = flags; if (w.err_flag) atomicOr(w.err_flag, flags); }
        w.smp_state[2 * set] = base;
        w.smp_state[2 * set + 1] = finished ? -1 : attempts;
    }
}


// ---- 1b. chunked sampler: one set's draw stream cut into chunks that many CTAs walk at once ----------------
// The serial chain p -> p + consumed(p) enters chunk c (draw positions [c_begin, c_end)) at c_begin + e with a small
// offset e (the last attempt of chunk c-1 overshoots c_begin by fewer draws than it consumed).  consumed(p) depends on
// the draws alone — duplicates among the four indices — not on the correspondences, so:
//   map kernel     — per chunk, the function e -> exit offset into chunk c+1 for EVERY e < CH_K, by pointer jumping over
//                    the chunk's windows (no checkSubset, no point loads).  With large n nearly every attempt consumes
//                    exactly four draws, so chains of different residues mod 4 do not meet for tens of thousands of
//                    draws: waiting for convergence does not work, carrying all entries through does.
//   entry kernel   — one CTA per set composes the maps in chunk order (entry(0) = 0): the true entry of every chunk.
//   chunk kernel   — every CTA walks its chunk from its true entry window by window like the serial kernel and leaves
//                    its accepted positions in a list.
//   stitch kernel  — one thread per set walks the chunk summaries in order, re-checks exit(c-1) == entry(c), applies
//                    the 10000-consecutive-failures rule and the end of the round; a scatter kernel numbers the samples.
// Anything unusual (an exit offset >= CH_K, a failure run that could reach 10000, ...) hands the set to the serial kernel.
constexpr int CH_WINDOWS = 8;
constexpr int CH_DRAWS = CH_WINDOWS * SW;             // 16 384 draw positions per chunk
constexpr int CH_LIST = CH_DRAWS / 4 + 8;             // accepted attempts per chunk (an attempt consumes >= 4 draws)
constexpr int CH_K = 64;                              // entry offsets carried through a chunk
constexpr int64_t CHUNKED_MIN_ITERS = 32768;       // rounds shorter than this stay on the one-CTA-per-set kernel

struct ChunkOut { int64_t entry, exit; int32_t n_ok, n_nodes, head, tail; int32_t flags, pad; };   // flags: 1 table short, 2 unsafe

__global__ void __launch_bounds__(SMP_THREADS)
ransac_sample_map_kernel(RansacWork w, int round_base, int n_chunks, uint8_t* __restrict__ maps)
{
    const int set = blockIdx.y, chunk = blockIdx.x;
    const int n = w.counts_n[set];
    uint8_t* map = maps + ((size_t)set * n_chunks + chunk) * CH_K;
    if (n <= 4) { if (threadIdx.x < CH_K) map[threadIdx.x] = 255; return; }
    __shared__ int32_t s_draw[SW + SW_TAIL];
    __shared__ uint16_t jump[2][SW];
    __shared__ uint8_t cur_e[CH_K];
    const int64_t B0 = round_base == 0 ? 0 : w.smp_state[2 * set];
    const int64_t c_begin = B0 + (int64_t)chunk * CH_DRAWS;
    const TabGet slow{ w.rng_tab, w.rng_len, (uint32_t)n };
    if (threadIdx.x < CH_K) cur_e[threadIdx.x] = (uint8_t)threadIdx.x;
    constexpr uint16_t BAD = 0xffff;
    for (int k = 0; k < CH_WINDOWS; k++) {
        const int64_t base = c_begin + (int64_t)k * SW;
        __syncthreads();
        for (int j = threadIdx.x; j < SW + SW_TAIL; j += SMP_THREADS) {
            const int64_t pp = base + j;
            s_draw[j] = pp < w.rng_len ? (int32_t)(w.rng_tab[pp] % (uint32_t)n) : -1;
        }
        __syncthreads();
        auto get = [&](int64_t pos) -> int {
            const int64_t j = pos - base;
            return (j >= 0 && j < SW + SW_TAIL) ? s_draw[j] : slow(pos);
        };
        #pragma unroll 1
        for (int q = 0; q < SW_PER_THREAD; q++) {
            const int o = q * SMP_THREADS + threadIdx.x;
            int idx[4];
            const int c = draw_subset_g(get, base + o, idx);
            // values >= SW are terminal: SW + (offset into the next window), or BAD (table overrun / absurd consumption)
            jump[0][o] = (uint16_t)((c <= 0 || c >= 0x4000) ? BAD : o + c);
        }
        __syncthreads();
        int cur = 0;
        #pragma unroll 1
        for (int r = 0; r < SW_ROUNDS; r++) {
            #pragma unroll
            for (int q = 0; q < SW_PER_THREAD; q++) {
                const int o = q * SMP_THREADS + threadIdx.x;
                const uint16_t j = jump[cur][o];
                jump[cur ^ 1][o] = j < SW ? jump[cur][j] : j;
            }
            __syncthreads();
            cur ^= 1;
        }
        if (threadIdx.x < CH_K) {
            const uint8_t e = cur_e[threadIdx.x];
            uint8_t out = 255;
            if (e != 255) {
                const uint16_t t = jump[cur][e];
                if (t != BAD && t >= SW && t - SW < CH_K && t - SW < 255) out = (uint8_t)(t - SW);
            }
            cur_e[threadIdx.x] = out;
        }
    }
    __syncthreads();
    if (threadIdx.x < CH_K) map[threadIdx.x] = cur_e[threadIdx.x];
}

// one CTA per set: entry(0) = 0, entry(c+1) = map_c[entry(c)]; -1 from the first chunk whose map has no answer
constexpr int CH_ENTRY_BATCH = 64;
__global__ void __launch_bounds__(256)
ransac_sample_entry_kernel(int n_chunks, const uint8_t* __restrict__ maps, int32_t* __restrict__ entries)
{
    const int set = blockIdx.x;
    __shared__ uint32_t s_maps[CH_ENTRY_BATCH * CH_K / 4];
    __shared__ int32_t s_ent[CH_ENTRY_BATCH];
    __shared__ int s_e;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(maps + (size_t)set * n_chunks * CH_K);
    int32_t* ent = entries + (size_t)set * n_chunks;
    if (threadIdx.x == 0) s_e = 0;
    for (int c0 = 0; c0 < n_chunks; c0 += CH_ENTRY_BATCH) {
        const int m = min(CH_ENTRY_BATCH, n_chunks - c0);
        __syncthreads();
        for (int i = threadIdx.x; i < m * (CH_K / 4); i += blockDim.x) s_maps[i] = src[(size_t)c0 * (CH_K / 4) + i];
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint8_t* mp = reinterpret_cast<const uint8_t*>(s_maps);
            int e = s_e;
            for (int c = 0; c < m; c++) {
                s_ent[c] = e;
                if (e >= 0) { const uint8_t x = mp[c * CH_K + e]; e = x == 255 ? -1 : (int)x; }
            }
            s_e = e;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += blockDim.x) ent[c0 + i] = s_ent[i];
    }
}

__global__ void __launch_bounds__(SMP_THREADS)
ransac_sample_chunk_kernel(RansacWork w, int round_base, int n_chunks, const int32_t* __restrict__ entries,
                           ChunkOut* __restrict__ outs, int32_t* __restrict__ lists)
{
    const int set = blockIdx.y, chunk = blockIdx.x;
    const int n = w.counts_n[set];
    ChunkOut* out = outs + (size_t)set * n_chunks + chunk;
    int32_t* list = lists + ((size_t)set * n_chunks + chunk) * CH_LIST;
    if (n <= 4 || (round_base > 0 && (w.smp_state[2 * set + 1] < 0 || w.n_samples[set] < round_base))) {
        if (threadIdx.x == 0) { out->entry = out->exit = 0; out->n_ok = out->n_nodes = out->head = out->tail = 0; out->flags = 4; }
        return;                                                   // flags 4: nothing to do for this set
    }
    const float4* __restrict__ pts = w.pts + w.starts[set];
    __shared__ float4 spts[SMEM_PTS];
    __shared__ uint16_t info[SW];
    __shared__ int32_t s_draw[SW + SW_TAIL];
    __shared__ uint16_t jump[2][SW];
    __shared__ uint8_t reach[SW];
    __shared__ int s_wsum[SMP_THREADS / 32][2];
    __shared__ int s_last, s_first_ok, s_last_ok, s_bad;
    const bool staged = n <= SMEM_PTS;
    if (staged)
        for (int i = threadIdx.x; i < n; i += SMP_THREADS) spts[i] = pts[i];
    const int64_t B0 = round_base == 0 ? 0 : w.smp_state[2 * set];
    const int64_t c_begin = B0 + (int64_t)chunk * CH_DRAWS, c_end = c_begin + CH_DRAWS;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const TabGet slow{ w.rng_tab, w.rng_len, (uint32_t)n };
    int flags = 0;
    const int entry_off = entries[(size_t)set * n_chunks + chunk];    // chunk 0 enters exactly at B0 (offset 0)
    if (entry_off < 0) flags |= 2;                                // an earlier chunk's map had no answer: serial kernel
    int64_t base = c_begin + max(entry_off, 0);
    int sw_eff = (int)min((int64_t)SW, c_end - base);
    if (c_end + SW + SW_TAIL + 64 >= w.rng_len) flags |= 1;       // the table must cover the chunk and its look-ahead
    int n_ok_total = 0, n_nodes_total = 0, head = 0, run = 0;
    bool seen_ok = false;
    const int64_t entry = base;
    int64_t exit_pos = base;
    while (!flags) {
        __syncthreads();
        for (int j = threadIdx.x; j < SW + SW_TAIL; j += SMP_THREADS) {
            const int64_t pp = base + j;
            s_draw[j] = pp < w.rng_len ? (int32_t)(w.rng_tab[pp] % (uint32_t)n) : -1;
        }
        if (threadIdx.x == 0) { s_last = 0; s_first_ok = SW; s_last_ok = -1; s_bad = 0; }
        __syncthreads();
        auto get = [&](int64_t pos) -> int {
            const int64_t j = pos - base;
            return (j >= 0 && j < SW + SW_TAIL) ? s_draw[j] : slow(pos);
        };
        #pragma unroll 1
        for (int k = 0; k < SW_PER_THREAD; k++) {
            const int o = k * SMP_THREADS + threadIdx.x;
            uint16_t e = 0;
            if (o < sw_eff) {
                int idx[4];
                const int cons = draw_subset_g(get, base + o, idx);
                if (cons > 0 && cons < 0x7fff) {
                    float ms1[8], ms2[8];
                    #pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const float4 q = staged ? spts[idx[i]] : pts[idx[i]];
                        ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
                    }
                    e = (uint16_t)(cons | (check_subset4(ms1, ms2) ? 0x8000 : 0));
                }
            }
            info[o] = e;
            const int c = e & 0x7fff;
            jump[0][o] = (uint16_t)((o >= sw_eff || c == 0 || o + c >= sw_eff) ? SW : o + c);
            reach[o] = o == 0 ? 1 : 0;
        }
        __syncthreads();
        int cur = 0;
        #pragma unroll 1
        for (int r = 0; r < SW_ROUNDS; r++) {
            #pragma unroll
            for (int k = 0; k < SW_PER_THREAD; k++) {
                const int o = k * SMP_THREADS + threadIdx.x;
                const int j = jump[cur][o];
                if (reach[o] && j < SW) reach[j] = 1;
                jump[cur ^ 1][o] = (uint16_t)(j < SW ? jump[cur][j] : SW);
            }
            __syncthreads();
            cur ^= 1;
        }
        // rank the chain nodes (blocked layout, so ranks follow stream order)
        int n_reach = 0, n_ok = 0, mask_r = 0, mask_ok = 0;
        #pragma unroll
        for (int k = 0; k < SW_PER_THREAD; k++) {
            const int o = threadIdx.x * SW_PER_THREAD + k;
            if (reach[o]) {
                const uint16_t e = info[o];
                mask_r |= 1 << k; n_reach++;
                if ((e & 0x7fff) == 0) atomicExch(&s_bad, 1);
                if (e & 0x8000) { mask_ok |= 1 << k; n_ok++; atomicMin(&s_first_ok, o); atomicMax(&s_last_ok, o); }
                atomicMax(&s_last, o);
            }
        }
        int pre_r = n_reach, pre_ok = n_ok;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, pre_r, d), b2 = __shfl_up_sync(0xffffffffu, pre_ok, d);
            if (lane >= d) { pre_r += a; pre_ok += b2; }
        }
        if (lane == 31) { s_wsum[wid][0] = pre_r; s_wsum[wid][1] = pre_ok; }
        __syncthreads();
        int off_ok = 0, tot_r = 0, tot_ok = 0;
        #pragma unroll
        for (int q = 0; q < SMP_THREADS / 32; q++) {
            if (q < wid) off_ok += s_wsum[q][1];
            tot_r += s_wsum[q][0]; tot_ok += s_wsum[q][1];
        }
        const int excl_ok = off_ok + pre_ok - n_ok;
        const int first_ok = s_first_ok, last_ok = s_last_ok, last = s_last;
        if (s_bad) { flags |= 1; break; }
        int fails_head = 0, fails_tail = 0;
        {
            int h = 0, t = 0;
            #pragma unroll
            for (int k = 0; k < SW_PER_THREAD; k++) {
                const int o = threadIdx.x * SW_PER_THREAD + k;
                if ((mask_r >> k) & 1) { h += o < first_ok; t += o > last_ok; }
            }
            #pragma unroll
            for (int d = 16; d > 0; d >>= 1) { h += __shfl_xor_sync(0xffffffffu, h, d); t += __shfl_xor_sync(0xffffffffu, t, d); }
            __syncthreads();
            if (lane == 0) { s_wsum[wid][0] = h; s_wsum[wid][1] = t; }
            __syncthreads();
            #pragma unroll
            for (int q = 0; q < SMP_THREADS / 32; q++) { fails_head += s_wsum[q][0]; fails_tail += s_wsum[q][1]; }
        }
        // failure runs: `run` = consecutive failed chain nodes since the chunk's last accept (or since its entry).  A window
        // holds at most SW / 4 = 512 nodes, so a run of 10000 always spans windows and shows up in these sums.
        if (tot_ok > 0) {
            const int gap = run + fails_head;
            if (!seen_ok) head = gap;
            else if (gap >= 10000) { flags |= 2; break; }         // getSubset would have given up inside the chunk
            seen_ok = true; run = fails_tail;
        } else run += tot_r;
        if (seen_ok && run >= 10000) { flags |= 2; break; }
        {
            int r = n_ok_total + excl_ok;
            #pragma unroll
            for (int k = 0; k < SW_PER_THREAD; k++)
                if ((mask_ok >> k) & 1) { if (r < CH_LIST) list[r] = (int32_t)(base + threadIdx.x * SW_PER_THREAD + k); r++; }
        }
        n_ok_total += tot_ok; n_nodes_total += tot_r;
        base = base + last + (info[last] & 0x7fff);
        if (base >= c_end) { exit_pos = base; break; }
        sw_eff = (int)min((int64_t)SW, c_end - base);
        if (base + SW + SW_TAIL + 64 >= w.rng_len) { flags |= 1; break; }
    }
    if (threadIdx.x == 0) {
        out->entry = entry; out->exit = exit_pos; out->n_ok = n_ok_total; out->n_nodes = n_nodes_total;
        out->head = seen_ok ? head : run; out->tail = run; out->flags = flags | (n_ok_total > CH_LIST ? 2 : 0);
    }
}

// one thread per set walks the chunk summaries in order
__global__ void ransac_sample_stitch_kernel(RansacWork w, int round_base, int round_end, int n_chunks,
                                            const ChunkOut* __restrict__ outs, const int32_t* __restrict__ lists,
                                            int32_t* __restrict__ offsets, int* __restrict__ serial_flag)
{
    const int set = blockIdx.x * blockDim.x + threadIdx.x;
    if (set >= w.n_sets) return;
    const ChunkOut* o = outs + (size_t)set * n_chunks;
    int32_t* off = offsets + (size_t)set * n_chunks;
    serial_flag[set] = 0;
    for (int c = 0; c < n_chunks; c++) off[c] = -1;
    const int n = w.counts_n[set];
    if (round_base == 0) {
        w.niters_cur[set] = max(w.max_iters, 1); w.best_iter[set] = -1; w.best_count[set] = 0;
        w.n_samples[set] = 0; w.status_flags[set] = 0;
        w.smp_state[2 * set] = 0; w.smp_state[2 * set + 1] = 0;
    }
    if (o[0].flags & 4) return;
    int64_t expect = round_base == 0 ? 0 : w.smp_state[2 * set];
    int attempts = round_base == 0 ? 0 : (int)w.smp_state[2 * set + 1];
    int iter = round_base, flags = 0;
    bool finished = false, done = false, unsafe = false;
    for (int c = 0; c < n_chunks && !done; c++) {
        if (o[c].flags & 2) { unsafe = true; break; }
        if (o[c].flags & 1) { flags |= 1; finished = true; break; }
        if (o[c].entry != expect) { unsafe = true; break; }
        off[c] = iter;
        if (o[c].n_ok == 0) {
            attempts += o[c].n_nodes;
            if (attempts >= 10000) { unsafe = true; break; }      // exact give-up point: let the serial kernel find it
        } else {
            if (attempts + o[c].head >= 10000) { unsafe = true; break; }
            attempts = o[c].tail;
        }
        if (iter + o[c].n_ok >= round_end) {
            const int need = round_end - iter;                    // >= 1
            const int64_t p = lists[((size_t)set * n_chunks + c) * CH_LIST + need - 1];
            int idx[4];
            const int cons = draw_subset(w.rng_tab, w.rng_len, p, (uint32_t)n, idx);
            expect = p + cons; attempts = 0; iter = round_end; done = true;
        } else {
            iter += o[c].n_ok; expect = o[c].exit;
        }
    }
    if (unsafe) {
        serial_flag[set] = 1; if (w.chunk_serial_count) atomicAdd(w.chunk_serial_count, 1);
        for (int c = 0; c < n_chunks; c++) off[c] = -1;
        return;
    }
    if (!done && !finished) { flags |= 1; finished = true; }     // the chunks (= the draw table) ended before the round did
    w.n_samples[set] = iter;
    if (flags) { w.status_flags[set] = flags; if (w.err_flag) atomicOr(w.err_flag, flags); }
    w.smp_state[2 * set] = expect;
    w.smp_state[2 * set + 1] = finished ? -1 : attempts;
}

__global__ void ransac_sample_scatter_kernel(RansacWork w, int round_end, int n_chunks, const ChunkOut* __restrict__ outs,
                                             const int32_t* __restrict__ lists, const int32_t* __restrict__ offsets)
{
    const int set = blockIdx.y, chunk = blockIdx.x;
    const int o = offsets[(size_t)set * n_chunks + chunk];
    if (o < 0) return;
    const int cnt = outs[(size_t)set * n_chunks + chunk].n_ok;
    const int32_t* list = lists + ((size_t)set * n_chunks + chunk) * CH_LIST;
    int32_t* dst = w.sample_pos + (size_t)set * w.max_iters;
    for (int r = threadIdx.x; r < cnt; r += blockDim.x)
        if (o + r < round_end) dst[o + r] = list[r];
}

// ---- 2. hypothesis kernels: solve + score -----------------------------------------------------------
// Generic variant (CVG_HYP_MODE=3, kept as the plain restatement the others are checked against): the serial
// routine of homography_math.cuh per thread.  LtL and V (162 doubles, dynamically indexed) live in shared memory —
// as thread-local arrays they thrash L1 — element-major (element e of thread t at e*HYP_THREADS + t), so the
// divergent indices of 32 different Jacobi sweeps never conflict.
constexpr int JAC_DOUBLES = 162;

template <int S>
__device__ __forceinline__ bool solve_hypothesis(const RansacWork& w, const float4* __restrict__ pts, int n,
                                                 int32_t pos, float Hf[8], double* Hd, double* jac)
{
    int idx[4];
    draw_subset(w.rng_tab, w.rng_len, pos, (uint32_t)n, idx);
    float ms1[8], ms2[8];
    #pragma unroll
    for (int i = 0; i < 4; i++) {
        const float4 q = pts[idx[i]];
        ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
    }
    double H[9];
    Pts4 P{ ms1, ms2 };
    if (!run_kernel_seq<Pts4, S>(P, 4, H, jac, jac + 81 * S)) return false;
    #pragma unroll
    for (int i = 0; i < 8; i++) Hf[i] = (float)H[i];
    if (Hd) for (int i = 0; i < 9; i++) Hd[i] = H[i];
    return true;
}

constexpr int HYP_THREADS = 64;
constexpr int HYP_PTS = 512;
constexpr int HYP_SMEM = HYP_THREADS * JAC_DOUBLES * 8 + HYP_PTS * 16;

__global__ void __launch_bounds__(HYP_THREADS)
ransac_hyp_kernel(RansacWork w, int round_base)
{
    extern __shared__ double hyp_smem[];
    const int set = blockIdx.y;
    const int n = w.counts_n[set];
    const int n_samples = w.n_samples[set];
    const int iter0 = round_base + blockIdx.x * HYP_THREADS;
    // hypotheses at or beyond the adaptive niters (as known after the previous round) are never looked at
    if (iter0 >= n_samples || iter0 >= w.niters_cur[set]) return;
    const float4* __restrict__ pts = w.pts + w.starts[set];
    const int iter = iter0 + threadIdx.x;
    const bool active = iter < n_samples;
    float Hf[8];
    bool valid = false;
    if (active)
        valid = solve_hypothesis<HYP_THREADS>(w, pts, n, w.sample_pos[(size_t)set * w.max_iters + iter], Hf, nullptr,
                                              hyp_smem + threadIdx.x);
    if (!valid) {
        #pragma unroll
        for (int i = 0; i < 8; i++) Hf[i] = 0.f;
    }
    float4* spts = reinterpret_cast<float4*>(hyp_smem + HYP_THREADS * JAC_DOUBLES);
    int good = 0;
    for (int base = 0; base < n; base += HYP_PTS) {
        const int cnt = min(HYP_PTS, n - base);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += HYP_THREADS) spts[i] = pts[base + i];
        __syncthreads();
        #pragma unroll 4
        for (int i = 0; i < cnt; i++) {
            const float4 q = spts[i];                              // broadcast read
            const float e = reproj_err(Hf, q.x, q.y, q.z, q.w);
            good += (e <= w.thr2) ? 1 : 0;                         // NaN -> not an inlier
        }
    }
    if (active) w.counts[(size_t)set * w.max_iters + iter] = valid ? good : -1;
    if (w.scored_pts) {                                  // algorithmic traffic of the scoring: one float4 per (hypothesis, point)
        const unsigned bal = __ballot_sync(0xffffffffu, active && valid);
        if ((threadIdx.x & 31) == 0 && bal) atomicAdd(w.scored_pts, (unsigned long long)__popc(bal) * (unsigned long long)n);
    }
}

// Warp-per-hypothesis variant, used when a round holds too few hypotheses to hide the latency of
// thread-serial Jacobi sweeps (few image pairs in flight): the warp solves the DLT cooperatively
// (jacobi_warp.cuh), then its lanes score the correspondences with coalesced float4 reads and a
// warp-reduced count.  Bit-identical to ransac_hyp_kernel.
constexpr int HYPW_WARPS = 8;
constexpr int HYPW_SMEM_D = 81 + 81 + 9 + 72;       // doubles of scratch per warp

__global__ void __launch_bounds__(HYPW_WARPS * 32)
ransac_hyp_warp_kernel(RansacWork w, int round_base)
{
    __shared__ double smem[HYPW_WARPS][HYPW_SMEM_D];
    const int set = blockIdx.y;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = w.counts_n[set];
    const int n_samples = w.n_samples[set];
    const int iter = round_base + blockIdx.x * HYPW_WARPS + wid;
    if (iter >= n_samples || iter >= w.niters_cur[set]) return;          // warp-uniform
    const float4* __restrict__ pts = w.pts + w.starts[set];
    int idx[4];
    draw_subset(w.rng_tab, w.rng_len, w.sample_pos[(size_t)set * w.max_iters + iter], (uint32_t)n, idx);
    float ms1[8], ms2[8];
    #pragma unroll
    for (int i = 0; i < 4; i++) {
        const float4 q = pts[idx[i]];
        ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
    }
    double H[9];
    const bool valid = run_kernel4_warp(ms1, ms2, H, smem[wid]);
    int good = -1;
    if (valid) {
        float Hf[8];
        #pragma unroll
        for (int i = 0; i < 8; i++) Hf[i] = (float)H[i];
        int cnt = 0;
        for (int i = lane; i < n; i += 32) {
            const float4 q = pts[i];
            cnt += reproj_err(Hf, q.x, q.y, q.z, q.w) <= w.thr2 ? 1 : 0;
        }
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        good = cnt;
    }
    if (lane == 0) {
        w.counts[(size_t)set * w.max_iters + iter] = good;
        if (w.scored_pts && valid) atomicAdd(w.scored_pts, (unsigned long long)n);
        if (w.hyp_H && valid) {                                  // the finish kernel reads the winner's model from here
            float4* dst = reinterpret_cast<float4*>(w.hyp_H + ((size_t)set * w.max_iters + iter) * 8);
            dst[0] = make_float4((float)H[0], (float)H[1], (float)H[2], (float)H[3]);
            dst[1] = make_float4((float)H[4], (float)H[5], (float)H[6], (float)H[7]);
        }
    }
}

// Four hypotheses per warp (8-lane groups, jacobi9_g8): the variant for rounds that fill the chip, where
// the hypothesis kernel is bound by instruction issue and the rotation's scalar chain should be shared.
constexpr int HYPG_WARPS = 8;
constexpr int HYPG_SMEM = HYPG_WARPS * 4 * HYPW_SMEM_D * 8;      // 62 KB

__global__ void __launch_bounds__(HYPG_WARPS * 32)
ransac_hyp_g8_kernel(RansacWork w, int round_base)
{
    extern __shared__ double g8_smem[];
    const int set = blockIdx.y;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 3, j = lane & 7;
    const int n = w.counts_n[set];
    const int n_samples = w.n_samples[set];
    const int iter = round_base + (blockIdx.x * HYPG_WARPS + wid) * 4 + g;
    const bool live = iter < n_samples && iter < w.niters_cur[set];
    if (!__any_sync(0xffffffffu, live)) return;
    const float4* __restrict__ pts = w.pts + w.starts[set];
    float ms1[8], ms2[8];
    #pragma unroll
    for (int i = 0; i < 8; i++) { ms1[i] = 0.f; ms2[i] = 0.f; }
    if (live) {
        int idx[4];
        draw_subset(w.rng_tab, w.rng_len, w.sample_pos[(size_t)set * w.max_iters + iter], (uint32_t)n, idx);
        #pragma unroll
        for (int i = 0; i < 4; i++) {
            const float4 q = pts[idx[i]];
            ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
        }
    }
    double H[9];
    const bool valid = run_kernel4_g8(ms1, ms2, H, g8_smem + (size_t)(wid * 4 + g) * HYPW_SMEM_D, live);
    float Hf[8];
    #pragma unroll
    for (int i = 0; i < 8; i++) Hf[i] = valid ? (float)H[i] : 0.f;
    int cnt = 0;
    for (int i = j; i < n; i += 8) {                              // the four groups read the same 128 B per step
        const float4 q = pts[i];
        cnt += reproj_err(Hf, q.x, q.y, q.z, q.w) <= w.thr2 ? 1 : 0;
    }
    #pragma unroll
    for (int o = 4; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (live && j == 0) {
        w.counts[(size_t)set * w.max_iters + iter] = valid ? cnt : -1;
        if (w.scored_pts && valid) atomicAdd(w.scored_pts, (unsigned long long)n);
    }
}

// One hypothesis per THREAD with the register/predication-friendly Jacobi of jacobi_thread.cuh: the variant for
// rounds that fill the chip (>= a few thousand hypotheses).  A warp retires 32 rotations with 771 instructions
// where the 8-lane-group kernel needs ~2900.  224 threads x 126 doubles of matrix state = 220.5 KB of shared
// memory, one CTA per SM.  Hypotheses are numbered flat over (set, iteration) so CTAs stay full whatever the
// round length; lanes of one warp almost always share a set, so the scoring loop's float4 loads are warp-uniform
// (one L1 transaction, broadcast).  Bit-identical to the other hypothesis kernels.
#ifndef HYPT_THREADS_DEF
#define HYPT_THREADS_DEF 224
#define HYPT_CTAS_DEF 1
#endif
constexpr int HYPT_THREADS = HYPT_THREADS_DEF;
constexpr int HYPT_CTAS_PER_SM = HYPT_CTAS_DEF;
constexpr int HYPT_SMEM = HYPT_THREADS * JT_DOUBLES * 8;

struct WarpAny { __device__ __forceinline__ bool operator()(bool x) const { return __any_sync(0xffffffffu, x); } };

__global__ void __launch_bounds__(HYPT_THREADS, HYPT_CTAS_PER_SM)
ransac_hyp_t_kernel(RansacWork w, int round_base, int round_len)
{
    extern __shared__ double jt_smem[];
    const int64_t h0 = (int64_t)blockIdx.x * HYPT_THREADS;
    const int64_t h = h0 + threadIdx.x;
    const int set = (int)(h / round_len);
    const int iter = round_base + (int)(h - (int64_t)set * round_len);
    bool live = set < w.n_sets;
    int n = 0;
    const float4* __restrict__ pts = w.pts;
    if (live) {
        n = w.counts_n[set];
        live = iter < w.n_samples[set] && iter < w.niters_cur[set];
        pts = w.pts + w.starts[set];
    }
    if (!__syncthreads_or(live)) return;                        // block-uniform
    float ms1[8], ms2[8];
    #pragma unroll
    for (int i = 0; i < 8; i++) { ms1[i] = 0.f; ms2[i] = 0.f; }
    if (live) {
        int idx[4];
        draw_subset(w.rng_tab, w.rng_len, w.sample_pos[(size_t)set * w.max_iters + iter], (uint32_t)n, idx);
        #pragma unroll
        for (int i = 0; i < 4; i++) {
            const float4 q = pts[idx[i]];
            ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
        }
    }
    float Hf[8];
    bool valid;
    {
        double H[9];
        valid = run_kernel4_thread<HYPT_THREADS>(ms1, ms2, H, jt_smem + threadIdx.x, live, WarpAny());
        #pragma unroll
        for (int i = 0; i < 8; i++) Hf[i] = valid ? (float)H[i] : 0.f;
    }
    if (w.hyp_H) {
        // split mode: the model goes to HBM (32 B), ransac_score_kernel counts its inliers at full occupancy
        if (live) {
            float4* dst = reinterpret_cast<float4*>(w.hyp_H + ((size_t)set * w.max_iters + iter) * 8);
            dst[0] = make_float4(Hf[0], Hf[1], Hf[2], Hf[3]);
            dst[1] = make_float4(Hf[4], Hf[5], Hf[6], Hf[7]);
            w.counts[(size_t)set * w.max_iters + iter] = valid ? 0 : -1;
        }
        if (w.scored_pts) {                                  // statistics (timing enabled only): one atomic per warp, not per thread
            unsigned long long v = (live && valid) ? (unsigned long long)n : 0ull;
            #pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if ((threadIdx.x & 31) == 0 && v) atomicAdd(w.scored_pts, v);
        }
        return;
    }
    // ---- scoring: the matrix state is dead, the CTA's shared memory becomes a staging buffer for the
    //      correspondences of the (one or two, rarely more) sets its hypotheses belong to ----
    constexpr int STAGE_PTS = HYPT_SMEM / 16;                   // 14 112 correspondences
    float4* stage = reinterpret_cast<float4*>(jt_smem);
    const int set_first = (int)(h0 / round_len);
    const int set_last = min((int)((h0 + HYPT_THREADS - 1) / round_len), w.n_sets - 1);
    int cnt = 0;
    for (int s = set_first; s <= set_last; s++) {
        const int ns = w.counts_n[s];
        const float4* __restrict__ ps = w.pts + w.starts[s];
        const bool mine = live && valid && set == s;
        for (int base = 0; base < ns; base += STAGE_PTS) {
            const int m = min(STAGE_PTS, ns - base);
            __syncthreads();                                    // previous contents (matrix state or chunk) are consumed
            for (int i = threadIdx.x; i < m; i += HYPT_THREADS) stage[i] = ps[base + i];
            __syncthreads();
            if (mine) {
                #pragma unroll 4
                for (int i = 0; i < m; i++) {
                    const float4 q = stage[i];                  // same address in every lane: broadcast
                    cnt += reproj_err(Hf, q.x, q.y, q.z, q.w) <= w.thr2 ? 1 : 0;     // NaN -> not an inlier
                }
            }
        }
    }
    if (live) {
        w.counts[(size_t)set * w.max_iters + iter] = valid ? cnt : -1;
        if (w.scored_pts && valid) atomicAdd(w.scored_pts, (unsigned long long)n);
    }
}

// Scoring of the models ransac_hyp_t_kernel left in hyp_H: one hypothesis per thread, a CTA = SCORE_THREADS
// consecutive iterations of ONE set x one slice of its correspondences (blockIdx.z), staged in shared memory and read
// as warp-uniform float4 broadcasts.  The solve kernel holds 7 warps per SM (its matrix state fills shared memory);
// here a CTA needs 32 KB, so the fp32 pipe sees 48+ warps.  Slices add their counts with atomicAdd (integer: order-free).
constexpr int SCORE_THREADS = 256;
constexpr int SCORE_STAGE = 2048;
__global__ void __launch_bounds__(SCORE_THREADS)
ransac_score_kernel(RansacWork w, int round_base, int round_len, int n_slices, int tiles)
{
    __shared__ float4 stage[SCORE_STAGE];
    const int set = (int)(blockIdx.x / (unsigned)tiles);         // sets on x: no 65535 limit on their number
    const int r = (int)(blockIdx.x % (unsigned)tiles) * SCORE_THREADS + threadIdx.x;
    const int iter = round_base + r;
    const int n = w.counts_n[set];
    const size_t slot = (size_t)set * w.max_iters + iter;
    bool live = r < round_len && iter < w.n_samples[set] && iter < w.niters_cur[set];
    if (live) live = w.counts[slot] >= 0;                        // -1: degenerate sample, no model
    if (!__syncthreads_or(live)) return;
    float Hf[8];
    if (live) {
        const float4* src = reinterpret_cast<const float4*>(w.hyp_H + slot * 8);
        const float4 a = src[0], b = src[1];
        Hf[0] = a.x; Hf[1] = a.y; Hf[2] = a.z; Hf[3] = a.w; Hf[4] = b.x; Hf[5] = b.y; Hf[6] = b.z; Hf[7] = b.w;
    } else {
        #pragma unroll
        for (int i = 0; i < 8; i++) Hf[i] = 0.f;
    }
    const int per = (n + n_slices - 1) / n_slices;
    const int p0 = min(n, (int)blockIdx.z * per), p1 = min(n, p0 + per);
    const float4* __restrict__ ps = w.pts + w.starts[set];
    const float thr2 = w.thr2;
    int cnt = 0;
    for (int base = p0; base < p1; base += SCORE_STAGE) {
        const int m = min(SCORE_STAGE, p1 - base);
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += SCORE_THREADS) stage[i] = ps[base + i];
        __syncthreads();
        if (live) {
            int i = 0;
            #pragma unroll 2
            for (; i + 4 <= m; i += 4)
                cnt += count_inliers4(Hf, stage[i], stage[i + 1], stage[i + 2], stage[i + 3], thr2);
            for (; i < m; i++) {
                const float4 q = stage[i];
                cnt += reproj_err(Hf, q.x, q.y, q.z, q.w) <= thr2 ? 1 : 0;     // NaN -> not an inlier
            }
        }
    }
    if (live && cnt) {
        if (n_slices == 1) w.counts[slot] = cnt; else atomicAdd(&w.counts[slot], cnt);
    }
}

// ---- 3. select kernel: the serial scan of RANSACPointSetRegistrator::run --------------------------
// cv::RANSACUpdateNumIters(confidence, (double)(n - good) / n, mp, niters) for the whole warp (same arguments in every lane),
// mp = w.model_points.
// log(1 - confidence) comes from the host; log(1 - (1 - ep)^mp) comes from the host-verified table when the entry is listed,
// else from CUDA's log / pow with a check that neither the cap comparison nor cvRound is within nit_margin of flipping
// (then the pair is sent to the host and the call repeats the verify stage, see run_ransac in api.cu).
__device__ int update_num_iters_checked(const RansacWork& w, int n, int good, int niters, int lane)
{
    int found = -1;
    for (int i = lane; i < w.nit_n; i += 32)
        if (w.nit_tab[i].n == n && w.nit_tab[i].good == good && w.nit_tab[i].mp == w.model_points) found = i;
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) found = max(found, __shfl_xor_sync(0xffffffffu, found, o));
    double ep = (double)(n - good) / n;
    ep = ep > 0. ? ep : 0.; ep = ep < 1. ? ep : 1.;
    const double num = w.log_num;
    double denom; bool zero;
    if (found >= 0) { denom = w.nit_tab[found].denom_log; zero = w.nit_tab[found].zero != 0; }
    else {
        const double d0 = 1. - (w.model_points == 4 ? pow(1. - ep, 4.0) : w.model_points == 3 ? pow(1. - ep, 3.0)
                                                                                                 : pow(1. - ep, 2.0));
        zero = d0 < DBL_MIN;
        denom = zero ? -1. : log(d0);
    }
    int result;
    if (zero) result = 0;
    else if (denom >= 0 || -num >= niters * (-denom)) result = niters;
    else result = (int)rint(num / denom);            // cvRound: round half to even
    if (found < 0 && w.nit_req) {
        bool unsure = zero || !(denom < 0);           // never reached with good >= mp; let the host decide if it is
        if (!unsure) {
            // q >= niters: the cap wins and nothing is rounded; only a quotient within the margin of the cap, or — below the
            // cap — within the margin of a half-integer, could come out differently with the host's log / pow
            const double q = num / denom;
            const double m = w.nit_margin * ((double)niters + 1.);
            unsure = fabs(q - (double)niters) < m || (q < (double)niters && fabs(q - floor(q) - 0.5) < m);
        }
        if (unsure && lane == 0) {
            const int slot = atomicAdd(w.nit_req_n, 1);
            if (slot < w.nit_req_cap) w.nit_req[slot] = make_int2(n, good);
            if (w.err_flag) atomicOr(w.err_flag, 2);
        }
    }
    return result;
}

__global__ void ransac_select_kernel(RansacWork w, int round_base, int round_len)
{
    const int set = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (set >= w.n_sets) return;
    const int n = w.counts_n[set];
    const int n_samples = w.n_samples[set];
    const int32_t* __restrict__ counts = w.counts + (size_t)set * w.max_iters;
    int niters = w.niters_cur[set];
    int best = w.best_count[set], best_iter = w.best_iter[set];
    const int floor_good = w.model_points - 1;                     // good > max(best, modelPoints - 1)
    int base = round_base;
    const int end = min(round_base + round_len, n_samples);
    while (base < niters && base < end) {
        const int it = base + lane;
        const int c = (it < end) ? counts[it] : -1;
        int start = 0;
        for (;;) {
            const bool cand = lane >= start && it < niters && it < end && c > max(best, floor_good);
            const unsigned bal = __ballot_sync(0xffffffffu, cand);
            if (!bal) break;
            const int f = __ffs(bal) - 1;
            best = __shfl_sync(0xffffffffu, c, f);
            best_iter = base + f;
            if (!(w.flags & CVG_RANSAC_NO_EARLY_STOP))
                niters = update_num_iters_checked(w, n, best, niters, lane);
            start = f + 1;
        }
        base += 32;
    }
    if (lane == 0) {
        w.best_iter[set] = best_iter;
        w.best_count[set] = best;
        w.niters_cur[set] = niters;
        // value of `iter` when the reference loop exits
        w.iters_run[set] = n <= w.model_points ? 0 : min(max(niters, best_iter + 1), n_samples);
    }
}

// Without the adaptive stop (CVG_RANSAC_NO_EARLY_STOP) niters never changes, so the serial scan reduces to "first
// iteration with the largest count, if it beats the running best and modelPoints - 1": a block-wide argmax, one CTA per set.
constexpr int SELP_THREADS = 256;
__global__ void __launch_bounds__(SELP_THREADS)
ransac_select_all_kernel(RansacWork w, int round_base, int round_len)
{
    const int set = blockIdx.x;
    const int n = w.counts_n[set];
    const int n_samples = w.n_samples[set];
    const int32_t* __restrict__ counts = w.counts + (size_t)set * w.max_iters;
    const int end = min(min(round_base + round_len, n_samples), w.niters_cur[set]);
    // key = (count, first index wins): larger count first, then smaller index
    long long best = -1;
    for (int it = round_base + (int)threadIdx.x; it < end; it += SELP_THREADS) {
        const long long key = ((long long)counts[it] << 32) | (unsigned int)(0x7fffffff - it);
        best = key > best ? key : best;
    }
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const long long ob = __shfl_xor_sync(0xffffffffu, best, o); best = ob > best ? ob : best; }
    __shared__ long long s_best[SELP_THREADS / 32];
    if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < SELP_THREADS / 32; k++) best = s_best[k] > best ? s_best[k] : best;
        int bc = w.best_count[set], bi = w.best_iter[set];
        if (best >= 0) {
            const int c = (int)(best >> 32), it = 0x7fffffff - (int)(unsigned int)best;
            if (c > max(bc, w.model_points - 1)) { bc = c; bi = it; }
        }
        w.best_count[set] = bc; w.best_iter[set] = bi;
        const int niters = w.niters_cur[set];
        w.iters_run[set] = n <= w.model_points ? 0 : min(max(niters, bi + 1), n_samples);
    }
}

// ---- block reductions (parallel mode of the finish kernel) ----------------------------------------
__device__ __forceinline__ double shfl_down_d(double v, int o)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_down_sync(0xffffffffu, lo, o);
    hi = __shfl_down_sync(0xffffffffu, hi, o);
    return __hiloint2double(hi, lo);
}

// sums vals[0..K) over the block; result valid in every thread (through out[]); fixed order
template <int K>
__device__ void block_sum(double* vals, double* s_part /*[4*K]*/, double* s_out /*[K]*/)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    #pragma unroll
    for (int k = 0; k < K; k++) {
        double v = vals[k];
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = v + shfl_down_d(v, o);
        if (lane == 0) s_part[wid * K + k] = v;
    }
    __syncthreads();
    if (threadIdx.x < K) {
        double v = s_part[threadIdx.x];
        #pragma unroll
        for (int q = 1; q < (int)(blockDim.x >> 5); q++) v = v + s_part[q * K + threadIdx.x];
        s_out[threadIdx.x] = v;
    }
    __syncthreads();
    #pragma unroll
    for (int k = 0; k < K; k++) vals[k] = s_out[k];
    __syncthreads();
}

struct FinishShared {
    double part[4 * 56];
    double out[56];
    LmState lm;
    double H[9];
    double scratch_a[81], scratch_v[81], scratch_w[9];
    double jac[JAC_DOUBLES];
    double sums[8];
    double J[2 * EXACT_MAX_INLIERS * 9];        // exact mode: Jacobian rows of the current evaluation
    double r[2 * EXACT_MAX_INLIERS];            //             residuals
    float Hf[8];
    int flag;
    int warp_cnt[RS_THREADS / 32];
    int base_cnt;
};

// S, rmax and optionally A, v at parameters h, reduced over the block (parallel mode)
__device__ double lm_eval_block(const float4* __restrict__ pts, const int32_t* __restrict__ sel, int count,
                                const double* h, double* A, double* v, double* rmax, FinishShared& sh)
{
    double acc[56];
    #pragma unroll
    for (int k = 0; k < 56; k++) acc[k] = 0;
    double rm = 0;
    const bool wantJ = A != nullptr;
    for (int i = threadIdx.x; i < count; i += (int)blockDim.x) {
        const float4 q = pts[sel[i]];
        double r0, r1, J0[9], J1[9];
        refine_row(h, q.x, q.y, q.z, q.w, r0, r1, wantJ ? J0 : nullptr, wantJ ? J1 : nullptr);
        acc[55] += r0 * r0; acc[55] += r1 * r1;
        rm = fmax(rm, fmax(fabs(r0), fabs(r1)));
        if (wantJ) {
            int e = 0;
            #pragma unroll
            for (int j = 0; j < 9; j++) {
                #pragma unroll
                for (int k = j; k < 9; k++) { acc[e] += J0[j] * J0[k]; acc[e] += J1[j] * J1[k]; e++; }
                acc[45 + j] += J0[j] * r0; acc[45 + j] += J1[j] * r1;
            }
        }
    }
    // max via the same machinery (monotone: reduce as a sum of one-hot is not possible) -> separate
    acc[54] = 0;
    block_sum<56>(acc, sh.part, sh.out);
    // rmax: warp + block max
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) rm = fmax(rm, shfl_down_d(rm, o));
    if ((threadIdx.x & 31) == 0) sh.part[threadIdx.x >> 5] = rm;
    __syncthreads();
    rm = fmax(fmax(sh.part[0], sh.part[1]), fmax(sh.part[2], sh.part[3]));
    __syncthreads();
    if (wantJ) {
        int e = 0;
        for (int j = 0; j < 9; j++) {
            for (int k = j; k < 9; k++) { A[j * 9 + k] = acc[e]; A[k * 9 + j] = acc[e]; e++; }
            v[j] = acc[45 + j];
        }
    }
    if (rmax) *rmax = rm;
    return acc[55];
}

// Exact-order evaluation (n_inl <= EXACT_MAX_INLIERS): rows are computed in parallel, then every sum is
// accumulated by ONE thread in OpenCV's order (mulTransposed: sequential over rows; gemm: 4 interleaved
// accumulators below 100 rows; norm: the AVX2 pattern) — 56 independent sums on 56 threads.
__device__ double lm_eval_exact(const float4* __restrict__ pts, const int32_t* __restrict__ sel, int count,
                                const double* h, bool wantJ, double* A, double* v, double* rmax, FinishShared& sh)
{
    const int tid = threadIdx.x;
    const int rows = 2 * count;
    for (int i = tid; i < count; i += (int)blockDim.x) {
        const float4 q = pts[sel[i]];
        double r0, r1, J0[9], J1[9];
        refine_row(h, q.x, q.y, q.z, q.w, r0, r1, wantJ ? J0 : nullptr, wantJ ? J1 : nullptr);
        sh.r[2 * i] = r0; sh.r[2 * i + 1] = r1;
        if (wantJ) {
            #pragma unroll
            for (int j = 0; j < 9; j++) { sh.J[(2 * i) * 9 + j] = J0[j]; sh.J[(2 * i + 1) * 9 + j] = J1[j]; }
        }
    }
    __syncthreads();
    if (wantJ && tid < 45) {                              // upper triangle entry (j,k) of J^T J
        int j = 0, e = tid;
        while (e >= 9 - j) { e -= 9 - j; j++; }
        const int k = j + e;
        double s = 0;
        for (int row = 0; row < rows; row++) s += sh.J[row * 9 + j] * sh.J[row * 9 + k];
        sh.out[tid] = s;
    } else if (wantJ && tid >= 45 && tid < 54) {          // J^T r entry (56 sums on the first 56 threads: any block of >= 64 works)
        const int j = tid - 45;
        double s;
        if (rows < 100) {
            double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
            int k = 0;
            for (; k <= rows - 4; k += 4) {
                s0 += sh.J[k * 9 + j] * sh.r[k]; s1 += sh.J[(k + 1) * 9 + j] * sh.r[k + 1];
                s2 += sh.J[(k + 2) * 9 + j] * sh.r[k + 2]; s3 += sh.J[(k + 3) * 9 + j] * sh.r[k + 3];
            }
            for (; k < rows; k++) s0 += sh.J[k * 9 + j] * sh.r[k];
            s = ((s0 + s1) + s2) + s3;
        } else {
            s = 0;
            for (int k = 0; k < rows; k++) s += sh.J[k * 9 + j] * sh.r[k];
        }
        sh.out[45 + j] = s;
    } else if (tid == 54) {                               // |r|^2 in cv::norm's order
        NormL2SqrAcc na; na.init();
        for (int k = 0; k < rows; k++) na.push(sh.r[k]);
        sh.out[54] = na.finish();
    } else if (tid == 55) {
        double rm = 0;
        for (int k = 0; k < rows; k++) { const double q = fabs(sh.r[k]); if (q > rm) rm = q; }
        sh.out[55] = rm;
    }
    __syncthreads();
    if (wantJ) {
        int e = 0;
        for (int j = 0; j < 9; j++) {
            for (int k = j; k < 9; k++) { A[j * 9 + k] = sh.out[e]; A[k * 9 + j] = sh.out[e]; e++; }
            v[j] = sh.out[45 + j];
        }
    }
    if (rmax) *rmax = sh.out[55];
    const double S = sh.out[54];
    __syncthreads();
    return S;
}

// lm_step / lm_update with the 9x9 eigen-solves run cooperatively by warp 0 (all 32 lanes call)
// (both return the number of rotations of their eigen-solve in *rotations, 0 for none)
__device__ void lm_step_warp(LmState& st, FinishShared& sh, int* rotations)
{
    const int lane = threadIdx.x & 31;
    double* Ap = sh.part;                                  // 81 doubles of scratch
    for (int e = lane; e < 81; e += 32) Ap[e] = st.A[e] + ((e / 9 == e % 9) ? st.lambda * st.D[e / 9] : 0.0);
    __syncwarp();
    *rotations = solve_eig9_warp(Ap, st.v, st.d, sh.scratch_a, sh.scratch_v, sh.scratch_w);
    if (lane < 9) st.xd[lane] = st.x[lane] - st.d[lane];
    __syncwarp();
}

__device__ bool lm_update_warp(LmState& st, double Sd, FinishShared& sh, int* rotations)
{
    const double Rlo = 0.25, Rhi = 0.75;
    const int lane = threadIdx.x & 31;
    *rotations = 0;
    double temp_d[9];
    for (int i = 0; i < 9; i++) {
        const double s = dot4acc(st.A + i * 9, st.d, 9);
        temp_d[i] = -1 * s + 2 * st.v[i];
    }
    const double dS = dot_unrolled(st.d, temp_d, 9);
    const double R = (st.S - Sd) / (fabs(dS) > DBL_EPSILON ? dS : 1);
    double lambda = st.lambda, lc = st.lc;
    if (R > Rhi) {
        lambda *= 0.5;
        if (lambda < lc) lambda = 0;
    } else if (R < Rlo) {
        const double t = dot_unrolled(st.d, st.v, 9);
        double nu = (Sd - st.S) / (fabs(t) > DBL_EPSILON ? t : 1) + 2;
        nu = nu > 2. ? nu : 2.;
        nu = nu < 10. ? nu : 10.;
        if (lambda == 0) {
            const double maxval = invert_eig_max_diag9_warp(st.A, sh.scratch_a, sh.scratch_v, sh.scratch_w, rotations);
            lambda = lc = 1. / maxval;
            nu *= 0.5;
        }
        lambda *= nu;
    }
    __syncwarp();
    if (lane == 0) { st.lambda = lambda; st.lc = lc; }
    __syncwarp();
    return Sd < st.S;
}

// ---- 4. finish kernel -----------------------------------------------------------------------------
// Phase probe (-DFIN_PROF, off in the product build): thread 0 of every set's CTA logs each phase as it ends, after the
// phase's barrier, into g_fin_prof: (phase id | rotations << 8, SM cycles since the previous mark).  Entry 0 is the whole
// set: (FP_TOTAL | n_inl << 8, nanoseconds of %globaltimer).  cvg_finish_profile (below) copies the log to the host.
#ifdef FIN_PROF
enum FinPhase { FP_TOTAL = 0, FP_COMPACT, FP_DLT_SUMS, FP_DLT_LTL, FP_REFIT_EIG, FP_EVAL_J, FP_LM_SOLVE, FP_EVAL_XD,
                FP_LM_UPDATE, FP_LM_PROCEED, FP_MASK };
constexpr int FP_SETS = 256, FP_EVENTS = 96;
__device__ long long g_fin_prof[FP_SETS][FP_EVENTS][2];
__device__ int g_fin_prof_n[FP_SETS];
#define FPROF_BEGIN long long fp_t = clock64(), fp_ns = 0; int fp_n = 1; \
    if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(fp_ns));
#define FPROF(phase, rot) if (tid == 0 && set < FP_SETS && fp_n < FP_EVENTS) { \
        const long long t_ = clock64(); g_fin_prof[set][fp_n][0] = (phase) | ((long long)(rot) << 8); \
        g_fin_prof[set][fp_n][1] = t_ - fp_t; fp_n++; fp_t = t_; }
#define FPROF_END(n_inl) if (tid == 0 && set < FP_SETS) { long long ns_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_)); \
        g_fin_prof[set][0][0] = FP_TOTAL | ((long long)(n_inl) << 8); g_fin_prof[set][0][1] = ns_ - fp_ns; g_fin_prof_n[set] = fp_n; }
#else
#define FPROF_BEGIN
#define FPROF(phase, rot)
#define FPROF_END(n_inl)
#endif
__global__ void __launch_bounds__(RS_THREADS)
ransac_finish_kernel(RansacWork w)
{
    const int set = blockIdx.x;
    const int n = w.counts_n[set];
    const int64_t start = w.starts[set];
    const float4* __restrict__ pts = w.pts + start;
    uint8_t* mask = w.mask + start;
    uint8_t* rmask = w.ransac_mask ? w.ransac_mask + start : nullptr;
    int32_t* sel = w.sel + start;
    double* Hout = w.H + (size_t)set * 9;
    __shared__ FinishShared sh;
    const int tid = threadIdx.x;

    auto fail = [&]() {
        for (int i = tid; i < n; i += (int)blockDim.x) { mask[i] = 0; if (rmask) rmask[i] = 0; }
        if (tid < 9) Hout[tid] = 0.0;
        if (tid == 0) w.found[set] = 0;
    };
    if (n < 4) { fail(); return; }
    if (n == 4) {                                            // B.1: direct runKernel, mask of ones, no LM
        if (tid == 0) {
            PtsStrided P{ pts, nullptr };
            sh.flag = run_kernel_seq(P, 4, sh.H, sh.scratch_a, sh.scratch_v) ? 1 : 0;
        }
        __syncthreads();
        if (!sh.flag) { fail(); return; }
        if (tid < 4) { mask[tid] = 1; if (rmask) rmask[tid] = 1; }
        if (tid < 9) Hout[tid] = sh.H[tid];
        if (tid == 0) w.found[set] = 1;
        return;
    }
    const int best_iter = w.best_iter[set];
    if (best_iter < 0) { fail(); return; }

    // The winner's model.  Its mask needs the fp32 model only, and that is what the solve kernel left in hyp_H (8 floats, the
    // (float) of the fp64 H it computed): no second eigen-solve.  The fp64 H itself is needed when nothing refines it
    // (CVG_RANSAC_NO_REFINE) or when the DLT refit on the inliers is degenerate and LM starts from it: solved again then.
    const bool have_model = w.hyp_H != nullptr && w.hyp_H_complete && !(w.flags & CVG_RANSAC_NO_REFINE);
    auto solve_winner = [&]() {                              // warp 0, cooperatively (bit-identical to the hypothesis kernels)
        int idx[4];
        draw_subset(w.rng_tab, w.rng_len, w.sample_pos[(size_t)set * w.max_iters + best_iter], (uint32_t)n, idx);
        float ms1[8], ms2[8];
        #pragma unroll
        for (int i = 0; i < 4; i++) {
            const float4 q = pts[idx[i]];
            ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
        }
        double H[9];
        // scratch_a, scratch_v, scratch_w, jac are contiguous: 333 doubles >= the 243 run_kernel4_warp needs
        run_kernel4_warp(ms1, ms2, H, sh.scratch_a);
        if (tid == 0) {
            for (int i = 0; i < 9; i++) sh.H[i] = H[i];
            for (int i = 0; i < 8; i++) sh.Hf[i] = (float)H[i];
        }
    };
    if (have_model) {
        if (tid < 8) sh.Hf[tid] = w.hyp_H[((size_t)set * w.max_iters + best_iter) * 8 + tid];
    } else if (tid < 32) solve_winner();
    if (tid == 0) sh.base_cnt = 0;
    __syncthreads();
    FPROF_BEGIN
    float Hf[8];
    #pragma unroll
    for (int i = 0; i < 8; i++) Hf[i] = sh.Hf[i];
    const int lane = tid & 31, wid = tid >> 5;
    for (int base = 0; base < n; base += (int)blockDim.x) {   // ordered compaction of inlier indices
        const int i = base + tid;
        bool in = false;
        if (i < n) {
            const float4 q = pts[i];
            in = reproj_err(Hf, q.x, q.y, q.z, q.w) <= w.thr2;
            if (rmask) rmask[i] = in ? 1 : 0;
            if (w.flags & CVG_RANSAC_NO_REFINE) mask[i] = in ? 1 : 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) sh.warp_cnt[wid] = __popc(bal);
        __syncthreads();
        int off = sh.base_cnt;
        for (int k = 0; k < wid; k++) off += sh.warp_cnt[k];
        if (in) sel[off + __popc(bal & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (tid == 0) { int t = 0; for (int k = 0; k < (int)(blockDim.x >> 5); k++) t += sh.warp_cnt[k]; sh.base_cnt += t; }
        __syncthreads();
    }
    const int n_inl = sh.base_cnt;
    FPROF(FP_COMPACT, 0)
    if (w.flags & CVG_RANSAC_NO_REFINE) {
        if (tid < 9) Hout[tid] = sh.H[tid];
        if (tid == 0) w.found[set] = 1;
        return;
    }
    if (n_inl > 0) {
        const bool exact = n_inl <= EXACT_MAX_INLIERS;
        // ---- B.7: DLT refit on the inliers ----
        double cmx, cmy, cMx, cMy, smx, smy, sMx, sMy;
        if (exact) {
            // every sum by one thread, sequentially over the inliers (OpenCV's order)
            if (tid < 4) {
                double s0 = 0;
                for (int i = 0; i < n_inl; i++) {
                    const float4 q = pts[sel[i]];
                    s0 += tid == 0 ? q.z : tid == 1 ? q.w : tid == 2 ? q.x : q.y;
                }
                sh.sums[tid] = s0 / n_inl;
            }
            __syncthreads();
            cmx = sh.sums[0]; cmy = sh.sums[1]; cMx = sh.sums[2]; cMy = sh.sums[3];
            if (tid < 4) {
                const double cc = sh.sums[tid];
                double s0 = 0;
                for (int i = 0; i < n_inl; i++) {
                    const float4 q = pts[sel[i]];
                    s0 += fabs((tid == 0 ? q.z : tid == 1 ? q.w : tid == 2 ? q.x : q.y) - cc);
                }
                sh.sums[4 + tid] = s0;
            }
            __syncthreads();
            smx = sh.sums[4]; smy = sh.sums[5]; sMx = sh.sums[6]; sMy = sh.sums[7];
        } else {
            double s[4] = { 0, 0, 0, 0 };
            for (int i = tid; i < n_inl; i += (int)blockDim.x) {
                const float4 q = pts[sel[i]];
                s[0] += q.z; s[1] += q.w; s[2] += q.x; s[3] += q.y;
            }
            block_sum<4>(s, sh.part, sh.out);
            cmx = s[0] / n_inl; cmy = s[1] / n_inl; cMx = s[2] / n_inl; cMy = s[3] / n_inl;
            s[0] = s[1] = s[2] = s[3] = 0;
            for (int i = tid; i < n_inl; i += (int)blockDim.x) {
                const float4 q = pts[sel[i]];
                s[0] += fabs(q.z - cmx); s[1] += fabs(q.w - cmy); s[2] += fabs(q.x - cMx); s[3] += fabs(q.y - cMy);
            }
            block_sum<4>(s, sh.part, sh.out);
            smx = s[0]; smy = s[1]; sMx = s[2]; sMy = s[3];
        }
        FPROF(FP_DLT_SUMS, 0)
        const bool dlt_ok = !(fabs(smx) < DBL_EPSILON || fabs(smy) < DBL_EPSILON ||
                              fabs(sMx) < DBL_EPSILON || fabs(sMy) < DBL_EPSILON);
        if (!dlt_ok && have_model) {                         // block-uniform: LM starts from the RANSAC model in fp64
            if (tid < 32) solve_winner();
            __syncthreads();
        }
        if (dlt_ok) {
            smx = n_inl / smx; smy = n_inl / smy; sMx = n_inl / sMx; sMy = n_inl / sMy;
            double* LtL = sh.scratch_a;
            if (exact) {
                if (tid < 45) {                               // one upper-triangle entry per thread, sequential over points
                    int j = 0, e = tid;
                    while (e >= 9 - j) { e -= 9 - j; j++; }
                    const int k = j + e;
                    double acc = 0;
                    for (int i = 0; i < n_inl; i++) {
                        const float4 q = pts[sel[i]];
                        const double x = (q.z - cmx) * smx, y = (q.w - cmy) * smy;
                        const double X = (q.x - cMx) * sMx, Y = (q.y - cMy) * sMy;
                        const double Lx[9] = { X, Y, 1, 0, 0, 0, -x * X, -x * Y, -x };
                        const double Ly[9] = { 0, 0, 0, X, Y, 1, -y * X, -y * Y, -y };
                        acc += Lx[j] * Lx[k] + Ly[j] * Ly[k];
                    }
                    LtL[j * 9 + k] = acc; LtL[k * 9 + j] = acc;
                }
            } else {
                double L[45];
                #pragma unroll
                for (int k = 0; k < 45; k++) L[k] = 0;
                for (int i = tid; i < n_inl; i += (int)blockDim.x) {
                    const float4 q = pts[sel[i]];
                    const double x = (q.z - cmx) * smx, y = (q.w - cmy) * smy;
                    const double X = (q.x - cMx) * sMx, Y = (q.y - cMy) * sMy;
                    const double Lx[9] = { X, Y, 1, 0, 0, 0, -x * X, -x * Y, -x };
                    const double Ly[9] = { 0, 0, 0, X, Y, 1, -y * X, -y * Y, -y };
                    int e = 0;
                    #pragma unroll
                    for (int j = 0; j < 9; j++)
                        #pragma unroll
                        for (int k = j; k < 9; k++) { L[e] += Lx[j] * Lx[k] + Ly[j] * Ly[k]; e++; }
                }
                block_sum<45>(L, sh.part, sh.out);
                if (tid == 0) {
                    int e = 0;
                    for (int j = 0; j < 9; j++)
                        for (int k = j; k < 9; k++) { LtL[j * 9 + k] = L[e]; LtL[k * 9 + j] = L[e]; e++; }
                }
            }
            __syncthreads();
            FPROF(FP_DLT_LTL, 0)
            int rot = 0;
            if (tid < 32) {
                rot = jacobi9_warp(LtL, sh.scratch_w, sh.scratch_v);
                if (tid == 0) {
                    const double invHnorm[9] = { 1. / smx, 0, cmx, 0, 1. / smy, cmy, 0, 0, 1 };
                    const double Hnorm2[9] = { sMx, 0, -cMx * sMx, 0, sMy, -cMy * sMy, 0, 0, 1 };
                    double Vl[9], Htemp[9], H0[9];
                    for (int i = 0; i < 9; i++) Vl[i] = sh.scratch_v[72 + i];
                    mat3mul(invHnorm, Vl, Htemp);
                    mat3mul(Htemp, Hnorm2, H0);
                    const double sc = 1. / H0[8];
                    for (int i = 0; i < 9; i++) sh.H[i] = H0[i] * sc;
                }
            }
            __syncthreads();
            FPROF(FP_REFIT_EIG, rot)
        }
        // ---- B.8: LMSolver (9 parameters, 10 iterations); reductions by the block, eigen-solves by warp 0 ----
        LmState& st = sh.lm;
        if (tid < 9) st.x[tid] = sh.H[tid];
        __syncthreads();
        {
            double A[81], v[9], rmax;
            const double S = exact ? lm_eval_exact(pts, sel, n_inl, st.x, true, A, v, &rmax, sh)
                                   : lm_eval_block(pts, sel, n_inl, st.x, A, v, &rmax, sh);
            if (tid == 0) {
                for (int i = 0; i < 81; i++) st.A[i] = A[i];
                for (int i = 0; i < 9; i++) st.v[i] = v[i];
                st.S = S; st.rmax = rmax;
                lm_begin(st);
            }
            __syncthreads();
            FPROF(FP_EVAL_J, 0)
        }
        for (;;) {
            int rot = 0;
            if (tid < 32) lm_step_warp(st, sh, &rot);
            __syncthreads();
            FPROF(FP_LM_SOLVE, rot)
            const double Sd = exact ? lm_eval_exact(pts, sel, n_inl, st.xd, false, nullptr, nullptr, nullptr, sh)
                                    : lm_eval_block(pts, sel, n_inl, st.xd, nullptr, nullptr, nullptr, sh);
            FPROF(FP_EVAL_XD, 0)
            if (tid < 32) {
                const bool acc = lm_update_warp(st, Sd, sh, &rot);
                if (tid == 0) sh.flag = acc ? 1 : 0;
            }
            __syncthreads();
            FPROF(FP_LM_UPDATE, rot)
            if (sh.flag) {
                if (tid < 9) st.x[tid] = st.xd[tid];
                __syncthreads();
                double A[81], v[9], rmax;
                const double S = exact ? lm_eval_exact(pts, sel, n_inl, st.x, true, A, v, &rmax, sh)
                                       : lm_eval_block(pts, sel, n_inl, st.x, A, v, &rmax, sh);
                if (tid == 0) {
                    for (int i = 0; i < 81; i++) st.A[i] = A[i];
                    for (int i = 0; i < 9; i++) st.v[i] = v[i];
                    st.S = S; st.rmax = rmax;
                }
                __syncthreads();
                FPROF(FP_EVAL_J, 0)
            }
            if (tid == 0) sh.flag = lm_proceed(st, 10) ? 1 : 0;
            __syncthreads();
            FPROF(FP_LM_PROCEED, 0)
            if (!sh.flag) break;
        }
        if (tid == 0) {
            const double sc = 1. / st.x[8];
            for (int i = 0; i < 9; i++) sh.H[i] = st.x[i] * sc;
        }
        __syncthreads();
        // B.9: returned mask = err(H_final) <= thr^2 over ALL correspondences
        #pragma unroll
        for (int i = 0; i < 8; i++) Hf[i] = (float)sh.H[i];
        for (int i = tid; i < n; i += (int)blockDim.x) {
            const float4 q = pts[i];
            mask[i] = reproj_err(Hf, q.x, q.y, q.z, q.w) <= w.thr2 ? 1 : 0;
        }
        FPROF(FP_MASK, 0)
        FPROF_END(n_inl)
    } else {
        for (int i = tid; i < n; i += (int)blockDim.x) mask[i] = 0;
        if (have_model) {                                    // never reached with a winner of >= 4 inliers; keep H defined
            if (tid < 32) solve_winner();
            __syncthreads();
        }
    }
    if (tid < 9) Hout[tid] = sh.H[tid];
    if (tid == 0) w.found[set] = 1;
}

#ifdef FIN_PROF
// Copies the phase log of the last finish launches (sets 0 .. n_sets-1, FP_EVENTS entries of two int64 each per set, then
// one int32 entry count per set) to the host and clears the counts.  Exported only by a -DFIN_PROF build.
extern "C" int cvg_finish_profile(long long* log, int* counts, int n_sets)
{
    if (n_sets < 0 || n_sets > FP_SETS) return -1;
    if (cudaMemcpyFromSymbol(log, g_fin_prof, sizeof(long long) * 2 * FP_EVENTS * n_sets) != cudaSuccess) return -1;
    if (cudaMemcpyFromSymbol(counts, g_fin_prof_n, sizeof(int) * n_sets) != cudaSuccess) return -1;
    static int zero[FP_SETS];
    return cudaMemcpyToSymbol(g_fin_prof_n, zero, sizeof(zero)) == cudaSuccess ? FP_EVENTS : -1;
}
#endif

// layout of the chunked sampler's scratch inside one allocation; returns the total size
int64_t ransac_chunk_scratch_bytes(int n_sets, int n_chunks, size_t* outs, size_t* lists, size_t* offsets, size_t* serial,
                                   size_t* maps, size_t* entries)
{
    size_t o = 0;
    *outs = o;    o += (size_t)n_sets * n_chunks * sizeof(ChunkOut);
    *lists = o;   o += (size_t)n_sets * n_chunks * CH_LIST * sizeof(int32_t);
    *offsets = o; o += (size_t)n_sets * n_chunks * sizeof(int32_t);
    *entries = o; o += (size_t)n_sets * n_chunks * sizeof(int32_t);
    *serial = o;  o += ((size_t)n_sets * sizeof(int) + 63) / 64 * 64;
    *maps = o;    o += (size_t)n_sets * n_chunks * CH_K + 64;
    return (int64_t)o;
}
int ransac_chunks_for_table(int64_t rng_len)
{
    const int64_t c = (rng_len - 2 * SW - SW_TAIL - 128) / CH_DRAWS;
    return c < 0 ? 0 : (c > 1000000 ? 1000000 : (int)c);
}

// ---- self test 0: rcp_rn_fastpath == __frcp_rn on every float of the fast range (both signs) ----------------
__global__ void selftest_rcp_kernel(unsigned long long* mismatches)
{
    const uint32_t stride = gridDim.x * blockDim.x;
    unsigned long long bad = 0;
    // |x| in [2^-126, 2^126): bit patterns 0x00800000 .. 0x7E7FFFFF, and the same with the sign bit
    for (uint64_t b = 0x00800000ull + blockIdx.x * blockDim.x + threadIdx.x; b < 0x7E800000ull; b += stride) {
        #pragma unroll
        for (uint32_t sgn = 0; sgn < 2; sgn++) {
            const float x = __uint_as_float((uint32_t)b | (sgn << 31));
            if (__float_as_uint(rcp_rn_fastpath(x)) != __float_as_uint(__frcp_rn(x))) bad++;
            if (__float_as_uint(__frcp_rn(x)) != __float_as_uint(__fdiv_rn(1.f, x))) bad++;
        }
    }
    if (bad) atomicAdd(mismatches, bad);
}
int launch_selftest_rcp(unsigned long long* d_mismatches, cudaStream_t st)
{
    selftest_rcp_kernel<<<148 * 16, 256, 0, st>>>(d_mismatches);
    return 1;
}

// ---- self test 1: the warp-cooperative 9x9 routines (jacobi_warp.cuh) == the serial ones (homography_math.cuh) ----------
// One warp per matrix; lane 0 builds the matrix from its index (no host data) and runs the serial routine on the device.
// Every output double is compared bit for bit: W and V of jacobi, x of solve, the returned maximum of invert.
struct StRng {
    uint64_t s;
    __device__ uint64_t next()
    {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    __device__ double unif() { return (double)(next() >> 11) * 0x1.0p-53; }     // [0, 1)
    __device__ int below(int n) { return (int)(next() % (uint64_t)n); }
};

// LtL of a normalised DLT over n correspondences (a near-affine map with 30 % outliers), as the refit builds it
__device__ void selftest_dlt(StRng& r, int n, double* LtL)
{
    const uint64_t seed = r.next();
    auto point = [&](int i, float& Mx, float& My, float& mx, float& my) {
        StRng q{ seed + (uint64_t)i * 0x2545F4914F6CDD1Dull };
        Mx = (float)(640 * q.unif()); My = (float)(480 * q.unif());
        if (q.unif() < 0.3) { mx = (float)(640 * q.unif()); my = (float)(480 * q.unif()); }
        else { mx = (float)(0.9 * Mx + 0.05 * My + 20 + q.unif() - 0.5); my = (float)(-0.04 * Mx + 1.1 * My - 7 + q.unif() - 0.5); }
    };
    double cMx = 0, cMy = 0, cmx = 0, cmy = 0, sMx = 0, sMy = 0, smx = 0, smy = 0;
    float Mx, My, mx, my;
    for (int i = 0; i < n; i++) { point(i, Mx, My, mx, my); cmx += mx; cmy += my; cMx += Mx; cMy += My; }
    cmx /= n; cmy /= n; cMx /= n; cMy /= n;
    for (int i = 0; i < n; i++) {
        point(i, Mx, My, mx, my);
        smx += fabs(mx - cmx); smy += fabs(my - cmy); sMx += fabs(Mx - cMx); sMy += fabs(My - cMy);
    }
    smx = n / smx; smy = n / smy; sMx = n / sMx; sMy = n / sMy;
    for (int e = 0; e < 81; e++) LtL[e] = 0;
    for (int i = 0; i < n; i++) { point(i, Mx, My, mx, my); dlt_accumulate_point(LtL, Mx, My, mx, my, cMx, cMy, cmx, cmy, sMx, sMy, smx, smy); }
}

__device__ void selftest_matrix(int idx, double* M, double* b)
{
    StRng r{ 0x5EEDull * 1000003ull + (uint64_t)idx };
    switch (idx % 5) {
    case 0: selftest_dlt(r, 4, M); break;                                    // a 4-point sample
    case 1: selftest_dlt(r, 5 + r.below(3996), M); break;                    // a refit over 5 .. 4000 inliers
    case 2: {                                                                // LM: J^T J + lambda * diag(J^T J)
        for (int e = 0; e < 81; e++) M[e] = 0;
        const int rows = 10 + r.below(400);
        for (int q = 0; q < rows; q++) {
            double J[9];
            for (int j = 0; j < 9; j++) J[j] = (2 * r.unif() - 1) * (j < 6 ? 1.0 : 1e-3);
            for (int j = 0; j < 9; j++) for (int k = j; k < 9; k++) M[j * 9 + k] += J[j] * J[k];
        }
        const double lambda = pow(10.0, -6 + 8 * r.unif());
        for (int j = 0; j < 9; j++) M[j * 10] = M[j * 10] + lambda * M[j * 10];
        break;
    }
    case 3: {                                                                // small integers: tied pivot candidates
        for (int j = 0; j < 9; j++) for (int k = j; k < 9; k++) M[j * 9 + k] = (double)(r.below(5) - 2) * (j == k ? -2 : 1);
        break;
    }
    default: {                                                               // zeros in the upper triangle
        const double pz = r.unif();
        for (int j = 0; j < 9; j++)
            for (int k = j; k < 9; k++) M[j * 9 + k] = (k > j && r.unif() < pz) ? 0.0 : 2 * r.unif() - 1;
        break;
    }
    }
    for (int j = 0; j < 9; j++) for (int k = 0; k < j; k++) M[j * 9 + k] = M[k * 9 + j];
    for (int j = 0; j < 9; j++) b[j] = 2 * r.unif() - 1;
}

constexpr int STJ_WARPS = 4;
constexpr int STJ_DOUBLES = 81 * 5 + 9 * 4;
__global__ void __launch_bounds__(STJ_WARPS * 32) selftest_jacobi_kernel(unsigned long long* mismatches, int n_mats)
{
    __shared__ double sm[STJ_WARPS][STJ_DOUBLES];
    const int lane = threadIdx.x & 31;
    double* M = sm[threadIdx.x >> 5];
    double* a = M + 81; double* v = a + 81; double* sa = v + 81; double* sv = sa + 81;
    double* w = sv + 81; double* b = w + 9; double* x = b + 9; double* xs = x + 9;
    unsigned long long bad = 0;
    for (int m = blockIdx.x * STJ_WARPS + (threadIdx.x >> 5); m < n_mats; m += gridDim.x * STJ_WARPS) {
        if (lane == 0) selftest_matrix(m, M, b);
        __syncwarp();
        for (int e = lane; e < 81; e += 32) a[e] = M[e];
        __syncwarp();
        jacobi9_warp(a, w, v);
        if (lane == 0) {
            double ws[9];
            for (int e = 0; e < 81; e++) sa[e] = M[e];
            jacobi<9>(sa, ws, sv);
            for (int i = 0; i < 9; i++) bad += __double_as_longlong(w[i]) != __double_as_longlong(ws[i]);
            for (int e = 0; e < 81; e++) bad += __double_as_longlong(v[e]) != __double_as_longlong(sv[e]);
        }
        __syncwarp();
        solve_eig9_warp(M, b, x, a, v, w);
        if (lane == 0) {
            solve_eig<9>(M, b, xs, sa, sv);
            for (int i = 0; i < 9; i++) bad += __double_as_longlong(x[i]) != __double_as_longlong(xs[i]);
        }
        __syncwarp();
        const double mv = invert_eig_max_diag9_warp(M, a, v, w);
        if (lane == 0) bad += __double_as_longlong(mv) != __double_as_longlong(invert_eig_max_diag<9>(M, sa, sv));
        __syncwarp();
    }
    if (lane == 0 && bad) atomicAdd(mismatches, bad);
}
int launch_selftest_jacobi(unsigned long long* d_mismatches, int n_mats, cudaStream_t st)
{
    selftest_jacobi_kernel<<<(n_mats + STJ_WARPS - 1) / STJ_WARPS, STJ_WARPS * 32, 0, st>>>(d_mismatches, n_mats);
    return 1;
}

int ransac_set_device_attrs(char* err, size_t errlen)
{
    cudaError_t e = cudaFuncSetAttribute(ransac_hyp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HYP_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ransac_hyp_g8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HYPG_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ransac_hyp_t_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HYPT_SMEM);
    if (e != cudaSuccess) { snprintf(err, errlen, "cudaFuncSetAttribute(ransac kernels): %s", cudaGetErrorString(e)); return 1; }
    return 0;
}

int ransac_round_len(const RansacWork& w)
{
    // Hypotheses are solved and scored in rounds; after each round the serial selection scan advances, so rounds
    // beyond the adaptive stop (RANSACUpdateNumIters) cost one early exit per warp.  A round is a latency-bound
    // launch (~135 dependent rotations per matrix whatever the kernel), so it is made long enough to fill the chip:
    // at least 256 iterations per set, and n_sets x round_len >= one full wave of the thread-per-hypothesis kernel.
    static const int round_env = getenv("CVG_ROUND_LEN") ? atoi(getenv("CVG_ROUND_LEN")) : 0;
    const int n_sms = w.n_sms > 0 ? w.n_sms : 148;
    int round_len = w.max_iters;
    if (!(w.flags & CVG_RANSAC_NO_EARLY_STOP)) {
        // wave_div engines share the GPU (lanes of one context working on sub-batches of a call): each sizes its rounds
        // to its share, so that the sum of the concurrent rounds is still one wave and no lane solves hypotheses far
        // beyond its sets' adaptive stop
        const int64_t wave = (int64_t)n_sms * HYPT_THREADS * HYPT_CTAS_PER_SM / std::max(1, w.wave_div);
        int64_t fill = wave / w.n_sets / 32 * 32;              // rounded down: n_sets x round_len must not spill into a second wave
        if (fill < 256) {
            // many sets: a round of 256 iterations is several waves; make it a whole number of them (13 350 real pairs in
            // calls of 445 sets: 288 iterations = 3.9 waves and 7 rounds instead of 256 = 3.4 waves — 4 wave times — and 8)
            const int64_t k = (256 * (int64_t)w.n_sets + wave - 1) / wave;
            fill = k * wave / w.n_sets / 32 * 32;
        }
        round_len = (int)std::min<int64_t>(std::max<int64_t>(256, fill), w.max_iters);
        if (round_env > 0) round_len = std::min(round_env, w.max_iters);
    }
    return round_len;
}

int launch_ransac_sample(const RansacWork& w, int rb, int len, cudaStream_t st)
{
    if (rb == 0 && w.chunk_outs && w.n_chunks > 1 && (int64_t)len >= CHUNKED_MIN_ITERS) {
        // a huge single round (the no-early-stop throughput mode): cut every set's draw stream into chunks
        ChunkOut* outs = static_cast<ChunkOut*>(w.chunk_outs);
        ransac_sample_map_kernel<<<dim3((unsigned)w.n_chunks, (unsigned)w.n_sets), SMP_THREADS, 0, st>>>(w, rb, w.n_chunks, w.chunk_maps);
        ransac_sample_entry_kernel<<<w.n_sets, 256, 0, st>>>(w.n_chunks, w.chunk_maps, w.chunk_entries);
        ransac_sample_chunk_kernel<<<dim3((unsigned)w.n_chunks, (unsigned)w.n_sets), SMP_THREADS, 0, st>>>(w, rb, w.n_chunks, w.chunk_entries,
                                                                                                          outs, w.chunk_lists);
        ransac_sample_stitch_kernel<<<(w.n_sets + 63) / 64, 64, 0, st>>>(w, rb, rb + len, w.n_chunks, outs, w.chunk_lists,
                                                                        w.chunk_offsets, w.chunk_serial);
        ransac_sample_scatter_kernel<<<dim3((unsigned)w.n_chunks, (unsigned)w.n_sets), 256, 0, st>>>(w, rb + len, w.n_chunks, outs,
                                                                                                 w.chunk_lists, w.chunk_offsets);
        ransac_sample_kernel<4><<<w.n_sets, SMP_THREADS, 0, st>>>(w, rb, rb + len, w.chunk_serial);   // sets the stitch rejected
        return 6;
    }
    ransac_sample_kernel<4><<<w.n_sets, SMP_THREADS, 0, st>>>(w, rb, rb + len, nullptr);
    return 1;
}

int launch_ransac_hyp(const RansacWork& w, int hb, int hlen, cudaStream_t st, const cudaEvent_t* ev, bool* hyp_complete)
{
    static const int hyp_mode = getenv("CVG_HYP_MODE") ? atoi(getenv("CVG_HYP_MODE")) : 0;   // experiments: 1 warp, 2 g8, 3 thread (generic), 4 thread
    const int n_sms = w.n_sms > 0 ? w.n_sms : 148;
    int launches = 1;
    if (ev) cudaEventRecord(ev[0], st);
    // Measured on B200 (round 1).  13 350 real pairs (3.4 M hypotheses per round), whole verify stage: generic
    // thread-per-hypothesis 612 ms, warp-per-hypothesis 1436 ms, four-per-warp 498 ms.  64 synthetic 8k x 8k pairs
    // (16 384 hypotheses per round), hypothesis kernels per step: warp 4.15 ms, four-per-warp 2.41 ms.
    // One set alone (256 hypotheses): warp 0.30 ms, generic thread 1.1 ms.
    const int64_t hyps = (int64_t)hlen * w.n_sets;
    const int mode = hyp_mode ? hyp_mode : (hyps <= 4096 ? 1 : 4);
    if (mode == 2 || mode == 3) *hyp_complete = false;     // the A/B kernels do not leave their models in hyp_H
    if (mode == 1) {                                       // a handful of hypotheses: latency of one matrix counts
        dim3 grid((hlen + HYPW_WARPS - 1) / HYPW_WARPS, w.n_sets);
        ransac_hyp_warp_kernel<<<grid, HYPW_WARPS * 32, 0, st>>>(w, hb);
    } else if (mode == 2) {                                // four matrices per warp
        dim3 grid((hlen + HYPG_WARPS * 4 - 1) / (HYPG_WARPS * 4), w.n_sets);
        ransac_hyp_g8_kernel<<<grid, HYPG_WARPS * 32, HYPG_SMEM, st>>>(w, hb);
    } else if (mode == 3) {                                // generic serial routine, one thread per hypothesis
        dim3 grid((hlen + HYP_THREADS - 1) / HYP_THREADS, w.n_sets);
        ransac_hyp_kernel<<<grid, HYP_THREADS, HYP_SMEM, st>>>(w, hb);
    } else {                                               // the chip is full: one thread per hypothesis
        const int64_t blocks = (hyps + HYPT_THREADS - 1) / HYPT_THREADS;
        ransac_hyp_t_kernel<<<(unsigned)blocks, HYPT_THREADS, HYPT_SMEM, st>>>(w, hb, hlen);
    }
    if (ev) cudaEventRecord(ev[1], st);
    if (mode == 4 && w.hyp_H) {
        // slices of the correspondences so that the launch holds >= ~6 CTAs per SM (or one slice per 512 points)
        const int tiles = (hlen + SCORE_THREADS - 1) / SCORE_THREADS;
        const int64_t ctas = (int64_t)tiles * w.n_sets;
        int n_slices = (int)std::min<int64_t>(std::max<int64_t>(1, ((int64_t)n_sms * 6 + ctas - 1) / ctas), std::max(1, w.max_n / 512));
        n_slices = std::max(1, std::min(n_slices, 64));
        ransac_score_kernel<<<dim3((unsigned)ctas, 1, (unsigned)n_slices), SCORE_THREADS, 0, st>>>(w, hb, hlen, n_slices, tiles);
        launches += 1;
    }
    if (ev) cudaEventRecord(ev[2], st);
    return launches;
}

int launch_ransac_select(const RansacWork& w, int rb, int len, cudaStream_t st)
{
    const int warps_per_block = 4;
    if (w.flags & CVG_RANSAC_NO_EARLY_STOP)
        ransac_select_all_kernel<<<w.n_sets, SELP_THREADS, 0, st>>>(w, rb, len);
    else
        ransac_select_kernel<<<(w.n_sets + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(w, rb, len);
    return 1;
}

int launch_ransac_finish(const RansacWork& w, bool hyp_complete, cudaStream_t st)
{
    // Sets of a few dozen correspondences (the real dataset: 445 sets per call, n <= 127) take the exact path, which is
    // warp 0's serial eigen-solves plus 56 single-thread sums: with 64 threads per CTA four CTAs fit an SM (206 registers)
    // and the call's sets run in one wave instead of two.  Every loop of the kernel strides by blockDim.x.
    const int finish_threads = w.max_n <= 512 ? 64 : RS_THREADS;
    RansacWork wf = w;
    wf.hyp_H_complete = hyp_complete ? 1 : 0;
    ransac_finish_kernel<<<w.n_sets, finish_threads, 0, st>>>(wf);
    return 1;
}

int launch_ransac(const RansacWork& w, cudaStream_t st, cudaEvent_t* hyp_events, int* n_hyp_rounds)
{
    if (n_hyp_rounds) *n_hyp_rounds = 0;
    if (w.n_sets <= 0) return 0;
    const int round_len = ransac_round_len(w);
    int launches = 0, round = 0;
    bool hyp_complete = w.hyp_H != nullptr;
    for (int rb = 0; rb < w.max_iters; rb += round_len, round++) {
        const int len = w.max_iters - rb < round_len ? w.max_iters - rb : round_len;
        launches += launch_ransac_sample(w, rb, len, st);
        const bool timed = hyp_events != nullptr && round < 16;
        const cudaEvent_t ev[3] = { timed ? hyp_events[2 * round] : nullptr, timed ? hyp_events[2 * round + 1] : nullptr,
                                    timed ? hyp_events[32 + round] : nullptr };
        launches += launch_ransac_hyp(w, rb, len, st, timed ? ev : nullptr, &hyp_complete);
        if (timed) *n_hyp_rounds = round + 1;
        launches += launch_ransac_select(w, rb, len, st);
    }
    launches += launch_ransac_finish(w, hyp_complete, st);
    return launches;
}

// ---- cv::estimateAffine2D / estimateAffinePartial2D (RANSAC): solve + score, finish -------------------
// The two affine methods share the sampler (ransac_sample_kernel<MP>), the select scan and the niters verification with
// findHomography, and one pair of kernels below, instantiated for each model description (AffineModel, PartialModel).
// A minimal solve is a closed form of ~40 fp64 operations, so one kernel solves and scores: a CTA is SCORE_THREADS
// consecutive iterations of one set x one slice of its correspondences (blockIdx.z), as in ransac_score_kernel; every
// thread re-solves its hypothesis from the sample (cheaper than a round trip through HBM) and adds its slice's count to
// counts[] (zeroed before the launch) with an integer atomicAdd.
//
// A model description gives the sample size MP and the closed-form solve (2x3 M from MP points), the N parameters LMSolver
// refines and their map to and from M, and the refine callback's residuals and Jacobian entries for one correspondence
// q = (Mx, My, X, Y): row 2i is the x residual, row 2i + 1 the y residual.
struct AffineModel {            // estimateAffine2D: Affine2DEstimatorCallback, Affine2DRefineCallback; x = M
    static constexpr int MP = 3, N = 6;
    __device__ static void solve(const float* from, const float* to, double* M) { affine_solve(from, to, M); }
    __device__ static void params(const double* M, double* x) { for (int i = 0; i < 6; i++) x[i] = M[i]; }
    __device__ static void matrix(const double* x, double* M) { for (int i = 0; i < 6; i++) M[i] = x[i]; }
    __device__ static void residuals(const double* h, const float4& q, double& r0, double& r1)
    {
        const double Mx = q.x, My = q.y;
        r0 = h[0] * Mx + h[1] * My + h[2] - q.z;
        r1 = h[3] * Mx + h[4] * My + h[5] - q.w;
    }
    // row 2i is (X, Y, 1, 0, 0, 0), row 2i + 1 is (0, 0, 0, X, Y, 1)
    __device__ static double jac(int row, int j, const float4& q)
    {
        const int c = j - 3 * (row & 1);
        return c == 0 ? (double)q.x : c == 1 ? (double)q.y : c == 2 ? 1.0 : 0.0;
    }
};

struct PartialModel {           // estimateAffinePartial2D: AffinePartial2DEstimatorCallback, AffinePartial2DRefineCallback
    static constexpr int MP = 2, N = 4;
    __device__ static void solve(const float* from, const float* to, double* M) { affine_partial_solve(from, to, M); }
    // x = (a, b, tx, ty) = (M00, M10, M02, M12); M = [a, -b, tx; b, a, ty] (the solve's M maps back to itself, bit for bit)
    __device__ static void params(const double* M, double* x) { x[0] = M[0]; x[1] = M[3]; x[2] = M[2]; x[3] = M[5]; }
    __device__ static void matrix(const double* x, double* M)
    {
        M[0] = x[0]; M[1] = -x[1]; M[2] = x[2]; M[3] = x[1]; M[4] = x[0]; M[5] = x[3];
    }
    __device__ static void residuals(const double* h, const float4& q, double& r0, double& r1)
    {
        const double Mx = q.x, My = q.y;
        r0 = h[0] * Mx - h[1] * My + h[2] - q.z;
        r1 = h[1] * Mx + h[0] * My + h[3] - q.w;
    }
    // row 2i is (X, -Y, 1, 0), row 2i + 1 is (Y, X, 0, 1)
    __device__ static double jac(int row, int j, const float4& q)
    {
        if (row & 1) return j == 0 ? (double)q.y : j == 1 ? (double)q.x : j == 2 ? 0.0 : 1.0;
        return j == 0 ? (double)q.x : j == 1 ? -(double)q.y : j == 2 ? 1.0 : 0.0;
    }
};

template <class Model>
__device__ __forceinline__ void affine_solve_sample(const RansacWork& w, const float4* __restrict__ pts, int n, int32_t pos,
                                                    double M[6])
{
    constexpr int MP = Model::MP;
    int idx[MP];
    draw_subset_g<MP>(TabGet{ w.rng_tab, w.rng_len, (uint32_t)n }, pos, idx);
    float ms1[2 * MP], ms2[2 * MP];
    #pragma unroll
    for (int i = 0; i < MP; i++) {
        const float4 q = pts[idx[i]];
        ms1[2 * i] = q.x; ms1[2 * i + 1] = q.y; ms2[2 * i] = q.z; ms2[2 * i + 1] = q.w;
    }
    Model::solve(ms1, ms2, M);
}

template <class Model>
__global__ void __launch_bounds__(SCORE_THREADS)
ransac_affine_hyp_kernel(RansacWork w, int round_base, int round_len, int n_slices, int tiles)
{
    __shared__ float4 stage[SCORE_STAGE];
    const int set = (int)(blockIdx.x / (unsigned)tiles);
    const int r = (int)(blockIdx.x % (unsigned)tiles) * SCORE_THREADS + threadIdx.x;
    const int iter = round_base + r;
    const int n = w.counts_n[set];
    const size_t slot = (size_t)set * w.max_iters + iter;
    const bool live = r < round_len && iter < w.n_samples[set] && iter < w.niters_cur[set];
    if (!__syncthreads_or(live)) return;
    const float4* __restrict__ ps = w.pts + w.starts[set];
    float F[6];
    {
        double M[6];
        if (live) affine_solve_sample<Model>(w, ps, n, w.sample_pos[slot], M);
        #pragma unroll
        for (int i = 0; i < 6; i++) F[i] = live ? (float)M[i] : 0.f;
    }
    const int per = (n + n_slices - 1) / n_slices;
    const int p0 = min(n, (int)blockIdx.z * per), p1 = min(n, p0 + per);
    const float thr2 = w.thr2;
    int cnt = 0;
    for (int base = p0; base < p1; base += SCORE_STAGE) {
        const int m = min(SCORE_STAGE, p1 - base);
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += SCORE_THREADS) stage[i] = ps[base + i];
        __syncthreads();
        if (live) {
            #pragma unroll 4
            for (int i = 0; i < m; i++) {
                const float4 q = stage[i];                              // same address in every lane: broadcast
                cnt += affine_err(F, q.x, q.y, q.z, q.w) <= thr2 ? 1 : 0;   // NaN -> not an inlier
            }
        }
    }
    if (live && cnt) atomicAdd(&w.counts[slot], cnt);
}

// The refine's sums for N parameters: the upper triangle of J^T J (NT entries), J^T r (N), |r|^2 and (exact mode) max |r|
template <int N>
struct AffineShared {
    static constexpr int NT = N * (N + 1) / 2;
    double part[(RS_THREADS / 32) * (NT + N + 1)];
    double out[NT + N + 2];
    LmStateN<N> lm;
    double scratch_a[N * N], scratch_v[N * N];
    double r[2 * EXACT_MAX_INLIERS];            // exact mode: residuals of the current evaluation
    int flag;
    int warp_cnt[RS_THREADS / 32];
    int base_cnt;
};

// At x (wantJ): S = |r|^2, max |r|, A = J^T J (N x N) and v = J^T r, left in st.  At xd: Sd = |r|^2 in sh.out[0].  Up to
// EXACT_MAX_INLIERS inliers every sum is one thread's, in OpenCV's order (mulTransposed sequential over rows, gemm with
// 4 interleaved accumulators below 100 rows, norm in the AVX2 pattern); above, per-thread partial sums and block_sum.
template <class Model>
__device__ void affine_lm_eval(const float4* __restrict__ pts, const int32_t* __restrict__ sel, int count, const double* h,
                               bool wantJ, AffineShared<Model::N>& sh)
{
    constexpr int N = Model::N, NT = AffineShared<N>::NT;
    const int tid = threadIdx.x;
    double S, rm, A[NT], v[N];
    if (count <= EXACT_MAX_INLIERS) {
        const int rows = 2 * count;
        for (int i = tid; i < count; i += (int)blockDim.x) Model::residuals(h, pts[sel[i]], sh.r[2 * i], sh.r[2 * i + 1]);
        __syncthreads();
        if (wantJ && tid < NT) {                                 // upper triangle entry (j, k) of J^T J
            int j = 0, e = tid;
            while (e >= N - j) { e -= N - j; j++; }
            const int k = j + e;
            double s = 0;
            for (int row = 0; row < rows; row++) {
                const float4 q = pts[sel[row >> 1]];
                s += Model::jac(row, j, q) * Model::jac(row, k, q);
            }
            sh.out[tid] = s;
        } else if (wantJ && tid >= NT && tid < NT + N) {         // J^T r entry
            const int j = tid - NT;
            double s;
            if (rows < 100) {
                double s4[4] = { 0, 0, 0, 0 };
                const int full = rows & ~3;
                for (int row = 0; row < rows; row++)
                    s4[row < full ? (row & 3) : 0] += Model::jac(row, j, pts[sel[row >> 1]]) * sh.r[row];
                s = ((s4[0] + s4[1]) + s4[2]) + s4[3];
            } else {
                s = 0;
                for (int row = 0; row < rows; row++) s += Model::jac(row, j, pts[sel[row >> 1]]) * sh.r[row];
            }
            sh.out[NT + j] = s;
        } else if (tid == NT + N) {
            NormL2SqrAcc na; na.init();
            for (int row = 0; row < rows; row++) na.push(sh.r[row]);
            sh.out[NT + N] = na.finish();
        } else if (tid == NT + N + 1) {
            double m = 0;
            for (int row = 0; row < rows; row++) { const double q = fabs(sh.r[row]); if (q > m) m = q; }
            sh.out[NT + N + 1] = m;
        }
        __syncthreads();
        S = sh.out[NT + N]; rm = sh.out[NT + N + 1];
        if (wantJ) {
            for (int e = 0; e < NT; e++) A[e] = sh.out[e];
            for (int j = 0; j < N; j++) v[j] = sh.out[NT + j];
        }
        __syncthreads();
    } else {
        double acc[NT + N + 1];
        #pragma unroll
        for (int k = 0; k < NT + N + 1; k++) acc[k] = 0;
        rm = 0;
        // 64 partial sums whatever blockDim.x (64 or 128, chosen from the batch's largest set): threads 64.. add exact
        // zeros, so a set's M does not depend on the batch it came in
        for (int i = tid; tid < 64 && i < count; i += 64) {
            const float4 q = pts[sel[i]];
            double r0, r1;
            Model::residuals(h, q, r0, r1);
            acc[NT + N] += r0 * r0; acc[NT + N] += r1 * r1;
            rm = fmax(rm, fmax(fabs(r0), fabs(r1)));
            if (wantJ) {
                int e = 0;
                #pragma unroll
                for (int j = 0; j < N; j++) {
                    #pragma unroll
                    for (int k = j; k < N; k++) {
                        acc[e] += Model::jac(0, j, q) * Model::jac(0, k, q); acc[e] += Model::jac(1, j, q) * Model::jac(1, k, q); e++;
                    }
                    acc[NT + j] += Model::jac(0, j, q) * r0; acc[NT + j] += Model::jac(1, j, q) * r1;
                }
            }
        }
        block_sum<NT + N + 1>(acc, sh.part, sh.out);
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) rm = fmax(rm, shfl_down_d(rm, o));
        if ((tid & 31) == 0) sh.part[tid >> 5] = rm;
        __syncthreads();
        rm = sh.part[0];
        for (int q = 1; q < (int)(blockDim.x >> 5); q++) rm = fmax(rm, sh.part[q]);
        __syncthreads();
        S = acc[NT + N];
        for (int e = 0; e < NT; e++) A[e] = acc[e];
        for (int j = 0; j < N; j++) v[j] = acc[NT + j];
    }
    if (tid == 0) {
        LmStateN<N>& st = sh.lm;
        if (wantJ) {
            int e = 0;
            for (int j = 0; j < N; j++) {
                for (int k = j; k < N; k++) { st.A[j * N + k] = A[e]; st.A[k * N + j] = A[e]; e++; }
                st.v[j] = v[j];
            }
            st.S = S; st.rmax = rm;
        } else {
            sh.out[0] = S;                                       // Sd, read by thread 0 after the barrier below
        }
    }
    __syncthreads();
}

// One CTA per set: the winner re-solved in fp64, the returned mask from (float)M (RANSAC stage: the refine moves M, not the
// mask), the ordered compaction of its inliers and LMSolver with the model's refine callback for refine_iters iterations.
template <class Model>
__global__ void __launch_bounds__(RS_THREADS)
ransac_affine_finish_kernel(RansacWork w, int refine_iters)
{
    constexpr int MP = Model::MP, N = Model::N;
    const int set = blockIdx.x;
    const int n = w.counts_n[set];
    const int64_t start = w.starts[set];
    const float4* __restrict__ pts = w.pts + start;
    uint8_t* mask = w.mask + start;
    int32_t* sel = w.sel + start;
    double* Mout = w.H + (size_t)set * 6;
    __shared__ AffineShared<N> sh;
    LmStateN<N>& st = sh.lm;
    const int tid = threadIdx.x;
    if (n < MP || (n > MP && w.best_iter[set] < 0)) {           // cv2 returns an empty matrix
        for (int i = tid; i < n; i += (int)blockDim.x) mask[i] = 0;
        if (tid < 6) Mout[tid] = 0.0;
        if (tid == 0) w.found[set] = 0;
        return;
    }
    if (n == MP) {                                               // count == modelPoints: the closed form, mask all 1, no refine
        if (tid == 0) {
            float ms1[2 * MP], ms2[2 * MP];
            for (int i = 0; i < MP; i++) { ms1[2 * i] = pts[i].x; ms1[2 * i + 1] = pts[i].y; ms2[2 * i] = pts[i].z; ms2[2 * i + 1] = pts[i].w; }
            double M[6];
            Model::solve(ms1, ms2, M);
            for (int i = 0; i < 6; i++) Mout[i] = M[i];
            w.found[set] = 1;
        }
        if (tid < MP) mask[tid] = 1;
        return;
    }
    if (tid == 0) {
        double M[6];
        affine_solve_sample<Model>(w, pts, n, w.sample_pos[(size_t)set * w.max_iters + w.best_iter[set]], M);
        Model::params(M, st.x);
        sh.base_cnt = 0;
    }
    __syncthreads();
    float F[6];
    {
        double M[6];
        Model::matrix(st.x, M);
        #pragma unroll
        for (int i = 0; i < 6; i++) F[i] = (float)M[i];
    }
    const int lane = tid & 31, wid = tid >> 5;
    for (int base = 0; base < n; base += (int)blockDim.x) {       // mask + ordered compaction of the inlier indices
        const int i = base + tid;
        bool in = false;
        if (i < n) {
            const float4 q = pts[i];
            in = affine_err(F, q.x, q.y, q.z, q.w) <= w.thr2;
            mask[i] = in ? 1 : 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) sh.warp_cnt[wid] = __popc(bal);
        __syncthreads();
        int off = sh.base_cnt;
        for (int k = 0; k < wid; k++) off += sh.warp_cnt[k];
        if (in) sel[off + __popc(bal & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (tid == 0) { int t = 0; for (int k = 0; k < (int)(blockDim.x >> 5); k++) t += sh.warp_cnt[k]; sh.base_cnt += t; }
        __syncthreads();
    }
    const int n_inl = sh.base_cnt;
    if (refine_iters > 0 && n_inl > 0) {
        affine_lm_eval<Model>(pts, sel, n_inl, st.x, true, sh);
        if (tid == 0) lm_begin(st);
        for (;;) {
            if (tid == 0) lm_step(st, sh.scratch_a, sh.scratch_v);
            __syncthreads();
            affine_lm_eval<Model>(pts, sel, n_inl, st.xd, false, sh);
            if (tid == 0) sh.flag = lm_update(st, sh.out[0], sh.scratch_a, sh.scratch_v) ? 1 : 0;
            __syncthreads();
            if (sh.flag) {                                       // accepted: x = xd, A, v, S, rmax at x
                if (tid == 0) for (int i = 0; i < N; i++) st.x[i] = st.xd[i];
                __syncthreads();
                affine_lm_eval<Model>(pts, sel, n_inl, st.x, true, sh);
            }
            if (tid == 0) sh.flag = lm_proceed(st, refine_iters) ? 1 : 0;
            __syncthreads();
            if (!sh.flag) break;
        }
    }
    if (tid == 0) {
        double M[6];
        Model::matrix(st.x, M);
        for (int i = 0; i < 6; i++) Mout[i] = M[i];
        w.found[set] = 1;
    }
}

template <class Model>
static int launch_affine_model(const RansacWork& w, int refine_iters, cudaStream_t st)
{
    const int round_len = ransac_round_len(w);
    const int n_sms = w.n_sms > 0 ? w.n_sms : 148;
    int launches = 0;
    for (int rb = 0; rb < w.max_iters; rb += round_len) {
        const int len = w.max_iters - rb < round_len ? w.max_iters - rb : round_len;
        ransac_sample_kernel<Model::MP><<<w.n_sets, SMP_THREADS, 0, st>>>(w, rb, rb + len, nullptr);
        cudaMemset2DAsync(w.counts + rb, (size_t)w.max_iters * 4, 0, (size_t)len * 4, (size_t)w.n_sets, st);
        // slices of the correspondences so that the launch holds >= ~6 CTAs per SM (or one slice per 512 points)
        const int tiles = (len + SCORE_THREADS - 1) / SCORE_THREADS;
        const int64_t ctas = (int64_t)tiles * w.n_sets;
        int n_slices = (int)std::min<int64_t>(std::max<int64_t>(1, ((int64_t)n_sms * 6 + ctas - 1) / ctas), std::max(1, w.max_n / 512));
        n_slices = std::max(1, std::min(n_slices, 64));
        ransac_affine_hyp_kernel<Model><<<dim3((unsigned)ctas, 1, (unsigned)n_slices), SCORE_THREADS, 0, st>>>(w, rb, len, n_slices, tiles);
        launches += 2 + launch_ransac_select(w, rb, len, st);
    }
    ransac_affine_finish_kernel<Model><<<w.n_sets, w.max_n <= 512 ? 64 : RS_THREADS, 0, st>>>(w, refine_iters);
    return launches + 1;
}

int launch_affine(const RansacWork& w, int refine_iters, cudaStream_t st)
{
    if (w.n_sets <= 0) return 0;
    return w.model_points == 2 ? launch_affine_model<PartialModel>(w, refine_iters, st)
                               : launch_affine_model<AffineModel>(w, refine_iters, st);
}

// ---- gates + inlier gather: reference src/TestsDetector.cpp:74-94 ---------------------------------
__global__ void gates_kernel(GateWork g)
{
    const int pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (pair >= g.n_pairs) return;
    const int n = g.counts_n[pair];
    const int64_t start = g.starts[pair];
    const uint8_t* mask = g.mask + start;
    const float4* pts = g.pts + start;
    const bool found = n >= g.model_points && g.found[pair] != 0;
    int cnt = 0;
    if (found)
        for (int i = lane; i < n; i += 32) cnt += mask[i] ? 1 : 0;
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    // a 2x3 affine M (stride 6) is promoted to [M; 0 0 1]: its det3 is the area scale M00*M11 - M01*M10
    const double* Hs = g.H + (size_t)pair * g.h_stride;
    double H[9];
    #pragma unroll
    for (int i = 0; i < 6; i++) H[i] = found ? Hs[i] : 0.0;
    if (g.h_stride == 9) {
        #pragma unroll
        for (int i = 6; i < 9; i++) H[i] = found ? Hs[i] : 0.0;
    } else {
        H[6] = 0.0; H[7] = 0.0; H[8] = found ? 1.0 : 0.0;
    }
    const double det = found ? det3(H) : 0.0;
    int status;
    if (n < g.min_inliers) status = CVG_PAIR_LT4_MATCHES;                     // :74
    else if (!found) status = CVG_PAIR_H_EMPTY;                              // :79
    else if (cnt < g.min_inliers) status = CVG_PAIR_LT4_INLIERS;             // :81
    else {
        const double ad = fabs(det);                                          // :84, float constants promoted
        status = (ad < (double)g.det_lo || ad > (double)g.det_hi) ? CVG_PAIR_DET_REJECT : CVG_PAIR_ACCEPT;
    }
    if (lane == 0) {
        cvg_pair_result r;
        r.status = status; r.n_good = n; r.n_inliers = found ? cnt : 0;
        r.ransac_iters = g.iters_run ? g.iters_run[pair] : 0;
        for (int i = 0; i < 9; i++) r.H[i] = H[i];
        r.det = det;
        g.results[pair] = r;
    }
    if (g.inlier_xy) {
        // :87-94 — inlier scene points, in order, divided by scale when scale != 1.0f
        int written = 0;
        if (status == CVG_PAIR_ACCEPT) {
            const float scale = g.pair_scale ? g.pair_scale[pair] : 1.0f;
            float* out = g.inlier_xy + 2 * start;
            for (int base = 0; base < n; base += 32) {
                const int i = base + lane;
                const bool in = i < n && mask[i];
                const unsigned bal = __ballot_sync(0xffffffffu, in);
                if (in) {
                    const int o = written + __popc(bal & ((1u << lane) - 1));
                    float x = pts[i].z, y = pts[i].w;
                    if (scale != 1.0f) { x = __fdiv_rn(x, scale); y = __fdiv_rn(y, scale); }
                    out[2 * o] = x; out[2 * o + 1] = y;
                }
                written += __popc(bal);
            }
        }
        if (lane == 0) g.inlier_count[pair] = written;
    }
}

void launch_gates(const GateWork& g, cudaStream_t st)
{
    if (g.n_pairs <= 0) return;
    gates_kernel<<<(g.n_pairs + 3) / 4, 128, 0, st>>>(g);
}

// ---- compaction of ratio-test survivors into correspondences: reference src/TestsDetector.cpp:62-72 --
// one block per (segment, view) pair; output order = query order (block-wide ordered compaction)
constexpr int CMP_THREADS = 256;

__global__ void __launch_bounds__(CMP_THREADS)
compact_kernel(CompactWork c)
{
    const int pair = blockIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int seg = pair / c.n_views, view = pair % c.n_views;
    const int r0 = c.view_offsets[view], r1 = c.view_offsets[view + 1];
    const int64_t start = (int64_t)seg * c.n_query + r0;
    const int32_t* idx = c.idx + (size_t)seg * c.n_query * 2;
    const uint8_t* acc = c.accept + (size_t)seg * c.n_query;
    const float2* mk = reinterpret_cast<const float2*>(c.model_kpt);
    const float2* sk = reinterpret_cast<const float2*>(c.scene_kpt) + c.seg_kpt_offsets[seg];
    float4* out = c.pts + start;
    __shared__ int s_wcnt[CMP_THREADS / 32];
    __shared__ int s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int base = r0; base < r1; base += CMP_THREADS) {
        const int q = base + threadIdx.x;
        const bool in = q < r1 && acc[q];
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) s_wcnt[wid] = __popc(bal);
        __syncthreads();
        int off = s_base;
        for (int k = 0; k < wid; k++) off += s_wcnt[k];
        if (in) {
            const float2 a = mk[q];                           // model.keypoints[i][queryIdx].pt   :68
            const float2 b = sk[idx[2 * q]];                  // sceneKP[trainIdx].pt              :69
            out[off + __popc(bal & ((1u << lane) - 1))] = make_float4(a.x, a.y, b.x, b.y);
        }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < CMP_THREADS / 32; k++) t += s_wcnt[k]; s_base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { c.starts[pair] = start; c.n_good[pair] = s_base; }
}

void launch_compact(const CompactWork& c, cudaStream_t st)
{
    const int n = c.n_segments * c.n_views;
    if (n <= 0) return;
    compact_kernel<<<n, CMP_THREADS, 0, st>>>(c);
}

}  // namespace cvg
