// match_tc.cu — tensor-core match kernel for sm_100a: TMA -> shared memory -> tcgen05.mma -> TMEM ->
// fused per-query top-2 epilogue.  No distance matrix ever reaches HBM.
//
// Reference: BFMatcher(NORM_L2).knnMatch(view_desc, scene_desc, 2), src/TestsDetector.cpp:59-60.
// The accumulator is  acc' = 2 q.t - ||t||^2  (operands prepared by prep.cu; exact for integer
// descriptors), so the nearest train row maximises acc' and  d^2 = ||q||^2 - acc'.
//
// CTA = 576 threads, one CTA per SM, persistent over a static list of units (128 query rows x a run
// of 256-wide train tiles):
//   warp 0      TMA producer   : A tile (queries, resident per unit, double-buffered), a 4-stage ring of
//                                half-K B stages (256 train rows x 64 K, SWIZZLE_128B) and a 2-stage ring of the
//                                16-column norm augmentation (SWIZZLE_32B)
//   warp 1      MMA issuer     : per tile 8 x tcgen05.mma (M128 N256 K16, bf16 -> fp32) + 1 augmentation MMA
//                                into one of two 256-column TMEM accumulators; owns TMEM alloc
//   warps 2-17  epilogue       : tcgen05.ld 32x32b.x32 (thread = query row, 32 train columns per
//                                load), running top-2 per row kept in registers across the unit, four
//                                warps per TMEM lane quarter (64 columns each), merged at unit end
// Pipelines: a_full/a_empty, b_full/b_empty (TMA <-> MMA), t_full/t_empty (MMA <-> epilogue).
// Warps 0 and 1 walk their loops with all 32 lanes converged (every lane waits on the mbarriers) and ONE elect.sync lane
// issues: inside an `if (lane == 0)` region ptxas wraps each tcgen05.mma / commit / TMA instruction in an election loop
// and moves every descriptor through R2UR, ~250 instructions per tile instead of ~60 (DESIGN.md 4.1: 1.11 -> 0.96 ms).
//
// Cross-check form (KP = 1, BFMatcher(NORM_L2, crossCheck = true)): the same producer, MMA issuer and accumulator; the
// epilogue keeps each query row's nearest column and, per tile, reduces each train column to its nearest query row of the
// unit's view (redux.sync per warp, shared atomicMin over the four TMEM lane quarters, one global atomicMin per column and
// unit).  DESIGN.md 4.5.
//
// Pair mode (template PAIR, opt-in: CVG_MATCH_PAIR_MODE): the same kernel as clusters of two CTAs around
// tcgen05.mma.cta_group::2 (M256 N256 K16): each CTA holds its own query tile and half of every train stage, TMA loads
// are counted on the leader CTA's barriers, the leader issues the MMAs and multicasts its commits to both CTAs, both
// epilogues scan their own TMEM and arrive on the leader's barrier.  Bit-equal results; measured slower on B200
// (DESIGN.md 4.1), so the one-CTA form stays the default.
#include "common.cuh"
#include <cuda.h>
#include <string.h>
#include <stdlib.h>
#include <mutex>

namespace cvg {

constexpr int TC_EPI_WARPS = 16;                                 // 4 per TMEM lane quarter: 64 columns each per tile
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;                // 576
constexpr uint32_t A_ATOM_BYTES = TILE_M * 128;                   // 128 rows x 64 bf16          16 KB
constexpr uint32_t A_AUG_BYTES = TILE_M * KAUG * 2;               // 128 rows x 16 bf16           4 KB
constexpr uint32_t A_BYTES = 2 * A_ATOM_BYTES + A_AUG_BYTES;      //                             36 KB
// The train operand streams through two rings: 4 stages of [256 rows x 64 K] (one SWIZZLE_128B atom, 32 KB,
// released after its 4 MMAs) and 2 stages of the 16-column augmentation (8 KB).  Splitting K instead of N keeps
// the MMA at N=256 — an SS-mode MMA re-reads its A slice from shared memory for every instruction, and 64-row
// slices (measured) are 1.4x slower because they need 192 B/cycle of shared-memory bandwidth — while refills
// start twice as early as with whole 72 KB tiles, which hides the L2 latency of the next tile.
constexpr int B_STAGES = 4;                                       // half-K stages
constexpr uint32_t B_ATOM_BYTES = TILE_N * 128;                   // 256 rows x 64 bf16          32 KB
constexpr uint32_t B_AUG_BYTES = TILE_N * KAUG * 2;               //                              8 KB
// Pair mode (cta_group::2): two CTAs of a cluster run ONE M256 N256 MMA on two 128-row query tiles against the same
// train tiles.  Each CTA holds its own A tile and HALF of every B stage (128 train rows x 64 K = 16 KB), so a CTA pulls
// 36 KB instead of 72 KB per tile out of L2 — the single-CTA kernel is bound by L2 -> SM bandwidth (148 x 72 KB per
// 1.2 us tile = 17 TB/s wanted) — and the same 128 KB ring holds 8 stages (4 tiles of prefetch instead of 2).
constexpr int B_STAGES_PAIR = 8;
constexpr uint32_t B_HALF_BYTES = B_ATOM_BYTES / 2;               // 128 rows x 64 bf16          16 KB
constexpr uint32_t B_AUG_HALF_BYTES = B_AUG_BYTES / 2;            //                              4 KB
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;                       // shared::cluster address of the pair's even CTA
constexpr uint32_t OFF_A = 0;
constexpr uint32_t OFF_B = 2 * A_BYTES;                           //  72 KB
constexpr uint32_t OFF_BAUG = OFF_B + B_STAGES * B_ATOM_BYTES;    // 200 KB
constexpr uint32_t OFF_SCRATCH = OFF_BAUG + 2 * B_AUG_BYTES;      // 216 KB
constexpr uint32_t SCRATCH_BYTES = 3 * TILE_M * 16;                 // partial top-2 of column parts 1..3 at unit end
constexpr uint32_t OFF_SHARE = OFF_SCRATCH + SCRATCH_BYTES;         // running (best, second best) of every column part, per row
constexpr uint32_t SHARE_BYTES = 4 * TILE_M * 8;                    //                              4 KB
constexpr uint32_t OFF_BAR = OFF_SHARE + SHARE_BYTES;
// cross-check form: the row merge (3 parts x 128 rows x 8 B) and the 16 tile counters live in the scratch area, the column
// keys of four tiles (4 x 256 x 4 B) in the share area
constexpr uint32_t XC_MERGE_BYTES = 3 * TILE_M * 8;
static_assert(XC_MERGE_BYTES + 16 * 4 <= SCRATCH_BYTES && 4 * TILE_N * 4 <= SHARE_BYTES, "cross-check shared memory");
constexpr uint32_t TC_SMEM_SLACK = 512;                           // the dynamic window is 1024-aligned in practice; checked in the kernel
constexpr uint32_t TC_SMEM_BYTES = OFF_BAR + 512 + TC_SMEM_SLACK;
static_assert(TC_SMEM_BYTES <= 232448, "shared memory budget of one CTA (227 KB)");
#ifndef TC_ISSUER_UNROLL
#define TC_ISSUER_UNROLL 2                                        // stage loop of the MMA issuer: 1 = rolled
#endif
constexpr int kIssuerUnroll = TC_ISSUER_UNROLL;
#ifndef TC_ISSUER_WARP
#define TC_ISSUER_WARP 1
#endif
#ifndef TOP2_GROUPS_PER_TEST
#define TOP2_GROUPS_PER_TEST 4                                    // groups of 4 columns per filter test; same run: 1 -> 1.061 ms, 2 -> 0.957, 4 -> 0.949
#endif
constexpr float ABSENT_BELOW = -5.0e8f;                           // padded train rows carry -2^30

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a protocol bug must trap, not hang the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* dbg, int code)
{
    for (uint32_t spin = 0; !mbar_try_wait(bar, parity); spin++) {
        if (spin > (1u << 26)) {
            if (dbg) { dbg[0] = code; dbg[1] = (int)blockIdx.x; dbg[2] = (int)threadIdx.x; }
            __threadfence_system();
            __trap();
        }
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// pair mode: the load lands in this CTA's shared memory, its bytes are counted on the LEADER CTA's barrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(dst), "l"(map), "r"(bar & PEER_MASK), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar)
{
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" :: "r"(bar & PEER_MASK) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar)       // arrives on the barrier at this offset in BOTH CTAs
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ bool elect_one()                       // one lane of the (converged) warp
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "elect.sync _|p, 0xffffffff;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok));
    return ok != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t* r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptors (K-major).  Bits: [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4,
// [46,48) version = 1 (Blackwell), [61,64) layout type (2 = SWIZZLE_128B, 6 = SWIZZLE_32B).
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr)
{
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint64_t desc_sw32(uint32_t saddr)
{
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46) | (6ull << 61);
}
// instruction descriptor, kind::f16: D = F32 (bits 4-5 = 1), A = B = BF16 (bits 7-9, 10-12 = 1),
// both K-major (bits 15, 16 = 0), N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t TC_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE_N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
constexpr uint32_t TC_IDESC_PAIR = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE_N >> 3) << 17) | ((uint32_t)((2 * TILE_M) >> 4) << 24);

// Running top-2 (largest acc') of one query row over 32 more train columns.  `f` is the row's filter: no
// column with a value <= f can be one of the row's two best (f >= the warp's own second best b2, and it is
// raised further by what the other three column parts of the same rows have found, see the epilogue).  Maxima
// of groups of 4 columns are compared with it first, so a group costs ~2 instructions per lane unless one of
// the warp's 32 rows really has a candidate in it.  Strict > against the warp's own values keeps the earlier
// (lower) train index on ties, as cv::batchDistance's insertion does.
__device__ __forceinline__ void top2_insert4(const uint32_t* r4, int c, float& b1, int& i1, float& b2, int& i2, float& f)
{
    #pragma unroll
    for (int j = 0; j < 4; j++) {
        const float v = __uint_as_float(r4[j]);
        if (v > f) {
            if (v > b1) { b2 = b1; i2 = i1; b1 = v; i1 = c + j; }
            else        { b2 = v; i2 = c + j; }
            f = fmaxf(f, b2);
        }
    }
}

// The same for a group of 4 columns whose maximum gmax is known to exceed f.  Nearly always exactly ONE column of the group
// is a candidate, so the maximum is inserted without branches (its column = the first one equal to gmax) and only a second
// candidate in the same group — the largest of the other three still above the raised filter — takes the generic path.
// Inserting the maximum first gives the result of the ascending scan: among equal values the first column goes in first,
// and a smaller value that is inserted after a larger one lands where the ascending scan would have left it.
struct Top2State { float b1; int i1; float b2; int i2; float f; };
#ifndef TC_OUTLINE_SLOW
#define TC_OUTLINE_SLOW 0       // measured: the outlined slow path halves the kernel (3048 -> 1608 SASS instructions) but costs 7 % (call overhead)
#endif
#if TC_OUTLINE_SLOW
__device__ __noinline__
#else
__device__ __forceinline__
#endif
Top2State top2_insert_group_impl(float v0, float v1, float v2, float v3, int c, float gmax, Top2State st)
{
    float b1 = st.b1, b2 = st.b2, f = st.f; int i1 = st.i1, i2 = st.i2;
    int j = 3;
    j = (v2 == gmax) ? 2 : j; j = (v1 == gmax) ? 1 : j; j = (v0 == gmax) ? 0 : j;
    const bool top = gmax > b1;
    b2 = top ? b1 : gmax; i2 = top ? i1 : c + j;
    b1 = top ? gmax : b1; i1 = top ? c + j : i1;
    f = fmaxf(f, b2);
    const float w0 = j == 0 ? -INFINITY : v0, w1 = j == 1 ? -INFINITY : v1, w2 = j == 2 ? -INFINITY : v2, w3 = j == 3 ? -INFINITY : v3;
    if (fmaxf(fmaxf(w0, w1), fmaxf(w2, w3)) > f) {
        const float w[4] = { w0, w1, w2, w3 };
        #pragma unroll
        for (int k = 0; k < 4; k++) {
            const float v = w[k];
            if (v > f) {
                if (v > b1) { b2 = b1; i2 = i1; b1 = v; i1 = c + k; }
                else        { b2 = v; i2 = c + k; }
                f = fmaxf(f, b2);
            }
        }
    }
    return Top2State{ b1, i1, b2, i2, f };
}
__device__ __forceinline__ void top2_insert_group(const uint32_t* r4, int c, float gmax, float& b1, int& i1, float& b2, int& i2, float& f)
{
    const Top2State st = top2_insert_group_impl(__uint_as_float(r4[0]), __uint_as_float(r4[1]), __uint_as_float(r4[2]), __uint_as_float(r4[3]),
                                                c, gmax, Top2State{ b1, i1, b2, i2, f });
    b1 = st.b1; i1 = st.i1; b2 = st.b2; i2 = st.i2; f = st.f;
}

// A group of 8 columns whose maximum gmax exceeds f, as ONE straight-line region (the two groups of 4 used to be two divergent
// regions entered by different lanes one after the other): the column of the maximum is the lowest set bit of the mask of
// equal values, the insertion is a handful of selects, and a second candidate among the other seven — rare — takes the
// generic ascending loop.
__device__ __forceinline__ void top2_insert_group8(const uint32_t* r8, int c, float gmax, float& b1, int& i1, float& b2, int& i2, float& f)
{
    float v[8];
    #pragma unroll
    for (int k = 0; k < 8; k++) v[k] = __uint_as_float(r8[k]);
    unsigned eq = 0;
    #pragma unroll
    for (int k = 0; k < 8; k++) eq |= (v[k] == gmax) ? (1u << k) : 0u;
    const int j = __ffs((int)eq) - 1;
    const bool top = gmax > b1;
    b2 = top ? b1 : gmax; i2 = top ? i1 : c + j;
    b1 = top ? gmax : b1; i1 = top ? c + j : i1;
    f = fmaxf(f, b2);
    float w[8];
    #pragma unroll
    for (int k = 0; k < 8; k++) w[k] = (k == j) ? -INFINITY : v[k];
    const float rest = fmaxf(fmaxf(fmaxf(w[0], w[1]), fmaxf(w[2], w[3])), fmaxf(fmaxf(w[4], w[5]), fmaxf(w[6], w[7])));
    if (rest > f) {
        #pragma unroll
        for (int k = 0; k < 8; k++) {
            const float x = w[k];
            if (x > f) {
                if (x > b1) { b2 = b1; i2 = i1; b1 = x; i1 = c + k; }
                else        { b2 = x; i2 = c + k; }
                f = fmaxf(f, b2);
            }
        }
    }
}

#ifdef TC_PROF
__device__ int g_prof_entries[4];
#define PROF_ENTRY(k) { const unsigned am__ = __activemask(); if ((int)(threadIdx.x & 31) == __ffs(am__) - 1) { atomicAdd(&g_prof_entries[k], 1); atomicAdd(&g_prof_entries[k + 1], __popc(am__)); } }
#else
#define PROF_ENTRY(k)
#endif
__device__ __forceinline__ void top2_scan32(const uint32_t* r, int c0, float& b1, int& i1, float& b2, int& i2, float& f)
{
    float g[8];
    #pragma unroll
    for (int k = 0; k < 8; k++)
        g[k] = fmaxf(fmaxf(__uint_as_float(r[4 * k]), __uint_as_float(r[4 * k + 1])),
                     fmaxf(__uint_as_float(r[4 * k + 2]), __uint_as_float(r[4 * k + 3])));
    // one branch per 16 columns on the fast path (branch resolution was 17 % of the epilogue's stalls with one per 4)
    #pragma unroll
    for (int k = 0; k < 8; k += TOP2_GROUPS_PER_TEST) {
        float gm = g[k];
        #pragma unroll
        for (int e = 1; e < TOP2_GROUPS_PER_TEST; e++) gm = fmaxf(gm, g[k + e]);
        if (gm > f) {
            PROF_ENTRY(0)
#ifndef TOP2_INSERT8
#define TOP2_INSERT8 0                             // measured: one region per 8 columns 1.153 ms, two regions of 4 columns 1.102 ms
#endif
#if TOP2_INSERT8 && TOP2_GROUPS_PER_TEST == 2
            top2_insert_group8(r + 4 * k, c0 + 4 * k, gm, b1, i1, b2, i2, f);
#else
            #pragma unroll
            for (int e = 0; e < TOP2_GROUPS_PER_TEST; e++)
                if (g[k + e] > f) top2_insert_group(r + 4 * (k + e), c0 + 4 * (k + e), g[k + e], b1, i1, b2, i2, f);
#endif
        }
    }
}

// The first tile(s) of a unit: no filter exists yet, every group of columns holds candidates for every row, and the branchy
// scan above would run its slow path 16 times per tile with all 32 lanes diverging.  Here every column is inserted without
// a branch (strict >: ties keep the earlier column, as the ascending scan does).
__device__ __forceinline__ void top2_dense32(const uint32_t* r, int c0, float& b1, int& i1, float& b2, int& i2)
{
    #pragma unroll
    for (int j = 0; j < 32; j++) {
        const float v = __uint_as_float(r[j]);
        const bool gt1 = v > b1, gt2 = v > b2;
        b2 = gt1 ? b1 : (gt2 ? v : b2);
        i2 = gt1 ? i1 : (gt2 ? c0 + j : i2);
        b1 = gt1 ? v : b1;
        i1 = gt1 ? c0 + j : i1;
    }
}

__device__ __forceinline__ void share_store(uint32_t addr, float a, float b)
{
    asm volatile("st.volatile.shared.v2.f32 [%0], {%1, %2};" :: "r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void share_load(uint32_t addr, float& a, float& b)
{
    asm volatile("ld.volatile.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "r"(addr) : "memory");
}

// Candidate form for non-integer descriptors (the accumulator is then an approximation of 2 q.t - ||t||^2): the four
// largest values per row are kept; the fp32 re-rank (match_exact.cu) decides among them and proves, with an error
// bound, that no other column can belong to the two nearest.  Ties need no care here: a column that is dropped has
// a value <= the fourth kept one, which is all the bound uses.
__device__ __forceinline__ void top4_scan32(const uint32_t* r, int c0, float (&b)[4], int (&ix)[4], float& f)
{
    float g[8];
    #pragma unroll
    for (int k = 0; k < 8; k++)
        g[k] = fmaxf(fmaxf(__uint_as_float(r[4 * k]), __uint_as_float(r[4 * k + 1])),
                     fmaxf(__uint_as_float(r[4 * k + 2]), __uint_as_float(r[4 * k + 3])));
    #pragma unroll
    for (int k = 0; k < 8; k++) {
        if (g[k] > f) {
            #pragma unroll
            for (int j = 0; j < 4; j++) {
                const float v = __uint_as_float(r[4 * k + j]);
                if (v > f) {
                    const int id = c0 + 4 * k + j;
                    if (v > b[2]) {
                        b[3] = b[2]; ix[3] = ix[2];
                        if (v > b[1]) {
                            b[2] = b[1]; ix[2] = ix[1];
                            if (v > b[0]) { b[1] = b[0]; ix[1] = ix[0]; b[0] = v; ix[0] = id; }
                            else          { b[1] = v; ix[1] = id; }
                        } else { b[2] = v; ix[2] = id; }
                    } else { b[3] = v; ix[3] = id; }
                    f = fmaxf(f, b[3]);
                }
            }
        }
    }
}

// ---- cross-check epilogue (KP = 1) ----
// Nearest column of a row over 32 more columns: larger acc' wins, ties keep the lower column (the ascending scan's strict >).
__device__ __forceinline__ void xc_row_scan32(const uint32_t* r, int c0, float& b1, int& i1)
{
    float m = __uint_as_float(r[0]);
    #pragma unroll
    for (int k = 1; k < 32; k++) m = fmaxf(m, __uint_as_float(r[k]));
    if (m > b1) {
        int j = 31;
        #pragma unroll
        for (int k = 30; k >= 0; k--) j = (__uint_as_float(r[k]) == m) ? k : j;
        b1 = m; i1 = c0 + j;
    }
}
// Column keys of 32 columns for this warp's 32 rows, reduced over the warp and merged into the tile's shared slots.
// qbias = ||q||^2 + 2^23 (exact: ||q||^2 < 2^23 for rows of 0..255), so qbias - acc' = d^2 + 2^23 exactly and its float
// bits are 0x4B000000 + d^2: shifted left by 7 (the constant part wraps to 0x80000000) and or-ed with the row in the tile,
// the key orders by (d^2, row) and stays <= 0xBFFFFFFF.  Rows outside the unit's view have qbias = inf: key 0xC00000xx.
constexpr uint32_t XC_KEY_ABSENT = 0xC0000000u;
__device__ __forceinline__ void xc_col_keys32(const uint32_t* r, float qbias, uint32_t row, uint32_t* slots, int lane)
{
    #pragma unroll
    for (int k = 0; k < 32; k++) {
        const uint32_t key = (__float_as_uint(__fsub_rn(qbias, __uint_as_float(r[k]))) << 7) | row;
        const uint32_t m = __reduce_min_sync(0xffffffffu, key);
        if (lane == 0) atomicMin(&slots[k], m);
    }
}

struct TcMaps { CUtensorMap q, qaug, t, taug, qlo, tlo, th, taugh; };   // th / taugh: 128-row boxes of the train operand (pair mode)

// KP = 1: cross-check keys (integer descriptors), parts_out = XcOut (common.cuh: key layout); units of build_xc_plan.
// KP = 2: exact top-2 per row (integer descriptors), partial records Top2 with distances.
// KP = 4: four candidates per row and column part (non-integer descriptors), partial records Top4 with raw
//         accumulator values, slot (part_slot * 4 + column part).
// PAIR: launched as clusters of two CTAs (cta_group::2); unit 2p + r belongs to CTA r of the cluster that owns pair p, and
//       both units of a pair name the same train tiles.
// EXPB: the instance with the CVG_TC_EXP experiment switches; the product instance (EXPB = false) carries none of their
//       per-tile tests (~15 instructions per warp and tile in a loop that is bound by its instruction count).
template <int KP, bool PAIR, bool EXPB>
__global__ void __launch_bounds__(TC_THREADS, 1)
match_tc_kernel(const __grid_constant__ TcMaps maps, const float* __restrict__ qnorm,
                const MatchUnit* __restrict__ units, int n_units, void* __restrict__ parts_out,
                const int* __restrict__ gate_flag, int gate_want, int* dbg, int exp_mode_arg)
{
    const int exp_mode = EXPB ? exp_mode_arg : 0;
    // exp_mode (experiments only, set through CVG_TC_EXP): bit 0 = epilogue releases the accumulator without
    // scanning it, bit 1 = the producer re-arms ring stages without issuing the B loads
    if (gate_flag && *gate_flag != gate_want) return;
#ifdef TC_PROF
    if (blockIdx.x == 0 && threadIdx.x == 0 && dbg) {        // slow-path entries of the PREVIOUS launch: warp level, lane level
        dbg[34] = g_prof_entries[0]; dbg[35] = g_prof_entries[1];
        g_prof_entries[0] = 0; g_prof_entries[1] = 0;
    }
#endif
    constexpr bool SPLIT = KP == 4;                  // hi/lo split operands (non-integer descriptors)
    static_assert(!(SPLIT && PAIR), "pair mode serves the exact (integer descriptor) form only");
    constexpr int N_STAGES_PER_TILE = SPLIT ? 4 : 2;
    constexpr int NB = PAIR ? B_STAGES_PAIR : B_STAGES;                   // ring stages
    constexpr uint32_t STAGE_BYTES = PAIR ? B_HALF_BYTES : B_ATOM_BYTES;  // bytes of a ring stage in THIS CTA
    const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    // persistent loop: worker w of n_workers takes list entries w, w + n_workers, ...; an entry is a unit, or a pair of units
    const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int n_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_entries = PAIR ? n_units / 2 : n_units;
    auto unit_of = [&](int e) { return PAIR ? 2 * e + (int)cta_rank : e; };
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (smem_base - smem_u32(smem_raw));
    if (smem_base - smem_u32(smem_raw) > TC_SMEM_SLACK) {          // never seen: the window starts 1024-aligned
        if (dbg) { dbg[0] = 9; dbg[1] = (int)blockIdx.x; }
        __trap();
    }
    const uint32_t bar0 = smem_base + OFF_BAR;
    // barrier slots (8 bytes each)
    const uint32_t a_full = bar0, a_empty = bar0 + 16, t_full = bar0 + 32, t_empty = bar0 + 48;
    const uint32_t b_full = bar0 + 64, b_empty = bar0 + 64 + 8 * NB;
    constexpr int NG = PAIR ? 4 : 2;                                                // augmentation ring stages (pair: 4 KB each, as deep as the B ring)
    constexpr uint32_t G_BYTES = PAIR ? B_AUG_HALF_BYTES : B_AUG_BYTES;
    const uint32_t g_full = bar0 + 64 + 16 * NB, g_empty = g_full + 8 * NG;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 64 + 16 * NB + 16 * NG + 16);
    int* chunk_ctr = reinterpret_cast<int*>(smem + OFF_BAR + 480);      // [4]: next 64-column chunk of the unit, per TMEM lane quarter
    static_assert(64 + 16 * B_STAGES_PAIR + 16 * 4 + 16 + 8 <= 512, "barrier area");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; i++) chunk_ctr[i] = 0;
        for (int i = 0; i < 2; i++) {
            mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, 1);
            mbar_init(t_full + 8 * i, 1); mbar_init(t_empty + 8 * i, (PAIR ? 2 : 1) * TC_EPI_WARPS);   // pair: both CTAs' epilogues arrive on the leader's
        }
        for (int i = 0; i < NG; i++) { mbar_init(g_full + 8 * i, 1); mbar_init(g_empty + 8 * i, 1); }
        for (int i = 0; i < NB; i++) { mbar_init(b_full + 8 * i, 1); mbar_init(b_empty + 8 * i, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        if constexpr (PAIR) {                            // the same warp of both CTAs
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" :: "r"(smem_u32(tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" :: "r"(smem_u32(tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();          // the peer's barriers are initialised before anything is sent to them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
#if TC_ISSUER_WARP
        const bool el = elect_one();                 // all lanes walk the loop and wait, one issues (see the MMA issuer)
        {
#else
        constexpr bool el = true;
        if (lane == 0) {
#endif
            auto expect_tx = [&](uint32_t bar, uint32_t bytes) { if (el) mbar_expect_tx(bar, bytes); };
            auto load = [&](uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) { if (el) tma_load_2d(dst, map, c0, c1, bar); };
            auto load_pair = [&](uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) { if (el) tma_load_2d_pair(dst, map, c0, c1, bar); };
            auto arrive = [&](uint32_t bar) { if (el) mbar_arrive(bar); };
            uint32_t ua = 0, bs = 0, tcnt = 0;
            for (int e = worker; e < n_entries; e += n_workers, ua++) {
                const MatchUnit un = units[unit_of(e)];
                // KP == 2: A tile (queries) double-buffered.  KP == 4 (split operands): one buffer holding the hi and lo
                // halves of 2q — [hi k 0-63][hi k 64-127][lo k 0-63][lo k 64-127][aug] = 68 KB in the same 72 KB region.
                const uint32_t ab = SPLIT ? 0u : (ua & 1);
                mbar_wait(a_empty + 8 * ab, (SPLIT ? (ua & 1) : ((ua >> 1) & 1)) ^ 1, dbg, 1);
                const uint32_t sa = smem_base + OFF_A + ab * A_BYTES;
                if constexpr (SPLIT) {
                    expect_tx(a_full, 4 * A_ATOM_BYTES + A_AUG_BYTES);
                    load(sa, &maps.q, 0, un.q_row0, a_full);
                    load(sa + A_ATOM_BYTES, &maps.q, 64, un.q_row0, a_full);
                    load(sa + 2 * A_ATOM_BYTES, &maps.qlo, 0, un.q_row0, a_full);
                    load(sa + 3 * A_ATOM_BYTES, &maps.qlo, 64, un.q_row0, a_full);
                    load(sa + 4 * A_ATOM_BYTES, &maps.qaug, 0, un.q_row0, a_full);
                } else if constexpr (PAIR) {
                    // both CTAs load their own query tile; the bytes of both are counted on the leader's barrier
                    if (leader) expect_tx(a_full + 8 * ab, 2 * A_BYTES);
                    load_pair(sa, &maps.q, 0, un.q_row0, a_full + 8 * ab);
                    load_pair(sa + A_ATOM_BYTES, &maps.q, 64, un.q_row0, a_full + 8 * ab);
                    load_pair(sa + 2 * A_ATOM_BYTES, &maps.qaug, 0, un.q_row0, a_full + 8 * ab);
                } else {
                    expect_tx(a_full + 8 * ab, A_BYTES);
                    load(sa, &maps.q, 0, un.q_row0, a_full + 8 * ab);
                    load(sa + A_ATOM_BYTES, &maps.q, 64, un.q_row0, a_full + 8 * ab);
                    load(sa + 2 * A_ATOM_BYTES, &maps.qaug, 0, un.q_row0, a_full + 8 * ab);
                }
                for (int t = 0; t < un.n_tiles; t++, tcnt++) {
                    const int row = un.t_row0 + t * TILE_N;
                    // ring stages of a tile: the two K halves of the train operand; split operands add the two K halves
                    // of its lo part (stages 2, 3)
                    #pragma unroll 1
                    for (int h = 0; h < N_STAGES_PER_TILE; h++, bs++) {
                        const uint32_t s = bs % NB;
                        mbar_wait(b_empty + 8 * s, ((bs / NB) & 1) ^ 1, dbg, 2);
                        if constexpr (PAIR) {
                            // this CTA's half of the stage: train rows [row + 128 r, +128) — accumulator columns 128 r ..
                            if ((exp_mode & 2) && bs >= NB) { if (leader) arrive(b_full + 8 * s); continue; }
                            if (leader) expect_tx(b_full + 8 * s, 2 * B_HALF_BYTES);
                            load_pair(smem_base + OFF_B + s * B_HALF_BYTES, &maps.th, 64 * (h & 1), row + (int)cta_rank * (TILE_N / 2),
                                             b_full + 8 * s);
                            continue;
                        }
                        if (!SPLIT && (exp_mode & 2) && bs >= B_STAGES) { arrive(b_full + 8 * s); continue; }
                        expect_tx(b_full + 8 * s, B_ATOM_BYTES);
                        load(smem_base + OFF_B + s * B_ATOM_BYTES, (SPLIT && h >= 2) ? &maps.tlo : &maps.t, 64 * (h & 1), row,
                                    b_full + 8 * s);
                    }
                    const uint32_t g = tcnt % NG;
                    mbar_wait(g_empty + 8 * g, ((tcnt / NG) & 1) ^ 1, dbg, 7);
                    if constexpr (PAIR) {
                        if (leader) expect_tx(g_full + 8 * g, 2 * B_AUG_HALF_BYTES);
                        load_pair(smem_base + OFF_BAUG + g * G_BYTES, &maps.taugh, 0, row + (int)cta_rank * (TILE_N / 2), g_full + 8 * g);
                        continue;
                    }
                    expect_tx(g_full + 8 * g, B_AUG_BYTES);
                    load(smem_base + OFF_BAUG + g * B_AUG_BYTES, &maps.taug, 0, row, g_full + 8 * g);
                }
            }
            if constexpr (PAIR) {
                // tail: the leader's last commits are multicast to this CTA's barriers as well; wait for the release of
                // every slot's last use so that nothing is still on its way here when the CTA exits
                for (int k = 0; k < NB; k++, bs++) mbar_wait(b_empty + 8 * (bs % NB), ((bs / NB) & 1) ^ 1, dbg, 12);
                for (int k = 0; k < NG; k++, tcnt++) mbar_wait(g_empty + 8 * (tcnt % NG), ((tcnt / NG) & 1) ^ 1, dbg, 13);
                for (int k = 0; k < 2; k++, ua++) mbar_wait(a_empty + 8 * (ua & 1), ((ua >> 1) & 1) ^ 1, dbg, 14);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
#if TC_ISSUER_WARP
        // the whole warp walks the loop and waits; one elected lane issues (the compiler then keeps the descriptor
        // arithmetic on the uniform datapath and needs no per-instruction election loop around tcgen05.mma / commit)
        const bool el = elect_one();
        if (leader) {
#else
        constexpr bool el = true;
        if (lane == 0 && leader) {                   // pair mode: the leader CTA issues for both
#endif
            uint32_t ua = 0, bs = 0, tc = 0;
#ifdef TC_PROF
            long long w_a = 0, w_t = 0, w_b = 0, w_g = 0, q0 = 0; const long long m_start = clock64();
#define MPROF_BEGIN q0 = clock64();
#define MPROF_END(acc) acc += clock64() - q0;
#else
#define MPROF_BEGIN
#define MPROF_END(acc)
#endif
            auto mma = [&](uint32_t d, uint64_t da, uint64_t db, uint32_t accumulate) {
                if (!el) return;
                if constexpr (PAIR) tc_mma_bf16_pair(d, da, db, TC_IDESC_PAIR, accumulate);
                else tc_mma_bf16(d, da, db, TC_IDESC, accumulate);
            };
            auto commit = [&](uint32_t bar) { if (!el) return; if constexpr (PAIR) tc_commit_pair(bar); else tc_commit(bar); };
            for (int e = worker; e < n_entries; e += n_workers, ua++) {
                const int n_tiles = units[unit_of(e)].n_tiles;
                const uint32_t ab = SPLIT ? 0u : (ua & 1);
                MPROF_BEGIN mbar_wait(a_full + 8 * ab, SPLIT ? (ua & 1) : ((ua >> 1) & 1), dbg, 3); MPROF_END(w_a)
                const uint32_t sa = smem_base + OFF_A + ab * A_BYTES;
                const uint64_t da_aug = desc_sw32(sa + (SPLIT ? 4 : 2) * A_ATOM_BYTES);
                for (int t = 0; t < n_tiles; t++, tc++) {
                    const uint32_t acc = tc & 1;
                    MPROF_BEGIN mbar_wait(t_empty + 8 * acc, ((tc >> 1) & 1) ^ 1, dbg, 5); MPROF_END(w_t)
                    const uint32_t d_tmem = tmem_base + acc * TILE_N;
                    #pragma unroll kIssuerUnroll
                    for (int h = 0; h < N_STAGES_PER_TILE; h++, bs++) {
                        const uint32_t s = bs % NB;
                        MPROF_BEGIN mbar_wait(b_full + 8 * s, (bs / NB) & 1, dbg, 4); MPROF_END(w_b)
                        tc_fence_after();
                        const uint32_t sb = smem_base + OFF_B + s * STAGE_BYTES;
                        // descriptors of the stage once, then + 2 per K step (the address field counts 16-byte units; stage and A
                        // buffers are 1024-aligned, so the 14-bit field cannot carry): fewer instructions on the one thread that
                        // feeds the tensor pipe and shares its scheduler with four busy epilogue warps
                        const uint64_t db0 = desc_sw128(sb);
                        const uint64_t da0 = desc_sw128(sa + (uint32_t)h * A_ATOM_BYTES);
                        #pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const uint32_t koff = (uint32_t)k * 32u;             // 16 bf16 = 32 B inside the swizzle atom
                            const uint64_t db = db0 + 2u * (uint32_t)k;
                            if constexpr (SPLIT) {
                                // 2q.t ~ hi.hi + lo.hi (stages 0, 1: train hi) + hi.lo (stages 2, 3: train lo)
                                const uint32_t kh = (uint32_t)(h & 1);
                                mma(d_tmem, desc_sw128(sa + kh * A_ATOM_BYTES + koff), db, (h | k) ? 1u : 0u);
                                if (h < 2) mma(d_tmem, desc_sw128(sa + (2 + kh) * A_ATOM_BYTES + koff), db, 1u);
                            } else {
                                mma(d_tmem, da0 + 2u * (uint32_t)k, db, (h | k) ? 1u : 0u);
                            }
                        }
                        commit(b_empty + 8 * s);         // ring stage reusable once these MMAs retire
                    }
                    {
                        const uint32_t g = tc % NG;
                        MPROF_BEGIN mbar_wait(g_full + 8 * g, (tc / NG) & 1, dbg, 8); MPROF_END(w_g)
                        tc_fence_after();
                        mma(d_tmem, da_aug, desc_sw32(smem_base + OFF_BAUG + g * G_BYTES), 1u);
                        commit(g_empty + 8 * g);
                    }
                    commit(t_full + 8 * acc);            // accumulator ready for the epilogue (of both CTAs)
                }
                commit(a_empty + 8 * ab);
            }
#ifdef TC_PROF
            if (el && (exp_mode & 32) && dbg && blockIdx.x == 0) {
                int* o = dbg + 28;
                o[0] = (int)tc; o[1] = (int)(w_a / 64); o[2] = (int)(w_t / 64); o[3] = (int)(w_b / 64); o[4] = (int)(w_g / 64); o[5] = (int)((clock64() - m_start) / 64);
            }
#endif
        }
    } else {
        // ===================== epilogue =====================
        const int ew = warp - 2;
        const int quarter = warp & 3;                    // TMEM lanes this warp may touch: 32*(warp%4)..
        const int part = ew >> 2;                        // which 64 columns of the 256-wide accumulator
        const int row_in_tile = quarter * 32 + lane;
        Top2* scratch = reinterpret_cast<Top2*>(smem + OFF_SCRATCH);
        // Every column part publishes its running (best, second best) per row; before each tile a warp raises its
        // filter to the second largest value any part has seen for the row.  Unsynchronised on purpose: a stale or
        // torn pair still consists of values of real columns with "second <= some other column of that part", so
        // the bound below is always <= the row's true second best.  Values equal to a foreign bound are kept
        // (the bound is lowered by one lattice step) because the foreign column may have the higher train index.
        const uint32_t share = smem_base + OFF_SHARE;
        const uint32_t my_share = share + (uint32_t)(part * TILE_M + row_in_tile) * 8u;
        // the accumulator barriers' addresses, held in a register: left to itself the compiler re-derives the shared-memory
        // window base (S2UR SR_CgaCtaId + four dependent instructions) in front of every tile's wait
        uint32_t t_full_r = t_full, t_empty_r = t_empty;
        uint32_t tmem_q = tmem_base + ((uint32_t)(quarter * 32) << 16);      // this warp's TMEM lane quarter (same treatment)
        asm volatile("" : "+r"(t_full_r), "+r"(t_empty_r), "+r"(tmem_q));
        if constexpr (KP == 1) {
            // the share area holds the column keys of four tiles, the scratch area the row merge and the tiles' counters
            reinterpret_cast<uint2*>(smem + OFF_SHARE)[ew * 32 + lane] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
            if (ew == 0 && lane < 16) reinterpret_cast<int*>(smem + OFF_SCRATCH + XC_MERGE_BYTES)[lane] = 0;
        } else {
            share_store(my_share, -INFINITY, -INFINITY);
        }
        asm volatile("bar.sync 1, %0;" :: "n"(32 * TC_EPI_WARPS) : "memory");
        if constexpr (KP == 2) {
            uint32_t tc = 0;
            // exp bit 5: cycle counts of the phases of this warp's tile loop, summed over its tiles (debug words 12..)
#ifdef TC_PROF
            const bool prof = (exp_mode & 32) != 0;
#else
            constexpr bool prof = false;
#endif
            long long c_wait = 0, c_ld = 0, c_share = 0, c_scan = 0, c_tiles = 0, c_flush = 0, c_unit = 0, t0 = 0, t1 = 0, tu = 0;
            const long long t_start = prof ? clock64() : 0;
            for (int e = worker; e < n_entries; e += n_workers) {
                if (prof) tu = clock64();
                const MatchUnit un = units[unit_of(e)];
                float b1 = -INFINITY, b2 = -INFINITY, f = (exp_mode & 4) ? INFINITY : -INFINITY;   // exp bit 2: nothing ever passes the filter
                int i1 = -1, i2 = -1;
                if (prof) { t1 = clock64(); c_unit += t1 - tu; }
                // Measured and rejected: two groups of 8 warps taking alternate tiles (128 columns per warp): 1.21 ms instead
                // of 1.10 ms per 64 pairs — the epilogue is bound by its instruction stream (~250 per warp and tile, four
                // warps per scheduler), not by the latency of one tile's chain.
#ifndef TC_DYNAMIC_PARTS
#define TC_DYNAMIC_PARTS 0                            // measured: 1.153 ms with dynamic parts, 1.114 ms with fixed ones (same run)
#endif
                // Dynamic column parts (experiment, off): the four warps of a TMEM lane quarter (the same 32 query rows) do not own a fixed 64-column
                // part of every tile; each takes the next unclaimed 64-column chunk of the unit from a shared counter.  The
                // accumulator of a tile goes back to the MMA issuer when its 16 chunks have been loaded, whoever loaded them: a
                // warp that is held up by a burst of candidates no longer holds up the tile, a faster warp of its quarter takes
                // the chunk it would have been late for.  Chunks are claimed in ascending order, so every warp still scans its
                // columns in ascending order (ties keep the earlier column) and the unit flush merges the four warps' records by
                // (value, index) as before.  A chunk of tile T can only be claimed after some warp finished a chunk of T - 1, i.e.
                // after t_full of T - 2 completed: the parity wait below cannot mistake an older phase for the one it needs.
                const uint32_t tc_unit0 = tc;
                const int n_chunks_unit = un.n_tiles * 4;
                for (int t_static = 0;; t_static++) {
                    int t, dpart;
                    if (TC_DYNAMIC_PARTS) {
                        int c = 0;
                        if (lane == 0) c = atomicAdd(&chunk_ctr[quarter], 1);
                        c = __shfl_sync(0xffffffffu, c, 0);
                        if (c >= n_chunks_unit) break;
                        t = c >> 2; dpart = c & 3;
                    } else {
                        if (t_static >= un.n_tiles) break;
                        t = t_static; dpart = part;
                    }
                    tc = tc_unit0 + (uint32_t)t;
                    const uint32_t acc = tc & 1;
                    if (prof) t0 = clock64();
                    // The filter update (what the other three column parts of these rows have found so far) runs BEFORE the wait for
                    // the next accumulator: a warp that has to wait anyway does it for free (same-run A/B: no slower than after the
                    // wait, and the accumulator goes back to the MMA issuer ~300 cycles earlier once it has arrived).
                    auto update_filter = [&]() {
                        if (t > 0 && !(exp_mode & 8)) {               // exp bit 3: no filter sharing between the column parts
                            float o1[3], o2[3];
                            #pragma unroll
                            for (int pp = 0; pp < 3; pp++) {
                                const int op = (part + 1 + pp) & 3;
                                share_load(share + (uint32_t)(op * TILE_M + row_in_tile) * 8u, o1[pp], o2[pp]);
                            }
                            // second largest of the four bests, and the largest of the four seconds
                            const float m1 = fmaxf(b1, o1[0]), n1 = fminf(b1, o1[0]);
                            const float m2 = fmaxf(o1[1], o1[2]), n2 = fminf(o1[1], o1[2]);
                            const float second_best = fmaxf(fminf(m1, m2), fmaxf(n1, n2));
                            const float foreign = fmaxf(fmaxf(second_best, o2[0]), fmaxf(o2[1], o2[2]));
                            // Strictly below the foreign bound, so that values equal to it pass the `>` tests.  This instance only ever
                            // sees integer-valued accumulators below 2^24 (section 4.1): foreign - 1 is exact and is the
                            // largest value of that lattice below the bound; padded columns (-2^30, where - 1 rounds away) are
                            // discarded at the flush anyway, and -inf stays -inf.  One FADD; the general form (largest float
                            // below the bound) cost ten instructions and a divergent branch per tile.
                            f = fmaxf(f, foreign - 1.0f);
                        }
                    };
#ifndef TC_SHARE_AFTER_WAIT
#define TC_SHARE_AFTER_WAIT 0                         // A/B: 1 = the round-1 order (wait, filter update, loads)
#endif
                    // (Measured and rejected: letting a warp that is late — accumulator already there — skip the update: its filter goes
                    // stale, it enters the slow path far more often and falls further behind: 1.11 -> 1.27 ms per 64 pairs.)
                    if (!TC_SHARE_AFTER_WAIT) update_filter();
                    if (prof) { t1 = clock64(); c_share += t1 - t0; t0 = t1; }
                    mbar_wait(t_full_r + 8 * acc, (tc >> 1) & 1, dbg, 6);
                    tc_fence_after();
                    if (prof) { t1 = clock64(); c_wait += t1 - t0; t0 = t1; c_tiles++; }
                    if (TC_SHARE_AFTER_WAIT) update_filter();
                    const uint32_t tbase = tmem_q + acc * TILE_N + dpart * 64;
                    const int col_base = un.t_local0 + t * TILE_N + dpart * 64;
                    if (!(exp_mode & 1)) {
                        uint32_t ra[32], rb[32];
                        tc_ld32(tbase, ra);                           // two loads in flight before the wait
                        tc_ld32(tbase + 32, rb);
                        tc_wait_ld();
                        if (prof) { t1 = clock64(); c_ld += t1 - t0; t0 = t1; }
                        // The warp's 64 columns are in registers: the accumulator goes back to the MMA issuer at once — before
                        // the filter update and before the scan — so that the next-but-one tile's MMAs start as early as they
                        // can (the MMA issuer waited 394 cycles per tile for this arrival when the filter update came first).
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) { if constexpr (PAIR) mbar_arrive_leader(t_empty_r + 8 * acc); else mbar_arrive(t_empty_r + 8 * acc); }
                        if (exp_mode & 16) {                          // exp bit 4: loads, no scan (the values are consumed by one OR chain)
                            uint32_t acc_or = 0;
                            #pragma unroll
                            for (int k = 0; k < 32; k++) acc_or |= ra[k] | rb[k];
                            if (acc_or == 0x12345678u) b1 = 1.f;
                        } else {
#ifndef TC_DENSE_TILES
#define TC_DENSE_TILES 0
#endif
                            if (t < TC_DENSE_TILES && !(exp_mode & 4)) {
                                top2_dense32(ra, col_base, b1, i1, b2, i2);
                                top2_dense32(rb, col_base + 32, b1, i1, b2, i2);
                                f = fmaxf(f, b2);
                            } else {
                                top2_scan32(ra, col_base, b1, i1, b2, i2, f);
                                top2_scan32(rb, col_base + 32, b1, i1, b2, i2, f);
                            }
                        }
                        share_store(my_share, b1, b2);
                        if (prof) { t1 = clock64(); c_scan += t1 - t0; }
                    } else {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) { if constexpr (PAIR) mbar_arrive_leader(t_empty_r + 8 * acc); else mbar_arrive(t_empty_r + 8 * acc); }
                    }
                }
                tc = tc_unit0 + (uint32_t)un.n_tiles;
                // ---- unit flush: merge the four column parts, convert to distances, write the partial ----
                if (prof) t0 = clock64();
                share_store(my_share, -INFINITY, -INFINITY);     // reset before the barriers below
                if (b1 < ABSENT_BELOW) { i1 = -1; }
                if (b2 < ABSENT_BELOW) { i2 = -1; }
                if (part > 0) {
                    Top2 o; o.d1 = b1; o.i1 = i1; o.d2 = b2; o.i2 = i2;
                    scratch[(part - 1) * TILE_M + row_in_tile] = o;
                }
                asm volatile("bar.sync 1, %0;" :: "n"(32 * TC_EPI_WARPS) : "memory");
                if (part == 0) {
                    if (lane == 0) chunk_ctr[quarter] = 0;        // every warp of the quarter has left the chunk loop; next unit starts at 0
                    // larger acc' first, ties -> lower train index
                    #pragma unroll
                    for (int pp = 0; pp < 3; pp++) {
                        const Top2 o = scratch[pp * TILE_M + row_in_tile];
                        const float cv[2] = { o.d1, o.d2 };
                        const int ci[2] = { o.i1, o.i2 };
                        #pragma unroll
                        for (int k = 0; k < 2; k++) {
                            const float v = cv[k]; const int i = ci[k];
                            if (i < 0) continue;
                            if (i1 < 0 || v > b1 || (v == b1 && i < i1)) { b2 = b1; i2 = i1; b1 = v; i1 = i; }
                            else if (i2 < 0 || v > b2 || (v == b2 && i < i2)) { b2 = v; i2 = i; }
                        }
                    }
                    const float qn = qnorm[un.q_row0 + row_in_tile];
                    Top2 out;
                    out.i1 = i1; out.i2 = i2;
                    out.d1 = i1 >= 0 ? sqrtf(fmaxf(qn - b1, 0.f)) : INFINITY;
                    out.d2 = i2 >= 0 ? sqrtf(fmaxf(qn - b2, 0.f)) : INFINITY;
                    reinterpret_cast<Top2*>(parts_out)[(size_t)un.part_slot * TILE_M + row_in_tile] = out;
                }
                asm volatile("bar.sync 1, %0;" :: "n"(32 * TC_EPI_WARPS) : "memory");
                if (prof) c_flush += clock64() - t0;
            }
            if (prof && dbg && blockIdx.x == 0 && lane == 0 && (ew == 0 || ew == 15)) {
                int* o = dbg + 12 + (ew == 0 ? 0 : 8);
                o[0] = (int)c_tiles; o[1] = (int)(c_wait / 64); o[2] = (int)(c_share / 64); o[3] = (int)(c_ld / 64); o[4] = (int)(c_scan / 64);
                o[5] = (int)(c_flush / 64); o[6] = (int)(c_unit / 64); o[7] = (int)((clock64() - t_start) / 64);
            }
        } else if constexpr (KP == 4) {
            uint32_t tc = 0;
            for (int e = worker; e < n_entries; e += n_workers) {
                const MatchUnit un = units[unit_of(e)];
                float b[4] = { -INFINITY, -INFINITY, -INFINITY, -INFINITY }, f = -INFINITY;
                int ix[4] = { -1, -1, -1, -1 };
                for (int t = 0; t < un.n_tiles; t++, tc++) {
                    const uint32_t acc = tc & 1;
                    mbar_wait(t_full_r + 8 * acc, (tc >> 1) & 1, dbg, 6);
                    tc_fence_after();
                    if (t > 0) {
                        // a part's fourth best is a lower bound of the row's fourth best: columns at or below it are no candidates
                        float foreign = -INFINITY;
                        #pragma unroll
                        for (int pp = 0; pp < 3; pp++) {
                            const int op = (part + 1 + pp) & 3;
                            float o1, o2;
                            share_load(share + (uint32_t)(op * TILE_M + row_in_tile) * 8u, o1, o2);
                            foreign = fmaxf(foreign, o2);
                        }
                        f = fmaxf(f, foreign);
                    }
                    const uint32_t tbase = tmem_q + acc * TILE_N + part * 64;
                    const int col_base = un.t_local0 + t * TILE_N + part * 64;
                    if (!(exp_mode & 1)) {
                        uint32_t ra[32], rb[32];
                        tc_ld32(tbase, ra);
                        tc_ld32(tbase + 32, rb);
                        tc_wait_ld();
                        top4_scan32(ra, col_base, b, ix, f);
                        top4_scan32(rb, col_base + 32, b, ix, f);
                        share_store(my_share, b[0], b[3]);
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) { if constexpr (PAIR) mbar_arrive_leader(t_empty_r + 8 * acc); else mbar_arrive(t_empty_r + 8 * acc); }
                }
                // ---- unit flush: every column part writes its own candidate record ----
                share_store(my_share, -INFINITY, -INFINITY);
                Top4 out;
                #pragma unroll
                for (int k = 0; k < 4; k++) { out.v[k] = b[k]; out.i[k] = b[k] < ABSENT_BELOW ? -1 : ix[k]; }
                reinterpret_cast<Top4*>(parts_out)[((size_t)un.part_slot * 4 + part) * TILE_M + row_in_tile] = out;
                asm volatile("bar.sync 1, %0;" :: "n"(32 * TC_EPI_WARPS) : "memory");     // all share slots reset before the next unit
            }
        } else {
            // Cross-check.  Column keys: tile tc's 256 columns have slots in buffer tc & 3; the four warps of a column part
            // (one per TMEM lane quarter) merge into them with atomicMin, and the last of the four to count itself in flushes
            // the 64 columns to global memory and resets the slots.  No per-tile barrier: a warp is at most two tiles ahead of
            // the slowest (the accumulator of tile T + 2 needs every warp's release of tile T), and the flusher of tile T
            // finishes it before it releases tile T + 1, so buffer tc & 3 is free again when tile tc + 4 arrives.
            uint32_t* colkeys = reinterpret_cast<uint32_t*>(smem + OFF_SHARE);                 // [4 tiles][256 columns]
            float2* rmerge = reinterpret_cast<float2*>(smem + OFF_SCRATCH);                    // [3 column parts][128 rows]
            int* colcnt = reinterpret_cast<int*>(smem + OFF_SCRATCH + XC_MERGE_BYTES);         // [4 tiles][4 column parts]
            const XcOut xo = *reinterpret_cast<const XcOut*>(parts_out);
            uint32_t tc = 0;
            for (int e = worker; e < n_entries; e += n_workers) {
                const MatchUnit un = units[unit_of(e)];
                const bool row_ok = row_in_tile < (un.pad1 & 255);
                const float qbias = row_ok ? __fadd_rn(qnorm[un.q_row0 + row_in_tile], 8388608.f) : INFINITY;
                // this unit's view slot and segment: column keys from the segment's first train row, row keys of the segment
                unsigned long long* ck = xo.colkey + (un.pad1 >> 8) * xo.t_total + (un.t_row0_f32 - un.t_local0 - xo.t_base);
                float b1 = -INFINITY;
                int i1 = -1;
                for (int t = 0; t < un.n_tiles; t++, tc++) {
                    const uint32_t acc = tc & 1;
                    mbar_wait(t_full_r + 8 * acc, (tc >> 1) & 1, dbg, 6);
                    tc_fence_after();
                    const uint32_t tbase = tmem_q + acc * TILE_N + part * 64;
                    const int col_base = un.t_local0 + t * TILE_N + part * 64;
                    uint32_t ra[32], rb[32];
                    tc_ld32(tbase, ra);
                    tc_ld32(tbase + 32, rb);
                    tc_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(t_empty_r + 8 * acc);
                    xc_row_scan32(ra, col_base, b1, i1);
                    xc_row_scan32(rb, col_base + 32, b1, i1);
                    uint32_t* slots = colkeys + (tc & 3) * TILE_N + part * 64;
                    xc_col_keys32(ra, qbias, (uint32_t)row_in_tile, slots, lane);
                    xc_col_keys32(rb, qbias, (uint32_t)row_in_tile, slots + 32, lane);
                    __syncwarp();
                    int last = 0;
                    if (lane == 0) {
                        __threadfence_block();
                        last = atomicAdd(&colcnt[(tc & 3) * 4 + part], 1) == 3;
                    }
                    if (__shfl_sync(0xffffffffu, last, 0)) {
                        __threadfence_block();
                        #pragma unroll
                        for (int h = 0; h < 2; h++) {
                            const uint32_t k = atomicExch(&slots[h * 32 + lane], 0xFFFFFFFFu);
                            const int col = col_base + h * 32 + lane;
                            if (k < XC_KEY_ABSENT && col < un.seg_cols)
                                atomicMin(&ck[col], ((unsigned long long)((k >> 7) & 0x7FFFFFu) << 32) | (uint32_t)(un.q_row0 + (int)(k & 127u)));
                        }
                        if (lane == 0) colcnt[(tc & 3) * 4 + part] = 0;
                    }
                }
                // ---- unit flush: merge the four column parts (larger acc', then lower column), one key per row ----
                if (b1 < ABSENT_BELOW) i1 = -1;
                if (part > 0) rmerge[(part - 1) * TILE_M + row_in_tile] = make_float2(b1, __int_as_float(i1));
                asm volatile("bar.sync 1, %0;" :: "n"(32 * TC_EPI_WARPS) : "memory");
                if (part == 0) {
                    #pragma unroll
                    for (int pp = 0; pp < 3; pp++) {
                        const float2 o = rmerge[pp * TILE_M + row_in_tile];
                        const int i = __float_as_int(o.y);
                        if (i >= 0 && (i1 < 0 || o.x > b1 || (o.x == b1 && i < i1))) { b1 = o.x; i1 = i; }
                    }
                    if (row_ok && i1 >= 0) {
                        const uint32_t d2 = __float_as_uint(__fsub_rn(qbias, b1)) - 0x4B000000u;
                        atomicMin(&xo.rowkey[un.part_slot * xo.row_stride + un.q_row0 + row_in_tile], ((unsigned long long)d2 << 32) | (uint32_t)i1);
                    }
                }
                asm volatile("bar.sync 1, %0;" :: "n"(32 * TC_EPI_WARPS) : "memory");
            }
        }
    }
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();          // both epilogues are done with TMEM, both producers have seen their tails
    else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" :: "r"(tmem_base) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" :: "r"(tmem_base) : "memory");
    }
}

// ---- host side ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

int tc_init(char* err, size_t errlen)
{
    static std::mutex mu;
    std::lock_guard<std::mutex> g(mu);
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
        snprintf(err, errlen, "cuTensorMapEncodeTiled not available: %s", cudaGetErrorString(e));
        return 1;
    }
    g_encode = (EncodeTiledFn)fn;
    return 0;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device property of a function: called once for every device a
// context is created on (api.cu, under its own mutex), with that device current.
int tc_set_device_attrs(char* err, size_t errlen)
{
    const void* fns[7] = { (const void*)match_tc_kernel<2, false, false>, (const void*)match_tc_kernel<2, false, true>,
                           (const void*)match_tc_kernel<4, false, false>, (const void*)match_tc_kernel<4, false, true>,
                           (const void*)match_tc_kernel<2, true, false>, (const void*)match_tc_kernel<2, true, true>,
                           (const void*)match_tc_kernel<1, false, false> };
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 7 && e == cudaSuccess; i++)
        e = cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES);
    if (e != cudaSuccess) {
        snprintf(err, errlen, "cudaFuncSetAttribute(match_tc_kernel): %s", cudaGetErrorString(e));
        return 1;
    }
    return 0;
}

static int make_map(CUtensorMap* m, const void* base, uint64_t rows, uint32_t cols, uint32_t box_cols,
                    uint32_t box_rows, CUtensorMapSwizzle sw, char* err, size_t errlen)
{
    cuuint64_t gdim[2] = { cols, rows };
    cuuint64_t gstride[1] = { (cuuint64_t)cols * 2 };
    cuuint32_t box[2] = { box_cols, box_rows };
    cuuint32_t estr[2] = { 1, 1 };
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(err, errlen, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%u", (int)r, (unsigned long long)rows, cols);
        return 1;
    }
    return 0;
}

static bool dbg_print_clusters() { return getenv("CVG_DEBUG") != nullptr; }

bool tc_pair_mode_enabled()
{
    static int on = -1;
    if (on < 0) { const char* e = getenv("CVG_TC_PAIR"); on = e ? (atoi(e) != 0) : 0; }
    return on != 0;
}

// The six (eight) tensor maps of a call, encoded on the host ahead of the launch so that nothing but the launch itself sits
// between the caller's timing events (cuTensorMapEncodeTiled costs a few microseconds each).
int tc_encode_maps(const TcOperands& op, int candidates, TcMapsOpaque* out, char* err, size_t errlen)
{
    static_assert(sizeof(TcMapsOpaque) >= sizeof(TcMaps), "TcMapsOpaque too small");
    if (tc_init(err, errlen)) return 1;
    TcMaps& maps = *reinterpret_cast<TcMaps*>(out);
    if (make_map(&maps.q, op.Qb, op.nq_pad, DIM, 64, TILE_M, CU_TENSOR_MAP_SWIZZLE_128B, err, errlen)) return 1;
    if (make_map(&maps.qaug, op.Qaug, op.nq_pad, KAUG, KAUG, TILE_M, CU_TENSOR_MAP_SWIZZLE_32B, err, errlen)) return 1;
    if (make_map(&maps.t, op.Tb, op.nt_pad, DIM, 64, TILE_N, CU_TENSOR_MAP_SWIZZLE_128B, err, errlen)) return 1;
    if (make_map(&maps.taug, op.Taug, op.nt_pad, KAUG, KAUG, TILE_N, CU_TENSOR_MAP_SWIZZLE_32B, err, errlen)) return 1;
    if (make_map(&maps.th, op.Tb, op.nt_pad, DIM, 64, TILE_N / 2, CU_TENSOR_MAP_SWIZZLE_128B, err, errlen)) return 1;
    if (make_map(&maps.taugh, op.Taug, op.nt_pad, KAUG, KAUG, TILE_N / 2, CU_TENSOR_MAP_SWIZZLE_32B, err, errlen)) return 1;
    maps.qlo = maps.q; maps.tlo = maps.t;
    if (candidates == 4) {
        if (!op.Qlo || !op.Tlo) { snprintf(err, errlen, "candidate path needs the lo operand halves"); return 1; }
        if (make_map(&maps.qlo, op.Qlo, op.nq_pad, DIM, 64, TILE_M, CU_TENSOR_MAP_SWIZZLE_128B, err, errlen)) return 1;
        if (make_map(&maps.tlo, op.Tlo, op.nt_pad, DIM, 64, TILE_N, CU_TENSOR_MAP_SWIZZLE_128B, err, errlen)) return 1;
    }
    return 0;
}

int launch_match_tc(const TcOperands& op, const TcMapsOpaque* encoded, const MatchUnit* units, int n_units, void* parts, int candidates,
                    const int* gate_flag, int gate_want, int* dbg, int n_sms, cudaStream_t st, char* err, size_t errlen,
                    bool paired)
{
    if (n_units <= 0) return 0;
    const TcMaps& maps = *reinterpret_cast<const TcMaps*>(encoded);
    const int grid = n_units < n_sms ? n_units : n_sms;
    static int exp_mode = -1;
    if (exp_mode < 0) { const char* e = getenv("CVG_TC_EXP"); exp_mode = e ? atoi(e) : 0; }
    if (candidates == 1)
        match_tc_kernel<1, false, false><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, 0);
    else if (candidates == 4) {
        if (exp_mode) match_tc_kernel<4, false, true><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, exp_mode);
        else match_tc_kernel<4, false, false><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, 0);
    }
    else if (paired && (n_units % 2) == 0 && n_sms >= 2) {
        // clusters of two CTAs (cta_group::2): consecutive units (2p, 2p + 1) share their train tiles
        const int n_pairs = n_units / 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(2 * (n_sms / 2))); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = TC_SMEM_BYTES; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        // The persistent loop deals entries to clusters statically, so every cluster of the grid must be resident at once:
        // a GPC with an odd number of free SMs leaves one without a partner, and a second wave would double the time.
        static int max_clusters = -1;
        if (max_clusters < 0) {
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, match_tc_kernel<2, true, false>, &cfg) != cudaSuccess || n <= 0) { cudaGetLastError(); n = n_sms / 2; }
            max_clusters = n < n_sms / 2 ? n : n_sms / 2;
            if (getenv("CVG_TC_PAIR_CLUSTERS")) max_clusters = atoi(getenv("CVG_TC_PAIR_CLUSTERS"));
            if (dbg_print_clusters()) fprintf(stderr, "cvgraft: match pair mode runs %d clusters of 2 CTAs (%d SMs)\n", max_clusters, n_sms);
        }
        const int clusters = n_pairs < max_clusters ? n_pairs : max_clusters;
        cfg.gridDim = dim3((unsigned)(2 * clusters));
        cudaError_t le = exp_mode
            ? cudaLaunchKernelEx(&cfg, match_tc_kernel<2, true, true>, maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, exp_mode)
            : cudaLaunchKernelEx(&cfg, match_tc_kernel<2, true, false>, maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, 0);
        if (le != cudaSuccess) {
            snprintf(err, errlen, "match_tc_kernel (pair mode) launch: %s", cudaGetErrorString(le));
            return 1;
        }
    } else if (exp_mode)
        match_tc_kernel<2, false, true><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, exp_mode);
    else
        match_tc_kernel<2, false, false><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(maps, op.qnorm, units, n_units, parts, gate_flag, gate_want, dbg, 0);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(err, errlen, "match_tc_kernel launch: %s", cudaGetErrorString(e));
        return 1;
    }
    return 0;
}

}  // namespace cvg
