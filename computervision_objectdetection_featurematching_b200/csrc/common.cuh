// common.cuh — shared declarations of libcvgraft's translation units.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cvgraft.h"

namespace cvg {

constexpr int DIM = CVG_DESC_DIM;       // 128
constexpr int KAUG = 16;                // extra K columns that fold ||t||^2 into the contraction
constexpr int TILE_M = 128;             // query rows per tile (TMEM lanes)
constexpr int TILE_N = 256;             // train rows per tile (TMEM columns of one accumulator)

// One unit of match work: 128 query rows against a run of train tiles of one segment (a segment is
// one scene / one train matrix).  A unit produces one partial top-2 record per query row.
struct MatchUnit {
    int32_t q_row0;          // first query row (multiple of TILE_M)
    int32_t t_row0;          // first train row in the concatenated, padded train matrix
    int32_t n_tiles;         // number of TILE_N-wide train tiles
    int32_t t_local0;        // index of t_row0 inside its segment (train index reported = local)
    int32_t part_slot;       // partial record block: parts[part_slot * TILE_M + row].  Cross-check plan: the segment index
    int32_t seg_cols;        // valid train rows of the segment (for masking the padded tail)
    int32_t t_row0_f32;      // first train row in the unpadded fp32 train matrix (exact kernel)
    int32_t pad1;            // knn2 plan: 0.  Cross-check plan: view slot << 8 | query rows of the unit in its view (1..128)
};

// Partial / final top-2 record of one query row.
struct __align__(16) Top2 {
    float d1; int32_t i1; float d2; int32_t i2;
};

// Candidate record of one query row and one column part of a unit (non-integer descriptors): raw accumulator
// values 2 q.t - ||t||^2 (approximate), largest first, and their train indices (-1 = absent).
struct __align__(16) Top4 {
    float v[4]; int32_t i[4];
};

// A train segment as the re-rank kernels see it.
struct SegDev {
    int64_t f32_row0;        // first row in the unpadded fp32 train matrix
    int32_t rows;            // valid train rows
    int32_t pad;
};

// Per (segment, row-block) directory entry for the merge kernel.
struct MergeEntry {
    int32_t first_slot;      // first partial slot
    int32_t n_slots;         // consecutive slots (ascending train order)
};

// ---- launchers (defined in the .cu files) --------------------------------------------------------
// prep.cu
void launch_prep_rows(const float* X, int n_rows, int n_pad, int is_train, __nv_bfloat16* Xb,
                      __nv_bfloat16* Xlo /*lo half: bf16(x - hi), zero for integer rows; or NULL*/, __nv_bfloat16* Xaug, float* norms, int* nonint_flag /*bit0 non-integer, bit1 non-finite*/,
                      int* tnmax_bits /*train side: max ||t||^2 as float bits, or NULL*/, cudaStream_t st);
struct PrepSeg { int64_t f32_row0; int64_t pad_row0; int32_t rows; int32_t pad; };   // ascending pad_row0
void launch_prep_train_segments(const float* X, const PrepSeg* segs_dev, int n_segs, int64_t rows_pad_total,
                                __nv_bfloat16* Xb, __nv_bfloat16* Xlo, __nv_bfloat16* Xaug, int* nonint_flag,
                                int* tnmax_bits, cudaStream_t st);
void launch_pack_points(const float* src_xy, const float* dst_xy, int64_t n, float4* pts, cudaStream_t st);

// match_exact.cu — fp32 SIMT kernel in cv::batchDistance's summation order
void launch_match_exact(const float* Q, int n_query, const float* T, const MatchUnit* units, int n_units,
                        Top2* parts, const int* gate_flag /*device flag: run only if *flag == gate_want, or NULL*/,
                        int gate_want, cudaStream_t st);

// Cross-check (BFMatcher(NORM_L2, crossCheck = true)): the match kernels leave, per (segment, query row), the
// (key << 32 | train index in the segment) of the row's nearest train row of that segment and, per (view slot, train
// column), the (key << 32 | absolute query row) of the column's nearest query row of that view, both reduced with atomicMin
// (~0 = none).  key = d^2 (tensor-core kernel, integer rows) or the float bits of cv2's distance (exact SIMT kernel);
// xc_finish turns d^2 into distance bits.  Layout (DESIGN.md 4.5): rowkey[seg * row_stride + absolute query row],
// colkey[view * t_total + fp32 train row - t_base]; the segment travels in MatchUnit::part_slot.  One train matrix is
// the case seg = 0, t_base = 0.
struct XcOut {
    unsigned long long* rowkey; unsigned long long* colkey;
    int64_t row_stride;                             // rows per segment block of rowkey
    int64_t t_total;                                // train rows of the call (the segments' rows, contiguous from t_base)
    int64_t t_base;                                 // fp32 row of the call's first train row
};
void launch_match_exact_xc(const float* Q, const float* T, const MatchUnit* units, int n_units, XcOut out,
                           const int* gate_flag /*skipped if *flag == 0 (the tensor-core kernel serves the call), or NULL*/,
                           cudaStream_t st);
struct XcFinish {
    XcOut keys;
    int row_begin, row_end;                         // query rows of the call (absolute)
    int n_segs, n_views, max_view_rows, max_seg_rows;
    const SegDev* views;                            // [n_views] query rows of each view slot (f32_row0 = first row)
    const SegDev* segs;                             // [n_segs] train rows of each segment (f32_row0 = first fp32 row)
    const float* Q; const float* T;                 // fp32 rows
    int* guard_counts;                              // [2] rows / columns redone by the d >= 2048 guard (zeroed by the caller)
    int* guard_total;                               // receives their sum
    int2* row_list; unsigned long long* row_g;      // [n_segs * nq], [2 * n_segs * nq]
    int2* col_list; unsigned long long* col_g;      // [n_views * t_total], [2 * n_views * t_total]
    const int* gate_flag;                           // the d^2 -> distance step runs only if *gate_flag == 0 (tensor-core path)
    // outputs.  accept == NULL: idx / dist [nq] of the one segment (cvg_match_cross_check).  Otherwise the knn2 layout the
    // fused path compacts: idx[2 * (seg * nq + i)] = train index, accept[seg * nq + i] = matched (dist unused)
    int32_t* idx; float* dist; uint8_t* accept;
    int n_sms;
};
// d^2 keys -> distance keys (the d >= 2048 rows and columns redone exactly), then the mutual test; returns the launch count
int launch_xc_finish(const XcFinish& w, cudaStream_t st);

// match_tc.cu — tcgen05 / TMEM / TMA kernel
struct TcOperands {
    const __nv_bfloat16* Qb; const __nv_bfloat16* Qaug; const float* qnorm; int nq_pad;
    const __nv_bfloat16* Tb; const __nv_bfloat16* Taug; int nt_pad;
    const __nv_bfloat16* Qlo; const __nv_bfloat16* Tlo;      // lo halves of the split operands (candidate path), or NULL
};
int  tc_init(char* err, size_t errlen);     // resolves cuTensorMapEncodeTiled; 0 = ok
int  tc_set_device_attrs(char* err, size_t errlen);       // dynamic shared memory opt-in on the CURRENT device
int  ransac_set_device_attrs(char* err, size_t errlen);   // same for the verify kernels
// candidates = 2: exact top-2 (Top2 parts[n_units][128]); 4: candidate records (Top4 parts[n_units][4][128]);
// 1: cross-check keys (parts = device XcOut, units of build_xc_plan).
// gate_flag (device, may be NULL): the kernel runs only if *gate_flag == gate_want.
// paired: the unit list is made of pairs (2p, 2p + 1) with the same train tiles (build_plan with an even number of row
// blocks): the exact form then runs as clusters of two CTAs with cta_group::2 MMAs.
struct alignas(64) TcMapsOpaque { unsigned char bytes[8 * 128]; };          // the CUtensorMaps of one call (match_tc.cu: TcMaps)
int  tc_encode_maps(const TcOperands& op, int candidates, TcMapsOpaque* out, char* err, size_t errlen);
int  launch_match_tc(const TcOperands& op, const TcMapsOpaque* encoded, const MatchUnit* units, int n_units, void* parts, int candidates,
                     const int* gate_flag, int gate_want, int* dbg, int n_sms,
                     cudaStream_t st, char* err, size_t errlen, bool paired = false);
bool tc_pair_mode_enabled();                 // CVG_TC_PAIR=1: pair mode for every context of the process (A/B runs); else per context flag

// merge.cu (in match_exact.cu)
void launch_merge(const Top2* parts, const MergeEntry* dir, int n_segments, int n_rowblocks, int n_query,
                  float ratio, int32_t* idx, float* dist, uint8_t* accept,
                  const int* gate_flag /*skipped if *flag == gate_skip, or NULL*/, int gate_skip, cudaStream_t st,
                  int* fb_count = nullptr /*guard: rows whose second distance is >= 2048 go to fb_list instead*/,
                  int2* fb_list = nullptr);
void launch_fallback_exact(const int* fb_count, const int2* fb_list, unsigned long long* fb_keys, const SegDev* segs,
                           int n_segments, int n_query, int max_seg_rows, float ratio, const float* Q, int q_row_begin,
                           const float* T, int32_t* idx, float* dist, uint8_t* accept, const int* gate_flag, int gate_want,
                           int n_sms, cudaStream_t st);
// candidate path: merge of Top4 records, fp32 re-rank with proof, exact fallback for the unproven rows
void launch_merge4_rerank(const Top4* parts4, const MergeEntry* dir, const SegDev* segs, int n_segments, int n_rowblocks,
                          int n_query, int max_seg_rows, float ratio, const float* Q, int q_row_begin, const float* T,
                          const float* qnorm, const int* tnmax_bits, int32_t* idx, float* dist, uint8_t* accept, int* fb_count,
                          int2* fb_list, unsigned long long* fb_keys /*[2][n_segments * n_query]*/,
                          const int* gate_flag, int gate_want, int n_sms, cudaStream_t st);
void launch_merge_parts(const float* dist_parts, const int32_t* idx_parts, int n_parts, int n_query, float ratio,
                        int32_t* idx, float* dist, uint8_t* accept, cudaStream_t st);
void launch_shift_index(const int32_t* idx_in, const float* dist_in, int n_query, int32_t idx_base,
                        float* dist, int32_t* idx, cudaStream_t st);

// ransac.cu
// RANSACUpdateNumIters depends on log() and pow() of the C library OpenCV runs on; CUDA's are up to 2 ulp away, which could
// move cvRound(num / denom) when the quotient sits within ~1e-12 of a half-integer.  The device therefore uses the HOST's
// log(1 - confidence), flags every evaluation whose rounding or cap decision is closer than `nit_margin` to a boundary, and
// the host answers those (n, good) pairs with its own libm values; the verify stage is then repeated with the table.
// An entry is keyed on (model points, n, good): homography (4), estimateAffine2D (3) and estimateAffinePartial2D (2) calls on
// one engine share its table.
struct NitEntry { int32_t n; int32_t good; double denom_log; int32_t zero; int32_t mp; };   // zero: 1 - (1-ep)^mp < DBL_MIN
struct RansacWork {
    const float4* pts;          // correspondence pool, (X, Y, x, y)
    const int64_t* starts;      // [P] first pool row of set k
    const int32_t* counts_n;    // [P] number of correspondences of set k
    int n_sets;
    int n_sms;                  // SMs of the device the work runs on
    int wave_div;               // engines sharing the GPU (>= 1): rounds are sized to 1 / wave_div of a wave
    int max_n;                  // upper bound of counts_n (host-known; sizes nothing, tunes launches)
    int max_iters;
    float thr2;                 // (float)(thr*thr)
    double conf;
    uint32_t flags;
    const uint32_t* rng_tab;    // raw cv::RNG outputs for the fixed seed, [rng_len]
    int64_t rng_len;
    // scratch
    int32_t* sample_pos;        // [P, max_iters] draw position where the accepted attempt starts
    int32_t* n_samples;         // [P]
    int32_t* counts;            // [P, max_iters]
    int32_t* best_iter;         // [P]
    int32_t* best_count;        // [P]
    int32_t* iters_run;         // [P]
    int32_t* niters_cur;        // [P] adaptive niters after the rounds scanned so far
    int64_t* smp_state;         // [P, 2] sampler state between rounds: next draw position, failure run (-1 = finished)
    unsigned long long* scored_pts;   // device counter: sum over scored hypotheses of n (or NULL)
    float* hyp_H;               // [P, max_iters, 8] fp32 models for ransac_score_kernel, or NULL = score inside the solve kernel
    int hyp_H_complete;         // every round's kernel left its models in hyp_H (set by launch_ransac for the finish kernel)
    int32_t* sel;               // [total] compacted inlier indices
    // outputs
    double* H;                  // [P, 9] (the affine methods: [P, 6])
    uint8_t* mask;              // [total]
    uint8_t* ransac_mask;       // [total] or NULL
    int32_t* found;             // [P]
    int32_t* status_flags;      // [P] bit0: rng table exhausted
    int* err_flag;              // one word, OR of all status_flags (or NULL); bit 1: niters entries were requested
    double log_num;             // log(max(1 - confidence, DBL_MIN)) from the host's libm
    const NitEntry* nit_tab; int nit_n;       // host-verified entries (usually none)
    int2* nit_req; int* nit_req_n; int nit_req_cap;   // (n, good) pairs the device asks the host about
    double nit_margin;          // distance to a decision boundary below which an evaluation is not trusted
    // chunked sampler scratch (huge single rounds; NULL / 0 = not available)
    void* chunk_outs; int32_t* chunk_lists; int32_t* chunk_offsets; int* chunk_serial; int n_chunks;
    uint8_t* chunk_maps; int32_t* chunk_entries; int* chunk_serial_count;
    int model_points;           // RANSAC modelPoints: 4 findHomography, 3 estimateAffine2D, 2 estimateAffinePartial2D
};
int64_t ransac_chunk_scratch_bytes(int n_sets, int n_chunks, size_t* outs, size_t* lists, size_t* offsets, size_t* serial,
                                   size_t* maps, size_t* entries);
int ransac_chunks_for_table(int64_t rng_len);
int launch_selftest_rcp(unsigned long long* d_mismatches, cudaStream_t st);
int launch_selftest_jacobi(unsigned long long* d_mismatches, int n_mats, cudaStream_t st);
// returns the number of kernel launches; hyp_events (optional, 48 events): [2r], [2r+1] bracket the solve kernel of round r,
// [32 + r] follows its score kernel
int  launch_ransac(const RansacWork& w, cudaStream_t st, cudaEvent_t* hyp_events = nullptr, int* n_hyp_rounds = nullptr);
// The phases launch_ransac loops over (the hypothesis-range sharded driver of multi.cu runs them too, with an exchange of
// the counts between hyp and select).  Each returns its number of kernel launches.
int  ransac_round_len(const RansacWork& w);                                    // iterations per round on one device
int  launch_ransac_sample(const RansacWork& w, int rb, int len, cudaStream_t st);   // samples of iterations [rb, rb + len)
// solve + score iterations [hb, hb + hlen); ev (optional, 3 events): before the solve kernel, after it, after the score
// kernel; *hyp_complete is cleared when the kernel used does not leave its models in hyp_H
int  launch_ransac_hyp(const RansacWork& w, int hb, int hlen, cudaStream_t st, const cudaEvent_t* ev, bool* hyp_complete);
int  launch_ransac_select(const RansacWork& w, int rb, int len, cudaStream_t st);   // serial scan of round [rb, rb + len)
int  launch_ransac_finish(const RansacWork& w, bool hyp_complete, cudaStream_t st);
// cv::estimateAffine2D(RANSAC) (w.model_points == 3) or cv::estimateAffinePartial2D(RANSAC) (2) for every set of w: the
// round-based sampler, one solve-and-score kernel per round, the select scan, then the finish kernel (winner's mask,
// compaction, 6- or 4-parameter LM of refine_iters iterations, none for 0).  M goes to w.H as 6 doubles per set.  Returns
// the number of kernel launches.
int  launch_affine(const RansacWork& w, int refine_iters, cudaStream_t st);

// detect glue (ransac.cu)
struct GateWork {
    int n_pairs;
    const float4* pts; const int64_t* starts; const int32_t* counts_n;   // per pair correspondences
    const uint8_t* mask; const int32_t* found; const double* H; const int32_t* iters_run;
    int model_points;                               // 4 homography, 3 / 2 the affine methods: fewer matches -> no model
    int h_stride;                                   // doubles per pair in H: 9 (3x3), 6 (2x3 M, promoted to 3x3 here)
    const float* pair_scale;                        // [n_pairs] or NULL
    int min_inliers; float det_lo, det_hi;
    cvg_pair_result* results;                       // [n_pairs] device
    float* inlier_xy;                               // [total, 2] compacted per pair at offsets, or NULL
    int32_t* inlier_count;                          // [n_pairs]
};
void launch_gates(const GateWork& g, cudaStream_t st);

// compaction of accepted matches into correspondences, per (segment, view) pair
struct CompactWork {
    int n_segments, n_views, n_query;
    const int32_t* view_offsets;                    // [V+1] device
    const float* model_kpt;                         // [n_query, 2]
    const float* scene_kpt;                         // concatenated scene keypoints
    const int64_t* seg_kpt_offsets;                 // [S+1] rows into scene_kpt
    const int32_t* idx; const uint8_t* accept;      // [S, n_query, 2], [S, n_query]
    float4* pts;                                    // [S * n_query] pool: pair (s,v) at s*n_query + view_offsets[v]
    int64_t* starts;                                // [S*V]
    int32_t* n_good;                                // [S*V]
};
void launch_compact(const CompactWork& c, cudaStream_t st);

}  // namespace cvg
