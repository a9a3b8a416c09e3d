/*
 * cvgraft.h — C ABI of libcvgraft: B200-native (sm_100a) descriptor matching + RANSAC homography.
 *
 * Drop-in boundary for the hot path of mattreturn1/ComputerVision_ObjectDetection_FeatureMatching.
 * The reference has no plugin/FFI interface; the seam is the pair of OpenCV calls inside
 * detectObjects() (reference include/TestsDetector.hpp:13-17):
 *
 *     matcher.knnMatch(model.descriptors[i], sceneDesc, knnMatches, 2)   src/TestsDetector.cpp:59-60
 *     ratio test + point gather                                          src/TestsDetector.cpp:62-72
 *     findHomography(objPts, scenePts, RANSAC, 5.0, inlierMask)          src/TestsDetector.cpp:77-78
 *     H.empty / countNonZero / determinant gates, inlier gather          src/TestsDetector.cpp:74,79-94
 *
 * plus the model hand-off after src/ModelsDetector.cpp:78-80 (descriptors uploaded once, resident
 * in HBM).  Each entry point below names the reference lines it replaces.  Semantics are those of
 * cv2 4.13.0 (SURVEY.md App. A/B); INTEGRATION.md shows the reference-side binding.
 *
 * Conventions: plain C, POD structs with a leading `size` field, int return codes (0 = ok), no
 * exceptions across the ABI.  Unless a name says `_dev`, every pointer is caller-owned HOST memory
 * and is not retained after the call returns (the asynchronous uploads and cvg_detect_scenes_submit
 * say how long theirs must stay valid).  A context belongs to one CUDA device (cvg_create) or to the
 * listed devices of one host (cvg_create_multi) and serves ONE caller thread: synchronous calls one at a
 * time, or several fused calls in flight through cvg_detect_scenes_submit / cvg_job_wait — the
 * context's lanes (internal engines with a worker thread each) overlap them on the GPU, so that one
 * call's latency-bound refit/LM kernel runs beside the next call's match and hypothesis kernels
 * (2.3 instead of 3.7 ms per batch of 64 pairs).  There is no CPU fallback: every entry point fails
 * with CVG_ERR_CUDA when no sm_100 device is present.
 */
#ifndef CVGRAFT_H
#define CVGRAFT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVG_DESC_DIM 128            /* SIFT descriptor length (reference: cv::SIFT, 128 x CV_32F)   */

/* return codes */
enum {
    CVG_OK = 0,
    CVG_ERR_INVALID = 1,            /* bad argument                                                  */
    CVG_ERR_CUDA = 2,               /* CUDA runtime/driver failure, see cvg_last_error()             */
    CVG_ERR_TOO_FEW_POINTS = 3,     /* findHomography with n < 4 (OpenCV throws, fundam.cpp)         */
    CVG_ERR_NOMEM = 4,
    CVG_ERR_LIMIT = 5               /* size beyond a documented limit                                */
};

/* per-pair gate outcome — reference src/TestsDetector.cpp:74 / :79 / :81 / :84 */
enum {
    CVG_PAIR_ACCEPT = 0,
    CVG_PAIR_LT4_MATCHES = 1,       /* goodMatches.size() < MIN_INLIERS            :74               */
    CVG_PAIR_H_EMPTY = 2,           /* H.empty()                                   :79               */
    CVG_PAIR_LT4_INLIERS = 3,       /* countNonZero(inlierMask) < MIN_INLIERS      :81               */
    CVG_PAIR_DET_REJECT = 4         /* fabs(determinant(H)) outside [0.1f, 10.0f]  :84               */
};

/* cvg_ransac_params.flags */
#define CVG_RANSAC_NO_EARLY_STOP 1u /* score all max_iters hypotheses, niters never shrinks          */
                                    /* (throughput mode of BASELINE config 5; not OpenCV semantics)  */
#define CVG_RANSAC_NO_REFINE     2u /* stop after the RANSAC stage: no DLT refit, no LM               */

/* cvg_create flags */
#define CVG_FORCE_EXACT_MATCH 1u    /* always use the fp32 SIMT match kernel (debug / A-B tests)     */
#define CVG_MATCH_PAIR_MODE   2u    /* exact tensor-core match as clusters of two CTAs (tcgen05      */
                                    /* cta_group::2, M = 256): same results; measured slower than    */
                                    /* the one-CTA form on B200 (DESIGN.md 4.1), kept for A-B runs   */

#define CVG_NITERS_ALL_ON_HOST 4u   /* every RANSACUpdateNumIters evaluation is answered by the host's libm (log, pow)    */
                                    /* instead of only those within 1e-10 of a rounding / cap boundary: same results,     */
                                    /* one extra pass of the verify stage per new (n, good) pair; for tests               */

typedef struct cvg_ctx cvg_ctx;
typedef struct cvg_models cvg_models;   /* resident model-view descriptor set                        */
typedef struct cvg_scenes cvg_scenes;   /* resident batch of scene descriptor sets (bench / multi-GPU)*/
typedef struct cvg_job cvg_job;         /* a fused call in flight (cvg_detect_scenes_submit)         */

/* findHomography(..., RANSAC, threshold, mask, maxIters, confidence) — src/TestsDetector.cpp:23,78 */
typedef struct cvg_ransac_params {
    uint32_t size;                  /* = sizeof(cvg_ransac_params)                                   */
    uint32_t flags;
    double threshold;               /* RANSAC_THRESHOLD = 5.0            src/TestsDetector.cpp:23    */
    double confidence;              /* OpenCV default 0.995                                          */
    int32_t max_iters;              /* OpenCV default 2000                                           */
    int32_t reserved;
} cvg_ransac_params;

/* constants of detectObjects() — src/TestsDetector.cpp:21-25 */
typedef struct cvg_detect_params {
    uint32_t size;                  /* = sizeof(cvg_detect_params)                                   */
    float ratio;                    /* MATCH_RATIO_THRESHOLD = 0.9f                       :21        */
    int32_t min_inliers;            /* MIN_INLIERS = 4                                    :22        */
    float det_lo;                   /* HOMOGRAPHY_DET_THRESHOLD = 0.1f                    :24        */
    float det_hi;                   /* HOMOGRAPHY_DET_UPPER_THRESHOLD = 10.0f             :25        */
    int32_t reserved;
    cvg_ransac_params ransac;
} cvg_detect_params;

typedef struct cvg_pair_result {
    int32_t status;                 /* CVG_PAIR_*                                                    */
    int32_t n_good;                 /* matches that passed the ratio test                            */
    int32_t n_inliers;              /* countNonZero(inlierMask) (0 when no H)                        */
    int32_t ransac_iters;           /* RANSAC iterations the reference loop would have run           */
    double H[9];                    /* row-major 3x3, H[8] == 1; zeros when status is LT4/H_EMPTY     */
    double det;                     /* determinant(H)                                                */
} cvg_pair_result;

void cvg_ransac_params_default(cvg_ransac_params* p);
void cvg_detect_params_default(cvg_detect_params* p);

/* ---- context -------------------------------------------------------------------------------- */
int  cvg_create(cvg_ctx** out, int device, unsigned flags);
/* One context over several GPUs of this host (SURVEY 8b row 1, 8e): single process, one device context and one
 * worker thread per listed GPU, one NCCL communicator per GPU (ncclCommInitAll; libnccl is resolved at run time).
 * On such a context: cvg_models_upload replicates the model set on every GPU; cvg_scenes_upload* deals a batch's
 * scenes to the GPUs by cost (batches of fewer than 2 x n_devices scenes stay whole and take the GPUs in turn);
 * cvg_detect_scenes* / _submit run every device's share concurrently and return results in the caller's order —
 * pair sharding of the loop nest of src/TestsDetector.cpp:38,58,99 under src/Output.cpp:23-57, no data-path
 * collective; cvg_match_knn2_sharded is the train-tile sharded match with its one all-gather.  The other entry
 * points (cvg_match_knn2, cvg_find_homography, cvg_detect_pairs, cvg_dev_*) run on the first listed GPU.
 * A device may be listed more than once (logical shards on one GPU, used by the single-GPU tests); NCCL refuses
 * such a communicator, so the exchange then runs as device-to-device copies (cvg_exchange_kind: "memcpy"). */
int  cvg_create_multi(cvg_ctx** out, const int* devices, int n_devices, unsigned flags);
int  cvg_num_devices(const cvg_ctx* ctx);
const char* cvg_exchange_kind(const cvg_ctx* ctx);   /* "nccl", "memcpy", or "none" for a one-device context */
void cvg_destroy(cvg_ctx* ctx);
/* Lanes: engines (stream + scratch + one internal worker thread each) of the context's GPU.  A synchronous
 * cvg_detect_scenes* call splits its batch into up to min(n_lanes, 3) sub-batches that run concurrently, so that one
 * sub-batch's latency-bound refit/LM kernel runs under another's match and hypothesis kernels; calls below ~2^25
 * distance evaluations per lane are not split.  cvg_detect_scenes_submit hands whole batches to the lanes in turn.
 * n_lanes = 1: everything on the context's own stream, on the caller's thread; 0: default (3, env CVG_LANES); up to
 * 8.  A synchronous call uses at most 3 of them (env CVG_SPLIT_LANES).  More lanes (and as many calls in flight) pay
 * off when the host has cores to spare: 6 lanes +7 %, 8 lanes +12 % on one GPU with 16 vCPUs, but -20 % on 8 GPUs
 * sharing 32 vCPUs (profiles/README.md). */
int  cvg_set_lanes(cvg_ctx* ctx, int n_lanes);
const char* cvg_last_error(void);   /* thread-local message of the last failing call                 */
/* Page-locked host memory for callers without CUDA headers: buffers handed to the *_async uploads are copied
 * by DMA while the GPU computes only if they are page-locked (pageable memory is staged, which serialises). */
void* cvg_host_alloc(size_t bytes);
void  cvg_host_free(void* p);
const char* cvg_version(void);

/* ---- model set: replaces nothing, hooks after src/ModelsDetector.cpp:78-80 -------------------
 * desc [N,128] row-major fp32 (all views concatenated), kpt_xy [N,2] (KeyPoint.pt),
 * view_offsets [V+1] row ranges per view, view_model [V] owning ObjectModel index (may be NULL).
 * The copy is converted once and stays resident in HBM until cvg_models_free. */
int  cvg_models_upload(cvg_ctx* ctx, const float* desc, const float* kpt_xy,
                       const int32_t* view_offsets, const int32_t* view_model, int n_views,
                       cvg_models** out);
void cvg_models_free(cvg_ctx* ctx, cvg_models* models);
int  cvg_models_num_views(const cvg_models* models);
int  cvg_models_num_rows(const cvg_models* models);

/* ---- match stage: replaces src/TestsDetector.cpp:59-60 (+ the compare of :67) ----------------
 * BFMatcher(NORM_L2).knnMatch(query, train, k=2) for the rows of one view (view >= 0) or of all
 * views (view == -1) against `train` [n_train,128].  Outputs, per query row i in order:
 *   idx[2i..2i+1]  nearest / second nearest train index, -1 where OpenCV returns a shorter list
 *   dist[2i..2i+1] their L2 distances (fp32, as DMatch.distance)
 *   accept[i]      m.size()==2 && m[0].distance < ratio*m[1].distance   (may be NULL)
 * Ties resolve to the lower train index; NaN/inf distances are never returned (App. A.1-A.4). */
int  cvg_match_knn2(cvg_ctx* ctx, const cvg_models* models, int view,
                    const float* train, int n_train, float ratio,
                    int32_t* idx, float* dist, uint8_t* accept);

/* Same for an arbitrary query matrix [n_query,128] in host memory. */
int  cvg_match_knn2_raw(cvg_ctx* ctx, const float* query, int n_query,
                        const float* train, int n_train, float ratio,
                        int32_t* idx, float* dist, uint8_t* accept);

/* ---- verify stage: replaces src/TestsDetector.cpp:77-79 --------------------------------------
 * findHomography(src, dst, RANSAC, p->threshold, mask, p->max_iters, p->confidence).
 * H gets the 3x3 CV_64F result (zeros if none), mask [n] the returned inlier mask, *found = 0 iff
 * OpenCV returns an empty H.  n < 4 -> CVG_ERR_TOO_FEW_POINTS.  ransac_mask (may be NULL) receives
 * the mask of the winning RANSAC hypothesis before refit/LM. */
int  cvg_find_homography(cvg_ctx* ctx, const float* src_xy, const float* dst_xy, int n,
                         const cvg_ransac_params* p, double H[9], uint8_t* mask, int* found,
                         uint8_t* ransac_mask);

/* Batched form: P independent point sets, set k = rows [offsets[k], offsets[k+1]) of src/dst.
 * Sets with fewer than 4 points report found=0.  iters (may be NULL) [P] = RANSAC iterations. */
int  cvg_find_homography_batch(cvg_ctx* ctx, const float* src_xy, const float* dst_xy,
                               const int64_t* offsets, int n_sets, const cvg_ransac_params* p,
                               double* H /*[P,9]*/, uint8_t* mask, int32_t* found /*[P]*/,
                               int32_t* iters /*[P]*/, uint8_t* ransac_mask);

/* ---- fused path: replaces the body of the view loop, src/TestsDetector.cpp:58-95 -------------
 * All views of the resident model set against one scene (descriptors [n_train,128] + keypoints
 * [n_train,2]).  per_view [V]: status, counts, H, det.  inlier_scene_xy receives, view after view,
 * the scene points of the inliers of ACCEPTED views divided by `scale` when scale != 1.0f
 * (:87-94, :48-55); inlier_offsets [V+1] delimits them.  Capacity of inlier_scene_xy: n_rows of the
 * model set x 2 floats.  Either may be NULL. */
int  cvg_detect_pairs(cvg_ctx* ctx, const cvg_models* models,
                      const float* scene_desc, const float* scene_kpt_xy, int n_train, float scale,
                      const cvg_detect_params* p, cvg_pair_result* per_view,
                      float* inlier_scene_xy, int32_t* inlier_offsets);

/* ---- resident scene batches (inputs already in HBM; used by bench.py `value` and the shards) --
 * cvg_scenes_upload copies S scene descriptor sets (concatenated, offsets [S+1]) to the device
 * once.  cvg_detect_scenes then runs every view of `models` against every scene: S*V pairs, no
 * host->device input traffic.  per_pair is [S*V] (scene-major).  scales [S] may be NULL (=1). */
int  cvg_scenes_upload(cvg_ctx* ctx, const float* desc, const float* kpt_xy,
                       const int64_t* offsets, int n_scenes, cvg_scenes** out);
void cvg_scenes_free(cvg_ctx* ctx, cvg_scenes* scenes);
/* cvg_detect_scenes plus the inlier scene points of every ACCEPTED pair (the consumer of the hot path,
 * src/TestsDetector.cpp:87-94 -> :112-248): inlier_scene_xy receives them pair after pair (scene-major, then view),
 * divided by the scene's scale when it is != 1.0f; inlier_offsets [S*V+1] delimits them.  Capacity of
 * inlier_scene_xy: S x n_rows of the model set x 2 floats.  All five scaled versions of a test image form one
 * batch, so one call covers the whole loop nest of detectObjects for that image (:38, :99-100, :58). */
int  cvg_detect_scenes_inliers(cvg_ctx* ctx, const cvg_models* models, const cvg_scenes* scenes,
                               const float* scales, const cvg_detect_params* p, cvg_pair_result* per_pair,
                               float* inlier_scene_xy, int64_t* inlier_offsets);
/* Streaming form for a caller that walks a list of test images (reference src/Output.cpp:27-47):
 * cvg_scenes_upload_async enqueues the copy and the operand conversion on the context's copy stream
 * and returns at once, so the upload of batch k+1 overlaps cvg_detect_scenes of batch k.  The host
 * arrays must stay valid and unchanged until cvg_scenes_wait or the first cvg_detect_scenes on the
 * handle has returned (use pinned memory for a truly asynchronous copy).  cvg_detect_scenes orders
 * itself after the upload on the device; cvg_scenes_wait is optional. */
int  cvg_scenes_upload_async(cvg_ctx* ctx, const float* desc, const float* kpt_xy,
                             const int64_t* offsets, int n_scenes, cvg_scenes** out);
int  cvg_scenes_wait(cvg_ctx* ctx, cvg_scenes* scenes);
/* Same for uint8 descriptor rows [N,128] (cv::SIFT::create(..., descriptorType = CV_8U), or SIFT's CV_32F output —
 * whose values are integers 0..255 — narrowed by the caller): a quarter of the host->device bytes of the fp32 form
 * (SURVEY 8f-3); widened to fp32 on the device, results identical. */
int  cvg_scenes_upload_u8_async(cvg_ctx* ctx, const uint8_t* desc, const float* kpt_xy,
                                const int64_t* offsets, int n_scenes, cvg_scenes** out);
int  cvg_detect_scenes(cvg_ctx* ctx, const cvg_models* models, const cvg_scenes* scenes,
                       const float* scales, const cvg_detect_params* p, cvg_pair_result* per_pair);
/* Asynchronous pair (SURVEY 8b "async _submit/_wait"): submit enqueues the fused call on one of the context's lanes
 * and returns at once; cvg_job_wait blocks until its results are in the caller's buffers, returns the call's code
 * and frees the job.  A single-threaded caller that walks a list of test images (src/Output.cpp:27-47) keeps two or
 * three jobs in flight — submit image k+1, wait image k, run the consumer on k — and the GPU overlaps one job's
 * refit/LM kernel with the next job's match and hypothesis kernels.  Output buffers, `models` and `scenes` must stay
 * valid until the wait; `scales` and `p` are copied.  Every job must be waited for before cvg_destroy. */
int  cvg_detect_scenes_submit(cvg_ctx* ctx, const cvg_models* models, const cvg_scenes* scenes, const float* scales,
                              const cvg_detect_params* p, cvg_pair_result* per_pair, float* inlier_scene_xy,
                              int64_t* inlier_offsets, cvg_job** job);
int  cvg_job_wait(cvg_ctx* ctx, cvg_job* job);

/* ---- train-tile sharded match over the GPUs of a cvg_create_multi context (BASELINE config 5) ---
 * knnMatch(query, train, 2) + ratio test for host matrices of any size that fits the GPUs together: GPU g gets
 * train rows [g*T, (g+1)*T) (T = ceil(n_train / n_devices) rounded up to 256) and the whole query matrix, computes
 * its local top-2 with global train indices, then ONE exchange step — ncclAllGather of (distance, index) pairs,
 * 16 B per query and GPU — and the lexicographic (distance, index) merge that reproduces OpenCV's tie rule for
 * any number of shards.  Same outputs as cvg_match_knn2_raw; replaces src/TestsDetector.cpp:59-72. */
int  cvg_match_knn2_sharded(cvg_ctx* ctx, const float* query, int n_query, const float* train, int n_train,
                            float ratio, int32_t* idx, float* dist, uint8_t* accept);

/* ---- device-pointer building blocks (multi-GPU train-tile sharding, BASELINE config 5) --------
 * All pointers are DEVICE memory of the context's GPU; `stream` is a cudaStream_t (NULL = default).
 * cvg_dev_match_top2: local top-2 of every query row against this rank's train tile, as
 *   distances dist [nq,2] (fp32, +inf where absent) and GLOBAL train indices idx [nq,2]
 *   (local index + train_index_base, -1 where absent).
 * cvg_dev_merge_top2: merge `n_parts` such partial results (layout [n_parts][nq][2]) in the
 *   lexicographic (distance, idx) order that reproduces OpenCV's tie rule (SURVEY App. A.2), then
 *   emit idx/dist/accept. */
int  cvg_dev_match_top2(cvg_ctx* ctx, void* stream, const float* query_dev, int n_query,
                        const float* train_dev, int n_train, int32_t train_index_base,
                        float* dist_dev, int32_t* idx_dev);
int  cvg_dev_merge_top2(cvg_ctx* ctx, void* stream, const float* dist_parts_dev,
                        const int32_t* idx_parts_dev, int n_parts, int n_query, float ratio,
                        int32_t* idx_dev, float* dist_dev, uint8_t* accept_dev);

/* ---- introspection for tests / bench --------------------------------------------------------- */
/* Which match path served the last match call on this context: 1 = tcgen05 tensor-core kernel, exact (integer
 * descriptors, what SIFT emits); 3 = tcgen05 kernel on hi/lo split bf16 operands keeping four candidates per row,
 * then an fp32 re-rank in cv::batchDistance's summation order that proves the answer with an error bound
 * (non-integer descriptors; unproven rows are redone exactly); 2 = exact fp32 SIMT kernel (CVG_FORCE_EXACT_MATCH,
 * non-finite values); 0 = none yet.  Results are cv2's bit for bit on every path. */
int  cvg_last_match_path(const cvg_ctx* ctx);
/* Rows of the last path-3 call that the re-rank could not prove and the exact fallback kernel redid. */
int  cvg_last_match_fallback_rows(const cvg_ctx* ctx);
/* Path 1 selects a unit's columns by d^2, OpenCV orders by sqrtf(d^2); the two differ only from d = 2048 on, where
 * neighbouring integer d^2 round to one float (u8 rows reach d = 2885; SIFT rows, norm 512, stay below 1024).
 * Rows whose second distance reaches 2048 are redone by the exact kernels, which compare rounded distances:
 * how many rows of the last path-1 call that was.  When the norms of both sides are known on the host and
 * ||q|| + ||t|| < 2047 the guard is not even enqueued. */
int  cvg_last_match_guard_rows(const cvg_ctx* ctx);
/* Verify calls with CVG_RANSAC_NO_EARLY_STOP and max_iters >= 32768 cut every set's cv::RNG draw stream into
 * chunks walked by many CTAs (same samples as the serial walk).  Returns how many sets of the last such call
 * were handed back to the one-CTA-per-set sampler, or -1 if the last verify call did not use the chunked sampler. */
int  cvg_last_sampler_serial_sets(const cvg_ctx* ctx);
/* The context's cudaStream_t (all of its GPU work is issued there); lets a harness record its own
 * CUDA events around calls. */
void* cvg_stream(const cvg_ctx* ctx);
/* Number of kernel launches issued by this context since creation (bench.py's gpu_launches). */
int64_t cvg_launch_count(const cvg_ctx* ctx);
/* Device times in milliseconds of the last call, measured with CUDA events on the context's stream
 * (0 if timing disabled): match_ms = the match kernel launch alone (tcgen05 or exact), ransac_ms =
 * verify-stage kernels, total_ms = first match launch to last gate launch. */
int  cvg_set_timing(cvg_ctx* ctx, int enabled);
int  cvg_last_timing(const cvg_ctx* ctx, float* match_ms, float* ransac_ms, float* total_ms);
/* Verify-stage detail of the last fused call (timing enabled): summed device time of the hypothesis
 * kernel launches, their number, and the number of (hypothesis, correspondence) pairs they scored —
 * 16 bytes each is the algorithmic traffic of the scoring (SURVEY.md section 8d). */
int  cvg_last_hyp_stats(const cvg_ctx* ctx, float* hyp_ms, int* hyp_launches, uint64_t* scored_points);
/* hyp_ms above covers the solve kernel (4-point DLT, one launch per round); the inlier counting of those models runs in
 * ransac_score_kernel, one launch per round as well: its summed device time in the last fused call. */
int  cvg_last_score_ms(const cvg_ctx* ctx, float* score_ms);
/* Error model of device faults.  The kernels never hang: every wait on a barrier is bounded and ends in a trap.  A trap (or
 * any other device-side fault) is reported by the call that synchronises — CVG_ERR_CUDA, cvg_last_error() says so — and it
 * leaves the process' CUDA context in a sticky error state: every later call on that GPU fails the same way, none hangs.
 * Recovery: cvg_destroy the contexts of that GPU (model sets and scene batches die with them), then cvg_device_reset(device)
 * — cudaDeviceReset, which also voids every other CUDA user's state in the process — and cvg_create again.  Whether the
 * driver hands the device back to the SAME process is up to the system: on this pool's B200 boxes it answers "device busy or
 * unavailable" (cvg_device_reset then returns CVG_ERR_CUDA and says so) and the process has to be restarted; a new process
 * gets the GPU at once. */
int  cvg_device_reset(int device);
/* Device self tests.  which = 0: the reciprocal the scoring kernel writes out by hand (MUFU.RCP + one Newton step) against
 * __frcp_rn and against 1.f / x on EVERY float with 2^-126 <= |x| < 2^126; *mismatches must come back 0. */
int  cvg_selftest(cvg_ctx* ctx, int which, uint64_t* mismatches);
/* Debugging aid: with CVG_TRACE=1 in the environment the library timestamps its uploads and fused calls on their streams;
 * this prints the device timeline to stderr and clears it. */
void cvg_trace_dump(void);
/* Debugging aid: the context's device status words (row kinds, match path, counters, kernel debug words; csrc/ctx.cuh). */
int  cvg_debug_words(const cvg_ctx* ctx, int* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* CVGRAFT_H */
