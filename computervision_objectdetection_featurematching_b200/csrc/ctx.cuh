// ctx.cuh — internal object layout of libcvgraft's handles (cvg_ctx, cvg_models, cvg_scenes, cvg_job) and the
// engine-level functions that api.cu implements and multi.cu (lanes, jobs, multi-device contexts) drives.
#pragma once
#include "common.cuh"
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

int cvg_set_err(int code, const char* fmt, ...);      // thread-local message of cvg_last_error(); returns code

#define CU_CHECK(call)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return cvg_set_err(CVG_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                               __FILE__, __LINE__);                                            \
    } while (0)

// grow-only device buffer
struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// grow-only page-locked host buffer (device -> host results land here by DMA, without a staging copy inside the driver)
struct HostBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Freed device buffers are kept for reuse: cudaMalloc/cudaFree cost milliseconds and serialise the
// device, which would dominate a streaming caller that uploads a scene batch per step.
struct BufPool {
    std::vector<DevBuf> free_list;
    cudaError_t acquire(DevBuf& b, size_t bytes)
    {
        if (b.cap >= bytes) return cudaSuccess;
        if (b.p) { release(b); }
        int best = -1;
        for (int i = 0; i < (int)free_list.size(); i++)
            if (free_list[i].cap >= bytes && (best < 0 || free_list[i].cap < free_list[best].cap)) best = i;
        // a buffer serves requests down to two thirds of its size: the buffers of a streaming caller (fp32 rows, bf16 operands,
        // u8 rows: 4 : 2 : 1) then stay with their own kind instead of stealing each other's and forcing a cudaMalloc
        if (best >= 0 && free_list[best].cap <= bytes + bytes / 2 + (1 << 20)) {
            b = free_list[best];
            free_list.erase(free_list.begin() + best);
            return cudaSuccess;
        }
        return b.ensure(bytes);
    }
    void release(DevBuf& b)
    {
        if (!b.p) return;
        if (free_list.size() >= 256) {              // bounded: the buffer that has waited longest goes (sizes of a
            free_list.front().release();            // streaming caller drift; keeping the smallest ones thrashed)
            free_list.erase(free_list.begin());
        }
        free_list.push_back(b);
        b.p = nullptr; b.cap = 0;
    }
    void clear() { for (DevBuf& b : free_list) b.release(); free_list.clear(); }
};

struct SegInfo { int rows; int64_t f32_row0; int64_t pad_row0; int ct; };

struct TrainSet {                      // a prepared set of train segments on the device
    int n_segs = 0;
    std::vector<SegInfo> segs;
    int64_t rows_total = 0, rows_pad_total = 0;
    int max_rows = 0;
    float* d_f32 = nullptr;            // [rows_total, 128]
    __nv_bfloat16* d_b = nullptr;      // [rows_pad_total, 128]
    __nv_bfloat16* d_blo = nullptr;    // [rows_pad_total, 128] lo half of the split operand (zero for integer rows)
    __nv_bfloat16* d_aug = nullptr;    // [rows_pad_total, 16]
    float* d_kpt = nullptr;            // [rows_total, 2] or null
    int64_t* d_kpt_offsets = nullptr;  // [S+1]
    int nonint = -1;                   // host-known row-kind bits of prep_rows_kernel (-1 unknown: decided on the device)
    int* d_tnmax = nullptr;            // device word: max ||t||^2 as float bits (error bound of the candidate path)
};

struct cvg_models {
    int n_rows = 0, n_pad = 0, n_views = 0;
    std::vector<int32_t> view_offsets, view_model;
    float* d_f32 = nullptr; __nv_bfloat16* d_b = nullptr; __nv_bfloat16* d_blo = nullptr; __nv_bfloat16* d_aug = nullptr;
    float* d_norm = nullptr; float* d_kpt = nullptr; int32_t* d_view_offsets = nullptr;
    int nonint = 0;
    float max_norm2 = 0.f;             // largest ||q||^2 of the set (host-known: decides whether d >= 2048 can occur at all)
    uint64_t uid = 0;                  // process-unique id: key of the cached match plan (addresses get reused)
    int device = -1;                   // device the buffers live on
    std::vector<cvg_models*> replicas; // multi-device context: one resident copy per device (this object is the shell)
};

struct cvg_scenes {
    TrainSet ts;
    DevBuf f32, b, blo, aug, kpt, kptoff, u8, segtab;
    int* d_flag = nullptr;             // non-integer flag of this batch (tail of kptoff)
    cudaEvent_t ready = nullptr;       // set by cvg_scenes_upload_async: upload + conversion finished
    float max_norm2 = -1.f;            // largest ||t||^2 of the batch when the host knows it (synchronous upload), else -1
    std::vector<int64_t> offsets_copy; // the caller's offsets (the library keeps no caller pointer beyond the call)
    // multi-device context: the batch is dealt to the devices scene by scene (this object is the shell)
    std::vector<cvg_scenes*> subs;     // per device, or null when the device got no scene
    std::vector<int> dev_of_scene, local_of_scene;
    int n_scenes_total = 0;
};

struct Lane;
struct MultiState;

struct cvg_ctx {
    int device = 0; unsigned flags = 0; int n_sms = 148;
    cudaStream_t stream = nullptr;
    // uploads of cvg_scenes_upload_async (overlap with compute) take these in turn: the operand conversion kernels of one
    // batch then run under the host -> device copy of the next
    cudaStream_t copy_stream[3] = { nullptr, nullptr, nullptr }; unsigned next_copy = 0;
    HostBuf inl_h, cnt_h, res_h;                       // inlier pool, counts, per-pair results + status words of the last fused call (page-locked)
    int* d_flags = nullptr;            // [0] train row kinds, [1] query row kinds, [2] match path (0 tensor exact, 1 tensor
                                       // candidates + re-rank, 2 exact SIMT), [3] raw-query kinds, [4] RNG table short,
                                       // [5] max ||t||^2 bits, [6] fallback row count, [7] rows the d >= 2048 guard redid, [8..16) kernel debug words,
                                       // [17] sets the chunked sampler handed to the serial one, [18] max ||q||^2 bits (models upload), [19] niters entries to verify,
                                       // [20..22) rows / columns the cross-check guard redid
    uint32_t* d_rng = nullptr; int64_t rng_len = 0;
    int last_match_path = 0; int64_t launches = 0;
    int timing = 0; float t_match = 0, t_ransac = 0, t_total = 0;
    cudaEvent_t ev[6] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    cudaEvent_t hyp_ev[48] = {};                       // [2r], [2r+1]: solve kernel of round r; [32 + r]: after its score kernel
    int hyp_rounds = 0; float t_hyp = 0, t_score = 0; int hyp_launches = 0; unsigned long long scored_pts = 0;
    unsigned long long* d_scored = nullptr;
    // scratch
    DevBuf q_f32, q_b, q_blo, q_aug, q_norm;           // raw-query path
    DevBuf t_f32, t_b, t_blo, t_aug, t_kpt, t_kptoff, t_segtab;  // per-call train path
    DevBuf units, dir, parts, idx, dist, accept;
    DevBuf parts4, segdev, fb;                         // candidate path: Top4 records, segment table, unproven rows
    DevBuf hypH;                                       // fp32 models of the current round(s), read by ransac_score_kernel
    DevBuf chunk;                                      // chunked sampler scratch (huge no-early-stop rounds)
    DevBuf plan_units, plan_dir;                       // match plan of the fused path, cached by (model set, scene shapes)
    DevBuf xc;                                         // cross-check: XcOut, row keys, column keys
    bool last_chunked = false;                         // the last verify call used the chunked sampler (d_flags[17] = sets it handed back)
    uint64_t plan_models_uid = 0; std::vector<int> plan_shape; int plan_units_n = 0;   // keyed on cvg_models::uid: addresses get reused
    DevBuf pts, starts, counts_n, sample_pos, n_samples, counts, best_iter, best_count, iters_run, niters_cur, smp_state, sel;
    DevBuf H, mask, rmask, found, sflags, results, inl_xy, inl_cnt, scales, src, dst;
    DevBuf nit, nitreq;                                // host-verified RANSACUpdateNumIters entries, the device's requests (run_ransac)
    std::vector<cvg::NitEntry> nit_host;
    int nit_mp = 4;                                    // model points of the last verify stage (keys its niters requests)
    BufPool pool;                                      // recycled buffers of freed scene batches
    // Small host->device parameter blocks of the fused path go through a mapped pinned staging area read by a
    // copy kernel, not through cudaMemcpyAsync: the H2D copy engine may be busy for milliseconds with the next
    // scene batch (cvg_scenes_upload_async) and would hold the compute stream behind it.
    uint8_t* stage_h = nullptr; uint8_t* stage_d = nullptr; size_t stage_cap = 0, stage_used = 0; bool stage_fallback = false;
    int wave_div = 1;                  // how many engines share this GPU right now (sizes the RANSAC rounds)
    cudaEvent_t sync_ev = nullptr;     // blocking-sync event a lane's worker sleeps on (sync_and_check)
    bool blocking_sync = false;        // this engine's current work is a pipelined job: sleep, do not spin, while the GPU works
    // lanes: engines of the same device, each driven by its own worker thread, that serve the sub-batches of one
    // synchronous fused call and the jobs of cvg_detect_scenes_submit (multi.cu)
    cvg_ctx* parent = nullptr;         // set on a lane / device engine
    std::vector<struct Lane*> lanes; int lanes_cfg = -1; unsigned next_lane = 0;
    int64_t split_min_cost = -1;
    struct MultiState* multi = nullptr;   // multi-device context (cvg_create_multi): this object is the shell
};

// ---- a worker thread with a FIFO of closures ---------------------------------------------------------
struct Worker {
    std::thread th; std::mutex m; std::condition_variable cv; std::deque<std::function<void()>> q; bool stop = false;
    Worker() { th = std::thread([this] { run(); }); }
    ~Worker() { { std::lock_guard<std::mutex> g(m); stop = true; } cv.notify_all(); if (th.joinable()) th.join(); }
    void post(std::function<void()> f) { { std::lock_guard<std::mutex> g(m); q.push_back(std::move(f)); } cv.notify_one(); }
    void run()
    {
        for (;;) {
            std::function<void()> f;
            { std::unique_lock<std::mutex> g(m); cv.wait(g, [this] { return stop || !q.empty(); }); if (q.empty()) return; f = std::move(q.front()); q.pop_front(); }
            f();
        }
    }
};

// completion of one piece of posted work
struct Done {
    std::mutex m; std::condition_variable cv; bool done = false; int rc = 0; std::string err;
    void set(int code, const char* msg) { { std::lock_guard<std::mutex> g(m); done = true; rc = code; if (code && msg) err = msg; } cv.notify_all(); }
    int wait() { std::unique_lock<std::mutex> g(m); cv.wait(g, [this] { return done; }); return rc; }
};

struct Lane { cvg_ctx* eng = nullptr; Worker* worker = nullptr; };

// the engine behind a public handle: the context itself, or device 0 of a multi-device shell (multi.cu)
cvg_ctx* cvg_primary(cvg_ctx* c);
const cvg_ctx* cvg_primary(const cvg_ctx* c);
const cvg_models* cvg_models_on(const cvg_models* m, const cvg_ctx* eng);   // the replica on eng's device (or m itself)

// ---- engine-level entry points (api.cu): one device, one stream, synchronous, caller's thread ------------
int  eng_create(cvg_ctx** out, int device, unsigned flags);
void eng_destroy(cvg_ctx* c);
int  eng_models_upload(cvg_ctx* c, const float* desc, const float* kpt_xy, const int32_t* view_offsets,
                       const int32_t* view_model, int n_views, cvg_models** out);
void eng_models_free(cvg_ctx* c, cvg_models* m);
int  eng_scenes_upload(cvg_ctx* c, const float* desc, const uint8_t* desc_u8, const float* kpt_xy, const int64_t* offsets,
                       int n_scenes, cvg_scenes** out, bool async, const int64_t* src_row0 = nullptr);
void eng_scenes_free(cvg_ctx* c, cvg_scenes* sc);
int  eng_scenes_wait(cvg_ctx* c, cvg_scenes* sc);
// scenes [s0, s1) of a resident batch against every view: per_pair [(s1 - s0) * V]; pool / cnt (may be NULL) receive the
// inlier scene points packed pair after pair (scene-major, then view) and the inlier counts per pair.  `c` may be any
// engine of the device that holds the scenes and the models.
int  eng_detect_range(cvg_ctx* c, const cvg_models* m, cvg_scenes* sc, int s0, int s1, const float* scales,
                      const cvg_detect_params* p, cvg_pair_result* per_pair, std::vector<float>* pool,
                      std::vector<int32_t>* cnt);
// the caller's cvg_detect_params (either size, include/cvgraft.h) checked and copied in full into *out; every entry point
// hands the copy on, never the caller's pointer
int  check_detect_params(const cvg_detect_params* p, cvg_detect_params* out);
int  check_params(const cvg_ransac_params* p);
int  sync_and_check(cvg_ctx* c);                        // waits for the engine's stream; names the device on a fault
// verify stage building blocks (the hypothesis-range sharded driver of multi.cu runs one engine per device through them)
int  ensure_rng(cvg_ctx* c, int max_iters, int64_t min_len = 0);   // the engine's cv::RNG draw table: >= max_iters * 48 and min_len
// scratch, flags and parameters of a verify stage over n_sets sets of the pool; counts gets counts_slack extra entries
int  eng_ransac_work(cvg_ctx* c, const float4* d_pts, const int64_t* d_starts, const int32_t* d_counts_n, int n_sets,
                     int max_n, int64_t pool_rows, const cvg_ransac_params* p, bool want_rmask, int counts_slack,
                     cvg::RansacWork* out, int model_points = 4);
int  nit_add_requests(cvg_ctx* c, std::vector<cvg::NitEntry>& tab, size_t* added);   // the engine's niters requests into tab
int  nit_upload(cvg_ctx* c);                            // c->nit_host to the device (stream-ordered, synchronised)

