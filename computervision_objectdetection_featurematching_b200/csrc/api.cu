// api.cu — the C ABI of libcvgraft (include/cvgraft.h): context, resident model/scene sets and the
// host-side orchestration of the match and verify kernels.  No CPU fallback exists: every entry point
// needs a CUDA device and fails loudly otherwise.
#include "ctx.cuh"
#include <atomic>
#include <string.h>
#include <stdlib.h>
#include <unistd.h>
#include <stdarg.h>
#include <math.h>
#include <float.h>

using namespace cvg;

static thread_local char g_err[512] = "";

int cvg_set_err(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define set_err cvg_set_err

// ---- device timeline for debugging (CVG_TRACE=1): timestamps on the streams, dumped by cvg_trace_dump -----------------
struct TraceEv { cudaEvent_t ev; const char* tag; int id; int dev; };
static std::mutex g_trace_mu;
static std::vector<TraceEv> g_trace;
static bool trace_on() { static const bool on = getenv("CVG_TRACE") && atoi(getenv("CVG_TRACE")); return on; }
void cvg_trace_mark(cudaStream_t st, const char* tag, int id)
{
    if (!trace_on()) return;
    TraceEv t; t.tag = tag; t.id = id; cudaGetDevice(&t.dev);
    if (cudaEventCreate(&t.ev) != cudaSuccess) return;
    cudaEventRecord(t.ev, st);
    std::lock_guard<std::mutex> g(g_trace_mu);
    if (g_trace.size() < 100000) g_trace.push_back(t);
}
extern "C" void cvg_trace_dump(void)
{
    std::lock_guard<std::mutex> g(g_trace_mu);
    if (g_trace.empty()) return;
    for (const TraceEv& t : g_trace) cudaEventSynchronize(t.ev);
    for (const TraceEv& t : g_trace) {
        float ms = 0; cudaEventElapsedTime(&ms, g_trace[0].ev, t.ev);
        fprintf(stderr, "trace %10.3f ms  dev %d  %-14s %d\n", ms, t.dev, t.tag, t.id);
    }
    for (const TraceEv& t : g_trace) cudaEventDestroy(t.ev);
    g_trace.clear();
}

__global__ void stage_copy_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src, size_t n16)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

// dst must be 16-byte aligned device memory with room for bytes rounded up to 16.
static cudaError_t h2d_small(cvg_ctx* c, void* dst, const void* src, size_t bytes)
{
    const size_t padded = (bytes + 15) & ~(size_t)15;
    if (!c->stage_h || c->stage_used + padded > c->stage_cap || ((uintptr_t)dst & 15)) {
        c->stage_fallback = true;                          // caller synchronises before its host source goes away
        return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream);
    }
    uint8_t* h = c->stage_h + c->stage_used;
    memcpy(h, src, bytes);
    const uint8_t* d = c->stage_d + c->stage_used;
    c->stage_used += padded;
    const size_t n16 = padded / 16;
    const int blocks = (int)std::min<size_t>((n16 + 255) / 256, 64);
    stage_copy_kernel<<<blocks, 256, 0, c->stream>>>(reinterpret_cast<uint4*>(dst), reinterpret_cast<const uint4*>(d), n16);
    c->launches++;
    return cudaGetLastError();
}

extern "C" {

const char* cvg_last_error(void) { return g_err; }
const char* cvg_version(void) { return "cvgraft 0.1.0 (sm_100a)"; }

void cvg_ransac_params_default(cvg_ransac_params* p)
{
    memset(p, 0, sizeof *p);
    p->size = sizeof *p; p->flags = 0; p->threshold = 5.0; p->confidence = 0.995; p->max_iters = 2000;
}

void cvg_detect_params_default(cvg_detect_params* p)
{
    memset(p, 0, sizeof *p);
    p->size = sizeof *p; p->ratio = 0.9f; p->min_inliers = 4; p->det_lo = 0.1f; p->det_hi = 10.0f;
    cvg_ransac_params_default(&p->ransac);
}

}  // extern "C"

// Opt-in attributes (dynamic shared memory) belong to a (function, device) pair: set once per device of the process.
static std::mutex g_dev_mu;
static bool g_dev_done[64] = {};
static void device_forget(int device) { std::lock_guard<std::mutex> g(g_dev_mu); if (device >= 0 && device < 64) g_dev_done[device] = false; }
static int device_init_once(int device, char* err, size_t errlen)
{
    std::mutex& mu = g_dev_mu; bool* done = g_dev_done;
    std::lock_guard<std::mutex> g(mu);
    if (device >= 0 && device < 64 && done[device]) return 0;
    if (tc_init(err, errlen)) return 1;
    if (tc_set_device_attrs(err, errlen)) return 1;
    if (ransac_set_device_attrs(err, errlen)) return 1;
    if (device >= 0 && device < 64) done[device] = true;
    return 0;
}

int eng_create(cvg_ctx** out, int device, unsigned flags)
{
    if (!out) return set_err(CVG_ERR_INVALID, "cvg_create: out is NULL");
    *out = nullptr;
    // more hardware work queues than the default 8: a context runs up to 1 + lanes compute streams and 2 copy streams, and
    // streams that share a queue serialise.  Only effective when the process has not initialised CUDA yet; never overrides.
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return set_err(CVG_ERR_CUDA, "cvg_create: no CUDA device (%s); libcvgraft has no CPU fallback",
                       cudaGetErrorString(e));
    if (device < 0 || device >= n_dev) return set_err(CVG_ERR_INVALID, "cvg_create: device %d of %d", device, n_dev);
    CU_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return set_err(CVG_ERR_CUDA, "cvg_create: device %d is sm_%d%d; libcvgraft is built for sm_100a only",
                       device, prop.major, prop.minor);
    char err[256];
    if (device_init_once(device, err, sizeof err)) return set_err(CVG_ERR_CUDA, "%s", err);
    cvg_ctx* c = new cvg_ctx();
    c->device = device; c->flags = flags; c->n_sms = prop.multiProcessorCount;
    int rc = [&]() -> int {
        CU_CHECK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        CU_CHECK(cudaMalloc(&c->d_flags, 64 * sizeof(int)));
        CU_CHECK(cudaMemset(c->d_flags, 0, 64 * sizeof(int)));
        for (int i = 0; i < 6; i++) CU_CHECK(cudaEventCreate(&c->ev[i]));
        for (int i = 0; i < 48; i++) CU_CHECK(cudaEventCreate(&c->hyp_ev[i]));
        CU_CHECK(cudaMalloc(&c->d_scored, 8));
        CU_CHECK(cudaMemset(c->d_scored, 0, 8));
        CU_CHECK(cudaEventCreateWithFlags(&c->sync_ev, cudaEventBlockingSync | cudaEventDisableTiming));
        return CVG_OK;
    }();
    if (rc) { eng_destroy(c); return rc; }                  // a half-built engine releases what it got
    c->stage_cap = 4u << 20;
    if (cudaHostAlloc((void**)&c->stage_h, c->stage_cap, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void**)&c->stage_d, c->stage_h, 0) != cudaSuccess) {
        cudaGetLastError(); c->stage_h = nullptr; c->stage_cap = 0;       // falls back to cudaMemcpyAsync
    }
    *out = c;
    return CVG_OK;
}

void eng_destroy(cvg_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (int i = 0; i < 3; i++) if (c->copy_stream[i]) cudaStreamSynchronize(c->copy_stream[i]);
    DevBuf* bufs[] = { &c->q_f32, &c->q_b, &c->q_blo, &c->q_aug, &c->q_norm, &c->t_f32, &c->t_b, &c->t_blo, &c->t_aug, &c->t_segtab, &c->t_kpt, &c->t_kptoff,
                       &c->units, &c->dir, &c->parts, &c->parts4, &c->segdev, &c->fb, &c->plan_units, &c->plan_dir, &c->chunk, &c->hypH, &c->idx, &c->dist, &c->accept, &c->pts, &c->starts, &c->counts_n,
                       &c->sample_pos, &c->n_samples, &c->counts, &c->best_iter, &c->best_count, &c->iters_run, &c->niters_cur, &c->smp_state, &c->sel,
                       &c->H, &c->mask, &c->rmask, &c->found, &c->sflags, &c->results, &c->inl_xy, &c->inl_cnt,
                       &c->scales, &c->src, &c->dst, &c->nit, &c->nitreq };
    for (DevBuf* b : bufs) b->release();
    c->pool.clear();
    if (c->d_flags) cudaFree(c->d_flags);
    if (c->d_rng) cudaFree(c->d_rng);
    for (int i = 0; i < 6; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (int i = 0; i < 48; i++) if (c->hyp_ev[i]) cudaEventDestroy(c->hyp_ev[i]);
    if (c->d_scored) cudaFree(c->d_scored);
    if (c->stage_h) cudaFreeHost(c->stage_h);
    if (c->sync_ev) cudaEventDestroy(c->sync_ev);
    if (c->stream) cudaStreamDestroy(c->stream);
    for (int i = 0; i < 3; i++) if (c->copy_stream[i]) cudaStreamDestroy(c->copy_stream[i]);
    c->inl_h.release(); c->cnt_h.release(); c->res_h.release();
    delete c;
}

extern "C" {

int cvg_debug_words(const cvg_ctx* c0, int* out, int n)
{
    const cvg_ctx* c = cvg_primary(c0);
    if (!c || !out || n < 0 || n > 64) return set_err(CVG_ERR_INVALID, "cvg_debug_words: bad argument");
    CU_CHECK(cudaSetDevice(c->device));
    CU_CHECK(cudaMemcpy(out, c->d_flags, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return CVG_OK;
}

int cvg_device_reset(int device)
{
    // cudaDeviceReset: the only way out of a sticky error.  Every handle of this device (contexts, model sets, scene batches,
    // cvg_host_alloc memory) is void afterwards; so is every other CUDA user's state in this process.
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceReset();
    cudaGetLastError();
    device_forget(device);
    // after a fault the driver tears the channel down asynchronously: the device reports "busy or unavailable" for a moment
    for (int attempt = 0; attempt < 20; attempt++) {
        e = cudaSetDevice(device);
        if (e == cudaSuccess) e = cudaFree(nullptr);             // forces a fresh primary context
        if (e == cudaSuccess) break;
        cudaGetLastError();
        usleep(100 * 1000);
    }
    if (e != cudaSuccess)
        return set_err(CVG_ERR_CUDA, "cudaDeviceReset(%d): %s — this driver does not hand the device back to a process that "
                       "faulted on it; restart the process", device, cudaGetErrorString(e));
    return CVG_OK;
}

void* cvg_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void cvg_host_free(void* p) { if (p) cudaFreeHost(p); }

// Introspection reads the engine that served the caller's last direct call: the context itself, or device 0 of a
// multi-device context (cvg_primary).
int cvg_last_match_path(const cvg_ctx* c0) { const cvg_ctx* c = cvg_primary(c0); return c ? c->last_match_path : 0; }
static int read_flag_word(const cvg_ctx* c, int word)
{
    int n = 0;
    cudaSetDevice(c->device);
    cudaMemcpy(&n, c->d_flags + word, 4, cudaMemcpyDeviceToHost);
    return n;
}
int cvg_last_match_fallback_rows(const cvg_ctx* c0)
{
    const cvg_ctx* c = cvg_primary(c0);
    return (!c || c->last_match_path != 3) ? 0 : read_flag_word(c, 6);
}
int cvg_last_match_guard_rows(const cvg_ctx* c0)
{
    const cvg_ctx* c = cvg_primary(c0);
    return (!c || c->last_match_path != 1) ? 0 : read_flag_word(c, 7);
}
int cvg_last_sampler_serial_sets(const cvg_ctx* c0)
{
    const cvg_ctx* c = cvg_primary(c0);
    return (!c || !c->last_chunked) ? -1 : read_flag_word(c, 17);
}
void* cvg_stream(const cvg_ctx* c0) { const cvg_ctx* c = cvg_primary(c0); return c ? (void*)c->stream : nullptr; }
int cvg_last_hyp_stats(const cvg_ctx* c0, float* hyp_ms, int* hyp_launches, uint64_t* scored_points)
{
    const cvg_ctx* c = cvg_primary(c0);
    if (!c) return CVG_ERR_INVALID;
    if (hyp_ms) *hyp_ms = c->t_hyp;
    if (hyp_launches) *hyp_launches = c->hyp_launches;
    if (scored_points) *scored_points = c->scored_pts;
    return CVG_OK;
}
int cvg_selftest(cvg_ctx* c0, int which, uint64_t* mismatches)
{
    cvg_ctx* c = cvg_primary(c0);
    if (!c || !mismatches || which != 0) return set_err(CVG_ERR_INVALID, "cvg_selftest: bad argument");
    CU_CHECK(cudaSetDevice(c->device));
    CU_CHECK(cudaMemsetAsync(c->d_scored, 0, 8, c->stream));
    c->launches += launch_selftest_rcp(c->d_scored, c->stream);
    unsigned long long n = 0;
    CU_CHECK(cudaMemcpyAsync(&n, c->d_scored, 8, cudaMemcpyDeviceToHost, c->stream));
    CU_CHECK(cudaStreamSynchronize(c->stream));
    *mismatches = n;
    return CVG_OK;
}
int cvg_last_score_ms(const cvg_ctx* c0, float* score_ms)
{
    const cvg_ctx* c = cvg_primary(c0);
    if (!c || !score_ms) return CVG_ERR_INVALID;
    *score_ms = c->t_score;
    return CVG_OK;
}
int cvg_set_timing(cvg_ctx* c0, int enabled) { cvg_ctx* c = cvg_primary(c0); if (!c) return CVG_ERR_INVALID; c->timing = enabled; return CVG_OK; }
int cvg_last_timing(const cvg_ctx* c0, float* m, float* r, float* t)
{
    const cvg_ctx* c = cvg_primary(c0);
    if (!c) return CVG_ERR_INVALID;
    if (m) *m = c->t_match;
    if (r) *r = c->t_ransac;
    if (t) *t = c->t_total;
    return CVG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// internals
// ---------------------------------------------------------------------------------------------------
static int round_up(int v, int m) { return (v + m - 1) / m * m; }

constexpr int64_t RNG_TABLE_CAP = 1LL << 28;                    // 1 GiB of draws
constexpr int NIT_REQ_CAP = 16384;                              // (n, good) pairs a call may ask the host about per attempt

// The raw cv::RNG stream of the fixed seed as a device table.  An accepted 4-point sample costs 4 draws plus the
// draws of the attempts checkSubset rejected before it (5-8 attempts on outlier-heavy sets), so the table is sized
// at 48 draws per iteration; a call that still runs out grows it (min_len) and repeats the verify stage.
static int ensure_rng(cvg_ctx* c, int max_iters, int64_t min_len = 0)
{
    int64_t want = std::max<int64_t>(1 << 20, (int64_t)max_iters * 48 + (1 << 16));
    want = std::max(want, min_len);
    if (want > RNG_TABLE_CAP) want = RNG_TABLE_CAP;
    if (c->rng_len >= want) return CVG_OK;
    std::vector<uint32_t> tab((size_t)want);
    uint64_t state = 0xFFFFFFFFFFFFFFFFull;                     // RNG rng((uint64)-1), SURVEY App. B.2
    for (int64_t i = 0; i < want; i++) {
        state = (uint64_t)(uint32_t)state * 4164903690U + (uint32_t)(state >> 32);
        tab[(size_t)i] = (uint32_t)state;
    }
    CU_CHECK(cudaStreamSynchronize(c->stream));
    if (c->d_rng) cudaFree(c->d_rng);
    c->d_rng = nullptr; c->rng_len = 0;
    CU_CHECK(cudaMalloc(&c->d_rng, (size_t)want * 4));
    CU_CHECK(cudaMemcpyAsync(c->d_rng, tab.data(), (size_t)want * 4, cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaStreamSynchronize(c->stream));
    c->rng_len = want;
    return CVG_OK;
}

// Prepare (convert) a train set that is already in device fp32 memory.
static int prep_train(cvg_ctx* c, TrainSet& ts, DevBuf& b, DevBuf& blo, DevBuf& aug, DevBuf& segtab, int flag_slot,
                      bool pooled = false, cudaStream_t st = nullptr, int* d_flag = nullptr)
{
    if (!st) st = c->stream;
    if (!d_flag) d_flag = c->d_flags + flag_slot;
    if (!ts.d_tnmax) ts.d_tnmax = c->d_flags + 5;
    CU_CHECK(cudaMemsetAsync(ts.d_tnmax, 0, 4, st));
    const size_t nb = (size_t)std::max<int64_t>(ts.rows_pad_total, 1) * DIM * 2;
    const size_t na = (size_t)std::max<int64_t>(ts.rows_pad_total, 1) * KAUG * 2;
    if (pooled) { CU_CHECK(c->pool.acquire(b, nb)); CU_CHECK(c->pool.acquire(blo, nb)); CU_CHECK(c->pool.acquire(aug, na)); }
    else { CU_CHECK(b.ensure(nb)); CU_CHECK(blo.ensure(nb)); CU_CHECK(aug.ensure(na)); }
    ts.d_b = b.as<__nv_bfloat16>(); ts.d_blo = blo.as<__nv_bfloat16>(); ts.d_aug = aug.as<__nv_bfloat16>();
    if (ts.n_segs == 1) {
        const SegInfo& s = ts.segs[0];
        launch_prep_rows(ts.d_f32 + s.f32_row0 * DIM, s.rows, s.ct * TILE_N, 1, ts.d_b, ts.d_blo, ts.d_aug, nullptr, d_flag,
                         ts.d_tnmax, st);
        c->launches++;
    } else if (ts.n_segs > 1) {
        // one launch for the whole batch: the segment table rides in front of the augmentation buffer's slack
        std::vector<PrepSeg> tab((size_t)ts.n_segs);
        for (int i = 0; i < ts.n_segs; i++) tab[(size_t)i] = PrepSeg{ ts.segs[(size_t)i].f32_row0, ts.segs[(size_t)i].pad_row0, ts.segs[(size_t)i].rows, 0 };
        if (pooled) CU_CHECK(c->pool.acquire(segtab, tab.size() * sizeof(PrepSeg)));
        else CU_CHECK(segtab.ensure(tab.size() * sizeof(PrepSeg)));
        CU_CHECK(cudaMemcpyAsync(segtab.p, tab.data(), tab.size() * sizeof(PrepSeg), cudaMemcpyHostToDevice, st));   // pageable: staged before return
        launch_prep_train_segments(ts.d_f32, segtab.as<PrepSeg>(), ts.n_segs, ts.rows_pad_total, ts.d_b, ts.d_blo, ts.d_aug,
                                   d_flag, ts.d_tnmax, st);
        c->launches++;
    }
    CU_CHECK(cudaGetLastError());
    return CVG_OK;
}

static void layout_segments(TrainSet& ts, const int64_t* offsets, int n)
{
    ts.n_segs = n; ts.segs.resize(n);
    int64_t pad = 0; int mx = 0;
    for (int s = 0; s < n; s++) {
        SegInfo& g = ts.segs[s];
        g.rows = (int)(offsets[s + 1] - offsets[s]);
        g.f32_row0 = offsets[s];
        g.ct = (g.rows + TILE_N - 1) / TILE_N;
        g.pad_row0 = pad;
        pad += (int64_t)g.ct * TILE_N;
        mx = std::max(mx, g.rows);
    }
    ts.rows_total = offsets[n]; ts.rows_pad_total = pad; ts.max_rows = mx;
}

struct QuerySide {
    const float* d_f32; const __nv_bfloat16* d_b; const __nv_bfloat16* d_blo; const __nv_bfloat16* d_aug; const float* d_norm;
    int row_begin, row_end;        // absolute rows matched
    int n_pad;                     // rows of the padded operand matrices
};

// Build the unit list for query rows [row_begin,row_end) x all segments.  Returns units sorted by size
// (largest first) and the merge directory [seg][rowblock].
static void build_plan(const QuerySide& q, const TrainSet& ts, int n_sms, std::vector<MatchUnit>& units,
                       std::vector<MergeEntry>& dir, int& n_rb)
{
    const int nq = q.row_end - q.row_begin;
    n_rb = (nq + TILE_M - 1) / TILE_M;
    int64_t total_tiles = 0;
    int max_ct = 1;
    for (const SegInfo& s : ts.segs) { total_tiles += (int64_t)n_rb * s.ct; max_ct = std::max(max_ct, s.ct); }
    // chunk length: minimise the estimated makespan (tiles per CTA incl. an A-reload cost of 0.5 tile)
    int best_ch = 1; double best_cost = 1e300;
    for (int ch = 1; ch <= max_ct; ch++) {
        int64_t n_units = 0;
        for (const SegInfo& s : ts.segs) n_units += (int64_t)n_rb * ((s.ct + ch - 1) / ch);
        const double waves = ceil((double)n_units / n_sms);
        const double cost = waves * (ch + 0.5);
        if (cost < best_cost - 1e-9) { best_cost = cost; best_ch = ch; }
    }
    units.clear(); dir.assign((size_t)ts.n_segs * n_rb, MergeEntry{ 0, 0 });
    // With an even number of row blocks the list is made of PAIRS: units (2p, 2p + 1) are row blocks (2i, 2i + 1) against
    // the same train tiles — what the cta_group::2 form of the match kernel needs (launch_match_tc, paired); any other
    // consumer sees an ordinary unit list.  Partial slots stay consecutive per (segment, row block) for the merge.
    const int group = (n_rb % 2 == 0) ? 2 : 1;
    int slot = 0;
    for (int s = 0; s < ts.n_segs; s++) {
        const SegInfo& g = ts.segs[s];
        const int n_chunks = (g.ct + best_ch - 1) / best_ch;
        const int slot0 = slot;
        for (int rb = 0; rb < n_rb; rb++) dir[(size_t)s * n_rb + rb] = MergeEntry{ slot0 + rb * n_chunks, n_chunks };
        slot += n_rb * n_chunks;
        for (int rb0 = 0; rb0 < n_rb; rb0 += group) {
            for (int ck = 0; ck < n_chunks; ck++) {
                // spread tiles evenly over the chunks of this segment
                const int t0 = (int)((int64_t)g.ct * ck / n_chunks), t1 = (int)((int64_t)g.ct * (ck + 1) / n_chunks);
                for (int rb = rb0; rb < rb0 + group; rb++) {
                    MatchUnit u;
                    u.q_row0 = q.row_begin + rb * TILE_M;
                    u.t_row0 = (int32_t)(g.pad_row0 + (int64_t)t0 * TILE_N);
                    u.n_tiles = t1 - t0;
                    u.t_local0 = t0 * TILE_N;
                    u.part_slot = slot0 + rb * n_chunks + ck;
                    u.seg_cols = g.rows;
                    u.t_row0_f32 = (int32_t)(g.f32_row0 + (int64_t)t0 * TILE_N);
                    u.pad1 = 0;
                    units.push_back(u);
                }
            }
        }
    }
    // largest first, groups kept together
    std::vector<int> order(units.size() / group);
    for (size_t i = 0; i < order.size(); i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return units[(size_t)a * group].n_tiles > units[(size_t)b * group].n_tiles; });
    std::vector<MatchUnit> sorted; sorted.reserve(units.size());
    for (int gi : order) for (int k = 0; k < group; k++) sorted.push_back(units[(size_t)gi * group + k]);
    units.swap(sorted);
}

// Match paths.  Host-side hints / cvg_last_match_path: 1 = tensor cores, exact (integer descriptors), 2 = exact fp32
// SIMT kernel, 3 = tensor cores, candidates + fp32 re-rank (non-integer descriptors), 0 = decided on the device.
// The device word d_flags[2] holds 0 / 1 / 2 for tensor-exact / tensor-candidates / SIMT.
static int path_from_kinds(unsigned ctx_flags, int q_kinds, int t_kinds)
{
    if (ctx_flags & CVG_FORCE_EXACT_MATCH) return 2;
    if (t_kinds < 0 || q_kinds < 0) return 0;
    const int k = q_kinds | t_kinds;
    return (k & 2) ? 2 : ((k & 1) ? 3 : 1);
}
static int path_from_device_word(int w) { return w == 0 ? 1 : (w == 1 ? 3 : 2); }

// Launch the match kernels for a plan already on the device.  With path_hint 0 all three variants are enqueued and
// gate themselves on d_flags[2]; no host round trip.
static int launch_match(cvg_ctx* c, const QuerySide& q, const TrainSet& ts, const MatchUnit* d_units, int n_units,
                        const MergeEntry* d_dir, int n_rb, float ratio, int path_hint, Top2* d_parts,
                        int32_t* d_idx, float* d_dist, uint8_t* d_accept, bool guard = true)
{
    const int nq = q.row_end - q.row_begin;
    const int* gate = path_hint == 0 ? c->d_flags + 2 : nullptr;
    const bool want_int = path_hint == 0 || path_hint == 1, want_cand = path_hint == 0 || path_hint == 3;
    const bool want_simt = path_hint == 0 || path_hint == 2;
    // guard: rows of the integer path whose second distance reaches 2048 are redone exactly (merge_kernel); the caller
    // switches it off when the norms of both sides prove that no distance can get there (SIFT: d <= 1024)
    guard = guard && want_int && n_units > 0;
    if ((want_cand || guard) && n_units > 0) {
        if (want_cand) CU_CHECK(c->parts4.ensure((size_t)n_units * 4 * TILE_M * sizeof(Top4)));
        CU_CHECK(c->segdev.ensure((size_t)ts.n_segs * sizeof(SegDev) + 16));
        CU_CHECK(c->fb.ensure((size_t)ts.n_segs * std::max(nq, 1) * (sizeof(int2) + 16)));   // row list + two key arrays
        std::vector<SegDev> sd((size_t)ts.n_segs);
        for (int s = 0; s < ts.n_segs; s++) sd[(size_t)s] = SegDev{ ts.segs[(size_t)s].f32_row0, ts.segs[(size_t)s].rows, 0 };
        CU_CHECK(h2d_small(c, c->segdev.p, sd.data(), sd.size() * sizeof(SegDev)));
        if (c->stage_fallback) CU_CHECK(cudaStreamSynchronize(c->stream));    // memcpy fallback: `sd` goes out of scope
    }
    TcOperands op{ q.d_b, q.d_aug, q.d_norm, q.n_pad, ts.d_b, ts.d_aug, (int)ts.rows_pad_total, q.d_blo, ts.d_blo };
    TcMapsOpaque maps_int, maps_cand;
    char err[256];
    if (n_units > 0 && want_int && tc_encode_maps(op, 2, &maps_int, err, sizeof err)) return set_err(CVG_ERR_CUDA, "%s", err);
    if (n_units > 0 && want_cand && tc_encode_maps(op, 4, &maps_cand, err, sizeof err)) return set_err(CVG_ERR_CUDA, "%s", err);
    if (c->timing) cudaEventRecord(c->ev[3], c->stream);
    if (n_units > 0) {
        if (want_int) {
            if (launch_match_tc(op, &maps_int, d_units, n_units, d_parts, 2, gate, 0, c->d_flags + 8, c->n_sms, c->stream, err, sizeof err,
                                (tc_pair_mode_enabled() || (c->flags & CVG_MATCH_PAIR_MODE)) && n_rb % 2 == 0))
                return set_err(CVG_ERR_CUDA, "%s", err);
            c->launches++;
        }
        if (want_cand) {
            if (launch_match_tc(op, &maps_cand, d_units, n_units, c->parts4.p, 4, gate, 1, c->d_flags + 8, c->n_sms, c->stream, err, sizeof err))
                return set_err(CVG_ERR_CUDA, "%s", err);
            c->launches++;
        }
        if (want_simt) {
            launch_match_exact(q.d_f32, q.row_end, ts.d_f32, d_units, n_units, d_parts, gate, 2, c->stream);
            c->launches++;
        }
    }
    if (c->timing) cudaEventRecord(c->ev[4], c->stream);
    const size_t n_rows_all = (size_t)ts.n_segs * std::max(nq, 1);
    if (want_int || want_simt || n_units == 0) {
        // without units (no train rows at all) nothing else writes the results: the merge runs ungated and emits -1
        launch_merge(d_parts, d_dir, ts.n_segs, n_rb, nq, ratio, d_idx, d_dist, d_accept, n_units == 0 ? nullptr : gate, 1,
                     c->stream, guard ? c->d_flags + 7 : nullptr, guard ? c->fb.as<int2>() : nullptr);
        c->launches++;
        if (guard) {
            // ungated: when another path served the call the merge did not run and the list is empty
            launch_fallback_exact(c->d_flags + 7, c->fb.as<int2>(), reinterpret_cast<unsigned long long*>(c->fb.as<int2>() + n_rows_all),
                                  c->segdev.as<SegDev>(), ts.n_segs, nq, ts.max_rows, ratio, q.d_f32, q.row_begin, ts.d_f32,
                                  d_idx, d_dist, d_accept, nullptr, 0, c->n_sms, c->stream);
            c->launches += 4;
        }
    }
    if (want_cand && n_units > 0) {
        launch_merge4_rerank(c->parts4.as<Top4>(), d_dir, c->segdev.as<SegDev>(), ts.n_segs, n_rb, nq, ts.max_rows, ratio, q.d_f32,
                             q.row_begin, ts.d_f32, q.d_norm, ts.d_tnmax ? ts.d_tnmax : c->d_flags + 5, d_idx, d_dist, d_accept,
                             c->d_flags + 6, c->fb.as<int2>(),
                             reinterpret_cast<unsigned long long*>(c->fb.as<int2>() + n_rows_all), gate, 1, c->n_sms, c->stream);
        c->launches += 5;
    }
    CU_CHECK(cudaGetLastError());
    return CVG_OK;
}

// d_flags[2] = match path word from the row kinds of both sides
__global__ void combine_flags_kernel(int* f, const int* train_flag, int extra_kinds_or_force, int ignore_query_flag = 0)
{
    // extra_kinds_or_force: host-known kinds of the query side (bits 0-1) or 4 = force the SIMT kernel
    const int k = *train_flag | (ignore_query_flag ? 0 : f[1]) | extra_kinds_or_force;
    f[2] = (k & 6) ? 2 : ((k & 1) ? 1 : 0);
}

// Verify stage on a device correspondence pool.
static int run_ransac(cvg_ctx* c, const float4* d_pts, const int64_t* d_starts, const int32_t* d_counts_n,
                      int n_sets, int max_n, int64_t pool_rows, const cvg_ransac_params* p, bool want_rmask)
{
    if (n_sets <= 0) return CVG_OK;
    int rc = ensure_rng(c, p->max_iters);
    if (rc) return rc;
    const int mi = std::max(p->max_iters, 1);
    CU_CHECK(c->sample_pos.ensure((size_t)n_sets * mi * 4));
    CU_CHECK(c->counts.ensure((size_t)n_sets * mi * 4));
    static const bool split_score = !(getenv("CVG_FUSED_SCORE") && atoi(getenv("CVG_FUSED_SCORE")));   // A/B: 1 = score inside the solve kernel
    if (split_score) CU_CHECK(c->hypH.ensure((size_t)n_sets * mi * 32));
    CU_CHECK(c->n_samples.ensure((size_t)n_sets * 4));
    CU_CHECK(c->best_iter.ensure((size_t)n_sets * 4));
    CU_CHECK(c->best_count.ensure((size_t)n_sets * 4));
    CU_CHECK(c->iters_run.ensure((size_t)n_sets * 4));
    CU_CHECK(c->niters_cur.ensure((size_t)n_sets * 4));
    CU_CHECK(c->smp_state.ensure((size_t)n_sets * 16));
    CU_CHECK(c->sflags.ensure((size_t)n_sets * 4));
    CU_CHECK(c->found.ensure((size_t)n_sets * 4));
    CU_CHECK(c->H.ensure((size_t)n_sets * 9 * 8));
    CU_CHECK(c->sel.ensure((size_t)std::max<int64_t>(pool_rows, 1) * 4));
    CU_CHECK(c->mask.ensure((size_t)std::max<int64_t>(pool_rows, 1)));
    if (want_rmask) CU_CHECK(c->rmask.ensure((size_t)std::max<int64_t>(pool_rows, 1)));
    RansacWork w;
    w.pts = d_pts; w.starts = d_starts; w.counts_n = d_counts_n; w.n_sets = n_sets; w.max_n = max_n;
    w.n_sms = c->n_sms; w.wave_div = std::max(1, c->wave_div);
    w.max_iters = mi;
    const double thr = p->threshold > 0 ? p->threshold : 3.0;        // defaultRANSACReprojThreshold
    w.thr2 = (float)(thr * thr);
    w.conf = p->confidence; w.flags = p->flags;
    w.rng_tab = c->d_rng; w.rng_len = c->rng_len;
    w.sample_pos = c->sample_pos.as<int32_t>(); w.n_samples = c->n_samples.as<int32_t>();
    w.hyp_H = split_score ? c->hypH.as<float>() : nullptr; w.hyp_H_complete = 0;
    w.counts = c->counts.as<int32_t>(); w.best_iter = c->best_iter.as<int32_t>();
    w.best_count = c->best_count.as<int32_t>(); w.iters_run = c->iters_run.as<int32_t>();
    w.niters_cur = c->niters_cur.as<int32_t>();
    w.smp_state = c->smp_state.as<int64_t>();
    w.sel = c->sel.as<int32_t>(); w.H = c->H.as<double>(); w.mask = c->mask.as<uint8_t>();
    w.ransac_mask = want_rmask ? c->rmask.as<uint8_t>() : nullptr;
    w.found = c->found.as<int32_t>(); w.status_flags = c->sflags.as<int32_t>();
    w.chunk_outs = nullptr; w.chunk_lists = nullptr; w.chunk_offsets = nullptr; w.chunk_serial = nullptr; w.n_chunks = 0;
    w.chunk_maps = nullptr; w.chunk_entries = nullptr; w.chunk_serial_count = nullptr;
    c->last_chunked = false;
    if ((p->flags & CVG_RANSAC_NO_EARLY_STOP) && mi >= 32768 && n_sets <= 65535) {     // sets ride on gridDim.y of the chunk kernels
        // one huge round: the draw stream of every set is walked by many CTAs at once (ransac_sample_chunk_kernel)
        const int n_chunks = ransac_chunks_for_table(c->rng_len);
        size_t o_outs, o_lists, o_off, o_ser, o_maps, o_ent;
        const int64_t bytes = ransac_chunk_scratch_bytes(n_sets, n_chunks, &o_outs, &o_lists, &o_off, &o_ser, &o_maps, &o_ent);
        if (n_chunks > 1 && bytes < (8LL << 30)) {
            CU_CHECK(c->chunk.ensure((size_t)bytes));
            uint8_t* b = c->chunk.as<uint8_t>();
            w.chunk_outs = b + o_outs; w.chunk_lists = reinterpret_cast<int32_t*>(b + o_lists);
            w.chunk_offsets = reinterpret_cast<int32_t*>(b + o_off); w.chunk_serial = reinterpret_cast<int*>(b + o_ser);
            w.chunk_maps = b + o_maps; w.chunk_entries = reinterpret_cast<int32_t*>(b + o_ent);
            w.n_chunks = n_chunks; w.chunk_serial_count = c->d_flags + 17;
            CU_CHECK(cudaMemsetAsync(c->d_flags + 17, 0, 4, c->stream));
            c->last_chunked = true;
        }
    }
    w.err_flag = c->d_flags + 4;
    CU_CHECK(cudaMemsetAsync(c->d_flags + 4, 0, 4, c->stream));
    // RANSACUpdateNumIters: the host's log(1 - confidence), the table of host-verified entries and the request list
    {
        double pc = p->confidence; pc = pc > 0. ? pc : 0.; pc = pc < 1. ? pc : 1.;
        const double one_minus = 1. - pc > DBL_MIN ? 1. - pc : DBL_MIN;
        w.log_num = log(one_minus);
        w.nit_margin = (c->flags & CVG_NITERS_ALL_ON_HOST) ? 1e300 : 1e-10;
        CU_CHECK(c->nitreq.ensure((size_t)NIT_REQ_CAP * sizeof(int2)));
        w.nit_req = c->nitreq.as<int2>(); w.nit_req_n = c->d_flags + 19; w.nit_req_cap = NIT_REQ_CAP;
        w.nit_tab = c->nit_host.empty() ? nullptr : c->nit.as<NitEntry>(); w.nit_n = (int)c->nit_host.size();
        CU_CHECK(cudaMemsetAsync(c->d_flags + 19, 0, 4, c->stream));
    }
    w.scored_pts = c->timing ? c->d_scored : nullptr;
    if (c->timing) CU_CHECK(cudaMemsetAsync(c->d_scored, 0, 8, c->stream));
    c->launches += launch_ransac(w, c->stream, c->timing ? c->hyp_ev : nullptr, &c->hyp_rounds);
    CU_CHECK(cudaGetLastError());
    return CVG_OK;
}

// The device asked about (n, good) pairs (err_flag bit 1): evaluate them with this host's libm — the functions OpenCV itself
// calls — and put them in the engine's table; the caller then repeats the verify stage.  Stream is idle (caller synchronised).
static int answer_nit_requests(cvg_ctx* c)
{
    int n_req = 0;
    CU_CHECK(cudaMemcpy(&n_req, c->d_flags + 19, 4, cudaMemcpyDeviceToHost));
    n_req = std::min(n_req, NIT_REQ_CAP);
    std::vector<int2> req((size_t)std::max(n_req, 0));
    if (n_req > 0) CU_CHECK(cudaMemcpy(req.data(), c->nitreq.p, (size_t)n_req * sizeof(int2), cudaMemcpyDeviceToHost));
    size_t added = 0;
    for (const int2& r : req) {
        bool have = false;
        for (const NitEntry& e : c->nit_host) if (e.n == r.x && e.good == r.y) { have = true; break; }
        if (have || r.x <= 0) continue;
        double ep = (double)(r.x - r.y) / r.x;                       // ptsetreg.cpp: (double)(count - goodCount) / count
        ep = ep > 0. ? ep : 0.; ep = ep < 1. ? ep : 1.;
        const double d0 = 1. - pow(1. - ep, 4);                      // modelPoints = 4
        NitEntry e; e.n = r.x; e.good = r.y; e.zero = d0 < DBL_MIN ? 1 : 0; e.denom_log = e.zero ? -1. : log(d0); e.pad = 0;
        c->nit_host.push_back(e); added++;
    }
    if (!added) return set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters: the device keeps asking about entries it already has");
    if (c->nit_host.size() > (1u << 20)) return set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters: verification table overflow");
    CU_CHECK(c->nit.ensure(c->nit_host.size() * sizeof(NitEntry)));
    CU_CHECK(cudaMemcpy(c->nit.p, c->nit_host.data(), c->nit_host.size() * sizeof(NitEntry), cudaMemcpyHostToDevice));
    return CVG_OK;
}

int check_params(const cvg_ransac_params* p)
{
    if (!p || p->size != sizeof(cvg_ransac_params)) return set_err(CVG_ERR_INVALID, "cvg_ransac_params: bad size field");
    if (!(p->confidence > 0 && p->confidence < 1)) return set_err(CVG_ERR_INVALID, "confidence must be in (0,1)");
    if (p->max_iters < 1 || p->max_iters > (1 << 24)) return set_err(CVG_ERR_LIMIT, "max_iters out of range [1, 2^24]");
    return CVG_OK;
}

static int sync_and_check(cvg_ctx* c)
{
    // The worker thread of a lane that serves a pipelined job sleeps on a blocking-sync event instead of spinning in
    // cudaStreamSynchronize: a context keeps up to 8 jobs in flight, and on a box with 8 GPUs their spinning threads would
    // outnumber the cores.  Sub-batches of a synchronous call and the caller's own thread keep the low-latency spin
    // (measured: sleeping workers cost a synchronous call 10 %).
    cudaError_t e;
    if (c->blocking_sync && c->sync_ev) {
        e = cudaEventRecord(c->sync_ev, c->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(c->sync_ev);
    } else e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        // A device-side trap (bounded mbarrier wait that ran out, see match_tc.cu) leaves the CUDA context of the whole
        // process in a sticky error state: every later call of every context on this device fails with the same code until
        // cvg_device_reset.  The kernels leave a code in d_flags[8..] before trapping, but device memory is unreadable now.
        return set_err(CVG_ERR_CUDA, "device execution failed: %s — the CUDA context of this process is unusable; destroy the "
                       "cvgraft contexts of device %d, call cvg_device_reset(%d) and create them again", cudaGetErrorString(e),
                       c->device, c->device);
    }
    return CVG_OK;
}

// ---- models ---------------------------------------------------------------------------------------
__global__ void max_norm_kernel(const float* __restrict__ norms, int n, int* __restrict__ out_bits)
{
    float m = 0.f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float v = norms[i];
        if (v > m) m = v;                                   // NaN never wins; +inf does (then nothing is "known safe")
    }
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out_bits, __float_as_int(m));   // non-negative floats order like ints
}

static std::atomic<uint64_t> g_models_uid{ 1 };

int eng_models_upload(cvg_ctx* c, const float* desc, const float* kpt_xy, const int32_t* view_offsets,
                      const int32_t* view_model, int n_views, cvg_models** out)
{
    if (!c || !out || !view_offsets || n_views < 0) return set_err(CVG_ERR_INVALID, "cvg_models_upload: bad argument");
    *out = nullptr;
    CU_CHECK(cudaSetDevice(c->device));
    const int n = view_offsets[n_views];
    if (n < 0 || (n > 0 && !desc)) return set_err(CVG_ERR_INVALID, "cvg_models_upload: bad row count / NULL desc");
    for (int v = 0; v < n_views; v++)
        if (view_offsets[v + 1] < view_offsets[v]) return set_err(CVG_ERR_INVALID, "view_offsets must be non-decreasing");
    cvg_models* m = new cvg_models();
    m->n_rows = n; m->n_views = n_views; m->device = c->device; m->uid = g_models_uid.fetch_add(1);
    m->n_pad = round_up(std::max(n, 1), TILE_M) + TILE_M;          // slack: a view's last tile may overrun
    m->view_offsets.assign(view_offsets, view_offsets + n_views + 1);
    if (view_model) m->view_model.assign(view_model, view_model + n_views);
    int flag[2] = { 0, 0 };
    const int rc = [&]() -> int {
        CU_CHECK(cudaMalloc(&m->d_f32, (size_t)m->n_pad * DIM * 4));
        CU_CHECK(cudaMalloc(&m->d_b, (size_t)m->n_pad * DIM * 2));
        CU_CHECK(cudaMalloc(&m->d_blo, (size_t)m->n_pad * DIM * 2));
        CU_CHECK(cudaMalloc(&m->d_aug, (size_t)m->n_pad * KAUG * 2));
        CU_CHECK(cudaMalloc(&m->d_norm, (size_t)m->n_pad * 4));
        CU_CHECK(cudaMalloc(&m->d_kpt, (size_t)std::max(n, 1) * 8));
        CU_CHECK(cudaMalloc(&m->d_view_offsets, (size_t)(n_views + 1) * 4));
        CU_CHECK(cudaMemsetAsync(m->d_f32, 0, (size_t)m->n_pad * DIM * 4, c->stream));
        if (n > 0) CU_CHECK(cudaMemcpyAsync(m->d_f32, desc, (size_t)n * DIM * 4, cudaMemcpyHostToDevice, c->stream));
        if (n > 0 && kpt_xy) CU_CHECK(cudaMemcpyAsync(m->d_kpt, kpt_xy, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        CU_CHECK(cudaMemcpyAsync(m->d_view_offsets, view_offsets, (size_t)(n_views + 1) * 4, cudaMemcpyHostToDevice, c->stream));
        CU_CHECK(cudaMemsetAsync(c->d_flags + 1, 0, 4, c->stream));
        CU_CHECK(cudaMemsetAsync(c->d_flags + 18, 0, 4, c->stream));
        launch_prep_rows(m->d_f32, n, m->n_pad, 0, m->d_b, m->d_blo, m->d_aug, m->d_norm, c->d_flags + 1, nullptr, c->stream);
        if (n > 0) max_norm_kernel<<<std::min(64, (n + 255) / 256), 256, 0, c->stream>>>(m->d_norm, n, c->d_flags + 18);
        c->launches += 2;
        CU_CHECK(cudaMemcpyAsync(&flag[0], c->d_flags + 1, 4, cudaMemcpyDeviceToHost, c->stream));
        CU_CHECK(cudaMemcpyAsync(&flag[1], c->d_flags + 18, 4, cudaMemcpyDeviceToHost, c->stream));
        CU_CHECK(cudaStreamSynchronize(c->stream));
        return CVG_OK;
    }();
    if (rc) { eng_models_free(c, m); return rc; }
    m->nonint = flag[0];
    memcpy(&m->max_norm2, &flag[1], 4);
    *out = m;
    return CVG_OK;
}

void eng_models_free(cvg_ctx* c, cvg_models* m)
{
    if (!m) return;
    if (c) cudaSetDevice(c->device); else if (m->device >= 0) cudaSetDevice(m->device);
    cudaFree(m->d_f32); cudaFree(m->d_b); cudaFree(m->d_blo); cudaFree(m->d_aug); cudaFree(m->d_norm); cudaFree(m->d_kpt);
    cudaFree(m->d_view_offsets);
    delete m;
}

extern "C" {

int cvg_models_num_views(const cvg_models* m) { return m ? m->n_views : 0; }
int cvg_models_num_rows(const cvg_models* m) { return m ? m->n_rows : 0; }

}  // extern "C"

// match `q` against a host train matrix; results to host
static int match_host_train(cvg_ctx* c, QuerySide q, int q_nonint, const float* train, int n_train, float ratio,
                            int32_t* idx, float* dist, uint8_t* accept)
{
    const int nq = q.row_end - q.row_begin;
    if (nq <= 0) return CVG_OK;
    if (n_train < 0 || (n_train > 0 && !train)) return set_err(CVG_ERR_INVALID, "bad train matrix");
    if (!idx || !dist) return set_err(CVG_ERR_INVALID, "idx/dist must not be NULL");
    TrainSet ts;
    const int64_t offs[2] = { 0, n_train };
    layout_segments(ts, offs, 1);
    CU_CHECK(c->t_f32.ensure((size_t)std::max(n_train, 1) * DIM * 4));
    ts.d_f32 = c->t_f32.as<float>();
    if (n_train > 0) CU_CHECK(cudaMemcpyAsync(ts.d_f32, train, (size_t)n_train * DIM * 4, cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaMemsetAsync(c->d_flags, 0, 4, c->stream));
    int rc = prep_train(c, ts, c->t_b, c->t_blo, c->t_aug, c->t_segtab, 0);
    if (rc) return rc;
    CU_CHECK(cudaMemcpyAsync(c->d_flags + 1, &q_nonint, 4, cudaMemcpyHostToDevice, c->stream));
    combine_flags_kernel<<<1, 1, 0, c->stream>>>(c->d_flags, c->d_flags, (c->flags & CVG_FORCE_EXACT_MATCH) ? 4 : 0);
    c->launches++;
    std::vector<MatchUnit> units; std::vector<MergeEntry> dir; int n_rb;
    build_plan(q, ts, c->n_sms, units, dir, n_rb);
    CU_CHECK(c->units.ensure(std::max<size_t>(units.size(), 1) * sizeof(MatchUnit)));
    CU_CHECK(c->dir.ensure(std::max<size_t>(dir.size(), 1) * sizeof(MergeEntry)));
    CU_CHECK(c->parts.ensure(std::max<size_t>(units.size(), 1) * TILE_M * sizeof(Top2)));
    CU_CHECK(c->idx.ensure((size_t)nq * 8)); CU_CHECK(c->dist.ensure((size_t)nq * 8)); CU_CHECK(c->accept.ensure((size_t)nq));
    if (!units.empty())
        CU_CHECK(cudaMemcpyAsync(c->units.p, units.data(), units.size() * sizeof(MatchUnit), cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaMemcpyAsync(c->dir.p, dir.data(), dir.size() * sizeof(MergeEntry), cudaMemcpyHostToDevice, c->stream));
    rc = launch_match(c, q, ts, c->units.as<MatchUnit>(), (int)units.size(), c->dir.as<MergeEntry>(), n_rb, ratio, 0,
                      c->parts.as<Top2>(), c->idx.as<int32_t>(), c->dist.as<float>(), c->accept.as<uint8_t>());
    if (rc) return rc;
    int flag = 0;
    CU_CHECK(cudaMemcpyAsync(idx, c->idx.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, c->stream));
    CU_CHECK(cudaMemcpyAsync(dist, c->dist.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, c->stream));
    if (accept) CU_CHECK(cudaMemcpyAsync(accept, c->accept.p, (size_t)nq, cudaMemcpyDeviceToHost, c->stream));
    CU_CHECK(cudaMemcpyAsync(&flag, c->d_flags + 2, 4, cudaMemcpyDeviceToHost, c->stream));
    rc = sync_and_check(c);
    if (rc) return rc;
    c->last_match_path = path_from_device_word(flag);
    if (c->timing) { cudaEventElapsedTime(&c->t_match, c->ev[3], c->ev[4]); c->t_ransac = 0; c->t_total = c->t_match; }
    return CVG_OK;
}

extern "C" {

int cvg_match_knn2(cvg_ctx* c, const cvg_models* m, int view, const float* train, int n_train, float ratio,
                   int32_t* idx, float* dist, uint8_t* accept)
{
    c = cvg_primary(c); m = cvg_models_on(m, c);
    if (!c || !m) return set_err(CVG_ERR_INVALID, "cvg_match_knn2: NULL context/models");
    if (view < -1 || view >= m->n_views) return set_err(CVG_ERR_INVALID, "cvg_match_knn2: view %d of %d", view, m->n_views);
    CU_CHECK(cudaSetDevice(c->device));
    QuerySide q{ m->d_f32, m->d_b, m->d_blo, m->d_aug, m->d_norm, 0, m->n_rows, m->n_pad };
    if (view >= 0) { q.row_begin = m->view_offsets[view]; q.row_end = m->view_offsets[view + 1]; }
    return match_host_train(c, q, m->nonint, train, n_train, ratio, idx, dist, accept);
}

int cvg_match_knn2_raw(cvg_ctx* c, const float* query, int n_query, const float* train, int n_train, float ratio,
                       int32_t* idx, float* dist, uint8_t* accept)
{
    c = cvg_primary(c);
    if (!c) return set_err(CVG_ERR_INVALID, "cvg_match_knn2_raw: NULL context");
    if (n_query < 0 || (n_query > 0 && !query)) return set_err(CVG_ERR_INVALID, "bad query matrix");
    if (n_query == 0) return CVG_OK;
    CU_CHECK(cudaSetDevice(c->device));
    const int n_pad = round_up(n_query, TILE_M);
    CU_CHECK(c->q_f32.ensure((size_t)n_pad * DIM * 4)); CU_CHECK(c->q_b.ensure((size_t)n_pad * DIM * 2));
    CU_CHECK(c->q_blo.ensure((size_t)n_pad * DIM * 2));
    CU_CHECK(c->q_aug.ensure((size_t)n_pad * KAUG * 2)); CU_CHECK(c->q_norm.ensure((size_t)n_pad * 4));
    CU_CHECK(cudaMemcpyAsync(c->q_f32.p, query, (size_t)n_query * DIM * 4, cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaMemsetAsync(c->d_flags + 3, 0, 4, c->stream));
    launch_prep_rows(c->q_f32.as<float>(), n_query, n_pad, 0, c->q_b.as<__nv_bfloat16>(), c->q_blo.as<__nv_bfloat16>(),
                     c->q_aug.as<__nv_bfloat16>(), c->q_norm.as<float>(), c->d_flags + 3, nullptr, c->stream);
    c->launches++;
    int qflag = 0;
    CU_CHECK(cudaMemcpyAsync(&qflag, c->d_flags + 3, 4, cudaMemcpyDeviceToHost, c->stream));
    CU_CHECK(cudaStreamSynchronize(c->stream));
    QuerySide q{ c->q_f32.as<float>(), c->q_b.as<__nv_bfloat16>(), c->q_blo.as<__nv_bfloat16>(), c->q_aug.as<__nv_bfloat16>(),
                 c->q_norm.as<float>(), 0, n_query, n_pad };
    return match_host_train(c, q, qflag, train, n_train, ratio, idx, dist, accept);
}

// ---- verify stage ---------------------------------------------------------------------------------
int cvg_find_homography_batch(cvg_ctx* c, const float* src_xy, const float* dst_xy, const int64_t* offsets,
                              int n_sets, const cvg_ransac_params* p, double* H, uint8_t* mask, int32_t* found,
                              int32_t* iters, uint8_t* ransac_mask)
{
    c = cvg_primary(c);
    if (!c || !offsets || n_sets < 0) return set_err(CVG_ERR_INVALID, "cvg_find_homography_batch: bad argument");
    int rc = check_params(p);
    if (rc) return rc;
    if (n_sets == 0) return CVG_OK;
    CU_CHECK(cudaSetDevice(c->device));
    const int64_t total = offsets[n_sets];
    if (total < 0 || (total > 0 && (!src_xy || !dst_xy))) return set_err(CVG_ERR_INVALID, "bad point arrays");
    std::vector<int64_t> starts(n_sets); std::vector<int32_t> cnts(n_sets);
    int max_n = 0;
    for (int k = 0; k < n_sets; k++) {
        const int64_t n = offsets[k + 1] - offsets[k];
        if (n < 0 || n > 0x7fffffff) return set_err(CVG_ERR_INVALID, "offsets must be non-decreasing");
        starts[k] = offsets[k]; cnts[k] = (int32_t)n; max_n = std::max(max_n, (int)n);
    }
    const size_t tot = (size_t)std::max<int64_t>(total, 1);
    CU_CHECK(c->src.ensure(tot * 8)); CU_CHECK(c->dst.ensure(tot * 8)); CU_CHECK(c->pts.ensure(tot * 16));
    CU_CHECK(c->starts.ensure((size_t)n_sets * 8)); CU_CHECK(c->counts_n.ensure((size_t)n_sets * 4));
    if (total > 0) {
        CU_CHECK(cudaMemcpyAsync(c->src.p, src_xy, (size_t)total * 8, cudaMemcpyHostToDevice, c->stream));
        CU_CHECK(cudaMemcpyAsync(c->dst.p, dst_xy, (size_t)total * 8, cudaMemcpyHostToDevice, c->stream));
    }
    CU_CHECK(cudaMemcpyAsync(c->starts.p, starts.data(), (size_t)n_sets * 8, cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaMemcpyAsync(c->counts_n.p, cnts.data(), (size_t)n_sets * 4, cudaMemcpyHostToDevice, c->stream));
    launch_pack_points(c->src.as<float>(), c->dst.as<float>(), total, c->pts.as<float4>(), c->stream);
    c->launches++;
    std::vector<int32_t> sflags(n_sets);
    for (int attempt = 0;; attempt++) {
        if (c->timing) cudaEventRecord(c->ev[0], c->stream);
        rc = run_ransac(c, c->pts.as<float4>(), c->starts.as<int64_t>(), c->counts_n.as<int32_t>(), n_sets, max_n, total, p,
                        ransac_mask != nullptr);
        if (rc) return rc;
        if (c->timing) cudaEventRecord(c->ev[1], c->stream);
        if (H) CU_CHECK(cudaMemcpyAsync(H, c->H.p, (size_t)n_sets * 72, cudaMemcpyDeviceToHost, c->stream));
        if (mask && total > 0) CU_CHECK(cudaMemcpyAsync(mask, c->mask.p, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
        if (ransac_mask && total > 0) CU_CHECK(cudaMemcpyAsync(ransac_mask, c->rmask.p, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
        if (found) CU_CHECK(cudaMemcpyAsync(found, c->found.p, (size_t)n_sets * 4, cudaMemcpyDeviceToHost, c->stream));
        if (iters) CU_CHECK(cudaMemcpyAsync(iters, c->iters_run.p, (size_t)n_sets * 4, cudaMemcpyDeviceToHost, c->stream));
        CU_CHECK(cudaMemcpyAsync(sflags.data(), c->sflags.p, (size_t)n_sets * 4, cudaMemcpyDeviceToHost, c->stream));
        rc = sync_and_check(c);
        if (rc) return rc;
        int bad = -1;
        for (int k = 0; k < n_sets && bad < 0; k++) if (sflags[k] & 1) bad = k;
        int words = 0;
        CU_CHECK(cudaMemcpy(&words, c->d_flags + 4, 4, cudaMemcpyDeviceToHost));
        if (bad < 0 && (words & 2)) {                               // niters entries to verify on the host, then again
            if (attempt >= 12) return set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters verification did not converge");
            rc = answer_nit_requests(c);
            if (rc) return rc;
            continue;
        }
        if (bad < 0) break;
        if (c->rng_len >= RNG_TABLE_CAP || attempt >= 4)
            return set_err(CVG_ERR_LIMIT, "set %d: RNG draw table exhausted (pathological rejection rate)", bad);
        rc = ensure_rng(c, p->max_iters, c->rng_len * 4);       // more draws, then the whole verify stage again
        if (rc) return rc;
    }
    if (c->timing) { cudaEventElapsedTime(&c->t_ransac, c->ev[0], c->ev[1]); c->t_match = 0; c->t_total = c->t_ransac; }
    return CVG_OK;
}

int cvg_find_homography(cvg_ctx* c, const float* src_xy, const float* dst_xy, int n, const cvg_ransac_params* p,
                        double H[9], uint8_t* mask, int* found, uint8_t* ransac_mask)
{
    if (n < 4) return set_err(CVG_ERR_TOO_FEW_POINTS, "findHomography needs at least 4 correspondences (got %d)", n);
    const int64_t offs[2] = { 0, n };
    int32_t f = 0;
    int rc = cvg_find_homography_batch(c, src_xy, dst_xy, offs, 1, p, H, mask, &f, nullptr, ransac_mask);
    if (found) *found = f;
    return rc;
}

}  // extern "C"

// ---- fused detect over a prepared train set --------------------------------------------------------
// host_needs_inliers: the inlier pool (pair (s, v) at s * n_rows + view_offsets[v]) and the per-pair counts are left in the
// engine's page-locked c->inl_h / c->cnt_h
static int detect_common(cvg_ctx* c, const cvg_models* m, cvg_scenes* cache, TrainSet& ts, const float* d_scales,
                         const cvg_detect_params* p, cvg_pair_result* per_pair, bool host_needs_inliers, bool guard = true)
{
    const int S = ts.n_segs, V = m->n_views, nq = m->n_rows;
    const int P = S * V;
    if (P == 0) return CVG_OK;
    QuerySide q{ m->d_f32, m->d_b, m->d_blo, m->d_aug, m->d_norm, 0, nq, m->n_pad };
    int n_units = 0, n_rb = 0;
    const MatchUnit* d_units; const MergeEntry* d_dir;
    // The match plan depends only on the model set and on the row counts of the scenes: a streaming caller whose
    // batches have the same shape (same number of descriptors per scene) reuses the plan already on the device.
    std::vector<int> shape((size_t)S);
    for (int i = 0; i < S; i++) shape[(size_t)i] = ts.segs[(size_t)i].rows;
    if (c->plan_models_uid == m->uid && c->plan_shape == shape && c->plan_units_n > 0) {
        n_units = c->plan_units_n; n_rb = (nq + TILE_M - 1) / TILE_M;
        d_units = c->plan_units.as<MatchUnit>(); d_dir = c->plan_dir.as<MergeEntry>();
    } else {
        std::vector<MatchUnit> units; std::vector<MergeEntry> dir;
        build_plan(q, ts, c->n_sms, units, dir, n_rb);
        CU_CHECK(c->plan_units.ensure(std::max<size_t>(units.size(), 1) * sizeof(MatchUnit) + 16));
        CU_CHECK(c->plan_dir.ensure(std::max<size_t>(dir.size(), 1) * sizeof(MergeEntry) + 16));
        if (!units.empty()) CU_CHECK(h2d_small(c, c->plan_units.p, units.data(), units.size() * sizeof(MatchUnit)));
        if (!dir.empty()) CU_CHECK(h2d_small(c, c->plan_dir.p, dir.data(), dir.size() * sizeof(MergeEntry)));
        if (c->stage_fallback) CU_CHECK(cudaStreamSynchronize(c->stream));    // memcpy fallback: host vectors go out of scope
        n_units = (int)units.size();
        d_units = c->plan_units.as<MatchUnit>(); d_dir = c->plan_dir.as<MergeEntry>();
        c->plan_models_uid = m->uid; c->plan_shape = shape; c->plan_units_n = n_units;
    }
    const size_t rows = (size_t)S * std::max(nq, 1);
    CU_CHECK(c->parts.ensure(std::max<size_t>(n_units, 1) * TILE_M * sizeof(Top2)));
    CU_CHECK(c->idx.ensure(rows * 8)); CU_CHECK(c->dist.ensure(rows * 8)); CU_CHECK(c->accept.ensure(rows));
    CU_CHECK(c->pts.ensure(rows * 16)); CU_CHECK(c->starts.ensure((size_t)P * 8)); CU_CHECK(c->counts_n.ensure((size_t)P * 4));
    CU_CHECK(c->results.ensure((size_t)P * sizeof(cvg_pair_result)));
    CU_CHECK(c->inl_cnt.ensure((size_t)P * 4));
    if (host_needs_inliers) {
        CU_CHECK(c->inl_xy.ensure(rows * 8));
        CU_CHECK(c->inl_h.ensure(rows * 8)); CU_CHECK(c->cnt_h.ensure((size_t)P * 4));
    }

    if (c->timing) cudaEventRecord(c->ev[0], c->stream);
    static std::atomic<int> det_id{ 0 };
    const int did = det_id.fetch_add(1);
    cvg_trace_mark(c->stream, "det_begin", did);
    const int path = path_from_kinds(c->flags, m->nonint, ts.nonint);
    if (path == 0) {
        combine_flags_kernel<<<1, 1, 0, c->stream>>>(c->d_flags, (cache && cache->d_flag) ? cache->d_flag : c->d_flags, m->nonint, 1);
        c->launches++;
    }
    int rc = launch_match(c, q, ts, d_units, n_units, d_dir, n_rb, p->ratio, path, c->parts.as<Top2>(),
                          c->idx.as<int32_t>(), c->dist.as<float>(), c->accept.as<uint8_t>(), guard);
    if (rc) return rc;
    CompactWork cw;
    cw.n_segments = S; cw.n_views = V; cw.n_query = nq; cw.view_offsets = m->d_view_offsets;
    cw.model_kpt = m->d_kpt; cw.scene_kpt = ts.d_kpt; cw.seg_kpt_offsets = ts.d_kpt_offsets;
    cw.idx = c->idx.as<int32_t>(); cw.accept = c->accept.as<uint8_t>();
    cw.pts = c->pts.as<float4>(); cw.starts = c->starts.as<int64_t>(); cw.n_good = c->counts_n.as<int32_t>();
    launch_compact(cw, c->stream);
    c->launches++;
    cvg_trace_mark(c->stream, "match_end", did);
    if (c->timing) cudaEventRecord(c->ev[1], c->stream);
    int max_view = 0;
    for (int v = 0; v < V; v++) max_view = std::max(max_view, m->view_offsets[v + 1] - m->view_offsets[v]);
    int flag = 0;
    for (int attempt = 0;; attempt++) {
        rc = run_ransac(c, c->pts.as<float4>(), c->starts.as<int64_t>(), c->counts_n.as<int32_t>(), P, max_view,
                        (int64_t)rows, &p->ransac, false);
        if (rc) return rc;
        GateWork g;
        g.n_pairs = P; g.pts = c->pts.as<float4>(); g.starts = c->starts.as<int64_t>(); g.counts_n = c->counts_n.as<int32_t>();
        g.mask = c->mask.as<uint8_t>(); g.found = c->found.as<int32_t>(); g.H = c->H.as<double>();
        g.iters_run = c->iters_run.as<int32_t>(); g.pair_scale = d_scales;
        g.min_inliers = p->min_inliers; g.det_lo = p->det_lo; g.det_hi = p->det_hi;
        g.results = c->results.as<cvg_pair_result>();
        g.inlier_xy = host_needs_inliers ? c->inl_xy.as<float>() : nullptr; g.inlier_count = c->inl_cnt.as<int32_t>();
        launch_gates(g, c->stream);
        c->launches++;
        cvg_trace_mark(c->stream, "det_end", did);
        if (c->timing) cudaEventRecord(c->ev[2], c->stream);
        CU_CHECK(cudaGetLastError());
        // Results travel through the engine's page-locked staging, never straight into the caller's (pageable) arrays: a
        // device -> host copy into pageable memory is staged by the driver behind EVERYTHING already queued on the device —
        // measured: with three calls and their uploads in flight, call k's results came back only when call k + 2 was done
        // and the H2D engine idled 4.4 ms in every 15 (e2e 7.0 instead of 5.1 ms per step).
        const size_t res_bytes = (size_t)P * sizeof(cvg_pair_result);
        CU_CHECK(c->res_h.ensure(res_bytes + 16));
        int* words_h = reinterpret_cast<int*>(c->res_h.as<uint8_t>() + res_bytes);     // [0] RNG table short, [1] match path word
        words_h[0] = 0; words_h[1] = 0;
        CU_CHECK(cudaMemcpyAsync(c->res_h.p, c->results.p, res_bytes, cudaMemcpyDeviceToHost, c->stream));
        if (host_needs_inliers) {
            // the whole pool (one slot range per pair) into the engine's page-locked staging; the callers pack it
            CU_CHECK(cudaMemcpyAsync(c->cnt_h.p, c->inl_cnt.p, (size_t)P * 4, cudaMemcpyDeviceToHost, c->stream));
            CU_CHECK(cudaMemcpyAsync(c->inl_h.p, c->inl_xy.p, rows * 8, cudaMemcpyDeviceToHost, c->stream));
        }
        CU_CHECK(cudaMemcpyAsync(&words_h[0], c->d_flags + 4, 4, cudaMemcpyDeviceToHost, c->stream));
        if (path == 0) CU_CHECK(cudaMemcpyAsync(&words_h[1], c->d_flags + 2, 4, cudaMemcpyDeviceToHost, c->stream));
        rc = sync_and_check(c);
        if (rc) return rc;
        memcpy(per_pair, c->res_h.p, res_bytes);
        const int rng_short = words_h[0];
        flag = words_h[1];
        if (!(rng_short & 1) && (rng_short & 2)) {                  // niters entries to verify on the host, then again
            if (attempt >= 12) return set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters verification did not converge");
            rc = answer_nit_requests(c);
            if (rc) return rc;
            continue;
        }
        if (!(rng_short & 1)) break;
        if (c->rng_len >= RNG_TABLE_CAP || attempt >= 4)
            return set_err(CVG_ERR_LIMIT, "RNG draw table exhausted (pathological rejection rate)");
        rc = ensure_rng(c, p->ransac.max_iters, c->rng_len * 4);   // more draws, then the verify stage again
        if (rc) return rc;
    }
    c->last_match_path = path == 0 ? path_from_device_word(flag) : path;
    if (c->timing) {
        c->t_hyp = 0; c->t_score = 0;
        for (int r = 0; r < c->hyp_rounds; r++) {
            float t = 0; cudaEventElapsedTime(&t, c->hyp_ev[2 * r], c->hyp_ev[2 * r + 1]); c->t_hyp += t;
            t = 0; cudaEventElapsedTime(&t, c->hyp_ev[2 * r + 1], c->hyp_ev[32 + r]); c->t_score += t;
        }
        c->hyp_launches = c->hyp_rounds;
        cudaMemcpy(&c->scored_pts, c->d_scored, 8, cudaMemcpyDeviceToHost);
        cudaEventElapsedTime(&c->t_match, c->ev[3], c->ev[4]);      // the match kernel(s) alone
        cudaEventElapsedTime(&c->t_ransac, c->ev[1], c->ev[2]);     // sample + hypothesis + select + finish + gates
        cudaEventElapsedTime(&c->t_total, c->ev[0], c->ev[2]);
    }
    return CVG_OK;
}

int check_detect_params(const cvg_detect_params* p)
{
    if (!p || p->size != sizeof(cvg_detect_params)) return set_err(CVG_ERR_INVALID, "cvg_detect_params: bad size field");
    return check_params(&p->ransac);
}

extern "C" {

int cvg_detect_pairs(cvg_ctx* c, const cvg_models* m, const float* scene_desc, const float* scene_kpt_xy, int n_train,
                     float scale, const cvg_detect_params* p, cvg_pair_result* per_view, float* inlier_scene_xy,
                     int32_t* inlier_offsets)
{
    c = cvg_primary(c); m = cvg_models_on(m, c);
    if (!c || !m || !per_view) return set_err(CVG_ERR_INVALID, "cvg_detect_pairs: NULL argument");
    int rc = check_detect_params(p);
    if (rc) return rc;
    if (n_train < 0 || (n_train > 0 && (!scene_desc || !scene_kpt_xy))) return set_err(CVG_ERR_INVALID, "bad scene arrays");
    CU_CHECK(cudaSetDevice(c->device));
    c->stage_used = 0; c->stage_fallback = false;
    const int V = m->n_views;
    TrainSet ts;
    const int64_t offs[2] = { 0, n_train };
    layout_segments(ts, offs, 1);
    CU_CHECK(c->t_f32.ensure((size_t)std::max(n_train, 1) * DIM * 4));
    CU_CHECK(c->t_kpt.ensure((size_t)std::max(n_train, 1) * 8));
    CU_CHECK(c->t_kptoff.ensure(16));
    CU_CHECK(c->scales.ensure((size_t)std::max(V, 1) * 4));
    ts.d_f32 = c->t_f32.as<float>(); ts.d_kpt = c->t_kpt.as<float>(); ts.d_kpt_offsets = c->t_kptoff.as<int64_t>();
    if (n_train > 0) {
        CU_CHECK(cudaMemcpyAsync(ts.d_f32, scene_desc, (size_t)n_train * DIM * 4, cudaMemcpyHostToDevice, c->stream));
        CU_CHECK(cudaMemcpyAsync(ts.d_kpt, scene_kpt_xy, (size_t)n_train * 8, cudaMemcpyHostToDevice, c->stream));
    }
    CU_CHECK(cudaMemcpyAsync(ts.d_kpt_offsets, offs, 16, cudaMemcpyHostToDevice, c->stream));
    std::vector<float> scales(std::max(V, 1), scale);
    CU_CHECK(cudaMemcpyAsync(c->scales.p, scales.data(), scales.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaMemsetAsync(c->d_flags, 0, 4, c->stream));
    rc = prep_train(c, ts, c->t_b, c->t_blo, c->t_aug, c->t_segtab, 0);
    if (rc) return rc;
    ts.nonint = -1;                                    // decided on the device
    const bool want_inl = inlier_scene_xy != nullptr && inlier_offsets != nullptr;
    rc = detect_common(c, m, nullptr, ts, c->scales.as<float>(), p, per_view, want_inl);
    if (rc) return rc;
    if (want_inl) {
        const float* pool = c->inl_h.as<float>(); const int32_t* cnt = c->cnt_h.as<int32_t>();
        int32_t o = 0;
        for (int v = 0; v < V; v++) {
            inlier_offsets[v] = o;
            const size_t start = (size_t)m->view_offsets[v];
            memcpy(inlier_scene_xy + 2 * (size_t)o, pool + 2 * start, (size_t)cnt[v] * 8);
            o += cnt[v];
        }
        inlier_offsets[V] = o;
    }
    return CVG_OK;
}

// uint8 descriptor rows (cv::SIFT with descriptorType = CV_8U) -> the fp32 rows every kernel reads
__global__ void u8_to_f32_kernel(const uchar4* __restrict__ in, float4* __restrict__ out, size_t n4)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const uchar4 v = in[i];
        out[i] = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
    }
}

}  // extern "C"

// src_row0 (may be NULL): scene s is read from rows [src_row0[s], src_row0[s] + rows of s) of the caller's arrays instead
// of rows [offsets[s], offsets[s + 1]) — a multi-device context hands every device its own, non-contiguous scenes.
int eng_scenes_upload(cvg_ctx* c, const float* desc, const uint8_t* desc_u8, const float* kpt_xy,
                      const int64_t* offsets, int n_scenes, cvg_scenes** out, bool async, const int64_t* src_row0)
{
    if (!c || !out || !offsets || n_scenes < 0) return set_err(CVG_ERR_INVALID, "cvg_scenes_upload: bad argument");
    *out = nullptr;
    CU_CHECK(cudaSetDevice(c->device));
    for (int s = 0; s < n_scenes; s++)
        if (offsets[s + 1] < offsets[s]) return set_err(CVG_ERR_INVALID, "offsets must be non-decreasing");
    const int64_t total = offsets[n_scenes];
    if (total > 0 && !desc && !desc_u8) return set_err(CVG_ERR_INVALID, "NULL desc");
    cvg_scenes* sc = new cvg_scenes();
    sc->n_scenes_total = n_scenes;
    sc->offsets_copy.assign(offsets, offsets + n_scenes + 1);   // the library's own copy: the caller's array may go away at once
    layout_segments(sc->ts, offsets, n_scenes);
    if (sc->ts.rows_pad_total > 0x7fffff00LL) { delete sc; return set_err(CVG_ERR_LIMIT, "scene batch too large (>2^31 padded rows)"); }
    cudaStream_t st = c->stream;
    if (async) {
        // copy streams are made on first use: only the engine that uploads needs them, and every stream beyond the
        // device's hardware queues (CUDA_DEVICE_MAX_CONNECTIONS, 8 by default) aliases with another one — a bulk copy
        // sharing a queue with a lane's compute stream serialises the two (measured: e2e 5.1 -> 7.0 ms per step)
        cudaStream_t& cs = c->copy_stream[c->next_copy++ % 2];
        if (!cs) CU_CHECK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        st = cs;
    }
    const int rc = [&]() -> int {
        CU_CHECK(c->pool.acquire(sc->f32, (size_t)std::max<int64_t>(total, 1) * DIM * 4));
        CU_CHECK(c->pool.acquire(sc->kpt, (size_t)std::max<int64_t>(total, 1) * 8));
        CU_CHECK(c->pool.acquire(sc->kptoff, (size_t)(n_scenes + 1) * 8 + 16));
        sc->ts.d_f32 = sc->f32.as<float>(); sc->ts.d_kpt = sc->kpt.as<float>(); sc->ts.d_kpt_offsets = sc->kptoff.as<int64_t>();
        sc->d_flag = reinterpret_cast<int*>(sc->kptoff.as<int64_t>() + (n_scenes + 1));
        sc->ts.d_tnmax = sc->d_flag + 1;
        static std::atomic<int> up_id{ 0 };
        const int tid = up_id.fetch_add(1);
        cvg_trace_mark(st, "h2d_begin", tid);
        // host -> device copies: one per array, or one per scene when the scenes are gathered from all over the caller's arrays
        auto h2d_rows = [&](void* dst, const void* src, size_t row_bytes) -> int {
            if (!src_row0) { CU_CHECK(cudaMemcpyAsync(dst, src, (size_t)total * row_bytes, cudaMemcpyHostToDevice, st)); return CVG_OK; }
            for (int s2 = 0; s2 < n_scenes; s2++) {
                const size_t rows = (size_t)(offsets[s2 + 1] - offsets[s2]);
                if (rows) CU_CHECK(cudaMemcpyAsync((uint8_t*)dst + (size_t)offsets[s2] * row_bytes, (const uint8_t*)src + (size_t)src_row0[s2] * row_bytes,
                                                   rows * row_bytes, cudaMemcpyHostToDevice, st));
            }
            return CVG_OK;
        };
        if (total > 0 && desc_u8) {                                 // a quarter of the PCIe bytes; widened on the device
            CU_CHECK(c->pool.acquire(sc->u8, (size_t)total * DIM));
            int r = h2d_rows(sc->u8.p, desc_u8, DIM);
            if (r) return r;
            const size_t n4 = (size_t)total * DIM / 4;
            u8_to_f32_kernel<<<(unsigned)std::min<size_t>((n4 + 255) / 256, (size_t)c->n_sms * 16), 256, 0, st>>>(
                sc->u8.as<uchar4>(), reinterpret_cast<float4*>(sc->ts.d_f32), n4);
            c->launches++;
        } else if (total > 0) { int r = h2d_rows(sc->ts.d_f32, desc, (size_t)DIM * 4); if (r) return r; }
        if (total > 0 && kpt_xy) { int r = h2d_rows(sc->ts.d_kpt, kpt_xy, 8); if (r) return r; }
        else if (total > 0) CU_CHECK(cudaMemsetAsync(sc->ts.d_kpt, 0, (size_t)total * 8, st));
        CU_CHECK(cudaMemcpyAsync(sc->ts.d_kpt_offsets, sc->offsets_copy.data(), (size_t)(n_scenes + 1) * 8, cudaMemcpyHostToDevice, st));
        CU_CHECK(cudaMemsetAsync(sc->d_flag, 0, 8, st));
        cvg_trace_mark(st, "h2d_end", tid);
        int r = prep_train(c, sc->ts, sc->b, sc->blo, sc->aug, sc->segtab, 0, true, st, sc->d_flag);
        if (r) return r;
        cvg_trace_mark(st, "prep_end", tid);
        if (async) {
            // the caller's buffers are read by the copy engine until `ready`; cvg_detect_scenes orders itself after it
            CU_CHECK(cudaEventCreateWithFlags(&sc->ready, cudaEventDisableTiming));
            CU_CHECK(cudaEventRecord(sc->ready, st));
            sc->ts.nonint = -1;                            // the match path is decided on the device from d_flag
        } else {
            int flag[2] = { 0, 0 };                        // row kinds, max ||t||^2 bits
            CU_CHECK(cudaMemcpyAsync(flag, sc->d_flag, 8, cudaMemcpyDeviceToHost, st));
            CU_CHECK(cudaStreamSynchronize(st));
            sc->ts.nonint = flag[0];
            memcpy(&sc->max_norm2, &flag[1], 4);
        }
        return CVG_OK;
    }();
    if (rc) { eng_scenes_free(c, sc); return rc; }
    *out = sc;
    return CVG_OK;
}

int eng_scenes_wait(cvg_ctx* c, cvg_scenes* sc)
{
    if (!c || !sc) return set_err(CVG_ERR_INVALID, "cvg_scenes_wait: NULL argument");
    if (!sc->ready) return CVG_OK;
    CU_CHECK(cudaSetDevice(c->device));
    CU_CHECK(cudaEventSynchronize(sc->ready));
    if (sc->ts.nonint < 0) {
        int flag[2] = { 0, 0 };
        CU_CHECK(cudaMemcpy(flag, sc->d_flag, 8, cudaMemcpyDeviceToHost));
        sc->ts.nonint = flag[0];
        memcpy(&sc->max_norm2, &flag[1], 4);
    }
    return CVG_OK;
}

void eng_scenes_free(cvg_ctx* c, cvg_scenes* sc)
{
    if (!sc) return;
    if (c) cudaSetDevice(c->device);
    if (sc->ready) { cudaEventSynchronize(sc->ready); cudaEventDestroy(sc->ready); sc->ready = nullptr; }
    if (c) {
        DevBuf* bufs[] = { &sc->f32, &sc->b, &sc->blo, &sc->aug, &sc->kpt, &sc->kptoff, &sc->u8, &sc->segtab };
        for (DevBuf* b : bufs) c->pool.release(*b);
    } else {
        sc->f32.release(); sc->b.release(); sc->blo.release(); sc->aug.release(); sc->u8.release(); sc->segtab.release(); sc->kpt.release(); sc->kptoff.release();
    }
    delete sc;
}

// Scenes [s0, s1) of a resident batch on engine `c` (the context itself, or one of its lanes: same device, own stream
// and scratch).  The sub-batch is a VIEW of the batch's train set: same device arrays, a slice of the segment list.
int eng_detect_range(cvg_ctx* c, const cvg_models* m, cvg_scenes* sc, int s0, int s1, const float* scales,
                     const cvg_detect_params* p, cvg_pair_result* per_pair, std::vector<float>* pool, std::vector<int32_t>* cnt)
{
    if (!c || !m || !sc || !per_pair) return set_err(CVG_ERR_INVALID, "cvg_detect_scenes: NULL argument");
    if (s0 < 0 || s1 > sc->ts.n_segs || s0 > s1) return set_err(CVG_ERR_INVALID, "cvg_detect_scenes: bad scene range");
    CU_CHECK(cudaSetDevice(c->device));
    const int S = s1 - s0, V = m->n_views;
    if (S * V == 0) return CVG_OK;
    c->stage_used = 0; c->stage_fallback = false;       // the engine's previous call has completed (calls are synchronous)
    if (sc->ready) CU_CHECK(cudaStreamWaitEvent(c->stream, sc->ready, 0));
    const float* d_scales = nullptr;
    if (scales) {
        std::vector<float> ps((size_t)S * V);
        for (int s = 0; s < S; s++) for (int v = 0; v < V; v++) ps[(size_t)s * V + v] = scales[s0 + s];
        CU_CHECK(c->scales.ensure(ps.size() * 4 + 16));
        CU_CHECK(h2d_small(c, c->scales.p, ps.data(), ps.size() * 4));
        if (c->stage_fallback) CU_CHECK(cudaStreamSynchronize(c->stream));
        d_scales = c->scales.as<float>();
    }
    TrainSet view = sc->ts;                              // device pointers shared; rows_pad_total stays (TMA map bounds)
    if (S != sc->ts.n_segs) {
        view.segs.assign(sc->ts.segs.begin() + s0, sc->ts.segs.begin() + s1);
        view.n_segs = S;
        view.d_kpt_offsets = sc->ts.d_kpt_offsets + s0;
        view.max_rows = 0;
        for (const SegInfo& g : view.segs) view.max_rows = std::max(view.max_rows, g.rows);
    }
    const bool want_inl = pool != nullptr && cnt != nullptr;
    // d >= 2048 needs ||q|| + ||t|| >= 2048: with both norms known on the host the guard kernels are not even enqueued
    const bool safe = sc->max_norm2 >= 0.f && sqrt((double)m->max_norm2) + sqrt((double)sc->max_norm2) < 2047.0;
    const int rc = detect_common(c, m, sc, view, d_scales, p, per_pair, want_inl, !safe);
    if (rc || !want_inl) return rc;
    // pack the pool pair after pair (scene-major, then view), on this engine's thread
    const float* hp = c->inl_h.as<float>(); const int32_t* hc = c->cnt_h.as<int32_t>();
    cnt->assign(hc, hc + (size_t)S * V);
    size_t total = 0;
    for (size_t i = 0; i < (size_t)S * V; i++) total += (size_t)hc[i];
    pool->resize(total * 2);
    size_t o = 0;
    for (int s = 0; s < S; s++)
        for (int v = 0; v < V; v++) {
            const size_t n = (size_t)hc[(size_t)s * V + v];
            memcpy(pool->data() + 2 * o, hp + 2 * ((size_t)s * m->n_rows + (size_t)m->view_offsets[v]), n * 8);
            o += n;
        }
    return CVG_OK;
}

extern "C" {

// ---- device-pointer building blocks -----------------------------------------------------------------
int cvg_dev_match_top2(cvg_ctx* c, void* stream, const float* query_dev, int n_query, const float* train_dev,
                       int n_train, int32_t train_index_base, float* dist_dev, int32_t* idx_dev)
{
    c = cvg_primary(c);
    if (!c || n_query < 0 || n_train < 0) return set_err(CVG_ERR_INVALID, "cvg_dev_match_top2: bad argument");
    if (n_query == 0) return CVG_OK;
    CU_CHECK(cudaSetDevice(c->device));
    cudaStream_t user = (cudaStream_t)stream;
    // order our stream after the caller's and back (the context owns its scratch and its stream)
    CU_CHECK(cudaEventRecord(c->ev[5], user));
    CU_CHECK(cudaStreamWaitEvent(c->stream, c->ev[5], 0));
    const int n_pad = round_up(n_query, TILE_M);
    CU_CHECK(c->q_b.ensure((size_t)n_pad * DIM * 2)); CU_CHECK(c->q_aug.ensure((size_t)n_pad * KAUG * 2));
    CU_CHECK(c->q_blo.ensure((size_t)n_pad * DIM * 2));
    CU_CHECK(c->q_norm.ensure((size_t)n_pad * 4));
    CU_CHECK(cudaMemsetAsync(c->d_flags, 0, 16, c->stream));
    launch_prep_rows(query_dev, n_query, n_pad, 0, c->q_b.as<__nv_bfloat16>(), c->q_blo.as<__nv_bfloat16>(),
                     c->q_aug.as<__nv_bfloat16>(), c->q_norm.as<float>(), c->d_flags + 1, nullptr, c->stream);
    c->launches++;
    TrainSet ts;
    const int64_t offs[2] = { 0, n_train };
    layout_segments(ts, offs, 1);
    ts.d_f32 = const_cast<float*>(train_dev);
    int rc = prep_train(c, ts, c->t_b, c->t_blo, c->t_aug, c->t_segtab, 0);
    if (rc) return rc;
    combine_flags_kernel<<<1, 1, 0, c->stream>>>(c->d_flags, c->d_flags, (c->flags & CVG_FORCE_EXACT_MATCH) ? 4 : 0);
    c->launches++;
    QuerySide q{ query_dev, c->q_b.as<__nv_bfloat16>(), c->q_blo.as<__nv_bfloat16>(), c->q_aug.as<__nv_bfloat16>(), c->q_norm.as<float>(), 0, n_query, n_pad };
    std::vector<MatchUnit> units; std::vector<MergeEntry> dir; int n_rb;
    build_plan(q, ts, c->n_sms, units, dir, n_rb);
    CU_CHECK(c->units.ensure(std::max<size_t>(units.size(), 1) * sizeof(MatchUnit)));
    CU_CHECK(c->dir.ensure(std::max<size_t>(dir.size(), 1) * sizeof(MergeEntry)));
    CU_CHECK(c->parts.ensure(std::max<size_t>(units.size(), 1) * TILE_M * sizeof(Top2)));
    CU_CHECK(c->idx.ensure((size_t)n_query * 8)); CU_CHECK(c->dist.ensure((size_t)n_query * 8));
    if (!units.empty()) CU_CHECK(cudaMemcpyAsync(c->units.p, units.data(), units.size() * sizeof(MatchUnit), cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaMemcpyAsync(c->dir.p, dir.data(), dir.size() * sizeof(MergeEntry), cudaMemcpyHostToDevice, c->stream));
    CU_CHECK(cudaStreamSynchronize(c->stream));
    // this entry point does not synchronise: the mapped staging area (reset by the next synchronous call) must not
    // carry parameter blocks that a still-queued copy kernel has to read
    const size_t stage_saved = c->stage_used;
    c->stage_used = c->stage_cap;
    rc = launch_match(c, q, ts, c->units.as<MatchUnit>(), (int)units.size(), c->dir.as<MergeEntry>(), n_rb, 0.9f, 0,
                      c->parts.as<Top2>(), c->idx.as<int32_t>(), c->dist.as<float>(), nullptr);
    c->stage_used = stage_saved;
    if (rc) return rc;
    launch_shift_index(c->idx.as<int32_t>(), c->dist.as<float>(), n_query, train_index_base, dist_dev, idx_dev, c->stream);
    c->launches++;
    CU_CHECK(cudaEventRecord(c->ev[5], c->stream));
    CU_CHECK(cudaStreamWaitEvent(user, c->ev[5], 0));
    return CVG_OK;
}

int cvg_dev_merge_top2(cvg_ctx* c, void* stream, const float* dist_parts_dev, const int32_t* idx_parts_dev, int n_parts,
                       int n_query, float ratio, int32_t* idx_dev, float* dist_dev, uint8_t* accept_dev)
{
    c = cvg_primary(c);
    if (!c || n_parts < 1 || n_query < 0) return set_err(CVG_ERR_INVALID, "cvg_dev_merge_top2: bad argument");
    CU_CHECK(cudaSetDevice(c->device));
    launch_merge_parts(dist_parts_dev, idx_parts_dev, n_parts, n_query, ratio, idx_dev, dist_dev, accept_dev,
                       (cudaStream_t)stream);
    c->launches++;
    CU_CHECK(cudaGetLastError());
    return CVG_OK;
}

}  // extern "C"
