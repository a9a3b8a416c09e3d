// multi.cu — what sits between the C ABI and the engines of api.cu:
//   * lanes: extra engines (own stream, own scratch, own worker thread) on the context's device.  A synchronous fused
//     call splits its scene batch into sub-batches that run concurrently on the lanes, so that one sub-batch's
//     latency-bound refit/LM kernel runs under another's match / solve / score kernels; cvg_detect_scenes_submit
//     hands whole batches to the lanes, so that a single-threaded caller pipelines calls (submit k+1, wait k).
//   * multi-device contexts (cvg_create_multi): one device context per listed GPU of the host, a resident model replica
//     per device, scene batches dealt to the devices by cost (pair sharding, SURVEY 8e-1: no data-path collective), and
//     cvg_match_knn2_sharded: train-tile sharding with ONE exchange step (ncclAllGather of 16 B per query and device
//     over NVLink) followed by the lexicographic (distance, index) merge (SURVEY 8e-2).
// Reference seam: the loop nest of detectObjects (src/TestsDetector.cpp:38,58,99) under processAllTestImages
// (src/Output.cpp:23-57), which carries no state from one (view, scene) pair to the next.
#include "ctx.cuh"
#include <dlfcn.h>
#include <stdlib.h>
#include <string.h>

using namespace cvg;

// ---- NCCL, resolved at run time (a process that already loaded NCCL, e.g. through torch, shares that copy) --------
typedef struct ncclComm* ncclComm_t;
struct NcclApi {
    int (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int /*ncclDataType_t*/, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
};
static NcclApi& nccl_api()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void* h = nullptr;
        for (const char* name : { "libnccl.so.2", "libnccl.so" }) { h = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
        if (!h) return;
        api.CommInitAll = (int (*)(ncclComm_t*, int, const int*))dlsym(h, "ncclCommInitAll");
        api.CommDestroy = (int (*)(ncclComm_t))dlsym(h, "ncclCommDestroy");
        api.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllGather");
        api.GroupStart = (int (*)())dlsym(h, "ncclGroupStart");
        api.GroupEnd = (int (*)())dlsym(h, "ncclGroupEnd");
        api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
        api.ok = api.CommInitAll && api.CommDestroy && api.AllGather && api.GroupStart && api.GroupEnd;
    });
    return api;
}
constexpr int NCCL_CHAR = 0;                               // ncclInt8 / ncclChar

struct MultiState {
    std::vector<int> devices;
    std::vector<cvg_ctx*> subs;                            // one device context (engine + lanes) per listed device
    std::vector<Worker*> workers;                          // one host thread per device for blocking per-device work
    std::vector<ncclComm_t> comms;                         // empty: exchange by device-to-device copies
    std::vector<DevBuf> loc_d, loc_i, all_d, all_i, qbuf, tbuf, out_idx, out_dist, out_acc;
    std::vector<cudaEvent_t> ev;
    unsigned next_dev = 0;
    const char* exchange = "none";
    // hypothesis-range sharded RANSAC: exchange steps of the last call and their device time on the first GPU; the first
    // GPU's timing events, five per round (solve start, solve end, score end, exchange start, exchange end)
    int n_exchanges = 0; float exchange_ms = 0.f;
    std::vector<cudaEvent_t> tev;
};

struct ChunkTask { int s0 = 0, s1 = 0; Done done; std::vector<float> pool; std::vector<int32_t> cnt; int match_path = 0; };

struct cvg_job {
    // single-device part
    cvg_ctx* ctx = nullptr; const cvg_models* m = nullptr; cvg_scenes* sc = nullptr;
    std::vector<ChunkTask*> chunks;
    std::vector<float> scales; bool have_scales = false;
    cvg_detect_params params;
    cvg_pair_result* per_pair = nullptr; float* inl_xy = nullptr; int64_t* inl_off = nullptr;
    // multi-device part: one sub-job per involved device, results scattered back into the caller's order at wait
    std::vector<cvg_job*> subs; std::vector<int> sub_dev;
    std::vector<std::vector<cvg_pair_result>> sub_res; std::vector<std::vector<float>> sub_xy; std::vector<std::vector<int64_t>> sub_off;
    const cvg_scenes* shell = nullptr; const cvg_models* shell_m = nullptr;
    ~cvg_job() { for (ChunkTask* t : chunks) delete t; for (cvg_job* j : subs) delete j; }
};

cvg_ctx* cvg_primary(cvg_ctx* c) { return (c && c->multi) ? c->multi->subs[0] : c; }
const cvg_ctx* cvg_primary(const cvg_ctx* c) { return (c && c->multi) ? c->multi->subs[0] : c; }
const cvg_models* cvg_models_on(const cvg_models* m, const cvg_ctx* eng)
{
    if (!m || m->replicas.empty() || !eng) return m;
    for (const cvg_models* r : m->replicas) if (r && r->device == eng->device) return r;
    return m->replicas[0];
}

// ---- lanes ------------------------------------------------------------------------------------------------
static int default_lanes()
{
    static const int n = [] { const char* e = getenv("CVG_LANES"); const int v = e ? atoi(e) : 3; return v < 1 ? 1 : (v > 8 ? 8 : v); }();
    return n;
}
static int lanes_of(const cvg_ctx* c) { return c->lanes_cfg > 0 ? c->lanes_cfg : default_lanes(); }

static int ensure_lanes(cvg_ctx* c, int n)
{
    while ((int)c->lanes.size() < n) {
        cvg_ctx* e = nullptr;
        const int rc = eng_create(&e, c->device, c->flags);
        if (rc) return rc;
        e->parent = c;
        Lane* l = new Lane();
        l->eng = e; l->worker = new Worker();
        c->lanes.push_back(l);
    }
    return CVG_OK;
}

static void destroy_lanes(cvg_ctx* c)
{
    for (Lane* l : c->lanes) { delete l->worker; eng_destroy(l->eng); delete l; }    // the worker drains its queue first
    c->lanes.clear();
}

// Sub-batches of a synchronous call: consecutive scene ranges of about equal cost (train rows), at most one per lane,
// and none at all for small calls (a split costs a thread hop per lane and shortens every launch).
static void plan_chunks(const cvg_ctx* c, const cvg_models* m, const cvg_scenes* sc, bool split, std::vector<std::pair<int, int>>& out)
{
    const int S = sc->ts.n_segs;
    out.clear();
    // a synchronous call gains nothing beyond three sub-batches (each ends in its own refit/LM chain; measured: 8 sub-batches
    // of 8 scenes halve the rate), pipelined jobs use every lane
    static const int max_split = [] { const char* e = getenv("CVG_SPLIT_LANES"); const int v = e ? atoi(e) : 3; return v < 1 ? 1 : v; }();
    int K = split ? std::min(std::min(lanes_of(c), max_split), S) : 1;
    const int64_t min_cost = c->split_min_cost >= 0 ? c->split_min_cost
                                                    : (getenv("CVG_SPLIT_MIN_COST") ? atoll(getenv("CVG_SPLIT_MIN_COST")) : (int64_t)1 << 25);
    const int64_t cost = sc->ts.rows_total * (int64_t)std::max(m->n_rows, 1);
    if (K > 1 && cost / K < min_cost) K = (int)std::max<int64_t>(1, cost / std::max<int64_t>(min_cost, 1));
    if (K <= 1) { out.push_back({ 0, S }); return; }
    int s = 0; int64_t done = 0;
    for (int k = 0; k < K && s < S; k++) {
        const int64_t target = sc->ts.rows_total * (k + 1) / K;
        int e = s;
        while (e < S && (done < target || e == s) && S - e > K - 1 - k) { done += sc->ts.segs[(size_t)e].rows; e++; }
        if (k == K - 1) e = S;
        if (e > s) out.push_back({ s, e });
        s = e;
    }
    if (s < S) out.back().second = S;
}

// Enqueue scenes x views of one device context on its lanes; returns without waiting.
static int dev_submit(cvg_ctx* c, const cvg_models* m, cvg_scenes* sc, const float* scales, const cvg_detect_params* p,
                      cvg_pair_result* per_pair, float* inl_xy, int64_t* inl_off, bool split, cvg_job** out)
{
    *out = nullptr;
    cvg_job* j = new cvg_job();
    j->ctx = c; j->m = m; j->sc = sc; j->params = *p; j->per_pair = per_pair; j->inl_xy = inl_xy; j->inl_off = inl_off;
    const int S = sc->ts.n_segs, V = m->n_views;
    if (scales) { j->scales.assign(scales, scales + S); j->have_scales = true; }
    std::vector<std::pair<int, int>> ranges;
    plan_chunks(c, m, sc, split, ranges);
    const int K = (int)ranges.size();
    const int need = split ? K : lanes_of(c);
    int rc = ensure_lanes(c, need);
    if (rc) { delete j; return rc; }
    const bool want_inl = inl_xy != nullptr && inl_off != nullptr;
    for (int k = 0; k < K; k++) {
        ChunkTask* t = new ChunkTask();
        t->s0 = ranges[(size_t)k].first; t->s1 = ranges[(size_t)k].second;
        j->chunks.push_back(t);
        // a split call occupies lanes 0..K-1 at once; pipelined jobs take the lanes in turn
        Lane* lane = c->lanes[split ? (size_t)k : (size_t)(c->next_lane++ % (unsigned)need)];
        cvg_ctx* eng = lane->eng;
        const int share = split ? K : need;
        lane->worker->post([=] {
            eng->wave_div = share;
            eng->blocking_sync = !split && need > 4;     // many lanes: their workers sleep while the GPU works (api.cu, sync_and_check)
            const int r = eng_detect_range(eng, m, sc, t->s0, t->s1, j->have_scales ? j->scales.data() : nullptr, &j->params,
                                           j->per_pair + (size_t)t->s0 * V, want_inl ? &t->pool : nullptr, want_inl ? &t->cnt : nullptr);
            t->match_path = eng->last_match_path;
            t->done.set(r, cvg_last_error());
        });
    }
    *out = j;
    return CVG_OK;
}

static int dev_wait(cvg_job* j)
{
    int rc = CVG_OK; std::string err;
    for (ChunkTask* t : j->chunks) {
        const int r = t->done.wait();
        if (r && !rc) { rc = r; err = t->done.err; }
    }
    if (rc) return cvg_set_err(rc, "%s", err.c_str());
    for (ChunkTask* t : j->chunks) j->ctx->last_match_path = std::max(t == j->chunks[0] ? 0 : j->ctx->last_match_path, t->match_path);
    if (j->inl_xy && j->inl_off) {
        // every chunk comes back packed pair after pair (eng_detect_range): concatenate in scene order
        const int V = j->m->n_views;
        int64_t o = 0;
        for (ChunkTask* t : j->chunks) {
            memcpy(j->inl_xy + 2 * (size_t)o, t->pool.data(), t->pool.size() * 4);
            for (size_t lp = 0; lp < t->cnt.size(); lp++) { j->inl_off[(size_t)t->s0 * V + lp] = o; o += t->cnt[lp]; }
        }
        j->inl_off[(size_t)j->sc->ts.n_segs * V] = o;
    }
    return CVG_OK;
}

// ---- multi-device: submit / wait ----------------------------------------------------------------------------
static int multi_submit(cvg_ctx* c, const cvg_models* m, const cvg_scenes* sc, const float* scales, const cvg_detect_params* p,
                        cvg_pair_result* per_pair, float* inl_xy, int64_t* inl_off, bool split, cvg_job** out)
{
    MultiState* ms = c->multi;
    *out = nullptr;
    if (m->replicas.size() != ms->subs.size() || sc->subs.size() != ms->subs.size())
        return cvg_set_err(CVG_ERR_INVALID, "models / scenes were not uploaded through this multi-device context");
    cvg_job* j = new cvg_job();
    j->ctx = c; j->shell = sc; j->shell_m = m; j->per_pair = per_pair; j->inl_xy = inl_xy; j->inl_off = inl_off;
    const int V = m->n_views;
    const bool want_inl = inl_xy != nullptr && inl_off != nullptr;
    const size_t nd = ms->subs.size();
    j->sub_res.resize(nd); j->sub_xy.resize(nd); j->sub_off.resize(nd);
    for (size_t d = 0; d < nd; d++) {
        cvg_scenes* sub = sc->subs[d];
        if (!sub) continue;
        const int Sd = sub->ts.n_segs;
        std::vector<float> sc_d;
        if (scales) { sc_d.resize((size_t)Sd); for (int s = 0; s < sc->n_scenes_total; s++) if (sc->dev_of_scene[(size_t)s] == (int)d) sc_d[(size_t)sc->local_of_scene[(size_t)s]] = scales[s]; }
        j->sub_res[d].resize((size_t)std::max(Sd * V, 1));
        if (want_inl) { j->sub_xy[d].resize((size_t)Sd * std::max(m->n_rows, 1) * 2); j->sub_off[d].resize((size_t)Sd * V + 1); }
        cvg_job* sj = nullptr;
        const int rc = dev_submit(ms->subs[d], m->replicas[d], sub, scales ? sc_d.data() : nullptr, p, j->sub_res[d].data(),
                                  want_inl ? j->sub_xy[d].data() : nullptr, want_inl ? j->sub_off[d].data() : nullptr, split, &sj);
        if (rc) { for (cvg_job* q : j->subs) dev_wait(q); delete j; return rc; }
        j->subs.push_back(sj); j->sub_dev.push_back((int)d);
    }
    *out = j;
    return CVG_OK;
}

static int multi_wait(cvg_job* j)
{
    int rc = CVG_OK; std::string err;
    for (cvg_job* sj : j->subs) {
        const int r = dev_wait(sj);
        if (r && !rc) { rc = r; err = cvg_last_error(); }
    }
    if (rc) return cvg_set_err(rc, "%s", err.c_str());
    const cvg_scenes* sc = j->shell; const cvg_models* m = j->shell_m;
    const int V = m->n_views, S = sc->n_scenes_total;
    const bool want_inl = j->inl_xy && j->inl_off;
    int64_t o = 0;
    for (int s = 0; s < S; s++) {
        const size_t d = (size_t)sc->dev_of_scene[(size_t)s]; const int ls = sc->local_of_scene[(size_t)s];
        memcpy(j->per_pair + (size_t)s * V, j->sub_res[d].data() + (size_t)ls * V, (size_t)V * sizeof(cvg_pair_result));
        if (!want_inl) continue;
        const int64_t a = j->sub_off[d][(size_t)ls * V], b = j->sub_off[d][(size_t)(ls + 1) * V];
        memcpy(j->inl_xy + 2 * (size_t)o, j->sub_xy[d].data() + 2 * (size_t)a, (size_t)(b - a) * 8);
        for (int v = 0; v < V; v++) j->inl_off[(size_t)s * V + v] = o + (j->sub_off[d][(size_t)ls * V + v] - a);
        o += b - a;
    }
    if (want_inl) j->inl_off[(size_t)S * V] = o;
    return CVG_OK;
}

static void multi_destroy(cvg_ctx* c)
{
    MultiState* ms = c->multi;
    if (!ms) return;
    for (Worker* w : ms->workers) delete w;
    NcclApi& na = nccl_api();
    for (size_t d = 0; d < ms->comms.size(); d++) if (ms->comms[d]) { cudaSetDevice(ms->devices[d]); na.CommDestroy(ms->comms[d]); }
    for (size_t d = 0; d < ms->subs.size(); d++) {
        cudaSetDevice(ms->devices[d]);
        for (std::vector<DevBuf>* v : { &ms->loc_d, &ms->loc_i, &ms->all_d, &ms->all_i, &ms->qbuf, &ms->tbuf, &ms->out_idx, &ms->out_dist, &ms->out_acc })
            if (d < v->size()) (*v)[d].release();
        if (d < ms->ev.size() && ms->ev[d]) cudaEventDestroy(ms->ev[d]);
        if (d == 0) for (cudaEvent_t e : ms->tev) cudaEventDestroy(e);
        if (ms->subs[d]) { destroy_lanes(ms->subs[d]); eng_destroy(ms->subs[d]); }
    }
    delete ms;
    c->multi = nullptr;
}

extern "C" {

// ---- context ------------------------------------------------------------------------------------------------
int cvg_create(cvg_ctx** out, int device, unsigned flags) { return eng_create(out, device, flags); }

int cvg_create_multi(cvg_ctx** out, const int* devices, int n_devices, unsigned flags)
{
    if (!out || !devices || n_devices < 1 || n_devices > 64) return cvg_set_err(CVG_ERR_INVALID, "cvg_create_multi: bad argument");
    *out = nullptr;
    cvg_ctx* shell = new cvg_ctx();
    shell->device = -1; shell->flags = flags;
    MultiState* ms = new MultiState();
    shell->multi = ms;
    ms->devices.assign(devices, devices + n_devices);
    const size_t nd = (size_t)n_devices;
    ms->subs.assign(nd, nullptr); ms->ev.assign(nd, nullptr);
    for (std::vector<DevBuf>* v : { &ms->loc_d, &ms->loc_i, &ms->all_d, &ms->all_i, &ms->qbuf, &ms->tbuf, &ms->out_idx, &ms->out_dist, &ms->out_acc }) v->resize(nd);
    for (size_t d = 0; d < nd; d++) {
        int rc = eng_create(&ms->subs[d], devices[d], flags);
        if (!rc && cudaEventCreateWithFlags(&ms->ev[d], cudaEventDisableTiming) != cudaSuccess) rc = cvg_set_err(CVG_ERR_CUDA, "cudaEventCreate failed");
        if (rc) { multi_destroy(shell); delete shell; return rc; }
        ms->subs[d]->parent = shell;
        ms->workers.push_back(new Worker());
    }
    // One NCCL communicator per device for the exchange step of the train-tile sharded match.  NCCL refuses a
    // communicator that names a GPU twice (logical devices on one GPU, as the single-GPU tests use): the exchange then
    // runs as device-to-device copies, which is also the fallback when libnccl cannot be loaded.
    bool distinct = true;
    for (size_t a = 0; a < nd; a++) for (size_t b = a + 1; b < nd; b++) if (devices[a] == devices[b]) distinct = false;
    ms->exchange = "memcpy";
    const char* no_nccl = getenv("CVG_NO_NCCL");
    if (nd > 1 && distinct && !(no_nccl && atoi(no_nccl)) && nccl_api().ok) {
        ms->comms.assign(nd, nullptr);
        const int r = nccl_api().CommInitAll(ms->comms.data(), n_devices, devices);
        if (r != 0) { ms->comms.clear(); cudaGetLastError(); }
        else ms->exchange = "nccl";
    }
    *out = shell;
    return CVG_OK;
}

int cvg_num_devices(const cvg_ctx* c) { return !c ? 0 : (c->multi ? (int)c->multi->subs.size() : 1); }
const char* cvg_exchange_kind(const cvg_ctx* c) { return (c && c->multi) ? c->multi->exchange : "none"; }

void cvg_destroy(cvg_ctx* c)
{
    if (!c) return;
    if (c->multi) { multi_destroy(c); delete c; return; }
    destroy_lanes(c);
    eng_destroy(c);
}

int cvg_set_lanes(cvg_ctx* c, int n_lanes)
{
    if (!c || n_lanes < 0 || n_lanes > 8) return cvg_set_err(CVG_ERR_INVALID, "cvg_set_lanes: 0 (default) .. 8");
    if (c->multi) { for (cvg_ctx* s : c->multi->subs) s->lanes_cfg = n_lanes ? n_lanes : -1; return CVG_OK; }
    c->lanes_cfg = n_lanes ? n_lanes : -1;
    return CVG_OK;
}

int64_t cvg_launch_count(const cvg_ctx* c)
{
    if (!c) return 0;
    int64_t n = 0;
    if (c->multi) { for (const cvg_ctx* s : c->multi->subs) n += cvg_launch_count(s); return n; }
    n = c->launches;
    for (const Lane* l : c->lanes) n += l->eng->launches;
    return n;
}

// ---- model set ------------------------------------------------------------------------------------------------
int cvg_models_upload(cvg_ctx* c, const float* desc, const float* kpt_xy, const int32_t* view_offsets,
                      const int32_t* view_model, int n_views, cvg_models** out)
{
    if (!c || !out) return cvg_set_err(CVG_ERR_INVALID, "cvg_models_upload: bad argument");
    if (!c->multi) return eng_models_upload(c, desc, kpt_xy, view_offsets, view_model, n_views, out);
    *out = nullptr;
    cvg_models* shell = new cvg_models();
    for (cvg_ctx* s : c->multi->subs) {                     // replicated: 7 MB for the reference's 89 views
        cvg_models* r = nullptr;
        const int rc = eng_models_upload(s, desc, kpt_xy, view_offsets, view_model, n_views, &r);
        if (rc) { for (size_t d = 0; d < shell->replicas.size(); d++) eng_models_free(c->multi->subs[d], shell->replicas[d]); delete shell; return rc; }
        shell->replicas.push_back(r);
    }
    const cvg_models* r0 = shell->replicas[0];
    shell->n_rows = r0->n_rows; shell->n_pad = r0->n_pad; shell->n_views = r0->n_views; shell->view_offsets = r0->view_offsets;
    shell->view_model = r0->view_model; shell->nonint = r0->nonint; shell->max_norm2 = r0->max_norm2; shell->uid = r0->uid;
    *out = shell;
    return CVG_OK;
}

void cvg_models_free(cvg_ctx* c, cvg_models* m)
{
    if (!m) return;
    if (!m->replicas.empty()) {
        for (size_t d = 0; d < m->replicas.size(); d++)
            eng_models_free((c && c->multi && d < c->multi->subs.size()) ? c->multi->subs[d] : nullptr, m->replicas[d]);
        delete m;
        return;
    }
    eng_models_free(c && !c->multi ? c : nullptr, m);
}

// ---- scene batches --------------------------------------------------------------------------------------------
static int scenes_upload_any(cvg_ctx* c, const float* desc, const uint8_t* desc_u8, const float* kpt_xy, const int64_t* offsets,
                             int n_scenes, cvg_scenes** out, bool async)
{
    if (!c || !out || !offsets || n_scenes < 0) return cvg_set_err(CVG_ERR_INVALID, "cvg_scenes_upload: bad argument");
    if (!c->multi) return eng_scenes_upload(c, desc, desc_u8, kpt_xy, offsets, n_scenes, out, async);
    *out = nullptr;
    MultiState* ms = c->multi;
    const size_t nd = ms->subs.size();
    for (int s = 0; s < n_scenes; s++)
        if (offsets[s + 1] < offsets[s]) return cvg_set_err(CVG_ERR_INVALID, "offsets must be non-decreasing");
    cvg_scenes* shell = new cvg_scenes();
    shell->n_scenes_total = n_scenes;
    shell->offsets_copy.assign(offsets, offsets + n_scenes + 1);
    shell->dev_of_scene.assign((size_t)n_scenes, 0); shell->local_of_scene.assign((size_t)n_scenes, 0);
    shell->subs.assign(nd, nullptr);
    std::vector<std::vector<int>> mine(nd);
    if ((size_t)n_scenes < 2 * nd) {
        // a small batch (the five scales of one test image) stays whole on one device, batches take the devices in turn:
        // the caller pipelines them with cvg_detect_scenes_submit
        const size_t d = ms->next_dev++ % nd;
        for (int s = 0; s < n_scenes; s++) mine[d].push_back(s);
    } else {
        // longest-processing-time-first by train rows (the cost of a scene is rows x model rows), ties to the lower device
        std::vector<int> order((size_t)n_scenes);
        for (int s = 0; s < n_scenes; s++) order[(size_t)s] = s;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return offsets[a + 1] - offsets[a] > offsets[b + 1] - offsets[b]; });
        std::vector<int64_t> load(nd, 0);
        for (int s : order) {
            size_t best = 0;
            for (size_t d = 1; d < nd; d++) if (load[d] < load[best]) best = d;
            mine[best].push_back(s); load[best] += offsets[s + 1] - offsets[s];
        }
        for (auto& v : mine) std::sort(v.begin(), v.end());
    }
    for (size_t d = 0; d < nd; d++) {
        if (mine[d].empty()) continue;
        std::vector<int64_t> off_d(mine[d].size() + 1, 0), src0(mine[d].size());
        for (size_t k = 0; k < mine[d].size(); k++) {
            const int s = mine[d][k];
            shell->dev_of_scene[(size_t)s] = (int)d; shell->local_of_scene[(size_t)s] = (int)k;
            src0[k] = offsets[s]; off_d[k + 1] = off_d[k] + (offsets[s + 1] - offsets[s]);
        }
        const int rc = eng_scenes_upload(ms->subs[d], desc, desc_u8, kpt_xy, off_d.data(), (int)mine[d].size(), &shell->subs[d], async,
                                         src0.data());
        if (rc) { for (size_t e = 0; e < nd; e++) if (shell->subs[e]) eng_scenes_free(ms->subs[e], shell->subs[e]); delete shell; return rc; }
    }
    *out = shell;
    return CVG_OK;
}

int cvg_scenes_upload(cvg_ctx* c, const float* desc, const float* kpt_xy, const int64_t* offsets, int n_scenes, cvg_scenes** out)
{
    return scenes_upload_any(c, desc, nullptr, kpt_xy, offsets, n_scenes, out, false);
}
int cvg_scenes_upload_async(cvg_ctx* c, const float* desc, const float* kpt_xy, const int64_t* offsets, int n_scenes, cvg_scenes** out)
{
    return scenes_upload_any(c, desc, nullptr, kpt_xy, offsets, n_scenes, out, true);
}
int cvg_scenes_upload_u8_async(cvg_ctx* c, const uint8_t* desc, const float* kpt_xy, const int64_t* offsets, int n_scenes, cvg_scenes** out)
{
    return scenes_upload_any(c, nullptr, desc, kpt_xy, offsets, n_scenes, out, true);
}

int cvg_scenes_wait(cvg_ctx* c, cvg_scenes* sc)
{
    if (!c || !sc) return cvg_set_err(CVG_ERR_INVALID, "cvg_scenes_wait: NULL argument");
    if (!c->multi) return eng_scenes_wait(c, sc);
    for (size_t d = 0; d < sc->subs.size(); d++)
        if (sc->subs[d]) { const int rc = eng_scenes_wait(c->multi->subs[d], sc->subs[d]); if (rc) return rc; }
    return CVG_OK;
}

void cvg_scenes_free(cvg_ctx* c, cvg_scenes* sc)
{
    if (!sc) return;
    if (!sc->subs.empty()) {
        for (size_t d = 0; d < sc->subs.size(); d++)
            if (sc->subs[d]) eng_scenes_free((c && c->multi && d < c->multi->subs.size()) ? c->multi->subs[d] : nullptr, sc->subs[d]);
        delete sc;
        return;
    }
    eng_scenes_free(c && !c->multi ? c : nullptr, sc);
}

// ---- fused path over resident scene batches ---------------------------------------------------------------------
int cvg_detect_scenes_submit(cvg_ctx* c, const cvg_models* m, const cvg_scenes* scenes, const float* scales,
                             const cvg_detect_params* p_in, cvg_pair_result* per_pair, float* inlier_scene_xy,
                             int64_t* inlier_offsets, cvg_job** job)
{
    if (!c || !m || !scenes || !per_pair || !job) return cvg_set_err(CVG_ERR_INVALID, "cvg_detect_scenes_submit: NULL argument");
    cvg_detect_params params;                          // the full layout: dev_submit copies it into the job
    const int rc = check_detect_params(p_in, &params);
    if (rc) return rc;
    const cvg_detect_params* p = &params;
    if (c->multi) return multi_submit(c, m, scenes, scales, p, per_pair, inlier_scene_xy, inlier_offsets, false, job);
    return dev_submit(c, m, const_cast<cvg_scenes*>(scenes), scales, p, per_pair, inlier_scene_xy, inlier_offsets, false, job);
}

int cvg_job_wait(cvg_ctx* c, cvg_job* job)
{
    if (!c || !job) return cvg_set_err(CVG_ERR_INVALID, "cvg_job_wait: NULL argument");
    const int rc = job->subs.empty() && !job->shell ? dev_wait(job) : multi_wait(job);
    delete job;
    return rc;
}

int cvg_detect_scenes_inliers(cvg_ctx* c, const cvg_models* m, const cvg_scenes* scenes, const float* scales,
                              const cvg_detect_params* p_in, cvg_pair_result* per_pair, float* inlier_scene_xy,
                              int64_t* inlier_offsets)
{
    if (!c || !m || !scenes || !per_pair) return cvg_set_err(CVG_ERR_INVALID, "cvg_detect_scenes: NULL argument");
    cvg_detect_params params;
    int rc = check_detect_params(p_in, &params);
    if (rc) return rc;
    const cvg_detect_params* p = &params;
    cvg_job* job = nullptr;
    if (c->multi) {
        rc = multi_submit(c, m, scenes, scales, p, per_pair, inlier_scene_xy, inlier_offsets, true, &job);
        if (rc) return rc;
        rc = multi_wait(job);
        delete job;
        return rc;
    }
    cvg_scenes* sc = const_cast<cvg_scenes*>(scenes);
    std::vector<std::pair<int, int>> ranges;
    plan_chunks(c, m, sc, true, ranges);
    if (ranges.size() <= 1) {
        // small call: the context's own engine, on the caller's thread
        c->wave_div = 1;
        const bool want_inl = inlier_scene_xy != nullptr && inlier_offsets != nullptr;
        std::vector<float> pool; std::vector<int32_t> cnt;
        rc = eng_detect_range(c, m, sc, 0, sc->ts.n_segs, scales, p, per_pair, want_inl ? &pool : nullptr, want_inl ? &cnt : nullptr);
        if (rc || !want_inl) return rc;
        memcpy(inlier_scene_xy, pool.data(), pool.size() * 4);
        int64_t o = 0;
        for (size_t pair = 0; pair < cnt.size(); pair++) { inlier_offsets[pair] = o; o += cnt[pair]; }
        inlier_offsets[cnt.size()] = o;
        return CVG_OK;
    }
    rc = dev_submit(c, m, sc, scales, p, per_pair, inlier_scene_xy, inlier_offsets, true, &job);
    if (rc) return rc;
    rc = dev_wait(job);
    delete job;
    return rc;
}

int cvg_detect_scenes(cvg_ctx* c, const cvg_models* m, const cvg_scenes* scenes, const float* scales,
                      const cvg_detect_params* p, cvg_pair_result* per_pair)
{
    return cvg_detect_scenes_inliers(c, m, scenes, scales, p, per_pair, nullptr, nullptr);
}

// ---- train-tile sharded match: SURVEY 8e-2, BASELINE config 5 ------------------------------------------------------
// Every device gets the whole query matrix and one contiguous, 256-aligned range of the train rows, computes its local
// top-2 per query with GLOBAL train indices (cvg_dev_match_top2), then ONE exchange: all-gather of the (distance, index)
// pairs, 16 B per query and device, and the lexicographic (distance, index) merge that reproduces OpenCV's tie rule
// whatever the number of shards (cvg_dev_merge_top2) — replaces src/TestsDetector.cpp:59-72 for one huge pair.
int cvg_match_knn2_sharded(cvg_ctx* c, const float* query, int n_query, const float* train, int n_train, float ratio,
                           int32_t* idx, float* dist, uint8_t* accept)
{
    if (!c || !c->multi) return cvg_set_err(CVG_ERR_INVALID, "cvg_match_knn2_sharded needs a context made by cvg_create_multi");
    if (n_query < 0 || n_train < 0 || (n_query > 0 && !query) || (n_train > 0 && !train) || !idx || !dist)
        return cvg_set_err(CVG_ERR_INVALID, "cvg_match_knn2_sharded: bad argument");
    if (n_query == 0) return CVG_OK;
    MultiState* ms = c->multi;
    const int nd = (int)ms->subs.size();
    int64_t per = ((int64_t)n_train + nd - 1) / nd;
    per = (per + TILE_N - 1) / TILE_N * TILE_N;
    std::vector<Done> done((size_t)nd);
    const size_t nq = (size_t)n_query;
    for (int d = 0; d < nd; d++) {
        ms->workers[(size_t)d]->post([=, &done] {
            cvg_ctx* e = ms->subs[(size_t)d];
            const int64_t a = std::min<int64_t>((int64_t)d * per, n_train), b = std::min<int64_t>(a + per, n_train);
            const int rc = [&]() -> int {
                CU_CHECK(cudaSetDevice(e->device));
                CU_CHECK(ms->qbuf[(size_t)d].ensure(nq * DIM * 4));
                CU_CHECK(ms->tbuf[(size_t)d].ensure((size_t)std::max<int64_t>(b - a, 1) * DIM * 4));
                CU_CHECK(ms->loc_d[(size_t)d].ensure(nq * 8)); CU_CHECK(ms->loc_i[(size_t)d].ensure(nq * 8));
                CU_CHECK(ms->all_d[(size_t)d].ensure(nq * 8 * nd)); CU_CHECK(ms->all_i[(size_t)d].ensure(nq * 8 * nd));
                CU_CHECK(cudaMemcpyAsync(ms->qbuf[(size_t)d].p, query, nq * DIM * 4, cudaMemcpyHostToDevice, e->stream));
                if (b > a) CU_CHECK(cudaMemcpyAsync(ms->tbuf[(size_t)d].p, train + (size_t)a * DIM, (size_t)(b - a) * DIM * 4, cudaMemcpyHostToDevice, e->stream));
                return cvg_dev_match_top2(e, e->stream, ms->qbuf[(size_t)d].as<float>(), n_query, ms->tbuf[(size_t)d].as<float>(), (int)(b - a),
                                          (int32_t)a, ms->loc_d[(size_t)d].as<float>(), ms->loc_i[(size_t)d].as<int32_t>());
            }();
            done[(size_t)d].set(rc, cvg_last_error());
        });
    }
    int rc = CVG_OK; std::string err;
    for (int d = 0; d < nd; d++) { const int r = done[(size_t)d].wait(); if (r && !rc) { rc = r; err = done[(size_t)d].err; } }
    if (rc) return cvg_set_err(rc, "%s", err.c_str());
    // ---- the exchange step -------------------------------------------------------------------------------------
    if (!ms->comms.empty()) {
        NcclApi& na = nccl_api();
        int r = na.GroupStart();
        for (int d = 0; d < nd && r == 0; d++) {
            cvg_ctx* e = ms->subs[(size_t)d];
            r = na.AllGather(ms->loc_d[(size_t)d].p, ms->all_d[(size_t)d].p, nq * 8, NCCL_CHAR, ms->comms[(size_t)d], e->stream);
            if (r == 0) r = na.AllGather(ms->loc_i[(size_t)d].p, ms->all_i[(size_t)d].p, nq * 8, NCCL_CHAR, ms->comms[(size_t)d], e->stream);
        }
        const int r2 = na.GroupEnd();
        if (r == 0) r = r2;
        if (r != 0) return cvg_set_err(CVG_ERR_CUDA, "ncclAllGather failed: %s", na.GetErrorString ? na.GetErrorString(r) : "?");
    } else {
        // logical devices on one GPU / no NCCL: the partial results travel to device 0 by device-to-device copies
        cvg_ctx* e0 = ms->subs[0];
        for (int d = 0; d < nd; d++) {
            cvg_ctx* e = ms->subs[(size_t)d];
            CU_CHECK(cudaSetDevice(e->device));
            CU_CHECK(cudaEventRecord(ms->ev[(size_t)d], e->stream));
            CU_CHECK(cudaSetDevice(e0->device));
            CU_CHECK(cudaStreamWaitEvent(e0->stream, ms->ev[(size_t)d], 0));
            CU_CHECK(cudaMemcpyPeerAsync(ms->all_d[0].as<uint8_t>() + (size_t)d * nq * 8, e0->device, ms->loc_d[(size_t)d].p, e->device, nq * 8, e0->stream));
            CU_CHECK(cudaMemcpyPeerAsync(ms->all_i[0].as<uint8_t>() + (size_t)d * nq * 8, e0->device, ms->loc_i[(size_t)d].p, e->device, nq * 8, e0->stream));
        }
    }
    // ---- merge on device 0, results to the host; the other devices only have to drain ----------------------------
    cvg_ctx* e0 = ms->subs[0];
    CU_CHECK(cudaSetDevice(e0->device));
    CU_CHECK(ms->out_idx[0].ensure(nq * 8)); CU_CHECK(ms->out_dist[0].ensure(nq * 8)); CU_CHECK(ms->out_acc[0].ensure(nq));
    rc = cvg_dev_merge_top2(e0, e0->stream, ms->all_d[0].as<float>(), ms->all_i[0].as<int32_t>(), nd, n_query, ratio,
                            ms->out_idx[0].as<int32_t>(), ms->out_dist[0].as<float>(), ms->out_acc[0].as<uint8_t>());
    if (rc) return rc;
    CU_CHECK(cudaMemcpyAsync(idx, ms->out_idx[0].p, nq * 8, cudaMemcpyDeviceToHost, e0->stream));
    CU_CHECK(cudaMemcpyAsync(dist, ms->out_dist[0].p, nq * 8, cudaMemcpyDeviceToHost, e0->stream));
    if (accept) CU_CHECK(cudaMemcpyAsync(accept, ms->out_acc[0].p, nq, cudaMemcpyDeviceToHost, e0->stream));
    for (int d = nd - 1; d >= 0; d--) {
        CU_CHECK(cudaSetDevice(ms->subs[(size_t)d]->device));
        CU_CHECK(cudaStreamSynchronize(ms->subs[(size_t)d]->stream));
    }
    return CVG_OK;
}

// ---- hypothesis-range sharded RANSAC: SURVEY 8e, BASELINE config 5 ------------------------------------------------------
// Every device holds the whole scan state of the one point set (points, draw table, samples, counts, best so far, adaptive
// niters) and runs the sampler and the serial select scan itself; only the solve + score kernels are split.  Round
// [rb, rb + len) is cut into G slices of S = ceil(len / G) iterations, device d solves and scores [rb + d*S, rb +
// min((d+1)*S, len)), and one exchange per round gives every device all counts of the round: an in-place ncclAllGather of S
// ints per device, or event-ordered peer copies.  The select kernels then scan exactly the counts one device would have
// computed, so the winner, the adaptive stop and the niters requests are the same everywhere.  The first device's finish
// kernel re-solves the winner from its own samples (bit-identical to the hypothesis kernels): no model crosses devices.
static int sharded_rounds(MultiState* ms, const std::vector<RansacWork>& w, int round_len, bool timing, int* at)
{
    const int G = (int)ms->subs.size();
    const int mi = w[0].max_iters;
    cvg_ctx* e0 = ms->subs[0];
    const int n_rounds = (mi + round_len - 1) / round_len;
    *at = 0;
    CU_CHECK(cudaSetDevice(e0->device));
    while (timing && (int)ms->tev.size() < 5 * n_rounds) {
        cudaEvent_t e;
        CU_CHECK(cudaEventCreate(&e));
        ms->tev.push_back(e);
    }
    if (timing) CU_CHECK(cudaEventRecord(e0->ev[0], e0->stream));
    bool hyp_complete = true;                                  // unused: the finish kernel re-solves the winner
    for (int rb = 0, round = 0; rb < mi; rb += round_len, round++) {
        const int len = std::min(round_len, mi - rb);
        const int S = (len + G - 1) / G;
        const cudaEvent_t* ev = timing ? ms->tev.data() + 5 * round : nullptr;
        for (int d = 0; d < G; d++) {
            cvg_ctx* e = ms->subs[(size_t)d];
            *at = d;
            CU_CHECK(cudaSetDevice(e->device));
            e->launches += launch_ransac_sample(w[(size_t)d], rb, len, e->stream);
            const int a = std::min(d * S, len), b = std::min((d + 1) * S, len);
            if (b > a) e->launches += launch_ransac_hyp(w[(size_t)d], rb + a, b - a, e->stream, d == 0 ? ev : nullptr, &hyp_complete);
            CU_CHECK(cudaGetLastError());
        }
        // ---- the exchange step: every device receives the round's G*S counts at counts[rb ...) ------------------------
        if (!ms->comms.empty()) {
            *at = 0;
            CU_CHECK(cudaSetDevice(e0->device));
            if (ev) CU_CHECK(cudaEventRecord(ev[3], e0->stream));
            NcclApi& na = nccl_api();
            int r = na.GroupStart();
            for (int d = 0; d < G && r == 0; d++) {
                int32_t* cnt = w[(size_t)d].counts + rb;               // in place: rank d sends its own slice
                r = na.AllGather(cnt + (size_t)d * S, cnt, (size_t)S * 4, NCCL_CHAR, ms->comms[(size_t)d], ms->subs[(size_t)d]->stream);
            }
            const int r2 = na.GroupEnd();
            if (r == 0) r = r2;
            if (r != 0) return cvg_set_err(CVG_ERR_CUDA, "ncclAllGather failed: %s", na.GetErrorString ? na.GetErrorString(r) : "?");
            CU_CHECK(cudaSetDevice(e0->device));
            if (ev) CU_CHECK(cudaEventRecord(ev[4], e0->stream));
        } else {
            for (int d = 0; d < G; d++) {
                *at = d;
                CU_CHECK(cudaSetDevice(ms->subs[(size_t)d]->device));
                CU_CHECK(cudaEventRecord(ms->ev[(size_t)d], ms->subs[(size_t)d]->stream));
            }
            for (int t = 0; t < G; t++) {
                cvg_ctx* et = ms->subs[(size_t)t];
                *at = t;
                CU_CHECK(cudaSetDevice(et->device));
                if (ev && t == 0) CU_CHECK(cudaEventRecord(ev[3], et->stream));
                for (int s = 0; s < G; s++) {
                    const int a = std::min(s * S, len), b = std::min((s + 1) * S, len);
                    if (s == t || b <= a) continue;
                    CU_CHECK(cudaStreamWaitEvent(et->stream, ms->ev[(size_t)s], 0));
                    CU_CHECK(cudaMemcpyPeerAsync(w[(size_t)t].counts + rb + a, et->device, w[(size_t)s].counts + rb + a,
                                                 ms->subs[(size_t)s]->device, (size_t)(b - a) * 4, et->stream));
                }
                if (ev && t == 0) CU_CHECK(cudaEventRecord(ev[4], et->stream));
            }
        }
        ms->n_exchanges++;
        for (int d = 0; d < G; d++) {
            cvg_ctx* e = ms->subs[(size_t)d];
            *at = d;
            CU_CHECK(cudaSetDevice(e->device));
            e->launches += launch_ransac_select(w[(size_t)d], rb, len, e->stream);
            CU_CHECK(cudaGetLastError());
        }
    }
    *at = 0;
    CU_CHECK(cudaSetDevice(e0->device));
    e0->launches += launch_ransac_finish(w[0], false, e0->stream);
    if (timing) CU_CHECK(cudaEventRecord(e0->ev[1], e0->stream));
    CU_CHECK(cudaGetLastError());
    if (timing) {
        e0->t_hyp = 0; e0->t_score = 0; ms->exchange_ms = 0;
        for (int r = 0; r < n_rounds; r++) {
            const cudaEvent_t* ev = ms->tev.data() + 5 * r;
            float t = 0;
            CU_CHECK(cudaEventSynchronize(ev[4]));
            CU_CHECK(cudaEventElapsedTime(&t, ev[0], ev[1])); e0->t_hyp += t;
            CU_CHECK(cudaEventElapsedTime(&t, ev[1], ev[2])); e0->t_score += t;
            CU_CHECK(cudaEventElapsedTime(&t, ev[3], ev[4])); ms->exchange_ms += t;
        }
        e0->hyp_rounds = n_rounds; e0->hyp_launches = n_rounds;
    }
    return CVG_OK;
}

int cvg_find_homography_sharded(cvg_ctx* c, const float* src_xy, const float* dst_xy, int n, const cvg_ransac_params* p,
                                double H[9], uint8_t* mask, int* found, int32_t* iters, uint8_t* ransac_mask)
{
    if (!c || !c->multi) return cvg_set_err(CVG_ERR_INVALID, "cvg_find_homography_sharded needs a context made by cvg_create_multi");
    if (n < 4) return cvg_set_err(CVG_ERR_TOO_FEW_POINTS, "findHomography needs at least 4 correspondences (got %d)", n);
    int rc = check_params(p);
    if (rc) return rc;
    if (!src_xy || !dst_xy) return cvg_set_err(CVG_ERR_INVALID, "cvg_find_homography_sharded: bad point arrays");
    MultiState* ms = c->multi;
    const int G = (int)ms->subs.size();
    cvg_ctx* e0 = ms->subs[0];
    const int mi = std::max(p->max_iters, 1);
    const bool timing = e0->timing != 0;
    ms->n_exchanges = 0; ms->exchange_ms = 0.f;
    int at = 0;                                                // the device the failing step ran on
    const int64_t start0 = 0; const int32_t n32 = n;
    std::vector<NitEntry> tab;                                 // the niters entries every device gets
    std::vector<int32_t> sflags((size_t)G), words((size_t)G);
    // every device's table to `tab`, where it differs (each engine keeps its entries unique: equal size = same set)
    auto share_table = [&]() -> int {
        for (int d = 0; d < G; d++) {
            cvg_ctx* e = ms->subs[(size_t)d];
            if (e->nit_host.size() == tab.size()) continue;
            at = d;
            CU_CHECK(cudaSetDevice(e->device));
            e->nit_host = tab;
            const int r = nit_upload(e);
            if (r) return r;
        }
        return CVG_OK;
    };
    rc = [&]() -> int {
        // points on every device, each device's draw table as long as the longest (the chunked sampler's layout and the
        // samples follow from the table's length), and one niters table: the union of the devices' tables
        int64_t rng_len = 0;
        for (int d = 0; d < G; d++) {
            cvg_ctx* e = ms->subs[(size_t)d];
            at = d;
            CU_CHECK(cudaSetDevice(e->device));
            CU_CHECK(e->src.ensure((size_t)n * 8)); CU_CHECK(e->dst.ensure((size_t)n * 8)); CU_CHECK(e->pts.ensure((size_t)n * 16));
            CU_CHECK(e->starts.ensure(8)); CU_CHECK(e->counts_n.ensure(4));
            CU_CHECK(cudaMemcpyAsync(e->src.p, src_xy, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
            CU_CHECK(cudaMemcpyAsync(e->dst.p, dst_xy, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
            CU_CHECK(cudaMemcpyAsync(e->starts.p, &start0, 8, cudaMemcpyHostToDevice, e->stream));
            CU_CHECK(cudaMemcpyAsync(e->counts_n.p, &n32, 4, cudaMemcpyHostToDevice, e->stream));
            launch_pack_points(e->src.as<float>(), e->dst.as<float>(), n, e->pts.as<float4>(), e->stream);
            e->launches++;
            int r = ensure_rng(e, mi);
            if (r) return r;
            rng_len = std::max(rng_len, e->rng_len);
            for (const NitEntry& x : e->nit_host) {
                bool have = false;
                for (const NitEntry& y : tab) if (x.n == y.n && x.good == y.good && x.mp == y.mp) { have = true; break; }
                if (!have) tab.push_back(x);
            }
        }
        for (int d = 0; d < G; d++) {
            at = d;
            CU_CHECK(cudaSetDevice(ms->subs[(size_t)d]->device));
            const int r = ensure_rng(ms->subs[(size_t)d], mi, rng_len);
            if (r) return r;
        }
        return share_table();
    }();
    for (int attempt = 0; rc == CVG_OK; attempt++) {
        std::vector<RansacWork> w((size_t)G);
        rc = [&]() -> int {
            for (int d = 0; d < G; d++) {
                cvg_ctx* e = ms->subs[(size_t)d];
                at = d;
                CU_CHECK(cudaSetDevice(e->device));
                // counts: the exchange writes G*S <= len + G - 1 entries from rb on
                const int r = eng_ransac_work(e, e->pts.as<float4>(), e->starts.as<int64_t>(), e->counts_n.as<int32_t>(), 1, n, n, p,
                                              ransac_mask != nullptr, G, &w[(size_t)d]);
                if (r) return r;
            }
            // adaptive stop: every device's slice of a round is the round one device would run; else one round
            int round_len = ransac_round_len(w[0]);
            if (!(p->flags & CVG_RANSAC_NO_EARLY_STOP)) round_len = (int)std::min<int64_t>((int64_t)G * round_len, mi);
            ms->n_exchanges = 0;
            int r = sharded_rounds(ms, w, round_len, timing, &at);
            if (r) return r;
            at = 0;
            CU_CHECK(cudaSetDevice(e0->device));
            if (H) CU_CHECK(cudaMemcpyAsync(H, e0->H.p, 72, cudaMemcpyDeviceToHost, e0->stream));
            if (mask) CU_CHECK(cudaMemcpyAsync(mask, e0->mask.p, (size_t)n, cudaMemcpyDeviceToHost, e0->stream));
            if (ransac_mask) CU_CHECK(cudaMemcpyAsync(ransac_mask, e0->rmask.p, (size_t)n, cudaMemcpyDeviceToHost, e0->stream));
            if (found) CU_CHECK(cudaMemcpyAsync(found, e0->found.p, 4, cudaMemcpyDeviceToHost, e0->stream));
            if (iters) CU_CHECK(cudaMemcpyAsync(iters, e0->iters_run.p, 4, cudaMemcpyDeviceToHost, e0->stream));
            for (int d = G - 1; d >= 0; d--) {
                cvg_ctx* e = ms->subs[(size_t)d];
                at = d;
                CU_CHECK(cudaSetDevice(e->device));
                CU_CHECK(cudaMemcpyAsync(&sflags[(size_t)d], e->sflags.p, 4, cudaMemcpyDeviceToHost, e->stream));
                CU_CHECK(cudaMemcpyAsync(&words[(size_t)d], e->d_flags + 4, 4, cudaMemcpyDeviceToHost, e->stream));
                r = sync_and_check(e);
                if (r) return r;
            }
            return CVG_OK;
        }();
        if (rc) break;
        // retry decisions on the union of the devices' flags
        bool short_tab = false; int want_nit = 0;
        for (int d = 0; d < G; d++) { short_tab = short_tab || (sflags[(size_t)d] & 1); want_nit |= words[(size_t)d] & 2; }
        if (!short_tab && want_nit) {                          // niters entries to verify on the host, then again
            if (attempt >= 12) return cvg_set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters verification did not converge");
            size_t added = 0;
            rc = [&]() -> int {
                for (int d = 0; d < G; d++) {
                    if (!(words[(size_t)d] & 2)) continue;
                    at = d;
                    CU_CHECK(cudaSetDevice(ms->subs[(size_t)d]->device));
                    size_t a = 0;
                    const int r = nit_add_requests(ms->subs[(size_t)d], tab, &a);
                    if (r) return r;
                    added += a;
                }
                if (!added) return cvg_set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters: the device keeps asking about entries it already has");
                if (tab.size() > (1u << 20)) return cvg_set_err(CVG_ERR_LIMIT, "RANSACUpdateNumIters: verification table overflow");
                return share_table();
            }();
            continue;
        }
        if (!short_tab) break;
        // a draw table ran out: every device's table grows to the same length, then the whole verify stage again
        const int64_t old_len = e0->rng_len;
        if (attempt >= 4) return cvg_set_err(CVG_ERR_LIMIT, "RNG draw table exhausted (pathological rejection rate)");
        rc = [&]() -> int {
            for (int d = 0; d < G; d++) {
                at = d;
                CU_CHECK(cudaSetDevice(ms->subs[(size_t)d]->device));
                const int r = ensure_rng(ms->subs[(size_t)d], mi, old_len * 4);
                if (r) return r;
            }
            return CVG_OK;
        }();
        if (rc == CVG_OK && e0->rng_len == old_len)            // at the size cap already
            return cvg_set_err(CVG_ERR_LIMIT, "RNG draw table exhausted (pathological rejection rate)");
    }
    if (rc) {
        const std::string msg = cvg_last_error();
        for (cvg_ctx* e : ms->subs) { cudaSetDevice(e->device); cudaStreamSynchronize(e->stream); }
        return cvg_set_err(rc, "cvg_find_homography_sharded, device %d: %s", ms->devices[(size_t)at], msg.c_str());
    }
    if (timing) {
        cudaSetDevice(e0->device);
        cudaEventElapsedTime(&e0->t_ransac, e0->ev[0], e0->ev[1]);
        e0->t_match = 0; e0->t_total = e0->t_ransac;
        cudaMemcpy(&e0->scored_pts, e0->d_scored, 8, cudaMemcpyDeviceToHost);   // the first GPU's share
    }
    return CVG_OK;
}

int cvg_last_exchange(const cvg_ctx* c, int* n_exchanges, float* exchange_ms)
{
    if (!c) return cvg_set_err(CVG_ERR_INVALID, "cvg_last_exchange: NULL context");
    if (n_exchanges) *n_exchanges = c->multi ? c->multi->n_exchanges : 0;
    if (exchange_ms) *exchange_ms = c->multi ? c->multi->exchange_ms : 0.f;
    return CVG_OK;
}

}  // extern "C"
