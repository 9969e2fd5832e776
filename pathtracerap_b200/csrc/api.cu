// api.cu - the C ABI of libptap.so (include/ptap.h): device context, arena, scene upload, render loop.
//
// Replaces Renderer::allocateOnGPU / renderLoop / renderImage / free (Renderer.cpp:15-148, 567-648) and
// GPUMemoryPool<T> (GPUMemoryPool.h:10-46).  Where the reference makes 12 cudaMallocManaged calls plus a managed
// copy of each pool object, and reaches every element through two dependent loads, this context owns ONE device
// arena per lifetime class (scene, frame), bump-allocated at 256 B alignment, and passes raw pointers by value.
// A whole iteration is enqueued without a host round trip: the active-ray count of every bounce lives in device
// memory (FrameState) and all kernels are persistent grids sized from the SM count.
#include <dlfcn.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "bvh_build.h"
#include "host_math.h"
#include "instance_math.h"
#include "kernels.cuh"

using namespace ptap;

namespace {

// Move-only owner of a CUDA handle (event, stream, device allocation): releases it when destroyed or given another one, and converts to
// the raw handle for the runtime's calls.  put() hands the runtime's create calls a place to write a new handle.
template <typename H> class Owned {
public:
    Owned() = default;
    Owned(Owned&& o) noexcept : h_(std::exchange(o.h_, nullptr)) {}
    ~Owned() { reset(); }
    void reset() { if (h_) release(h_); h_ = nullptr; }
    H* put() { reset(); return &h_; }
    operator H() const { return h_; }

private:
    static void release(cudaEvent_t e) { cudaEventDestroy(e); }
    static void release(cudaStream_t s) { cudaStreamDestroy(s); }
    static void release(void* p) { cudaFree(p); }
    H h_ = nullptr;
};
using Event = Owned<cudaEvent_t>;
using Stream = Owned<cudaStream_t>;
template <typename T> using DevMem = Owned<T*>;

// Bump allocation at 256 B alignment in one device allocation.  A buffer set is laid out by one function over an Arena& (its carve),
// which place() runs twice: a dry run that only counts the bytes, then, once they are reserved, the run that places the buffers.
struct Arena {
    DevMem<char> base;
    size_t cap = 0, used = 0;
    bool sizing = false;                 // a dry run: alloc() counts and returns nullptr
    cudaError_t reserve(size_t bytes)
    {
        used = 0;
        if (bytes <= cap) return cudaSuccess;
        cap = 0;
        const cudaError_t e = cudaMalloc(base.put(), bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    template <typename T> T* alloc(size_t count)
    {
        T* p = sizing ? nullptr : reinterpret_cast<T*>(base + used);
        used += (count * sizeof(T) + 255) & ~size_t(255);
        return p;
    }
    template <typename F> static size_t measure(F&& carve)
    {
        Arena dry;
        dry.sizing = true;
        carve(dry);
        return dry.used;
    }
    template <typename F> cudaError_t place(F&& carve)
    {
        const cudaError_t e = reserve(measure(carve));
        if (e == cudaSuccess) carve(*this);
        return e;
    }
};

}  // namespace

struct ptap_ctx {
    int device = 0;
    int sms = 148;
    // Multi-lane rendering (PTAP_LANES, default 4): iterations rotate over `lanes` wavefronts, each on its own stream, so that the drain
    // of one lane's persistent kernel (its last rays), its latency-bound scan and its ramp-up overlap the other lanes' kernels.
    // Film adds stay in iteration order (WaveDev::contrib + one ordered add per iteration).
    Stream streams[kMaxLanes];           // one per lane
    Stream& stream = streams[0];         // the context stream (lane 0's): everything but the other lanes of a render is enqueued here
    Event ev0, ev1, tm0, tm1;
    std::vector<Event> prof_events;
    std::vector<int> prof_kind;      // 0 generate, 1 trace, 2 shade  (pairs)
    size_t prof_used = 0;
    Arena scene_arena, frame_arena, scratch;
    SceneDev sc{};
    int lanes = 1;                       // lanes of the current render parameters
    int lanes_env = 0;                   // PTAP_LANES (0 = by frame size: kDefaultLanes, kSmallFrameLanes for frames of at most 2^20 pixels)
    WaveDev lane[kMaxLanes]{};           // valid for [0, lanes); iter_stride and contrib are set by each render for the lanes it uses
    float* contrib[kMaxLanes] = {};      // each lane's contribution buffer when lanes > 1 (WaveDev::contrib of a render on several lanes)
    Event e_fork, e_cache, e_join[kMaxLanes], e_gather[kMaxLanes];
    // host copies kept for the acceleration-structure builds
    std::vector<TriRec> h_tris;      // kept only when the BVH still has to be built here (no prebuilt one in the view)
    int ntris = 0;
    std::vector<PtapMesh> h_meshes;
    std::vector<PtapModel> h_models;
    std::vector<InstanceTrace> h_inst;
    InstanceTrace* d_inst = nullptr; TriRec* d_tris = nullptr; BvhNode* d_nodes = nullptr; size_t nodes_cap = 0; LeafTri* d_btris = nullptr; int* d_btid = nullptr;
    bool have_scene = false, have_grid = false, have_bvh = false, have_frame = false;
    int blas_nodes = 0, blas_depth = 0;   // BLAS nodes (the TLAS follows them in d_nodes) and BLAS levels of the BVH on the device
    int bvh_kind = -1;               // which builder made the BVH now on the device (PTAP_ACCEL_BVH / PTAP_ACCEL_BVH_DEVICE)
    int accel = PTAP_ACCEL_GRID_COMPAT;
    uint32_t flags = 0;
    bool cache_valid = false;
    int grid_trace = 0, grid_shade = 0, grid_gen = 0;
    int trace_ctas = 0;              // PTAP_TRACE_CTAS: CTAs per SM of the closest-hit kernels (0 = occupancy query)
    PtapStats stats{};
    PtapCamera camera{{0.0f, 0.0f, 920.0f}, {-10.0f, -4.0f, 900.0f}, {20.0f, 16.0f}, 0, 0u};      // Renderer.cpp:538-545
    std::vector<Event> iter_events;            // completion of every iteration of the last render call (PTAP_FLAG_ITER_TIMES)
    int iter_events_used = 0;
    std::vector<float> iter_ms;
    int emu_replay_ctas = 6, emu_walk_ctas = 2;
    Arena emu_arena; int emu_lanes = 0;          // PTAP_ACCEL_GRID_EMULATED: per-slot buffers of the render lanes
    DevMem<int2> d_tri_box; size_t tri_box_cap = 0; bool emu_ok = false;   // PTAP_ACCEL_GRID_EMULATED: per-triangle voxel boxes (own allocation)
    std::vector<int> h_grid_first, h_model_grid;     // first voxel of every grid on the device / grid of every model
    DevMem<int2> gd_cells; DevMem<int> gd_refs; size_t gd_ncells = 0, gd_nrefs = 0;   // grids built on the device (own allocation)
    void* nccl_comm = nullptr;                 // ptap_nccl_init
    Event e_peer;
    unsigned long long* d_stamps = nullptr;   // PTAP_FLAG_STAMP: (start, end) %globaltimer words of the closest-hit launches of the last render call
    int stamps_used = 0;
    bool render_pending = false;
    // ptap_query_*: scratch of their own (never an arena a render uses), the events that order them with the caller's stream, and
    // whether BVH occlusion takes the any-hit traversal.  Not an option of the ABI: an internal switch for the A/B measurement of
    // tools/bench_queries.py (PTAP_QUERY_ANYHIT=0 in the environment at ptap_create: closest hit + compare, the same answers)
    Arena query_arena;
    Event e_qin, e_qout;
    Arena update_arena;                  // ptap_update_models: the staged model records (never an arena a render uses)
    bool query_anyhit = true;
    std::string err;
};

namespace {

int fail(ptap_ctx* c, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (c) c->err = buf;
    return code;
}

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(ctx, (int)e_, "%s: %s", #call, cudaGetErrorString(e_));   \
    } while (0)

// fn(begin, end) over [0, n) on up to 8 host threads (the calling one included)
template <typename F> void parallelFor(int n, F fn)
{
    const int workers = n < (1 << 16) ? 1 : (int)std::min(8u, std::max(1u, std::thread::hardware_concurrency()));
    if (workers <= 1) { fn(0, n); return; }
    std::vector<std::thread> pool;
    const int chunk = (n + workers - 1) / workers;
    for (int w = 1; w < workers; ++w) pool.emplace_back([=]() { fn(std::min(n, w * chunk), std::min(n, (w + 1) * chunk)); });
    fn(0, std::min(n, chunk));
    for (std::thread& t : pool) t.join();
}

float4 row(const float* m, int r) { return make_float4(m[0 + r], m[4 + r], m[8 + r], m[12 + r]); }

constexpr int kMaxStamps = 8192;     // closest-hit launches of one render call that can be stamped (PTAP_FLAG_STAMP)

// emu: per-slot buffers of the emulated grid walk (PTAP_ACCEL_GRID_EMULATED only; see carveEmu / ensureEmuBuffers)
void launchTrace(ptap_ctx* c, FrameState* st, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, int round, int n_fixed,
                 const EmuBuf& emu, bool count_totals = false, cudaStream_t stream = nullptr, unsigned long long* stamp = nullptr)
{
    if (!stream) stream = c->stream;
    if (c->accel == PTAP_ACCEL_GRID_EMULATED) {
        // closest hit + the hits of the nearest model, then the replay of that model's walk (trace_emu.cu) ...
        launchTraceEmu(c->sc, O, D, hit, uv, counts, count_totals, st, round, n_fixed, c->grid_trace, c->sms * c->emu_replay_ctas, c->sms, stream, stamp, emu);
        // ... and the walk itself for the slots the replay could not confirm (the 0.3-0.6 % of rays on which the walk is not a closest-hit query)
        launchTraceGrid(c->sc, O, D, hit, uv, nullptr, false, st, round, n_fixed, c->sms, stream, nullptr, emu.list2);
    }
    else if (c->accel != PTAP_ACCEL_GRID_COMPAT) launchTraceBvh(c->sc, O, D, hit, uv, counts, count_totals, st, round, n_fixed, c->grid_trace, stream, stamp);
    else launchTraceGrid(c->sc, O, D, hit, uv, counts, count_totals, st, round, n_fixed, c->grid_trace, stream, stamp);
}

// Per-slot buffers of PTAP_ACCEL_GRID_EMULATED: hit count, kEmuHits x (triangle id, t), the list for the walk, the queue of replays in
// progress: 156 B per slot, plus 33 MB for the hits of grazing rays in k_emu_full.
// threads of a k_emu_full launch (one CTA per SM: it runs for ~0.5 % of the rays), each with kBigHits x 16 B of global memory for the hits of a grazing ray
size_t emuFullThreads(const ptap_ctx* c) { return (size_t)c->sms * kTraceBlock; }

EmuBuf carveEmu(const ptap_ctx* c, Arena& A, size_t n)
{
    EmuBuf e;
    e.n = A.alloc<int>(n); e.list = A.alloc<int>(n); e.list2 = A.alloc<int>(n); e.id = A.alloc<int>(n * kEmuHits); e.t = A.alloc<float>(n * kEmuHits); e.stride = (int)n;
    e.cont = A.alloc<uint4>(n * 5); e.cont_cap = (int)n;
    e.big = A.alloc<uint4>(emuFullThreads(c) * kBigHits);
    return e;
}

// The render lanes' buffers: one allocation of their own (the frame arena is sized before the acceleration structure is chosen), made
// the first time a frame is rendered through the emulation at this resolution.
int ensureEmuBuffers(ptap_ctx* ctx)
{
    if (ctx->accel != PTAP_ACCEL_GRID_EMULATED) return PTAP_OK;
    const size_t N = (size_t)ctx->lane[0].N;
    if (ctx->lane[0].emu.n && ctx->lane[0].emu.stride == (int)N && ctx->emu_lanes == ctx->lanes) return PTAP_OK;
    auto carve = [&](Arena& A) { for (int l = 0; l < ctx->lanes; ++l) ctx->lane[l].emu = carveEmu(ctx, A, N); };
    CK(ctx->emu_arena.place(carve));
    ctx->emu_lanes = ctx->lanes;
    return PTAP_OK;
}

void profMark(ptap_ctx* c, int kind)
{
    if (!(c->flags & PTAP_FLAG_PROFILE)) return;
    if (c->prof_used == c->prof_events.size()) {
        Event e; cudaEventCreate(e.put()); c->prof_events.push_back(std::move(e)); c->prof_kind.push_back(0);
    }
    c->prof_kind[c->prof_used] = kind;
    cudaEventRecord(c->prof_events[c->prof_used++], c->stream);
}

// zeroes the per-frame counters; what describes the uploaded scene and its acceleration structure stays
void resetStats(ptap_ctx* c)
{
    const PtapStats old = c->stats;
    c->stats = PtapStats{};
    c->stats.scene_bytes = old.scene_bytes; c->stats.ms_build = old.ms_build; c->stats.bvh_nodes = old.bvh_nodes; c->stats.bvh_depth = old.bvh_depth;
    c->stats.lanes = c->lanes;
}

// camera numbers into a wavefront descriptor: step = span / resolution in double, rounded once (Renderer.cpp:538-539, SAMPLESX = SAMPLESY = 1)
void applyCamera(const ptap_ctx* c, WaveDev& wv)
{
    wv.step_x = (float)((double)c->camera.span[0] / (double)wv.W);
    wv.step_y = (float)((double)c->camera.span[1] / (double)wv.H);
    for (int k = 0; k < 3; ++k) { wv.cam_o[k] = c->camera.origin[k]; wv.cam_p[k] = c->camera.plane_min[k]; }
    wv.jitter = c->camera.jitter; wv.jitter_seed = c->camera.jitter_seed;
}

int traceGridSize(ptap_ctx* c)
{
    int occ = c->accel == PTAP_ACCEL_GRID_EMULATED ? traceEmuOccupancy() : c->accel != PTAP_ACCEL_GRID_COMPAT ? traceBvhOccupancy() : traceGridOccupancy();
    if (c->trace_ctas > 0) occ = std::min(occ, c->trace_ctas);
    return c->sms * std::max(occ, 1);
}

// Length of the union of the intervals [first, second] (sorts them)
double unionLength(std::vector<std::pair<unsigned long long, unsigned long long>>& iv)
{
    std::sort(iv.begin(), iv.end());
    double len = 0.0; unsigned long long cur_b = 0, cur_e = 0; bool open = false;
    for (auto& x : iv) {
        if (!open) { cur_b = x.first; cur_e = x.second; open = true; }
        else if (x.first <= cur_e) cur_e = std::max(cur_e, x.second);
        else { len += (double)(cur_e - cur_b); cur_b = x.first; cur_e = x.second; }
    }
    if (open) len += (double)(cur_e - cur_b);
    return len;
}

int collect(ptap_ctx* ctx)
{
    if (!ctx->render_pending) return PTAP_OK;
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->render_pending = false;
    CK(cudaEventElapsedTime(&ctx->stats.ms_render, ctx->ev0, ctx->ev1));
    // counters summed over the lanes; the rounds reported are those of the latest iteration: of the lane with the latest iter_cur that
    // ran paths (ties to the lower lane)
    FrameState sum{}, last{};
    for (int l = 0; l < ctx->lanes; ++l) {
        FrameState f;
        CK(cudaMemcpy(&f, ctx->lane[l].st, sizeof f, cudaMemcpyDeviceToHost));
        if (l == 0 || (f.iter_cur > last.iter_cur && f.paths > 0)) last = f;
        sum.rays_traced += f.rays_traced; sum.rays_walked += f.rays_walked; sum.rays_reemulated += f.rays_reemulated; sum.paths += f.paths;
        sum.count_nodes += f.count_nodes; sum.count_tris += f.count_tris; sum.count_cells += f.count_cells; sum.count_refs += f.count_refs;
    }
    ctx->stats.rays_traced = (int64_t)sum.rays_traced;
    ctx->stats.rays_walked = (int64_t)sum.rays_walked;
    ctx->stats.rays_reemulated = (int64_t)sum.rays_reemulated;
    ctx->stats.paths = (int64_t)sum.paths;
    for (int i = 0; i < 16; ++i) ctx->stats.active_per_round[i] = i <= kMaxDepth ? last.n_active[i] : 0;
    const double rt = sum.rays_traced ? (double)sum.rays_traced : 1.0;
    ctx->stats.avg_nodes = (float)(sum.count_nodes / rt); ctx->stats.avg_tris = (float)(sum.count_tris / rt);
    ctx->stats.avg_cells = (float)(sum.count_cells / rt); ctx->stats.avg_refs = (float)(sum.count_refs / rt);
    ctx->stats.ms_generate = ctx->stats.ms_trace = ctx->stats.ms_shade = 0.f;
    for (size_t i = 0; i + 1 < ctx->prof_used; ++i) {          // event i -> i+1 spans the kernel of kind[i]
        float ms = 0.f;
        if (ctx->prof_kind[i] < 0) continue;
        cudaEventElapsedTime(&ms, ctx->prof_events[i], ctx->prof_events[i + 1]);
        if (ctx->prof_kind[i] == 0) ctx->stats.ms_generate += ms;
        else if (ctx->prof_kind[i] == 1) ctx->stats.ms_trace += ms;
        else ctx->stats.ms_shade += ms;
    }
    ctx->prof_used = 0;
    ctx->iter_ms.assign(ctx->iter_events_used, 0.f);
    for (int k = 0; k < ctx->iter_events_used; ++k) cudaEventElapsedTime(&ctx->iter_ms[k], ctx->ev0, ctx->iter_events[k]);
    ctx->iter_events_used = 0;
    ctx->stats.ms_trace_inflight = ctx->stats.ms_trace_sum = 0.f;
    if (ctx->stamps_used > 0 && ctx->d_stamps) {
        // closest-hit launches of the call as [start, end] intervals on the device's nanosecond clock: their summed lengths, and the length
        // of their union (time during which at least one closest-hit kernel was resident - lanes overlap, so the union is what a rate may
        // be divided by)
        std::vector<unsigned long long> h((size_t)ctx->stamps_used * 2);
        CK(cudaMemcpy(h.data(), ctx->d_stamps, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        std::vector<std::pair<unsigned long long, unsigned long long>> iv;
        double sum = 0.0;
        for (int k = 0; k < ctx->stamps_used; ++k)
            if (h[2 * k + 1] >= h[2 * k]) { iv.push_back({h[2 * k], h[2 * k + 1]}); sum += (double)(h[2 * k + 1] - h[2 * k]); }
        ctx->stats.ms_trace_inflight = (float)(unionLength(iv) * 1e-6); ctx->stats.ms_trace_sum = (float)(sum * 1e-6);
        ctx->stamps_used = 0;
    }
    return PTAP_OK;
}

struct TlasItem { float lo[3], hi[3]; int inst; };

float boxArea(const float* lo, const float* hi)
{
    const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return 2.f * (dx * dy + dy * dz + dz * dx);
}

// Median-split binary tree over the instances' world boxes (collapsed to 4-wide nodes afterwards); leaves are single instances
// (link ~(0x20000000 | model)).
int buildTlas(std::vector<TlasItem>& items, int b, int e, std::vector<Bvh2Node>& nodes, float* lo, float* hi)
{
    for (int k = 0; k < 3; ++k) { lo[k] = 3e38f; hi[k] = -3e38f; }
    for (int i = b; i < e; ++i)
        for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], items[i].lo[k]); hi[k] = std::max(hi[k], items[i].hi[k]); }
    if (e - b == 1) return ~(0x20000000 | items[b].inst);
    int axis = 0; float best = -1.f;
    for (int k = 0; k < 3; ++k) {
        float cmin = 3e38f, cmax = -3e38f;
        for (int i = b; i < e; ++i) { const float c = items[i].lo[k] + items[i].hi[k]; cmin = std::min(cmin, c); cmax = std::max(cmax, c); }
        if (cmax - cmin > best) { best = cmax - cmin; axis = k; }
    }
    const int mid = (b + e) / 2;
    std::nth_element(items.begin() + b, items.begin() + mid, items.begin() + e,
                     [axis](const TlasItem& x, const TlasItem& y) { return x.lo[axis] + x.hi[axis] < y.lo[axis] + y.hi[axis]; });
    const int me = (int)nodes.size();
    nodes.emplace_back();
    float l0[3], h0[3], l1[3], h1[3];
    int c0 = buildTlas(items, b, mid, nodes, l0, h0);
    int c1 = buildTlas(items, mid, e, nodes, l1, h1);
    if (boxArea(l1, h1) < boxArea(l0, h0)) {          // equal entry distances (origin inside both): visit the smaller box first
        std::swap(c0, c1);
        for (int k = 0; k < 3; ++k) { std::swap(l0[k], l1[k]); std::swap(h0[k], h1[k]); }
    }
    Bvh2Node& nd = nodes[me];
    nd.xy0 = make_float4(l0[0], h0[0], l0[1], h0[1]);
    nd.xy1 = make_float4(l1[0], h1[0], l1[1], h1[1]);
    nd.z01 = make_float4(l0[2], h0[2], l1[2], h1[2]);
    nd.link = make_int4(c0, c1, 0, 0);
    return me;
}

// Both builders write the scene arena's nodes in place: from then on the tree that was there is gone, and until the new one is complete
// (finishBvh) there is none to trace.  A build that fails - a tree too deep for the traversal stack, say - leaves the context without a
// BVH, and every entry point that would traverse one refuses (checkState).
void dropBvh(ptap_ctx* ctx)
{
    ctx->have_bvh = false; ctx->bvh_kind = -1; ctx->sc.tlas_root = -1;
}

// What an entry point needs of the context's state: an uploaded scene, render parameters, the acceleration structure of the current mode.
enum : unsigned { kScene = 1, kFrame = 2, kAccel = 4 };

// The state checks of the entry points, always in this order.  kAccel: the grid modes walk the grids; the BVH modes and the emulated grid
// walk traverse the BVH.
int checkState(ptap_ctx* ctx, const char* call, unsigned need)
{
    if ((need & kFrame) && (!ctx || !ctx->have_frame || ((need & kScene) && !ctx->have_scene)))
        return fail(ctx, PTAP_E_STATE, (need & kScene) ? "%s: scene and render parameters required" : "%s: no render parameters", call);
    if ((need & kScene) && (!ctx || !ctx->have_scene)) return fail(ctx, PTAP_E_STATE, "%s: no scene uploaded", call);
    if (need & kAccel) {
        if ((ctx->accel == PTAP_ACCEL_GRID_COMPAT || ctx->accel == PTAP_ACCEL_GRID_EMULATED) && !ctx->have_grid) return fail(ctx, PTAP_E_STATE, "%s: no grid in the uploaded scene", call);
        if (ctx->accel != PTAP_ACCEL_GRID_COMPAT && !ctx->have_bvh) return fail(ctx, PTAP_E_STATE, "%s: no BVH on the device (build_accel failed or was not called)", call);
    }
    return PTAP_OK;
}

// The preamble of an entry point that enqueues work: its state checks, then the context's device made current and a render still in
// flight collected.  Entry points that check arguments between the two call checkState first and enter(ctx) after.
int enter(ptap_ctx* ctx, const char* call = nullptr, unsigned need = 0)
{
    if (const int rc = checkState(ctx, call, need)) return rc;
    CK(cudaSetDevice(ctx->device));
    return collect(ctx);
}

// Times a build on the context stream into stats.ms_build: start() records its beginning, stop() its end, waits for it and stores the
// time.  A build that fails in between leaves ms_build as it was; the events go with the timer.
struct BuildTimer {
    ptap_ctx* ctx;
    Event b0, b1;
    int start() { CK(cudaEventCreate(b0.put())); CK(cudaEventCreate(b1.put())); CK(cudaEventRecord(b0, ctx->stream)); return PTAP_OK; }
    int stop() { CK(cudaEventRecord(b1, ctx->stream)); CK(cudaEventSynchronize(b1)); cudaEventElapsedTime(&ctx->stats.ms_build, b0, b1); return PTAP_OK; }
};

// The scene constants of the traversal from the instances' terms (instance_math.h), reduced over the models that have triangles:
// max_scale and max_pad over all of them, max_trans over the models up to and including the first whose matrices are not inverses.
void setSceneConstants(ptap_ctx* ctx, double max_scale, double max_pad, double max_trans, bool consistent)
{
    ctx->sc.tmin_world = -(float)((kEpsilon + 2e-4) * max_scale * 1.001 + max_pad + 1e-3);
    ctx->sc.prune = consistent ? 1.0003f : INFINITY;
    ctx->sc.tie = consistent ? 1.5e-4f : INFINITY;
    // residual of matrices that passed the check: |(M W - I) [o; 1]| <= 2e-5 * sqrt(3) * (|o|_1 + max |translation|); the kernel adds 1e-4 |o|_1
    ctx->sc.c_pad = (float)(4e-5 * max_trans + 1e-3);
}

// Second half of every BVH build: points every model at its mesh's root, derives the instances' world boxes from the BLAS root bounds
// (`roots[m]` = host copy of mesh m's root node), builds the TLAS over them behind the `nnodes` BLAS nodes and publishes the scene fields.
int finishBvh(ptap_ctx* ctx, const BvhNode* roots, const int* mesh_root, int nnodes, int blas_depth, size_t* tlas_bytes)
{
    const int nm = (int)ctx->h_models.size();
    std::vector<TlasItem> items;
    double max_scale = 0.0, max_pad = 0.0, max_trans = 1.0;
    bool consistent = true;
    for (int i = 0; i < nm; ++i) {
        const PtapModel& m = ctx->h_models[i];
        const int root = mesh_root[m.mesh_index];
        ctx->h_inst[i].grid.z = __builtin_bit_cast(float, root);
        if (root < 0) continue;
        InstanceBox b;
        if (!instanceBox(m.world_to_model, m.model_to_world, roots[m.mesh_index], b)) return fail(ctx, PTAP_E_INVALID, "model %d: world_to_model is singular", i);
        if (consistent) { max_trans = std::max(max_trans, b.trans); consistent = b.consistent; }
        TlasItem it; it.inst = i;
        for (int k = 0; k < 3; ++k) { it.lo[k] = b.lo[k]; it.hi[k] = b.hi[k]; }
        items.push_back(it);
        max_scale = std::max(max_scale, b.scale);
        max_pad = std::max(max_pad, b.pad);
    }
    std::vector<BvhNode> tlas;
    int tlas_root = -1, tlas_depth = 0;
    if (!items.empty()) {
        float lo[3], hi[3];
        std::vector<Bvh2Node> t2;
        const int link = buildTlas(items, 0, (int)items.size(), t2, lo, hi);
        if (link < 0) {                                   // a single instance: a root with one child
            Bvh2Node nd;
            nd.xy0 = make_float4(lo[0], hi[0], lo[1], hi[1]); nd.xy1 = nd.xy0;
            nd.z01 = make_float4(lo[2], hi[2], lo[2], hi[2]);
            nd.link = make_int4(link, link, 0, 0);
            t2.push_back(nd);
        }
        tlas_root = collapseBvh2(t2.data(), link < 0 ? (int)t2.size() - 1 : link, tlas, nnodes, 1, tlas_depth);
    }
    if (3 * (blas_depth + tlas_depth) + 8 > kBvhStack) return fail(ctx, PTAP_E_INVALID, "BVH too deep for the traversal stack (%d + %d levels, %d entries)", blas_depth, tlas_depth, kBvhStack);
    if (nnodes + tlas.size() > ctx->nodes_cap) return fail(ctx, PTAP_E_NOMEM, "BVH node storage exhausted");
    CK(cudaMemcpyAsync(ctx->d_inst, ctx->h_inst.data(), nm * sizeof(InstanceTrace), cudaMemcpyHostToDevice, ctx->stream));
    if (!tlas.empty()) CK(cudaMemcpyAsync(ctx->d_nodes + nnodes, tlas.data(), tlas.size() * sizeof(BvhNode), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));      // tlas is stack-owned
    if (tlas_bytes) *tlas_bytes = nm * sizeof(InstanceTrace) + tlas.size() * sizeof(BvhNode);
    ctx->sc.tlas_root = tlas_root;
    setSceneConstants(ctx, max_scale, max_pad, max_trans, consistent);
    ctx->blas_nodes = nnodes; ctx->blas_depth = blas_depth;
    ctx->have_bvh = true;
    return PTAP_OK;
}

// Copies a BVH (nodes, leaf order) into the scene arena, gathers the leaf-ordered triangle records, points every model at
// its mesh's root, derives the instances' world boxes from the BLAS root bounds and builds the TLAS over them.
int uploadBvh(ptap_ctx* ctx, const BvhNode* nodes, int nnodes, const int* tri_id, const int* mesh_root, size_t* bytes)
{
    const int nt = ctx->ntris, nm = (int)ctx->h_models.size();
    dropBvh(ctx);
    if ((size_t)nnodes > ctx->nodes_cap) return fail(ctx, PTAP_E_NOMEM, "BVH has more nodes than reserved (2 per triangle)");
    // range checks of every link and leaf-order entry: 90 MB of host memory for a 1.3 M-triangle scene, on every upload - spread over threads
    {
        std::atomic<int> bad_node{-1}, bad_leaf{-1}, bad_entry{-1};
        parallelFor(nnodes, [&](int b, int e) {
            for (int i = b; i < e; ++i)
                for (int k = 0; k < 4; ++k) {
                    const int l = nodes[i].link[k];
                    if (l >= nnodes) bad_node = i;
                    if (l < 0) { const int code = ~l, first = code >> 3, cnt = (code & 7) + 1; if (code >= 0x20000000 || first < 0 || first + cnt > nt) bad_leaf = i; }
                }
        });
        parallelFor(nt, [&](int b, int e) { for (int k = b; k < e; ++k) if (tri_id[k] < 0 || tri_id[k] >= nt) bad_entry = k; });
        if (bad_node >= 0) return fail(ctx, PTAP_E_INVALID, "BVH node %d: child index out of range", bad_node.load());
        if (bad_leaf >= 0) return fail(ctx, PTAP_E_INVALID, "BVH node %d: leaf range out of bounds", bad_leaf.load());
        if (bad_entry >= 0) return fail(ctx, PTAP_E_INVALID, "BVH leaf order entry %d out of range", bad_entry.load());
    }
    for (size_t m = 0; m < ctx->h_meshes.size(); ++m)
        if (mesh_root[m] >= nnodes) return fail(ctx, PTAP_E_INVALID, "mesh %d: BVH root out of range", (int)m);
    // Depth of every BLAS (the traversal stack is fixed-size).  Always computed from the nodes: a caller-supplied depth is only a hint that
    // must not be trusted (an understated one would overflow the per-thread stack); the pass also rejects cycles and shared nodes.
    int blas_depth = 0;
    {
        // the builders emit parents before children, so one forward sweep gives every node's level; any other order takes the stack walk
        std::vector<int> level(nnodes, 0);
        bool ordered = true;
        for (size_t m = 0; m < ctx->h_meshes.size(); ++m) {
            if (mesh_root[m] < 0) continue;
            if (level[mesh_root[m]]) return fail(ctx, PTAP_E_INVALID, "BVH node %d is the root of two meshes", mesh_root[m]);
            level[mesh_root[m]] = 1;
        }
        for (int i = 0; i < nnodes && ordered; ++i) {
            if (!level[i]) continue;
            blas_depth = std::max(blas_depth, level[i]);
            for (int k = 0; k < 4; ++k) {
                const int l = nodes[i].link[k];
                if (l < 0 || !slotUsed(nodes[i], k)) continue;
                if (l <= i) { ordered = false; break; }
                if (level[l]) return fail(ctx, PTAP_E_INVALID, "BVH node %d is reachable twice", l);
                level[l] = level[i] + 1;
            }
        }
        if (!ordered) {
            blas_depth = 0;
            std::vector<std::pair<int, int>> todo;
            std::vector<char> seen(nnodes, 0);
            for (size_t m = 0; m < ctx->h_meshes.size(); ++m) if (mesh_root[m] >= 0) todo.push_back({mesh_root[m], 1});
            while (!todo.empty()) {
                const auto [node, d] = todo.back(); todo.pop_back();
                if (seen[node]) return fail(ctx, PTAP_E_INVALID, "BVH node %d is reachable twice", node);
                seen[node] = 1;
                blas_depth = std::max(blas_depth, d);
                for (int k = 0; k < 4; ++k)
                    if (nodes[node].link[k] >= 0 && slotUsed(nodes[node], k)) todo.push_back({nodes[node].link[k], d + 1});
            }
        }
    }
    std::vector<BvhNode> roots(ctx->h_meshes.size());
    for (size_t m = 0; m < roots.size(); ++m)
        if (mesh_root[m] >= 0) roots[m] = nodes[mesh_root[m]];
    CK(cudaMemcpyAsync(ctx->d_nodes, nodes, (size_t)nnodes * sizeof(BvhNode), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_btid, tri_id, (size_t)nt * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    launchGatherTris(ctx->d_tris, ctx->d_btid, nt, ctx->d_btris, ctx->stream);     // leaf-order copies are made on the device
    size_t tb = 0;
    const int rc = finishBvh(ctx, roots.data(), mesh_root, nnodes, blas_depth, &tb);
    if (rc) return rc;
    if (bytes) *bytes = tb + (size_t)nnodes * sizeof(BvhNode) + (size_t)nt * sizeof(int);
    ctx->bvh_kind = PTAP_ACCEL_BVH;
    return PTAP_OK;
}

// PTAP_ACCEL_BVH_DEVICE: every mesh's BLAS is built on the GPU (bvh_device.cu) straight into the scene arena; only the root nodes come back
// to the host, for the TLAS.
int buildBvhOnDevice(ptap_ctx* ctx)
{
    const int nt = ctx->ntris, nmesh = (int)ctx->h_meshes.size();
    dropBvh(ctx);
    int max_tris = 0;
    for (const PtapMesh& m : ctx->h_meshes) max_tris = std::max(max_tris, m.t_end - m.t_start);
    CK(ctx->scratch.reserve(deviceBvhScratchBytes(max_tris)));
    std::vector<int> mesh_root(nmesh, -1);
    int nnodes = 0, leaf_base = 0, blas_depth = 0;
    for (int mi = 0; mi < nmesh; ++mi) {
        const PtapMesh& m = ctx->h_meshes[mi];
        const int n = m.t_end - m.t_start;
        if (n <= 0 || m.t_start < 0 || m.t_end > nt) continue;
        if ((size_t)nnodes + (size_t)n > ctx->nodes_cap || leaf_base + n > nt) return fail(ctx, PTAP_E_NOMEM, "device BVH build: node / leaf storage exhausted");
        int made = 0, depth = 0;
        std::string why;
        const int e = buildMeshBvhDevice(ctx->d_tris, m.t_start, m.t_end, m.bb_min, m.bb_max, nnodes, ctx->d_nodes + nnodes, leaf_base, ctx->d_btris, ctx->d_btid,
                                         ctx->scratch.base, ctx->scratch.cap, ctx->stream, &made, &depth, &why);
        if (e != 0) return fail(ctx, e, "device BVH build of mesh %d (%d triangles): %s", mi, n, why.empty() ? cudaGetErrorString((cudaError_t)e) : why.c_str());
        mesh_root[mi] = nnodes;
        nnodes += made; leaf_base += n; blas_depth = std::max(blas_depth, depth);
    }
    std::vector<BvhNode> roots(nmesh);
    for (int mi = 0; mi < nmesh; ++mi)
        if (mesh_root[mi] >= 0) CK(cudaMemcpyAsync(&roots[mi], ctx->d_nodes + mesh_root[mi], sizeof(BvhNode), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int rc = finishBvh(ctx, roots.data(), mesh_root.data(), nnodes, blas_depth, nullptr);
    if (rc) return rc;
    ctx->bvh_kind = PTAP_ACCEL_BVH_DEVICE;
    ctx->stats.bvh_nodes = nnodes; ctx->stats.bvh_depth = blas_depth;
    return PTAP_OK;
}

}  // namespace

extern "C" {

int ptap_create(int device, size_t arena_bytes, ptap_ctx** out)
{
    if (!out) return PTAP_E_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return PTAP_E_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return PTAP_E_NO_DEVICE;
    if (prop.major < 10) return PTAP_E_NO_DEVICE;              // sm_100a code only; no fallback path exists
    ptap_ctx* ctx = new ptap_ctx();
    ctx->device = device;
    ctx->sms = prop.multiProcessorCount;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(ctx->stream.put(), cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx; return PTAP_E_NO_DEVICE;
    }
    cudaEventCreate(ctx->ev0.put()); cudaEventCreate(ctx->ev1.put());
    auto envInt = [](const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; };
    ctx->sc.vote_tri = std::min(32, std::max(1, envInt("PTAP_VOTE_TRI", kVoteTri)));       // tuning knobs, see tools/tune_trace.py
    ctx->sc.vote_inst = std::min(32, std::max(1, envInt("PTAP_VOTE_INST", kVoteInst)));
    ctx->sc.vote_refill = std::min(32, std::max(1, envInt("PTAP_VOTE_REFILL", kVoteRefill)));
    ctx->sc.batch = std::max(1, envInt("PTAP_BATCH", kTraceBatch));
    ctx->sc.vote_grid = std::min(32, std::max(1, envInt("PTAP_VOTE_GRID", kVoteGrid)));
    ctx->sc.shade_sort = envInt("PTAP_SHADE_SORT", 0) != 0;
    ctx->lanes_env = std::min(kMaxLanes, std::max(0, envInt("PTAP_LANES", 0)));
    ctx->lanes = ctx->lanes_env ? ctx->lanes_env : kDefaultLanes;
    const int max_lanes = ctx->lanes_env ? ctx->lanes_env : kMaxLanes;      // streams and events for every lane a frame may use
    if (max_lanes > 1) {
        bool ok = cudaEventCreateWithFlags(ctx->e_fork.put(), cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(ctx->e_cache.put(), cudaEventDisableTiming) == cudaSuccess;
        for (int l = 0; l < max_lanes; ++l) {
            if (l > 0) ok = ok && cudaStreamCreateWithFlags(ctx->streams[l].put(), cudaStreamNonBlocking) == cudaSuccess;
            ok = ok && cudaEventCreateWithFlags(ctx->e_join[l].put(), cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(ctx->e_gather[l].put(), cudaEventDisableTiming) == cudaSuccess;
        }
        if (!ok) { ptap_destroy(ctx); return PTAP_E_NOMEM; }
    }      // measured slower on every workload (profiles/r01/README.md): opt-in
    ctx->trace_ctas = std::max(0, envInt("PTAP_TRACE_CTAS", 0));
    ctx->emu_replay_ctas = std::max(1, envInt("PTAP_EMU_REPLAY_CTAS", 6));     // CTAs per SM of k_emu_tail (k_emu_setup: twice as many); tuning only
    ctx->emu_walk_ctas = std::max(1, envInt("PTAP_EMU_WALK_CTAS", 2));
    ctx->sc.emu_refill = std::min(32, std::max(1, envInt("PTAP_EMU_REFILL", 8)));
    ctx->query_anyhit = envInt("PTAP_QUERY_ANYHIT", 1) != 0;
    if (cudaEventCreateWithFlags(ctx->e_qin.put(), cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(ctx->e_qout.put(), cudaEventDisableTiming) != cudaSuccess) {
        ptap_destroy(ctx); return PTAP_E_NOMEM;
    }
    if (arena_bytes) {                                          // caller-sized arena: split 1/4 scene, 3/4 frame
        if (ctx->scene_arena.reserve(arena_bytes / 4) != cudaSuccess || ctx->frame_arena.reserve(arena_bytes - arena_bytes / 4) != cudaSuccess) {
            ptap_destroy(ctx); return PTAP_E_NOMEM;
        }
    }
    *out = ctx;
    return PTAP_OK;
}

void ptap_destroy(ptap_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (const Stream& s : ctx->streams) if (s) cudaStreamSynchronize(s);
    if (ctx->nccl_comm) ptap_nccl_finalize(ctx);
    delete ctx;                          // the owners release the context's events, streams and device memory
}

const char* ptap_last_error(const ptap_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }
void* ptap_stream(ptap_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int ptap_upload_scene(ptap_ctx* ctx, const PtapSceneView* v)
{
    if (!ctx || !v || !v->models || !v->meshes || !v->vertices || !v->triangles || v->nmodels <= 0) return fail(ctx, PTAP_E_INVALID, "upload_scene: missing arrays");
    if (const int rc = enter(ctx)) return rc;
    const bool timing = getenv("PTAP_UPLOAD_TIMING") != nullptr;          // host-side phases of this call on stderr (diagnostics)
    const auto t_begin = std::chrono::steady_clock::now();
    auto t_last = t_begin;
    auto lap = [&](const char* what) {
        if (!timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "ptap_upload_scene: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    const int nm = v->nmodels, nt = v->ntriangles;
    const bool grid = v->grids && v->voxels && v->refs && v->ngrids > 0;
    // the scene arena is about to be overwritten: whatever was uploaded before is gone even if this call fails half-way
    ctx->have_scene = false; ctx->have_grid = false; ctx->have_bvh = false; ctx->bvh_kind = -1; ctx->cache_valid = false; ctx->emu_ok = false;
    ctx->sc.tlas_root = -1; ctx->sc.nmodels = 0;
    for (int i = 0; i < nm; ++i) {
        const PtapModel& m = v->models[i];
        if (m.mesh_index < 0 || m.mesh_index >= v->nmeshes) return fail(ctx, PTAP_E_INVALID, "model %d: mesh_index %d out of range", i, m.mesh_index);
        if (grid && (m.grid_index < 0 || m.grid_index >= v->ngrids)) return fail(ctx, PTAP_E_INVALID, "model %d: grid_index %d out of range", i, m.grid_index);
    }
    const bool prepacked = v->tri_recs && v->n_tri_recs == nt;      // ptap_scene_build_bvh / ptap_scene_pack_triangles made the records (indices checked there)
    if (!prepacked)
        for (int t = 0; t < nt; ++t)
            for (int k = 0; k < 3; ++k)
                if (v->triangles[t].v[k] < 0 || v->triangles[t].v[k] >= v->nvertices) return fail(ctx, PTAP_E_INVALID, "triangle %d: vertex index out of range", t);

    // ---- repack on the host (DESIGN.md "Data layout")
    std::vector<InstanceTrace> inst(nm);
    std::vector<InstanceShade> shade(nm);
    for (int i = 0; i < nm; ++i) {
        const PtapModel& m = v->models[i];
        InstanceTrace& it = inst[i];
        for (int r = 0; r < 3; ++r) { it.w2m[r] = row(m.world_to_model, r); it.m2w[r] = row(m.model_to_world, r); }
        it.bb_min = make_float4(0, 0, 0, 1); it.bb_max = make_float4(0, 0, 0, 1); it.grid = make_float4(1, 0, 0, 0);
        if (grid) {
            const PtapGrid& g = v->grids[m.grid_index];
            // the bbox is reached through the grid's creating model, not the traced one (Renderer.cpp:245-249)
            int owner = g.entity_index;
            if (owner < 0 || owner >= nm) return fail(ctx, PTAP_E_INVALID, "grid %d: entity_index %d out of range", m.grid_index, owner);
            const PtapMesh& mesh = v->meshes[v->models[owner].mesh_index];
            it.bb_min = make_float4(mesh.bb_min[0], mesh.bb_min[1], mesh.bb_min[2], g.width[0]);
            it.bb_max = make_float4(mesh.bb_max[0], mesh.bb_max[1], mesh.bb_max[2], g.width[1]);
            it.grid.x = g.width[2];
            it.grid.y = __builtin_bit_cast(float, (int)g.v_start);
        }
        float nmx[9];
        hm::normal_matrix(m.model_to_world, nmx);
        shade[i].nm0 = make_float4(nmx[0], nmx[1], nmx[2], m.mat.color[0]);
        shade[i].nm1 = make_float4(nmx[3], nmx[4], nmx[5], m.mat.color[1]);
        shade[i].nm2 = make_float4(nmx[6], nmx[7], nmx[8], m.mat.color[2]);
        shade[i].mat = make_int4(m.mat.type, 0, 0, 0);
    }
    const TriRec* recs = static_cast<const TriRec*>(v->tri_recs);
    if (!prepacked) {
        ctx->h_tris.resize(nt);
        makeTriRecs(v->vertices, v->triangles, nt, ctx->h_tris.data());
        recs = ctx->h_tris.data();
    } else ctx->h_tris.clear();
    ctx->ntris = nt;
    ctx->h_meshes.assign(v->meshes, v->meshes + v->nmeshes);
    ctx->h_models.assign(v->models, v->models + nm);
    ctx->h_grid_first.clear(); ctx->h_model_grid.clear();
    if (grid) {
        for (int g = 0; g < v->ngrids; ++g) ctx->h_grid_first.push_back(v->grids[g].v_start);
        for (int i = 0; i < nm; ++i) ctx->h_model_grid.push_back(v->models[i].grid_index);
    }

    std::vector<int2> cells;
    if (grid) {
        cells.resize(v->nvoxels);
        for (int i = 0; i < v->nvoxels; ++i) {
            // a voxel whose entity_type is not TRIANGLE is never tested (Renderer.cpp:226): store an empty range
            const bool tri = v->voxels[i].entity_type == 2;
            cells[i] = tri ? make_int2(v->voxels[i].start, v->voxels[i].end) : make_int2(0, 0);
            if (tri && (v->voxels[i].start < 0 || v->voxels[i].end > v->nrefs)) return fail(ctx, PTAP_E_INVALID, "voxel %d: ref range out of bounds", i);
        }
        for (int i = 0; i < v->nrefs; ++i)
            if (v->refs[i] < 0 || v->refs[i] >= nt) return fail(ctx, PTAP_E_INVALID, "ref %d: triangle index out of range", i);
        if (v->grid_dim[0] <= 0 || v->grid_dim[1] <= 0 || v->grid_dim[2] <= 0) return fail(ctx, PTAP_E_INVALID, "grid_dim must be positive");
        const long long ncell = (long long)v->grid_dim[0] * v->grid_dim[1] * v->grid_dim[2];
        for (int g = 0; g < v->ngrids; ++g)
            if (v->grids[g].v_start < 0 || v->grids[g].v_start + ncell > v->nvoxels) return fail(ctx, PTAP_E_INVALID, "grid %d: voxel range out of bounds", g);
    }

    lap("validate + repack (host)");
    // ---- one arena for everything scene-lifetime; BVH storage is reserved up front (2T-1 BLAS nodes + 2M TLAS nodes bound)
    const size_t nodes_cap = (size_t)std::max(nt, 1) * 2 + (size_t)nm * 2 + 2;
    InstanceTrace* d_inst; InstanceShade* d_shade; TriRec* d_tris; LeafTri* d_btris; float4* d_normals; int* d_btid; BvhNode* d_nodes;
    int2* d_cells = nullptr; int* d_refs = nullptr;
    auto carve = [&](Arena& A) {
        d_inst = A.alloc<InstanceTrace>(nm);
        d_shade = A.alloc<InstanceShade>(nm);
        d_tris = A.alloc<TriRec>(nt);
        d_btris = A.alloc<LeafTri>(nt);
        d_normals = A.alloc<float4>(nt);
        d_btid = A.alloc<int>(nt);
        d_nodes = A.alloc<BvhNode>(nodes_cap);
        if (grid) { d_cells = A.alloc<int2>(v->nvoxels); d_refs = A.alloc<int>(v->nrefs); }
    };
    CK(ctx->scene_arena.place(carve));
    CK(cudaMemcpyAsync(d_inst, inst.data(), nm * sizeof(InstanceTrace), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_shade, shade.data(), nm * sizeof(InstanceShade), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_tris, recs, (size_t)nt * sizeof(TriRec), cudaMemcpyHostToDevice, ctx->stream));
    launchExtractNormals(d_tris, nt, d_normals, ctx->stream);
    ctx->d_tris = d_tris;
    if (grid) {
        CK(cudaMemcpyAsync(d_cells, cells.data(), cells.size() * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(d_refs, v->refs, v->nrefs * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    }
    size_t bytes = nm * (sizeof(InstanceTrace) + sizeof(InstanceShade)) + (size_t)nt * sizeof(TriRec) +
                   (grid ? cells.size() * sizeof(int2) + (size_t)v->nrefs * sizeof(int) : 0);
    ctx->h_inst = inst;
    ctx->d_inst = d_inst; ctx->d_nodes = d_nodes; ctx->nodes_cap = nodes_cap; ctx->d_btris = d_btris; ctx->d_btid = d_btid;
    ctx->have_bvh = false; ctx->bvh_kind = -1;
    lap("enqueue scene copies");
    if (v->bvh_nodes && v->n_bvh_nodes > 0 && v->bvh_tri_id && v->bvh_mesh_root) {
        if (v->n_bvh_tris != nt || v->n_bvh_roots != v->nmeshes) return fail(ctx, PTAP_E_INVALID, "upload_scene: prebuilt BVH does not match the triangle / mesh counts");
        size_t bb = 0;
        int rc = uploadBvh(ctx, reinterpret_cast<const BvhNode*>(v->bvh_nodes), v->n_bvh_nodes, v->bvh_tri_id, v->bvh_mesh_root, &bb);
        if (rc) return rc;
        bytes += bb;
    }
    lap("BVH checks + TLAS (host)");
    CK(cudaStreamSynchronize(ctx->stream));
    lap("wait for the device");
    ctx->stats.scene_bytes = (int64_t)bytes;
    ctx->sc.inst = d_inst; ctx->sc.shade = d_shade; ctx->sc.tris = d_tris; ctx->sc.normals = d_normals;
    ctx->sc.cells = d_cells; ctx->sc.refs = d_refs; ctx->sc.nodes = d_nodes; ctx->sc.bvh_tris = d_btris; ctx->sc.bvh_tri_id = d_btid;
    ctx->sc.nmodels = nm; ctx->sc.gx = v->grid_dim[0]; ctx->sc.gy = v->grid_dim[1]; ctx->sc.gz = v->grid_dim[2];
    ctx->have_scene = true; ctx->have_grid = grid; ctx->cache_valid = false;
    ctx->accel = grid ? PTAP_ACCEL_GRID_COMPAT : PTAP_ACCEL_BVH;
    ctx->grid_trace = 0;
    return PTAP_OK;
}

int ptap_build_accel(ptap_ctx* ctx, int kind)
{
    if (const int rc = enter(ctx, "build_accel", kScene)) return rc;
    if (kind == PTAP_ACCEL_GRID_COMPAT) {
        if (!ctx->have_grid) return fail(ctx, PTAP_E_STATE, "build_accel: the uploaded scene carries no grids (call ptap_scene_build_grids first)");
    } else if (kind == PTAP_ACCEL_BVH) {
        if (!ctx->have_bvh || ctx->bvh_kind != PTAP_ACCEL_BVH) {
            BvhBuildResult res;
            if ((int)ctx->h_tris.size() != ctx->ntris) {        // the view brought prepacked records: read them back from the device
                ctx->h_tris.resize(ctx->ntris);
                CK(cudaMemcpyAsync(ctx->h_tris.data(), ctx->d_tris, (size_t)ctx->ntris * sizeof(TriRec), cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
            }
            buildSceneBvh(ctx->h_tris.data(), (int)ctx->h_tris.size(), ctx->h_meshes.data(), (int)ctx->h_meshes.size(), res);
            int rc = uploadBvh(ctx, res.nodes.data(), (int)res.nodes.size(), res.tri_id.data(), res.mesh_root.data(), nullptr);
            if (rc) return rc;
            CK(cudaStreamSynchronize(ctx->stream));
        }
    } else if (kind == PTAP_ACCEL_BVH_DEVICE) {
        if (ctx->bvh_kind != PTAP_ACCEL_BVH_DEVICE) {
            BuildTimer timer{ctx};
            int rc = timer.start();
            if (!rc) rc = buildBvhOnDevice(ctx);
            if (!rc) rc = timer.stop();
            if (rc) return rc;
        }
    } else if (kind == PTAP_ACCEL_GRID_EMULATED) {
        // the walk's results through the BVH (trace_emu.cu): needs the grids (their lists define the result), a BVH over the same triangles
        // (whichever builder made the one on the device; else the device builder), and lists of the shape the emulation relies on
        if (!ctx->have_grid) return fail(ctx, PTAP_E_STATE, "build_accel: the uploaded scene carries no grids (call ptap_scene_build_grids first)");
        if (!ctx->have_bvh) { const int rc = buildBvhOnDevice(ctx); if (rc) return rc; }
        if (!ctx->emu_ok) {
            const int nt = ctx->ntris, ng = (int)ctx->h_grid_first.size();
            if ((size_t)nt > ctx->tri_box_cap) {
                ctx->tri_box_cap = 0;
                CK(cudaMalloc(ctx->d_tri_box.put(), (size_t)std::max(nt, 1) * sizeof(int2)));
                ctx->tri_box_cap = (size_t)nt;
            }
            std::vector<int> range(2 * (size_t)std::max(ng, 1), 0);
            int ok = 0;
            const int e = gridTriBoxes(ctx->sc.cells, ctx->sc.refs, ng, ctx->h_grid_first.data(), ctx->sc.gx, ctx->sc.gy, ctx->sc.gz, nt, ctx->d_tri_box, range.data(), &ok, ctx->stream);
            if (e != 0) return fail(ctx, e, "build_accel: voxel boxes: %s", cudaGetErrorString((cudaError_t)e));
            if (!ok) return fail(ctx, PTAP_E_UNSUPPORTED, "build_accel: the voxel lists are not box-shaped ascending registrations of one grid per triangle; use PTAP_ACCEL_GRID_COMPAT");
            // every triangle a model's grid lists must belong to the model's own mesh (the BVH the emulation traverses is the mesh's)
            for (size_t i = 0; i < ctx->h_models.size(); ++i) {
                const int g = ctx->h_model_grid[i];
                const PtapMesh& mesh = ctx->h_meshes[ctx->h_models[i].mesh_index];
                if (range[2 * g] <= range[2 * g + 1] && (range[2 * g] < mesh.t_start || range[2 * g + 1] >= mesh.t_end))
                    return fail(ctx, PTAP_E_UNSUPPORTED, "build_accel: grid %d lists triangles outside the mesh of model %d; use PTAP_ACCEL_GRID_COMPAT", g, (int)i);
            }
            ctx->sc.tri_box = ctx->d_tri_box;
            ctx->emu_ok = true;
        }
    } else return fail(ctx, PTAP_E_INVALID, "build_accel: unknown kind %d", kind);
    ctx->accel = kind;
    ctx->cache_valid = false;
    ctx->grid_trace = traceGridSize(ctx);
    return PTAP_OK;
}

int ptap_update_models(ptap_ctx* ctx, const PtapModel* models, int32_t first, int32_t count)
{
    if (const int rc = checkState(ctx, "update_models", kScene)) return rc;
    const int nm = (int)ctx->h_models.size();
    if (count < 0 || first < 0 || first > nm - count) return fail(ctx, PTAP_E_INVALID, "update_models: models [%d, %d + %d) out of range (%d models)", first, first, count, nm);
    if (count == 0) return PTAP_OK;
    if (!models) return fail(ctx, PTAP_E_INVALID, "update_models: missing models");
    // every check before anything changes: a rejected call leaves the context tracing as before
    for (int k = 0; k < count; ++k) {
        const PtapModel& m = models[k];
        const PtapModel& was = ctx->h_models[first + k];
        if (m.mesh_index != was.mesh_index) return fail(ctx, PTAP_E_INVALID, "update_models: model %d: mesh_index %d differs from the uploaded %d (ptap_upload_scene changes it)", first + k, m.mesh_index, was.mesh_index);
        if (m.grid_index != was.grid_index) return fail(ctx, PTAP_E_INVALID, "update_models: model %d: grid_index %d differs from the uploaded %d (ptap_upload_scene changes it)", first + k, m.grid_index, was.grid_index);
        double w3[9], wi[9];
        linearPart(m.world_to_model, w3);
        if (!invert3(w3, wi)) return fail(ctx, PTAP_E_INVALID, "update_models: model %d: world_to_model is singular", first + k);
    }
    const bool tlas = ctx->have_bvh;
    int ninst = 0;                               // models with triangles: the leaves of the TLAS
    for (const InstanceTrace& it : ctx->h_inst) ninst += __builtin_bit_cast(int, it.grid.z) >= 0;
    if (tlas && (size_t)ctx->blas_nodes + std::max(ninst - 1, 1) > ctx->nodes_cap) return fail(ctx, PTAP_E_NOMEM, "update_models: BVH node storage exhausted");
    if (const int rc = enter(ctx)) return rc;

    // the host copies first: finishBvh and ptap_build_grids_device upload d_inst from h_inst
    std::copy(models, models + count, ctx->h_models.begin() + first);
    for (int k = 0; k < count; ++k)
        for (int r = 0; r < 3; ++r) { ctx->h_inst[first + k].w2m[r] = row(models[k].world_to_model, r); ctx->h_inst[first + k].m2w[r] = row(models[k].model_to_world, r); }
    ctx->cache_valid = false;
    auto failed = [&](int code, const char* what) {
        if (!tlas) return fail(ctx, code, "update_models: %s", what);
        dropBvh(ctx);
        return fail(ctx, code, "update_models: %s; the BVH was dropped: call ptap_build_accel", what);
    };
    PtapModel* staged = nullptr;
    cudaError_t e = ctx->update_arena.place([&](Arena& A) { staged = A.alloc<PtapModel>(count); });
    if (e == cudaSuccess) e = cudaMemcpyAsync(staged, models, (size_t)count * sizeof(PtapModel), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && tlas) e = ctx->scratch.reserve(std::max(ctx->scratch.cap, instanceUpdateScratchBytes(nm)));
    if (e != cudaSuccess) return failed((int)e, cudaGetErrorString(e));
    TlasBuild tb;
    std::string why;
    // the scene arena is the context's own: the records the shade kernel reads are rewritten in place
    int rc = updateInstancesDevice(ctx->d_inst, const_cast<InstanceShade*>(ctx->sc.shade), nm, staged, first, count, tlas ? ctx->d_nodes : nullptr,
                                   ctx->blas_nodes, ninst, ctx->scratch.base, ctx->scratch.cap, ctx->stream, &tb, &why);
    if (rc == 0) rc = (int)cudaStreamSynchronize(ctx->stream);
    if (rc != 0) return failed(rc, why.empty() ? cudaGetErrorString((cudaError_t)rc) : why.c_str());
    if (!tlas) return PTAP_OK;
    if (3 * (ctx->blas_depth + tb.depth) + 8 > kBvhStack) {
        char msg[160];
        snprintf(msg, sizeof msg, "BVH too deep for the traversal stack (%d + %d levels, %d entries)", ctx->blas_depth, tb.depth, kBvhStack);
        return failed(PTAP_E_INVALID, msg);
    }
    ctx->sc.tlas_root = tb.root;
    setSceneConstants(ctx, tb.max_scale, tb.max_pad, tb.max_trans, tb.consistent);
    return PTAP_OK;
}

int ptap_set_render_params(ptap_ctx* ctx, int32_t W, int32_t H, int32_t depth, uint32_t flags)
{
    if (!ctx || W <= 0 || H <= 0 || depth <= 0 || depth > kMaxDepth) return fail(ctx, PTAP_E_INVALID, "set_render_params: W,H > 0 and 1 <= depth <= %d required", kMaxDepth);
    if ((long long)W * H > (1ll << 30)) return fail(ctx, PTAP_E_INVALID, "set_render_params: too many pixels");
    if (const int rc = enter(ctx)) return rc;
    const int N = W * H;
    // small wavefronts leave more of the GPU idle per kernel: more of them in flight (measured: 512 x 512, 4 -> 8 lanes +10 %; 1920 x 1080 +0 %)
    ctx->lanes = ctx->lanes_env ? ctx->lanes_env : (N <= (1 << 20) ? kSmallFrameLanes : kDefaultLanes);
    const int ntiles = (N + kShadeTile - 1) / kShadeTile, nscan = (N + kScanSlots - 1) / kScanSlots;
    WaveDev& w0 = ctx->lane[0];
    w0 = WaveDev{};
    w0.W = W; w0.H = H; w0.N = N; w0.depth = depth; w0.ntiles = ntiles; w0.nscan = nscan;
    applyCamera(ctx, w0);
    w0.iter_stride = 1;
    // every lane: its queues, hits, scan state, counters and (several lanes) its contributions; lane 0 also the film, the first-hit cache,
    // uv and the stamps, which the other lanes share
    auto carve = [&](Arena& A) {
        for (int l = 0; l < ctx->lanes; ++l) {
            WaveDev& w = ctx->lane[l];
            if (l > 0) w = w0;
            for (int k = 0; k < 2; ++k) { w.O[k] = A.alloc<float4>(N); w.D[k] = A.alloc<float4>(N); w.C[k] = A.alloc<float4>(N); }
            w.hit = A.alloc<float4>(N);
            if (l == 0) { w.hit_cache = A.alloc<float4>(N); w.uv = A.alloc<float2>(N); w.film = A.alloc<float>((size_t)N * 3); }
            w.tile_status = A.alloc<unsigned long long>((size_t)nscan * kMaxDepth);
            w.tile_offset = A.alloc<int>(ntiles); w.tile_ballot = A.alloc<unsigned>(ntiles);
            w.perm = A.alloc<unsigned char>((size_t)nscan * kScanSlots);
            w.st = A.alloc<FrameState>(1);
            if (l == 0) ctx->d_stamps = A.alloc<unsigned long long>(2 * kMaxStamps);
            ctx->contrib[l] = ctx->lanes > 1 ? A.alloc<float>((size_t)N * 3) : nullptr;
        }
    };
    ctx->have_frame = false;              // the frame arena is about to be replaced: the last frame is gone even if this call fails
    CK(ctx->frame_arena.place(carve));
    ctx->stamps_used = 0;
    CK(cudaMemsetAsync(w0.film, 0, (size_t)N * 3 * sizeof(float), ctx->stream));   // initImageKernel, Renderer.cpp:557-565
    for (int l = 0; l < ctx->lanes; ++l) CK(cudaMemsetAsync(ctx->lane[l].st, 0, sizeof(FrameState), ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->flags = flags; ctx->cache_valid = false; ctx->have_frame = true;
    ctx->grid_shade = ctx->sms * std::max(shadeOccupancy(), 1);
    ctx->grid_gen = ctx->sms * 8;
    if (!ctx->grid_trace) ctx->grid_trace = traceGridSize(ctx);
    resetStats(ctx);
    return PTAP_OK;
}

int ptap_set_camera(ptap_ctx* ctx, const PtapCamera* cam)
{
    if (!ctx) return PTAP_E_INVALID;
    if (const int rc = enter(ctx)) return rc;
    const PtapCamera ref{{0.0f, 0.0f, 920.0f}, {-10.0f, -4.0f, 900.0f}, {20.0f, 16.0f}, 0, 0u};
    const PtapCamera c = cam ? *cam : ref;
    if (!(c.span[0] > 0.0f) || !(c.span[1] > 0.0f)) return fail(ctx, PTAP_E_INVALID, "set_camera: the image plane needs a positive extent");
    ctx->camera = c;
    ctx->cache_valid = false;
    if (ctx->have_frame)
        for (int l = 0; l < ctx->lanes; ++l) applyCamera(ctx, ctx->lane[l]);
    return PTAP_OK;
}

int ptap_render(ptap_ctx* ctx, int32_t iter_begin, int32_t iter_end)
{
    if (const int rc = checkState(ctx, "render", kScene | kFrame | kAccel)) return rc;
    if (iter_end < iter_begin) return fail(ctx, PTAP_E_INVALID, "render: empty iteration range");
    if (const int rc = enter(ctx)) return rc;
    if (const int rc = ensureEmuBuffers(ctx)) return rc;
    // jittered camera rays differ from iteration to iteration: the first-hit cache (Renderer.cpp:594-613) is meaningless then and is not used
    const bool cache = (ctx->flags & PTAP_FLAG_FIRST_HIT_CACHE) && !ctx->camera.jitter;
    // several lanes only for plain frames (the per-class event timing and the counting build stay on one stream)
    const int L = (ctx->flags & (PTAP_FLAG_PROFILE | PTAP_FLAG_COUNT)) ? 1 : std::max(1, std::min(ctx->lanes, iter_end - iter_begin));
    WaveDev* const lane = ctx->lane;
    for (int l = 0; l < L; ++l) { lane[l].iter_stride = L; lane[l].contrib = L > 1 ? ctx->contrib[l] : nullptr; }
    const bool stamping = (ctx->flags & PTAP_FLAG_STAMP) != 0;
    if (stamping) {
        // start words to all-ones (atomicMin), end words to zero (atomicMax): one interleaved pattern written by two strided memsets
        CK(cudaMemset2DAsync(ctx->d_stamps, 16, 0xff, 8, kMaxStamps, ctx->stream));
        CK(cudaMemset2DAsync(ctx->d_stamps + 1, 16, 0x00, 8, kMaxStamps, ctx->stream));
    }
    ctx->stamps_used = 0; ctx->iter_events_used = 0;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (L > 1) CK(cudaEventRecord(ctx->e_fork, ctx->stream));
    for (int l = 0; l < L; ++l) {
        if (l > 0) CK(cudaStreamWaitEvent(ctx->streams[l], ctx->e_fork, 0));
        launchSetIter(lane[l].st, iter_begin + l, ctx->streams[l]);
    }
    int64_t launches = L, trace_launches = 0;
    int cache_lane = -1;                 // lane whose stream produced the first-hit cache in this call; every other lane waits for e_cache once
    unsigned cache_waited = 0;
    for (int it = iter_begin; it < iter_end; ++it) {
        const int l = (it - iter_begin) % L;
        const WaveDev& wv = lane[l];
        cudaStream_t S = ctx->streams[l];
        profMark(ctx, 0);
        launchGenerate(wv, it, ctx->grid_gen, S); ++launches;
        int in = 0;
        for (int round = 0; round < wv.depth; ++round) {
            float4* hitbuf = (round == 0 && cache) ? wv.hit_cache : wv.hit;
            if (!(round == 0 && cache && ctx->cache_valid)) {                    // Renderer.cpp:594-620
                profMark(ctx, 1);
                unsigned long long* stamp = stamping && ctx->stamps_used < kMaxStamps ? ctx->d_stamps + 2 * (size_t)ctx->stamps_used++ : nullptr;
                launchTrace(ctx, wv.st, wv.O[in], wv.D[in], hitbuf, nullptr, nullptr, round, -1, wv.emu, (ctx->flags & PTAP_FLAG_COUNT) != 0, S, stamp); launches += ctx->accel == PTAP_ACCEL_GRID_EMULATED ? 5 : 1; ++trace_launches;
                if (L > 1 && round == 0 && cache) { CK(cudaEventRecord(ctx->e_cache, S)); cache_lane = l; cache_waited = 1u << l; }
            } else if (L > 1 && cache_lane >= 0 && !(cache_waited >> l & 1u)) {
                CK(cudaStreamWaitEvent(S, ctx->e_cache, 0)); cache_waited |= 1u << l;
            }
            profMark(ctx, 2);
            launchScan(ctx->sc, wv, round, hitbuf, wv.depth - round, -1, S); ++launches;
            launchShade(ctx->sc, wv, round, in, hitbuf, wv.depth - round, -1, 0, nullptr, ctx->grid_shade, S); ++launches;
            in ^= 1;
        }
        if (L > 1) {                     // film += this iteration's contributions, in iteration order across the lanes
            if (it > iter_begin) CK(cudaStreamWaitEvent(S, ctx->e_gather[(l + L - 1) % L], 0));
            launchFilmAdd(wv.film, wv.contrib, (size_t)wv.N * 3, S); ++launches;
            CK(cudaEventRecord(ctx->e_gather[l], S));
        }
        if (cache) ctx->cache_valid = true;
        if (ctx->flags & PTAP_FLAG_ITER_TIMES) {
            if (ctx->iter_events_used == (int)ctx->iter_events.size()) { Event e; CK(cudaEventCreate(e.put())); ctx->iter_events.push_back(std::move(e)); }
            CK(cudaEventRecord(ctx->iter_events[ctx->iter_events_used++], S));
        }
    }
    for (int l = 1; l < L; ++l) {
        CK(cudaEventRecord(ctx->e_join[l], ctx->streams[l]));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->e_join[l], 0));
    }
    profMark(ctx, -1);
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaGetLastError());
    ctx->stats.kernel_launches += launches;
    ctx->stats.trace_launches = trace_launches;
    ctx->render_pending = true;
    return PTAP_OK;
}

int ptap_sync(ptap_ctx* ctx)
{
    if (!ctx) return PTAP_E_INVALID;
    if (const int rc = enter(ctx)) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    return PTAP_OK;
}

int ptap_frame_begin(ptap_ctx* ctx)
{
    if (const int rc = enter(ctx, "frame_begin", kFrame)) return rc;
    CK(cudaMemsetAsync(ctx->lane[0].film, 0, (size_t)ctx->lane[0].N * 3 * sizeof(float), ctx->stream));
    for (int l = 0; l < ctx->lanes; ++l) CK(cudaMemsetAsync(ctx->lane[l].st, 0, sizeof(FrameState), ctx->stream));
    ctx->cache_valid = false;
    resetStats(ctx);
    return PTAP_OK;
}

// Device timer on the context stream: bench.py brackets its timed region with these.
int ptap_timer_start(ptap_ctx* ctx)
{
    if (!ctx) return PTAP_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->tm0) { CK(cudaEventCreate(ctx->tm0.put())); CK(cudaEventCreate(ctx->tm1.put())); }
    CK(cudaEventRecord(ctx->tm0, ctx->stream));
    return PTAP_OK;
}

int ptap_timer_stop(ptap_ctx* ctx, float* ms)
{
    if (!ctx || !ms || !ctx->tm0) return PTAP_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->tm1, ctx->stream));
    CK(cudaEventSynchronize(ctx->tm1));
    CK(cudaEventElapsedTime(ms, ctx->tm0, ctx->tm1));
    return PTAP_OK;
}

int ptap_film_reset(ptap_ctx* ctx)
{
    if (!ctx || !ctx->have_frame) return fail(ctx, PTAP_E_STATE, "film_reset: no render parameters");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->lane[0].film, 0, (size_t)ctx->lane[0].N * 3 * sizeof(float), ctx->stream));
    return PTAP_OK;
}

int ptap_read_film(ptap_ctx* ctx, float* rgb)
{
    if (!ctx || !ctx->have_frame || !rgb) return fail(ctx, PTAP_E_STATE, "read_film: no render parameters");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(rgb, ctx->lane[0].film, (size_t)ctx->lane[0].N * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    return ptap_sync(ctx);
}

int ptap_film_device_ptr(ptap_ctx* ctx, void** dev_ptr, size_t* nfloats)
{
    if (!ctx || !ctx->have_frame || !dev_ptr) return fail(ctx, PTAP_E_STATE, "film_device_ptr: no render parameters");
    *dev_ptr = ctx->lane[0].film;
    if (nfloats) *nfloats = (size_t)ctx->lane[0].N * 3;
    return PTAP_OK;
}

int ptap_film_add(ptap_ctx* ctx, const float* rgb)
{
    if (!ctx || !ctx->have_frame || !rgb) return fail(ctx, PTAP_E_STATE, "film_add: no render parameters");
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->lane[0].N * 3;
    float* tmp;
    CK(ctx->scratch.place([&](Arena& A) { tmp = A.alloc<float>(n); }));
    CK(cudaMemcpyAsync(tmp, rgb, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    launchFilmAdd(ctx->lane[0].film, tmp, n, ctx->stream);
    CK(cudaStreamSynchronize(ctx->stream));
    return PTAP_OK;
}

int ptap_get_stats(ptap_ctx* ctx, PtapStats* out)
{
    if (!ctx || !out) return PTAP_E_INVALID;
    if (const int rc = enter(ctx)) return rc;
    *out = ctx->stats;
    return PTAP_OK;
}

// Renderer::renderImage (Renderer.cpp:15-63).  The per-pixel conversion runs on the device (k_resolve_bmp), the bytes come back through
// a page-locked staging buffer, and the host only writes the header and the rows.
// `film`: W x H x 3 device floats (the context's film, or a resolved copy in the scratch arena); `d_bytes`: room for their bytes (prepareReadout)
static int writeBmpFrom(ptap_ctx* ctx, const float* film, unsigned char* d_bytes, int W, int H, const char* path, int32_t iters)
{
    const size_t nbytes = (size_t)3 * W * H;
    unsigned char* pinned = nullptr;
    CK(cudaHostAlloc((void**)&pinned, nbytes, cudaHostAllocDefault));
    const std::unique_ptr<unsigned char, cudaError_t (*)(void*)> h_bytes(pinned, cudaFreeHost);
    const float div = 1 / (float)iters;                                     // Renderer.cpp:42
    launchResolveBmp(film, nbytes, div, d_bytes, ctx->stream);
    cudaError_t e = cudaMemcpyAsync(h_bytes.get(), d_bytes, nbytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(ctx, (int)e, "write_bmp: %s", cudaGetErrorString(e));
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, PTAP_E_IO, "write_bmp: cannot open %s", path);
    unsigned char hdr[54] = {0};
    hdr[0] = 'B'; hdr[1] = 'M'; hdr[10] = 54; hdr[14] = 40; hdr[26] = 1; hdr[28] = 24;
    const int32_t fileSize = 54 + 3 * W * H, imageSize = 3 * W * H;
    memcpy(hdr + 2, &fileSize, 4); memcpy(hdr + 18, &W, 4); memcpy(hdr + 22, &H, 4); memcpy(hdr + 34, &imageSize, 4);
    // rows bottom-up as stored, no padding, bytes in (x, y, z) order exactly as the reference writes them (Renderer.cpp:45-53)
    const bool ok = fwrite(hdr, 1, 54, f) == 54 && fwrite(h_bytes.get(), 1, nbytes, f) == nbytes;
    fclose(f);
    if (!ok) return fail(ctx, PTAP_E_IO, "write_bmp: short write to %s", path);
    return PTAP_OK;
}

// The scratch of a read-out of the film at sx x sy samples per output pixel: when `resolved` is given, the film box-resolved into it;
// when `bytes` is given, room for the BMP bytes of the output
static int prepareReadout(ptap_ctx* ctx, int sx, int sy, const char* who, const float** resolved, unsigned char** bytes)
{
    const WaveDev& wv = ctx->lane[0];
    if (sx <= 0 || sy <= 0 || wv.W % sx || wv.H % sy) return fail(ctx, PTAP_E_INVALID, "%s: %d x %d samples do not divide the %d x %d film", who, sx, sy, wv.W, wv.H);
    const size_t nv = (size_t)(wv.W / sx) * (wv.H / sy) * 3;
    float* out = nullptr;
    auto carve = [&](Arena& A) {
        if (resolved) out = A.alloc<float>(nv);
        if (bytes) *bytes = A.alloc<unsigned char>(nv);
    };
    const cudaError_t e = ctx->scratch.place(carve);
    if (e != cudaSuccess) return fail(ctx, (int)e, "%s: %s", who, cudaGetErrorString(e));
    if (resolved) {
        launchResolveBox(wv.film, wv.W, wv.H, sx, sy, out, ctx->stream);
        *resolved = out;
    }
    return PTAP_OK;
}

int ptap_write_bmp_resolved(ptap_ctx* ctx, const char* path, int32_t iters, int32_t sx, int32_t sy)
{
    if (!ctx || !ctx->have_frame || !path || iters <= 0) return fail(ctx, PTAP_E_INVALID, "write_bmp: bad arguments");
    if (const int rc = enter(ctx)) return rc;
    const float* film = ctx->lane[0].film;              // 1 x 1: the film itself
    unsigned char* bytes = nullptr;
    if (const int rc = prepareReadout(ctx, sx, sy, "write_bmp_resolved", sx == 1 && sy == 1 ? nullptr : &film, &bytes)) return rc;
    return writeBmpFrom(ctx, film, bytes, ctx->lane[0].W / sx, ctx->lane[0].H / sy, path, iters);
}

int ptap_write_bmp(ptap_ctx* ctx, const char* path, int32_t iters) { return ptap_write_bmp_resolved(ctx, path, iters, 1, 1); }

int ptap_read_film_resolved(ptap_ctx* ctx, int32_t sx, int32_t sy, float* rgb)
{
    if (!ctx || !ctx->have_frame || !rgb) return fail(ctx, PTAP_E_STATE, "read_film_resolved: no render parameters");
    if (const int rc = enter(ctx)) return rc;
    const float* film = nullptr;
    if (const int rc = prepareReadout(ctx, sx, sy, "read_film_resolved", &film, nullptr)) return rc;
    CK(cudaMemcpyAsync(rgb, film, (size_t)(ctx->lane[0].W / sx) * (ctx->lane[0].H / sy) * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    return ptap_sync(ctx);
}

// ---- parity entry points -------------------------------------------------------------------------------------

// n rays of 6 host floats (origin, direction) into the O and D arrays the trace kernels read, on the context stream
static int uploadRays(ptap_ctx* ctx, const float* rays_od, int32_t n, float4* O, float4* D)
{
    std::vector<float4> hO(n), hD(n);
    for (int i = 0; i < n; ++i) {
        hO[i] = make_float4(rays_od[6 * (size_t)i], rays_od[6 * (size_t)i + 1], rays_od[6 * (size_t)i + 2], 0.f);
        hD[i] = make_float4(rays_od[6 * (size_t)i + 3], rays_od[6 * (size_t)i + 4], rays_od[6 * (size_t)i + 5], 0.f);
    }
    CK(cudaMemcpyAsync(O, hO.data(), n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(D, hD.data(), n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    return PTAP_OK;
}

static int traceImpl(ptap_ctx* ctx, const float* rays_od, int32_t n, PtapHit* out, int32_t* counts)
{
    if (!ctx || !ctx->have_scene || !rays_od || !out || n < 0) return fail(ctx, PTAP_E_STATE, "trace: scene and buffers required");
    if (const int rc = checkState(ctx, "trace", kAccel)) return rc;
    if (n == 0) return PTAP_OK;
    if (const int rc = enter(ctx)) return rc;
    float4 *O, *D, *hit; float2* uv; PtapHit* dout; int4* dcnt; FrameState* st; EmuBuf emu{};
    auto carve = [&](Arena& A) {
        O = A.alloc<float4>(n); D = A.alloc<float4>(n); hit = A.alloc<float4>(n);
        uv = A.alloc<float2>(n); dout = A.alloc<PtapHit>(n); dcnt = A.alloc<int4>(n);
        st = A.alloc<FrameState>(1);
        if (ctx->accel == PTAP_ACCEL_GRID_EMULATED) emu = carveEmu(ctx, A, n);
    };
    CK(ctx->scratch.place(carve));
    if (const int rc = uploadRays(ctx, rays_od, n, O, D)) return rc;
    CK(cudaMemsetAsync(st, 0, sizeof(FrameState), ctx->stream));
    if (!ctx->grid_trace) ctx->grid_trace = traceGridSize(ctx);
    launchTrace(ctx, st, O, D, hit, uv, counts ? dcnt : nullptr, 0, n, emu);
    launchResolveHits(ctx->sc, O, D, hit, uv, n, dout, ctx->stream);
    CK(cudaMemcpyAsync(out, dout, n * sizeof(PtapHit), cudaMemcpyDeviceToHost, ctx->stream));
    if (counts) CK(cudaMemcpyAsync(counts, dcnt, n * sizeof(int4), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    return PTAP_OK;
}

int ptap_trace(ptap_ctx* ctx, const float* rays_od, int32_t n, PtapHit* out) { return traceImpl(ctx, rays_od, n, out, nullptr); }
int ptap_trace_count(ptap_ctx* ctx, const float* rays_od, int32_t n, PtapHit* out, int32_t* counts) { return traceImpl(ctx, rays_od, n, out, counts); }

// ---- ray queries on device buffers (DESIGN.md 4.8) ---------------------------------------------------------------

static int checkQueryPtr(ptap_ctx* ctx, const char* call, const char* arg, const void* p, size_t align)
{
    if (!p) return fail(ctx, PTAP_E_INVALID, "%s: %s is NULL", call, arg);
    if ((uintptr_t)p % align) return fail(ctx, PTAP_E_INVALID, "%s: %s is not %zu-byte aligned", call, arg, align);
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();                                     // clear the sticky-free error of the failed query
        return fail(ctx, PTAP_E_INVALID, "%s: %s is not a pointer CUDA knows", call, arg);
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) return fail(ctx, PTAP_E_INVALID, "%s: %s is not device or managed memory", call, arg);
    if (a.device != ctx->device) return fail(ctx, PTAP_E_INVALID, "%s: %s is on device %d, the context on device %d", call, arg, a.device, ctx->device);
    return PTAP_OK;
}

// One implementation for both queries: validation, stream ordering (the caller's stream -> context stream -> the caller's stream), and chunks
// of at most kQueryChunk rays through the query arena, which is sized for one chunk and reused by every later call.
static int queryImpl(ptap_ctx* ctx, const char* call, const float* org, const float* dir, int32_t n, PtapHit* hits, uint8_t* occluded, void* stream)
{
    constexpr int kQueryChunk = 1 << 22;
    if (!ctx) return PTAP_E_INVALID;
    if (n < 0) return fail(ctx, PTAP_E_INVALID, "%s: n = %d", call, n);
    if (n == 0) return PTAP_OK;
    if (const int rc = checkState(ctx, call, kScene | kAccel)) return rc;
    CK(cudaSetDevice(ctx->device));          // no collect(): the stream orders a query after a render in flight; the host does not wait for it
    if (const int rc = checkQueryPtr(ctx, call, "org", org, 16)) return rc;
    if (const int rc = checkQueryPtr(ctx, call, "dir", dir, 16)) return rc;
    if (const int rc = hits ? checkQueryPtr(ctx, call, "hits", hits, alignof(PtapHit)) : checkQueryPtr(ctx, call, "occluded", occluded, 1)) return rc;
    const bool anyhit = occluded && ctx->query_anyhit && (ctx->accel == PTAP_ACCEL_BVH || ctx->accel == PTAP_ACCEL_BVH_DEVICE);
    const size_t chunk = std::min<size_t>((size_t)n, kQueryChunk);
    float4* hit; float2* uv = nullptr; FrameState* st; EmuBuf emu{};
    auto carve = [&](Arena& A) {
        hit = A.alloc<float4>(chunk);
        if (hits) uv = A.alloc<float2>(chunk);
        st = A.alloc<FrameState>(1);
        if (ctx->accel == PTAP_ACCEL_GRID_EMULATED) emu = carveEmu(ctx, A, chunk);
    };
    cudaStream_t S = ctx->stream, U = (cudaStream_t)stream;
    if (Arena::measure(carve) > ctx->query_arena.cap) CK(cudaStreamSynchronize(S));     // earlier queries may still read the arena being replaced
    CK(ctx->query_arena.place(carve));
    if (!ctx->grid_trace) ctx->grid_trace = traceGridSize(ctx);
    if (U && U != S) { CK(cudaEventRecord(ctx->e_qin, U)); CK(cudaStreamWaitEvent(S, ctx->e_qin, 0)); }
    const float4* O = reinterpret_cast<const float4*>(org);
    const float4* D = reinterpret_cast<const float4*>(dir);
    for (size_t off = 0; off < (size_t)n; off += chunk) {
        const int m = (int)std::min(chunk, (size_t)n - off);
        CK(cudaMemsetAsync(st, 0, sizeof(FrameState), S));    // arms the work-stealing cursor
        if (hits) {                                             // what ptap_trace launches, on device buffers
            launchTrace(ctx, st, O + off, D + off, hit, uv, nullptr, 0, m, emu, false, S);
            launchResolveHits(ctx->sc, O + off, D + off, hit, uv, m, hits + off, S);
        } else {
            if (anyhit) launchTraceBvhAny(ctx->sc, O + off, D + off, hit, st, m, ctx->grid_trace, S);
            else launchTrace(ctx, st, O + off, D + off, hit, nullptr, nullptr, 0, m, emu, false, S);   // grid modes: R0 may miss hits, no early exit
            launchResolveOccluded(ctx->sc, O + off, D + off, hit, m, occluded + off, S);
        }
    }
    CK(cudaGetLastError());
    if (U && U != S) { CK(cudaEventRecord(ctx->e_qout, S)); CK(cudaStreamWaitEvent(U, ctx->e_qout, 0)); }
    return PTAP_OK;
}

int ptap_query_closest(ptap_ctx* ctx, const float* org, const float* dir, int32_t n, PtapHit* hits, void* stream)
{
    return queryImpl(ctx, "query_closest", org, dir, n, hits, nullptr, stream);
}

int ptap_query_occluded(ptap_ctx* ctx, const float* org, const float* dir, int32_t n, uint8_t* occluded, void* stream)
{
    return queryImpl(ctx, "query_occluded", org, dir, n, nullptr, occluded, stream);
}

int ptap_shade(ptap_ctx* ctx, const PtapPathIn* paths, int32_t n, int32_t iter, int32_t remaining, PtapPathOut* out, int32_t* order, int32_t* n_alive)
{
    if (!ctx || !ctx->have_scene || !paths || !out || n <= 0 || remaining <= 0) return fail(ctx, PTAP_E_STATE, "shade: scene and buffers required");
    if (const int rc = enter(ctx)) return rc;
    const int ntiles = (n + kShadeTile - 1) / kShadeTile, nscan = (n + kScanSlots - 1) / kScanSlots;
    WaveDev wv{};
    float4* hit; int* slot_pos;
    auto carve = [&](Arena& A) {
        for (int k = 0; k < 2; ++k) { wv.O[k] = A.alloc<float4>(n); wv.D[k] = A.alloc<float4>(n); wv.C[k] = A.alloc<float4>(n); }
        hit = A.alloc<float4>(n);
        wv.film = A.alloc<float>((size_t)n * 3);
        slot_pos = A.alloc<int>(n);
        wv.tile_status = A.alloc<unsigned long long>(nscan);
        wv.tile_offset = A.alloc<int>(ntiles);
        wv.tile_ballot = A.alloc<unsigned>(ntiles);
        wv.perm = A.alloc<unsigned char>((size_t)nscan * kScanSlots);
        wv.st = A.alloc<FrameState>(1);
    };
    CK(ctx->scratch.place(carve));
    wv.N = n; wv.W = n; wv.H = 1; wv.depth = 1; wv.ntiles = ntiles; wv.nscan = nscan;
    std::vector<float4> hO(n), hD(n), hC(n), hH(n);
    for (int i = 0; i < n; ++i) {
        const PtapPathIn& p = paths[i];
        hO[i] = make_float4(p.orig[0], p.orig[1], p.orig[2], __builtin_bit_cast(float, i));   // film slot = path index
        hD[i] = make_float4(p.dir[0], p.dir[1], p.dir[2], 0.f);
        hC[i] = make_float4(p.color[0], p.color[1], p.color[2], 0.f);
        const bool miss = p.model < 0 || p.tri < 0;
        if (!miss && (p.model >= ctx->sc.nmodels || p.tri >= ctx->ntris)) return fail(ctx, PTAP_E_INVALID, "shade: path %d has ids out of range", i);
        hH[i] = make_float4(miss ? kFloatMax : p.dist, __builtin_bit_cast(float, p.tri), __builtin_bit_cast(float, p.model), 0.f);
    }
    CK(cudaMemcpyAsync(wv.O[0], hO.data(), n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(wv.D[0], hD.data(), n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(wv.C[0], hC.data(), n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(hit, hH.data(), n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(wv.film, 0, (size_t)n * 3 * sizeof(float), ctx->stream));
    CK(cudaMemsetAsync(wv.tile_status, 0, nscan * sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(wv.st, 0, sizeof(FrameState), ctx->stream));
    const int grid = ctx->sms * std::max(shadeOccupancy(), 1);
    launchScan(ctx->sc, wv, 0, hit, remaining, n, ctx->stream);
    launchShade(ctx->sc, wv, 0, 0, hit, remaining, n, iter, slot_pos, grid, ctx->stream);
    std::vector<float4> oO(n), oD(n), oC(n);
    std::vector<float> film((size_t)n * 3);
    std::vector<int> pos(n);
    FrameState fs;
    CK(cudaMemcpyAsync(oO.data(), wv.O[1], n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(oD.data(), wv.D[1], n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(oC.data(), wv.C[1], n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(film.data(), wv.film, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(pos.data(), slot_pos, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&fs, wv.st, sizeof fs, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    const int alive = fs.n_active[kMaxDepth + 1];
    if (n_alive) *n_alive = alive;
    for (int i = 0; i < n; ++i) {
        PtapPathOut& o = out[i];
        o.ipixel = paths[i].ipixel;
        if (pos[i] >= 0) {
            const int k = pos[i];
            if (k >= alive) return fail(ctx, PTAP_E_INVALID, "shade: compaction position out of range");
            o.alive = 1;
            o.orig[0] = oO[k].x; o.orig[1] = oO[k].y; o.orig[2] = oO[k].z;
            o.dir[0] = oD[k].x; o.dir[1] = oD[k].y; o.dir[2] = oD[k].z;
            o.color[0] = oC[k].x; o.color[1] = oC[k].y; o.color[2] = oC[k].z;
            if (__builtin_bit_cast(int, oO[k].w) != i) return fail(ctx, PTAP_E_INVALID, "shade: compaction lost the pixel id");
            if (order) order[k] = i;
        } else {
            o.alive = 0;
            memcpy(o.orig, paths[i].orig, 12); memcpy(o.dir, paths[i].dir, 12);
            o.color[0] = film[3 * (size_t)i]; o.color[1] = film[3 * (size_t)i + 1]; o.color[2] = film[3 * (size_t)i + 2];   // sqrt(throughput): the film contribution
        }
    }
    return PTAP_OK;
}

int ptap_bench_trace(ptap_ctx* ctx, const float* rays_od, int32_t n, int32_t reps, float* ms_per_launch)
{
    if (!ctx || !ctx->have_scene || !rays_od || n <= 0 || reps <= 0 || !ms_per_launch) return fail(ctx, PTAP_E_INVALID, "bench_trace: bad arguments");
    if (const int rc = enter(ctx, "bench_trace", kAccel)) return rc;
    float4 *O, *D, *hit; FrameState* st; EmuBuf emu{};
    auto carve = [&](Arena& A) {
        O = A.alloc<float4>(n); D = A.alloc<float4>(n); hit = A.alloc<float4>(n);
        st = A.alloc<FrameState>(1);
        if (ctx->accel == PTAP_ACCEL_GRID_EMULATED) emu = carveEmu(ctx, A, n);
    };
    CK(ctx->scratch.place(carve));
    if (const int rc = uploadRays(ctx, rays_od, n, O, D)) return rc;
    for (int w = 0; w < 3; ++w) { CK(cudaMemsetAsync(st, 0, sizeof(FrameState), ctx->stream)); launchTrace(ctx, st, O, D, hit, nullptr, nullptr, 0, n, emu); }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    for (int r = 0; r < reps; ++r) { CK(cudaMemsetAsync(st, 0, sizeof(FrameState), ctx->stream)); launchTrace(ctx, st, O, D, hit, nullptr, nullptr, 0, n, emu); }   // the memset re-arms the work-stealing cursor
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    *ms_per_launch = ms / reps;
    return PTAP_OK;
}

// Parity entry for the PRODUCTION closest-hit path.  ptap_trace launches the <UV = true> instantiations of the closest-hit kernels (it
// returns barycentrics); ptap_render launches <false, false>, a different code object, and leaves BVH hit distances to be evaluated by the
// consumer.  This call enqueues iteration `iter` exactly as ptap_render does on one lane - same launch wrappers, same arguments, the
// device-side ray counts - up to and including the closest-hit launch of round `round`, then returns that round's wavefront: the rays the
// kernel read (n x 6 floats), their pixels, and the hit records it wrote, resolved by the same consumer code k_shade uses for the
// deferred distance (exactHitDistance).  u, v are 0 (the production instantiation does not record them).  The film and the first-hit cache
// are left in an unspecified state: call ptap_frame_begin afterwards.
int ptap_render_probe(ptap_ctx* ctx, int32_t iter, int32_t round, float* rays_od, int32_t* pixels, PtapHit* hits, int32_t cap, int32_t* n_out)
{
    if (const int rc = checkState(ctx, "render_probe", kScene | kFrame | kAccel)) return rc;
    if (round < 0 || round >= ctx->lane[0].depth || !n_out || cap < 0) return fail(ctx, PTAP_E_INVALID, "render_probe: bad arguments");
    if (const int rc = enter(ctx)) return rc;
    if (const int rc = ensureEmuBuffers(ctx)) return rc;
    WaveDev& wv = ctx->lane[0];
    wv.iter_stride = 1; wv.contrib = nullptr;
    cudaStream_t S = ctx->stream;
    ctx->cache_valid = false;
    launchSetIter(wv.st, iter, S);
    launchGenerate(wv, iter, ctx->grid_gen, S);
    int in = 0;
    for (int r = 0; r <= round; ++r) {
        launchTrace(ctx, wv.st, wv.O[in], wv.D[in], wv.hit, nullptr, nullptr, r, -1, wv.emu, false, S);       // the instantiation ptap_render launches
        if (r == round) break;
        launchScan(ctx->sc, wv, r, wv.hit, wv.depth - r, -1, S);
        launchShade(ctx->sc, wv, r, in, wv.hit, wv.depth - r, -1, 0, nullptr, ctx->grid_shade, S);
        in ^= 1;
    }
    FrameState fs;
    CK(cudaMemcpyAsync(&fs, wv.st, sizeof fs, cudaMemcpyDeviceToHost, S));
    CK(cudaStreamSynchronize(S));
    CK(cudaGetLastError());
    const int n = fs.n_active[round];
    *n_out = n;
    if (n > cap) return fail(ctx, PTAP_E_INVALID, "render_probe: %d active rays, buffers hold %d", n, cap);
    if (n == 0) return PTAP_OK;
    PtapHit* dout;
    CK(ctx->scratch.place([&](Arena& A) { dout = A.alloc<PtapHit>(n); }));
    launchResolveHits(ctx->sc, wv.O[in], wv.D[in], wv.hit, nullptr, n, dout, S);
    std::vector<float4> hO(n), hD(n);
    CK(cudaMemcpyAsync(hO.data(), wv.O[in], n * sizeof(float4), cudaMemcpyDeviceToHost, S));
    CK(cudaMemcpyAsync(hD.data(), wv.D[in], n * sizeof(float4), cudaMemcpyDeviceToHost, S));
    if (hits) CK(cudaMemcpyAsync(hits, dout, n * sizeof(PtapHit), cudaMemcpyDeviceToHost, S));
    CK(cudaStreamSynchronize(S));
    CK(cudaGetLastError());
    for (int i = 0; i < n; ++i) {
        if (rays_od) {
            float* p = rays_od + 6 * (size_t)i;
            p[0] = hO[i].x; p[1] = hO[i].y; p[2] = hO[i].z; p[3] = hD[i].x; p[4] = hD[i].y; p[5] = hD[i].z;
        }
        if (pixels) pixels[i] = __builtin_bit_cast(int, hO[i].w);
    }
    return PTAP_OK;
}

int ptap_get_iteration_times(ptap_ctx* ctx, float* ms_since_start, int32_t cap, int32_t* n)
{
    if (!ctx || !n) return PTAP_E_INVALID;
    if (const int rc = enter(ctx)) return rc;
    *n = (int32_t)ctx->iter_ms.size();
    for (int k = 0; k < *n && k < cap && ms_since_start; ++k) ms_since_start[k] = ctx->iter_ms[k];
    return PTAP_OK;
}

// ---- multi-GPU: combining the per-GPU films (SURVEY.md 8e) ------------------------------------------------------------------------

// film(dst) += film(src), both contexts in this process (any two devices, or the same one).  The copy crosses NVLink as a peer copy
// ordered after everything enqueued on src so far; the add runs on dst's stream.  Calling this for src = rank 1, 2, ... in turn gives a
// FIXED order of float additions, so the reduced film is bit-reproducible (a tree or ring reduction is not).
int ptap_reduce_peer(ptap_ctx* dst, ptap_ctx* src)
{
    ptap_ctx* ctx = dst;
    if (!dst || !src || dst == src || !dst->have_frame || !src->have_frame) return fail(ctx, PTAP_E_STATE, "reduce_peer: two contexts with render parameters required");
    if (dst->lane[0].N != src->lane[0].N || dst->lane[0].W != src->lane[0].W) return fail(ctx, PTAP_E_INVALID, "reduce_peer: the films differ in size");
    const size_t n = (size_t)dst->lane[0].N * 3;
    CK(cudaSetDevice(src->device));
    if (!src->e_peer) CK(cudaEventCreateWithFlags(src->e_peer.put(), cudaEventDisableTiming));
    CK(cudaEventRecord(src->e_peer, src->stream));
    CK(cudaSetDevice(dst->device));
    if (!dst->e_peer) CK(cudaEventCreateWithFlags(dst->e_peer.put(), cudaEventDisableTiming));
    if (dst->device != src->device) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, dst->device, src->device) == cudaSuccess && can) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(src->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(ctx, (int)e, "reduce_peer: %s", cudaGetErrorString(e));
            cudaGetLastError();
        }
    }
    float* tmp;
    CK(dst->scratch.place([&](Arena& A) { tmp = A.alloc<float>(n); }));
    CK(cudaStreamWaitEvent(dst->stream, src->e_peer, 0));
    if (dst->device == src->device) CK(cudaMemcpyAsync(tmp, src->lane[0].film, n * sizeof(float), cudaMemcpyDeviceToDevice, dst->stream));
    else CK(cudaMemcpyPeerAsync(tmp, dst->device, src->lane[0].film, src->device, n * sizeof(float), dst->stream));
    CK(cudaEventRecord(dst->e_peer, dst->stream));
    launchFilmAdd(dst->lane[0].film, tmp, n, dst->stream);
    CK(cudaSetDevice(src->device));
    CK(cudaStreamWaitEvent(src->stream, dst->e_peer, 0));       // src may not reuse its film before the copy has read it
    CK(cudaSetDevice(dst->device));
    return PTAP_OK;
}

// One process per GPU: NCCL, resolved at run time (dlopen) so that libptap.so itself has no link-time dependency on it.
namespace {

struct NcclId { char internal[128]; };
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
};

NcclApi& nccl()
{
    static NcclApi a;
    if (a.lib || a.ok) return a;
    const char* names[] = {getenv("PTAP_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) { if (nm && *nm && (a.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break; }
    if (!a.lib) return a;
    a.GetUniqueId = reinterpret_cast<int (*)(NcclId*)>(dlsym(a.lib, "ncclGetUniqueId"));
    a.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(dlsym(a.lib, "ncclCommInitRank"));
    a.Reduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, int, void*, cudaStream_t)>(dlsym(a.lib, "ncclReduce"));
    a.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(a.lib, "ncclCommDestroy"));
    a.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(a.lib, "ncclGetErrorString"));
    a.ok = a.GetUniqueId && a.CommInitRank && a.Reduce && a.CommDestroy;
    return a;
}

}  // namespace

int ptap_nccl_unique_id(void* id128)
{
    if (!id128) return PTAP_E_INVALID;
    NcclApi& a = nccl();
    if (!a.ok) return PTAP_E_STATE;
    NcclId id; memset(&id, 0, sizeof id);
    const int rc = a.GetUniqueId(&id);
    memcpy(id128, &id, sizeof id);
    return rc == 0 ? PTAP_OK : PTAP_E_STATE;
}

int ptap_nccl_init(ptap_ctx* ctx, const void* id128, int32_t nranks, int32_t rank)
{
    if (!ctx || !id128 || nranks <= 0 || rank < 0 || rank >= nranks) return fail(ctx, PTAP_E_INVALID, "nccl_init: bad arguments");
    NcclApi& a = nccl();
    if (!a.ok) return fail(ctx, PTAP_E_STATE, "nccl_init: libnccl.so.2 could not be loaded (%s); set PTAP_NCCL_LIB", dlerror() ? dlerror() : "symbols missing");
    CK(cudaSetDevice(ctx->device));
    if (ctx->nccl_comm) ptap_nccl_finalize(ctx);
    NcclId id; memcpy(&id, id128, sizeof id);
    const int rc = a.CommInitRank(&ctx->nccl_comm, nranks, id, rank);
    if (rc != 0) { ctx->nccl_comm = nullptr; return fail(ctx, PTAP_E_STATE, "ncclCommInitRank: %s", a.GetErrorString ? a.GetErrorString(rc) : "error"); }
    return PTAP_OK;
}

int ptap_nccl_finalize(ptap_ctx* ctx)
{
    if (!ctx || !ctx->nccl_comm) return PTAP_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    nccl().CommDestroy(ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
    return PTAP_OK;
}

// ncclReduce(sum) of the film onto `root`, in place, ordered on the context stream after the render (no host synchronisation).
int ptap_reduce(ptap_ctx* ctx, int32_t root)
{
    if (!ctx || !ctx->have_frame) return fail(ctx, PTAP_E_STATE, "reduce: no render parameters");
    if (!ctx->nccl_comm) return fail(ctx, PTAP_E_STATE, "reduce: ptap_nccl_init has not been called");
    CK(cudaSetDevice(ctx->device));
    const int rc = nccl().Reduce(ctx->lane[0].film, ctx->lane[0].film, (size_t)ctx->lane[0].N * 3, /* ncclFloat32 */ 7, /* ncclSum */ 0, root, ctx->nccl_comm, ctx->stream);
    if (rc != 0) return fail(ctx, PTAP_E_STATE, "ncclReduce: %s", nccl().GetErrorString ? nccl().GetErrorString(rc) : "error");
    return PTAP_OK;
}

// Scene::addMeshesToGrid (Scene.cpp:318-396) on the device (grid_device.cu): one grid per distinct mesh in model order, exactly the
// assignment the reference makes (grid index != mesh index; the grid remembers its creating model, through which the traversal reads
// the mesh bounds, Renderer.cpp:245-249).  The view must be the one last uploaded (its vertices and triangles are read again: the voxel
// ranges need the original vertex positions, which the edge-form triangle records on the device do not reproduce bit for bit).
int ptap_build_grids_device(ptap_ctx* ctx, const PtapSceneView* v, int32_t gx, int32_t gy, int32_t gz)
{
    if (!ctx || !ctx->have_scene || !v || !v->vertices || !v->triangles || !v->meshes || !v->models) return fail(ctx, PTAP_E_STATE, "build_grids_device: uploaded scene and its view required");
    if (gx <= 0 || gy <= 0 || gz <= 0 || (long long)gx * gy * gz > (1ll << 27)) return fail(ctx, PTAP_E_INVALID, "build_grids_device: bad grid dimensions");
    if (v->ntriangles != ctx->ntris || v->nmodels != (int)ctx->h_models.size() || v->nmeshes != (int)ctx->h_meshes.size()) return fail(ctx, PTAP_E_INVALID, "build_grids_device: the view is not the uploaded scene");
    if (const int rc = enter(ctx)) return rc;
    BuildTimer timer{ctx};
    if (const int rc = timer.start()) return rc;
    const int nm = v->nmodels, nmesh = v->nmeshes, nt = v->ntriangles;
    const int gd[3] = {gx, gy, gz};
    const size_t ncell = (size_t)gx * gy * gz;
    // grid list, as Scene.cpp:322-339
    std::vector<int> grid_of_mesh(nmesh, -1), grid_mesh, grid_owner, model_grid(nm, -1);
    for (int i = 0; i < nm; ++i) {
        const int mi = v->models[i].mesh_index;
        if (mi < 0 || mi >= nmesh) return fail(ctx, PTAP_E_INVALID, "build_grids_device: model %d has no mesh", i);
        if (grid_of_mesh[mi] < 0) { grid_of_mesh[mi] = (int)grid_mesh.size(); grid_mesh.push_back(mi); grid_owner.push_back(i); }
        model_grid[i] = grid_of_mesh[mi];
    }
    const int ng = (int)grid_mesh.size();
    // vertex positions per triangle (9 floats), gathered on the host once
    std::vector<float> pos((size_t)nt * 9);
    for (int t = 0; t < nt; ++t)
        for (int k = 0; k < 3; ++k) {
            const int vi = v->triangles[t].v[k];
            if (vi < 0 || vi >= v->nvertices) return fail(ctx, PTAP_E_INVALID, "build_grids_device: triangle %d: vertex index out of range", t);
            memcpy(&pos[(size_t)t * 9 + 3 * k], v->vertices[vi].position, 12);
        }
    int max_tris = 1;
    for (int g = 0; g < ng; ++g) max_tris = std::max(max_tris, v->meshes[grid_mesh[g]].t_end - v->meshes[grid_mesh[g]].t_start);
    // phase 1: count the references of every grid
    DevMem<float> d_pos; DevMem<int> d_count, d_offset_all; DevMem<void> d_tmp;
    size_t tmp_bytes = gridDeviceTempBytes(max_tris, 1);
    CK(cudaMalloc(d_pos.put(), pos.size() * sizeof(float) + 16));
    CK(cudaMalloc(d_count.put(), (size_t)max_tris * sizeof(int)));
    CK(cudaMalloc(d_offset_all.put(), (size_t)std::max(nt, 1) * sizeof(int)));
    CK(cudaMalloc(d_tmp.put(), tmp_bytes));
    CK(cudaMemcpyAsync(d_pos, pos.data(), pos.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    std::vector<long long> npairs(ng, 0);
    std::vector<std::array<float, 3>> widths(ng);
    long long total = 0, max_pairs = 1;
    for (int g = 0; g < ng; ++g) {
        const PtapMesh& mesh = v->meshes[grid_mesh[g]];
        for (int k = 0; k < 3; ++k) widths[g][k] = (mesh.bb_max[k] - mesh.bb_min[k]) / gd[k];      // Scene.cpp:341-347
        const int n = std::max(0, mesh.t_end - mesh.t_start);
        CK((cudaError_t)gridDeviceCount(d_pos + (size_t)mesh.t_start * 9, mesh.t_start, n, mesh.bb_min, widths[g].data(), gd, d_count, d_offset_all + mesh.t_start,
                                        d_tmp, tmp_bytes, ctx->stream, &npairs[g]));
        total += npairs[g]; max_pairs = std::max(max_pairs, npairs[g]);
    }
    if (total > 0x7fffffffll) return fail(ctx, PTAP_E_NOMEM, "build_grids_device: %lld references exceed the 32-bit reference list", total);
    // phase 2: pairs, sort, cells
    ctx->gd_cells.reset(); ctx->gd_refs.reset(); d_tmp.reset();
    tmp_bytes = gridDeviceTempBytes(max_tris, max_pairs);
    DevMem<int> d_keys, d_vals, d_keys2;
    CK(cudaMalloc(d_tmp.put(), tmp_bytes));
    CK(cudaMalloc(d_keys.put(), (size_t)max_pairs * sizeof(int))); CK(cudaMalloc(d_vals.put(), (size_t)max_pairs * sizeof(int))); CK(cudaMalloc(d_keys2.put(), (size_t)max_pairs * sizeof(int)));
    CK(cudaMalloc(ctx->gd_cells.put(), (size_t)ng * ncell * sizeof(int2)));
    CK(cudaMalloc(ctx->gd_refs.put(), (size_t)std::max(total, 1ll) * sizeof(int)));
    ctx->gd_ncells = (size_t)ng * ncell; ctx->gd_nrefs = (size_t)total;
    long long ref_base = 0;
    for (int g = 0; g < ng; ++g) {
        const PtapMesh& mesh = v->meshes[grid_mesh[g]];
        const int n = std::max(0, mesh.t_end - mesh.t_start);
        CK((cudaError_t)gridDeviceFill(d_pos + (size_t)mesh.t_start * 9, mesh.t_start, n, mesh.bb_min, widths[g].data(), gd, d_offset_all + mesh.t_start, (int)npairs[g],
                                       d_keys, d_vals, d_keys2, d_tmp, tmp_bytes, (int)ref_base, ctx->gd_refs + ref_base, ctx->gd_cells + (size_t)g * ncell, ctx->stream));
        ref_base += npairs[g];
    }
    // instance records: mesh bounds through the grid's creating model, voxel widths, first voxel (as ptap_upload_scene does for host grids)
    for (int i = 0; i < nm; ++i) {
        const int g = model_grid[i];
        const PtapMesh& mesh = v->meshes[v->models[grid_owner[g]].mesh_index];
        InstanceTrace& it = ctx->h_inst[i];
        it.bb_min = make_float4(mesh.bb_min[0], mesh.bb_min[1], mesh.bb_min[2], widths[g][0]);
        it.bb_max = make_float4(mesh.bb_max[0], mesh.bb_max[1], mesh.bb_max[2], widths[g][1]);
        it.grid.x = widths[g][2];
        it.grid.y = __builtin_bit_cast(float, (int)((size_t)g * ncell));
    }
    CK(cudaMemcpyAsync(ctx->d_inst, ctx->h_inst.data(), nm * sizeof(InstanceTrace), cudaMemcpyHostToDevice, ctx->stream));
    if (const int rc = timer.stop()) return rc;
    ctx->sc.cells = ctx->gd_cells; ctx->sc.refs = ctx->gd_refs;
    ctx->h_grid_first.resize(ng); ctx->h_model_grid.assign(model_grid.begin(), model_grid.end()); ctx->emu_ok = false;
    for (int g = 0; g < ng; ++g) ctx->h_grid_first[g] = (int)((size_t)g * ncell);
    ctx->sc.gx = gx; ctx->sc.gy = gy; ctx->sc.gz = gz;
    ctx->have_grid = true; ctx->accel = PTAP_ACCEL_GRID_COMPAT; ctx->cache_valid = false;
    ctx->grid_trace = traceGridSize(ctx);
    return PTAP_OK;
}

// The grids now on the device in the reference's own layout (Voxel: start, end, entity_type; the reference list).  Two-call protocol:
// pass voxels / refs NULL to get the counts.
int ptap_read_grids(ptap_ctx* ctx, PtapVoxel* voxels, int32_t* refs, int32_t counts[2])
{
    if (!ctx || !ctx->have_grid || !ctx->gd_cells || !counts) return fail(ctx, PTAP_E_STATE, "read_grids: no device-built grids");
    CK(cudaSetDevice(ctx->device));
    counts[0] = (int32_t)ctx->gd_ncells; counts[1] = (int32_t)ctx->gd_nrefs;
    if (voxels) {
        std::vector<int2> h(ctx->gd_ncells);
        CK(cudaMemcpy(h.data(), ctx->gd_cells, h.size() * sizeof(int2), cudaMemcpyDeviceToHost));
        for (size_t c = 0; c < h.size(); ++c) { voxels[c].start = h[c].x; voxels[c].end = h[c].y; voxels[c].entity_type = 2; }
    }
    if (refs && ctx->gd_nrefs) CK(cudaMemcpy(refs, ctx->gd_refs, ctx->gd_nrefs * sizeof(int), cudaMemcpyDeviceToHost));
    return PTAP_OK;
}

}  // extern "C"
