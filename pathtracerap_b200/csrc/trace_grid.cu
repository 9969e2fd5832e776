// trace_grid.cu - closest hit through the reference's per-mesh uniform grid (PTAP_ACCEL_GRID_COMPAT).
//
// Replaces computeRaySceneIntersectionKernel and its helpers (Renderer.cpp:150-409) and is bit-compatible
// with them (oracle tier R0): same model loop, same slab test, same 3D-DDA with its early exit, same
// tolerant Moller-Trumbore predicate, every hit-deciding operation un-contracted (exact_math.cuh).
// What changes is everything around the arithmetic: the ray lives in registers instead of being written back
// to global memory per model (Renderer.cpp:381-384), the scene is SoA/AoSoA fetched as 16-byte vectors
// (TriRec, int2 cells) instead of 112 B of AoS gathers per test through two pointer hops, the flat normal and
// the 3x3 inverse-transpose are not evaluated in the loop at all (the kernel returns ids; the shade kernel
// looks the precomputed normal up), and the active count is read from device memory so that no host
// round trip separates the bounces.
#include "kernels.cuh"

namespace ptap {

namespace {

struct GridRay {
    V3 o, d, inv;
    float best_t;     // hit_info->impact_distance inside the current model
    int best_tri;
    float best_u, best_v;
};

// Renderer.cpp:174-215 without the normal (looked up later from the id)
template <bool COUNT>
__device__ __forceinline__ bool rayTriangle(const TriRec* __restrict__ tris, GridRay& r, int itri, int4& cnt)
{
    const float4 a = ldg4(&tris[itri].v0), b = ldg4(&tris[itri].e1), c = ldg4(&tris[itri].e2);
    if (COUNT) cnt.z++;
    const V3 v0 = v3(a), v0v1 = v3(b), v0v2 = v3(c);
    const V3 pvec = xcross(r.d, v0v2);
    const float det = xdot(v0v1, pvec);
    if (xabs(xsub(det, 0.0f)) < kEpsilon) return false;
    const float invDet = xdiv(1.0f, det);
    const V3 tvec = xsub(r.o, v0);
    const float u = xmul(xdot(tvec, pvec), invDet);
    if (u < (0.0f - kEpsilon) || u > (1.0f + kEpsilon)) return false;
    const V3 qvec = xcross(tvec, v0v1);
    const float v = xmul(xdot(r.d, qvec), invDet);
    if (v < (0.0f - kEpsilon) || xadd(u, v) > (1.0f + kEpsilon)) return false;
    const float t = xmul(xdot(v0v2, qvec), invDet);
    if (t < (0.0f - kEpsilon)) return false;
    if (r.best_t > t) { r.best_t = t; r.best_tri = itri; r.best_u = u; r.best_v = v; }
    return true;
}

}  // namespace

// Execution model: the same warp-wide state machine as k_trace_bvh (trace_bvh.cu), over the reference's own algorithm.  Each lane owns
// one ray and is in one of six states; a round counts the lanes per state with one warp reduction and runs a state's step when enough
// lanes wait for it (or when it is the most popular one), so that lanes at different models / voxels / triangles still share instructions:
//   MODEL  finish the previous model (model t -> world distance, nearest-model bookkeeping, Renderer.cpp:388-398), set up the next one
//          (Renderer.cpp:381-384) and run its slab test (Renderer.cpp:150-170, 252)
//   INIT   entry point, entry voxel and DDA increments (Renderer.cpp:254-311), fetch the first voxel
//   CELL   close the voxel just tested (Renderer.cpp:321-329: hit bookkeeping, early exit), take one DDA step (Renderer.cpp:331-357), fetch the voxel
//   TRI    one triangle reference of the current voxel (Renderer.cpp:217-236 -> 174-215)
//   DONE   retire the ray, refill the lane from the warp's batch of the work-stealing cursor
// Every arithmetic operation that decides a hit is the un-contracted one of the previous version of this kernel; only the schedule changed.
namespace {

enum : unsigned { G_MODEL = 0, G_INIT = 1, G_CELL = 2, G_TRI = 3, G_DONE = 4 };
enum : unsigned { F_INTERSECT = 1u, F_ANY = 2u, F_POST = 4u, F_MODEL_HIT = 8u };

}  // namespace

template <bool UV, bool COUNT>
__global__ void __launch_bounds__(kTraceBlock)
k_trace_grid(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit,
             float2* __restrict__ uv, int4* __restrict__ counts, FrameState* st, int round, int n_fixed, unsigned long long* __restrict__ stamp,
             const int* __restrict__ list)
{
    // list != null: the last launch of PTAP_ACCEL_GRID_EMULATED - only the slots k_emu_full (trace_emu.cu) handed over are walked
    const int n = list ? (int)st->n_walk[round] : n_fixed >= 0 ? n_fixed : st->n_active[round];
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_fixed < 0 && !list) st->rays_traced += (unsigned long long)n;
    if (blockIdx.x == 0 && threadIdx.x == 0 && list) st->rays_walked += (unsigned long long)n;
    if (stamp && threadIdx.x == 0) atomicMin(stamp, globalTimerNs());
    unsigned int* cursor = list ? &st->fetch_walk[round] : &st->fetch[round];
    const int GX = sc.gx, GY = sc.gy, GZ = sc.gz;
    unsigned long long tot_x = 0, tot_y = 0, tot_z = 0;
    int4 cnt = make_int4(0, 0, 0, 0);

    unsigned state = G_DONE, flags = 0;
    int i = -1, im = -1;
    V3 bo = v3(0, 0, 0), bd = v3(0, 0, 0);
    GridRay r; r.o = v3(0, 0, 0); r.d = v3(0, 0, 1); r.inv = v3(0, 0, 0); r.best_t = kFloatMax; r.best_tri = -1; r.best_u = 0.0f; r.best_v = 0.0f;
    float g_dist = kFloatMax, g_t = 0.0f, g_u = 0.0f, g_v = 0.0f;
    int g_model = -1, g_tri = -1;
    int ix = 0, iy = 0, iz = 0, cx = 0, cy = 0, cz = 0, vox0 = 0, ri = 0, rend = 0;
    float tmx = kFloatMax, tmy = kFloatMax, tmz = kFloatMax, dx = kFloatMax, dy = kFloatMax, dz = kFloatMax;
    float t_entry = 0.0f;
    WarpBatch work;
    const int vote = sc.vote_grid;

    for (;;) {
        // ---- who waits for what
        const bool live = state != G_DONE || i >= 0 || !work.exhausted;
        const unsigned sum = __reduce_add_sync(kFull, live ? 1u << (6u * state) : 0u);
        if (sum == 0u) break;
        const int n_model = sum & 63u, n_init = (sum >> 6) & 63u, n_cell = (sum >> 12) & 63u, n_tri = (sum >> 18) & 63u, n_done = (sum >> 24) & 63u;
        const int n_top = max(max(n_model, n_init), max(max(n_cell, n_tri), n_done));      // the most popular state always runs: progress
        const int need = min(vote, n_top);

        // ---- TRI: one triangle reference of the current voxel
        if (state == G_TRI && n_tri >= need) {
            const int itri = __ldg(&sc.refs[ri]);
            if (COUNT) cnt.y++;
            if (rayTriangle<COUNT>(sc.tris, r, itri, cnt)) flags |= F_ANY;
            if (++ri == rend) { state = G_CELL; flags |= F_POST; }
        }
        // ---- CELL: close the tested voxel, step the DDA, fetch the next voxel
        if (state == G_CELL && n_cell >= need) {
            bool leave = false;
            if (flags & F_POST) {
                if (flags & F_ANY) { cx = ix; cy = iy; cz = iz; flags |= F_INTERSECT; }
                flags &= ~(F_POST | F_ANY);
                if ((flags & F_INTERSECT) && (abs(cx - ix) > 2 || abs(cy - iy) > 2 || abs(cz - iz) > 2)) { leave = true; flags |= F_MODEL_HIT; }   // Renderer.cpp:326-329
                if (!leave) {
                    if (tmx < tmy && tmx < tmz) {
                        ix += r.d.x > 0.0f ? 1 : -1;
                        if (ix == (r.d.x > 0.0f ? GX : -1) || tmx >= kFloatMax) leave = true; else tmx = xadd(tmx, dx);
                    } else if (tmy < tmz) {
                        iy += r.d.y > 0.0f ? 1 : -1;
                        if (iy == (r.d.y > 0.0f ? GY : -1) || tmy >= kFloatMax) leave = true; else tmy = xadd(tmy, dy);
                    } else {
                        iz += r.d.z > 0.0f ? 1 : -1;
                        if (iz == (r.d.z > 0.0f ? GZ : -1) || tmz >= kFloatMax) leave = true; else tmz = xadd(tmz, dz);
                    }
                    if (leave && (flags & F_INTERSECT)) flags |= F_MODEL_HIT;                   // `return is_intersect`
                }
            }
            if (leave) state = G_MODEL;
            else {
                const int2 cell = __ldg(&sc.cells[vox0 + ix + iy * GX + iz * GX * GY]);
                if (COUNT) cnt.x++;
                if (cell.x < cell.y) { ri = cell.x; rend = cell.y; state = G_TRI; }
                else flags |= F_POST;                                                          // empty voxel: nothing to test, close it next round
            }
        }
        // ---- INIT: entry point, entry voxel, DDA increments
        if (state == G_INIT && n_init >= need) {
            const InstanceTrace* __restrict__ inst = &sc.inst[im];
            const float4 bbmin_wx = ldg4(&inst->bb_min), bbmax_wy = ldg4(&inst->bb_max), gridrec = ldg4(&inst->grid);
            const V3 mn = v3(bbmin_wx);
            const float wx = bbmin_wx.w, wy = bbmax_wy.w, wz = gridrec.x;
            vox0 = __float_as_int(gridrec.y);
            const V3 p = xadd(r.o, xscale(r.d, t_entry));
            if (xsub(p.x, mn.x) < -kEpsilon || xsub(p.y, mn.y) < -kEpsilon || xsub(p.z, mn.z) < -kEpsilon) state = G_MODEL;    // Renderer.cpp:256-259
            else {
                ix = f2i_x86(xdiv(xabs(xadd(xsub(p.x, mn.x), kEpsilon)), wx));
                iy = f2i_x86(xdiv(xabs(xadd(xsub(p.y, mn.y), kEpsilon)), wy));
                iz = f2i_x86(xdiv(xabs(xadd(xsub(p.z, mn.z), kEpsilon)), wz));
                ix = min(max(ix, 0), GX - 1); iy = min(max(iy, 0), GY - 1); iz = min(max(iz, 0), GZ - 1);
                tmx = kFloatMax; tmy = kFloatMax; tmz = kFloatMax; dx = kFloatMax; dy = kFloatMax; dz = kFloatMax;
                if (r.d.x != 0) {
                    const int nx = r.d.x > 0.0f ? ix + 1 : ix;
                    dx = xabs(xmul(wx, r.inv.x));
                    tmx = xmul(xsub(xadd(mn.x, xmul((float)nx, wx)), p.x), r.inv.x);
                }
                if (r.d.y != 0) {
                    const int ny = r.d.y > 0.0f ? iy + 1 : iy;
                    dy = xabs(xmul(wy, r.inv.y));
                    tmy = xmul(xsub(xadd(mn.y, xmul((float)ny, wy)), p.y), r.inv.y);
                }
                if (r.d.z != 0) {
                    const int nz = r.d.z > 0.0f ? iz + 1 : iz;
                    dz = xabs(xmul(wz, r.inv.z));
                    tmz = xmul(xsub(xadd(mn.z, xmul((float)nz, wz)), p.z), r.inv.z);
                }
                cx = 0; cy = 0; cz = 0;
                const int2 cell = __ldg(&sc.cells[vox0 + ix + iy * GX + iz * GX * GY]);
                if (COUNT) cnt.x++;
                if (cell.x < cell.y) { ri = cell.x; rend = cell.y; state = G_TRI; }
                else { state = G_CELL; flags |= F_POST; }
            }
        }
        // ---- MODEL: finish the previous model, set up the next one, slab test against the mesh bounds
        if (state == G_MODEL && n_model >= need) {
            if (flags & F_MODEL_HIT) {
                const InstanceTrace* __restrict__ inst = &sc.inst[im];
                const V3 nd = xnormalize(r.d);                                   // Renderer.cpp:388
                const V3 pm = xadd(r.o, xscale(nd, r.best_t));                   // Renderer.cpp:389
                const V3 pw = xmat4(ldg4(&inst->m2w[0]), ldg4(&inst->m2w[1]), ldg4(&inst->m2w[2]), pm, 1.0f);   // :390
                const float dist = xlength(xsub(pw, bo));                        // Renderer.cpp:391
                if (g_dist > dist) {                                             // Renderer.cpp:393-398
                    g_dist = dist; g_model = im; g_tri = r.best_tri; g_t = r.best_t;
                    if (UV) { g_u = r.best_u; g_v = r.best_v; }
                }
            }
            flags = 0;
            if (++im >= sc.nmodels) state = G_DONE;
            else {
                const InstanceTrace* __restrict__ inst = &sc.inst[im];
                const float4 w0 = ldg4(&inst->w2m[0]), w1 = ldg4(&inst->w2m[1]), w2 = ldg4(&inst->w2m[2]);
                r.o = xmat4(w0, w1, w2, bo, 1.0f);                                   // Renderer.cpp:381
                r.d = xnormalize(xmat4(w0, w1, w2, bd, 0.0f));                       // Renderer.cpp:382
                r.inv = v3(xdiv(1.0f, r.d.x), xdiv(1.0f, r.d.y), xdiv(1.0f, r.d.z)); // Renderer.cpp:383
                r.best_t = kFloatMax; r.best_tri = -1; r.best_u = 0.0f; r.best_v = 0.0f;   // Renderer.cpp:384
                const V3 mn = v3(ldg4(&inst->bb_min)), mx = v3(ldg4(&inst->bb_max));
                // Renderer.cpp:150-170
                const float t1 = r.d.x == 0.0f ? kFloatMin : xmul(xsub(mn.x, r.o.x), r.inv.x);
                const float t2 = r.d.x == 0.0f ? kFloatMax : xmul(xsub(mx.x, r.o.x), r.inv.x);
                const float t3 = r.d.y == 0.0f ? kFloatMin : xmul(xsub(mn.y, r.o.y), r.inv.y);
                const float t4 = r.d.y == 0.0f ? kFloatMax : xmul(xsub(mx.y, r.o.y), r.inv.y);
                const float t5 = r.d.z == 0.0f ? kFloatMin : xmul(xsub(mn.z, r.o.z), r.inv.z);
                const float t6 = r.d.z == 0.0f ? kFloatMax : xmul(xsub(mx.z, r.o.z), r.inv.z);
                const float tmin = max_std(max_std(min_std(t1, t2), min_std(t3, t4)), min_std(t5, t6));
                const float tmax = min_std(min_std(max_std(t1, t2), max_std(t3, t4)), max_std(t5, t6));
                if (!(tmax < 0 || tmin > tmax)) { t_entry = tmin; state = G_INIT; }      // else: stay in MODEL, the next round takes the next model
            }
        }
        // ---- DONE: retire finished rays, refill the lanes from the warp's batch
        if (n_done > 0 && n_done >= need) {
            const bool s_done = state == G_DONE;
            const unsigned m_done = __ballot_sync(kFull, s_done && live);
            if (s_done && i >= 0) {
                const bool found = g_dist < kFloatMax;                               // Renderer.cpp:402-408
                hit[i] = make_float4(found ? g_dist : kFloatMax, __int_as_float(found ? g_tri : -1), __int_as_float(found ? g_model : -1), g_t);
                if (UV && uv) uv[i] = make_float2(g_u, g_v);
                if (COUNT) { if (counts) counts[i] = cnt; tot_x += cnt.x; tot_y += cnt.y; tot_z += cnt.z; }
                i = -1;
            }
            work.fetch(cursor, sc.batch, n);
            int next;
            if (work.claim(m_done, s_done && live, next)) {
                i = list ? __ldg(&list[next]) : next;
                bo = v3(O[i]); bd = v3(D[i]);
                g_dist = kFloatMax; g_model = -1; g_tri = -1; g_t = 0.0f; g_u = 0.0f; g_v = 0.0f;
                if (COUNT) cnt = make_int4(0, 0, 0, 0);
                im = -1; flags = 0;
                state = G_MODEL;
            }
            work.advance(m_done);
        }
    }
    if (stamp && (threadIdx.x & 31) == 0) atomicMax(stamp + 1, globalTimerNs());
    if (COUNT) {        // counting build: per-warp totals into the frame state (never used for timing)
        warpTotalAdd(&st->count_cells, tot_x); warpTotalAdd(&st->count_refs, tot_y); warpTotalAdd(&st->count_tris, tot_z);
    }
}

void launchTraceGrid(const SceneDev& sc, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, bool count_totals,
                     FrameState* st, int round, int n_fixed, int grid, cudaStream_t stream, unsigned long long* stamp, const int* list)
{
    if (counts || count_totals) k_trace_grid<true, true><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, stamp, list);
    else if (uv) k_trace_grid<true, false><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, stamp, list);
    else k_trace_grid<false, false><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, stamp, list);
}

int traceGridOccupancy()
{
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_trace_grid<false, false>, kTraceBlock, 0);
    return nb;
}

}  // namespace ptap
