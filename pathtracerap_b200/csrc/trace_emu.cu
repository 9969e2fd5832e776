// trace_emu.cu - the reference's grid walk (oracle tier R0), answered through the BVH (PTAP_ACCEL_GRID_EMULATED).
//
// computeRayGridIntersection (Renderer.cpp:238-360) is not a closest-hit query: it walks the voxels of a model's 25^3 grid from the point
// where the ray enters the mesh box, tests every triangle LISTED in a voxel along the whole ray, remembers the last voxel in which some
// listed triangle was hit, and stops once it is more than two voxels away from that one (or leaves the grid).  The model's answer is the
// nearest hit among the triangles it happened to test.  0.3-0.6 % of the rays get a different answer than brute force, and the drop-in
// Renderer has to reproduce those too.  Walking the grid costs ~40 voxels and ~32 triangle tests per ray in eleven models (k_trace_grid:
// 940 warp instructions per ray at 12.6 of 32 lanes, issue-bound; three attempts to make the walk itself cheaper bought nothing,
// profiles/r02).  The same answer follows from three facts:
//   1. Only triangles the ray actually hits (predicate true, Renderer.cpp:174-215) influence a walk: a miss neither sets the voxel's hit
//      flag nor updates the nearest hit.  Every model's answer is therefore one of the ray's real hits, and no answer can be nearer than
//      the exact closest hit D* (tier R1: model m*, parameter t*).
//   2. Scene::addMeshesToGrid lists a triangle in every voxel of an index BOX (Scene.cpp:357-374); grid_device.cu derives that box per
//      triangle from the lists on the device and verifies the shape.  Given the set H of ALL hits of the ray in one model (typically 1-4
//      triangles), "does voxel v list a triangle the ray hits" is |H| box tests, so that model's walk can be REPLAYED without reading a
//      voxel or testing a triangle: the reference's own slab test, entry point, entry voxel and DDA stepping (every operation
//      un-contracted, as in k_trace_grid), its hit-voxel bookkeeping and early exit, the hits of H taking effect in the order the walk
//      meets them (first voxel along the path that lists them, ascending triangle id inside a voxel: that order decides exact-t ties).
//   3. If the replayed walk of m* returns t* (bit for bit), the reference's answer for the ray is m* with the walk's triangle: every other
//      model's answer is a real hit, hence not nearer (with one exception, handled in k_trace_emu: `ambiguous` instances), and a model
//      with a lower index that tied at D* would itself have been m* (the closest-hit rule breaks ties towards the lower model index
//      exactly as Renderer.cpp:393 does in model order).
// Launches: k_trace_emu is k_trace_bvh's state machine (TLAS pruning by the nearest hit so far, cross-instance ranking, deferred exact
// distance) except that inside an instance the ray interval never shrinks and every hit is recorded; the hits of the currently nearest
// instance are kept (two buffers in shared memory that swap roles) and written out with the closest hit.  k_emu_setup + k_emu_tail then
// replay the walk of that model (see there for why two kernels) and either confirm the hit - fixing the triangle id when the walk's tie
// rule differs - or append the slot to a list.  Rays on the list - those where the walk misses the closest hit (the 0.3-0.6 %), any
// (ray, model) with more than kEmuHits hits, and the ambiguous ones of fact 3 - are answered by the walk itself (k_trace_grid in list
// mode, last launch), so the result is exact whatever the geometry.  api.cu refuses this mode (and keeps the walk) when the lists on the
// device are not box-shaped, not ascending, or list triangles outside the mesh of a model that uses the grid.  The first version ran the
// replay inside this kernel's exit step and was slower than the walk: a 30-step loop for the two or three lanes that leave an instance
// together.
// Parity: tests/test_gpu_emulated.py, tests/test_gpu_production.py[emu] (bit-equal to the oracle's R0 and to k_trace_grid: fixtures, random
// rays, every round of the production path, whole films, and scenes that force the list path).
#include "bvh_traverse.cuh"

namespace ptap {

using namespace bvh;

namespace {

#ifndef PTAP_EMU_MIN_CTAS
#define PTAP_EMU_MIN_CTAS 7
#endif
#ifndef PTAP_EMU_FULL_BATCH
#define PTAP_EMU_FULL_BATCH 8
#endif
constexpr int kFullBatch = PTAP_EMU_FULL_BATCH;   // list entries a warp of k_emu_full takes per fetch: few, so that a short list spreads over all warps (the kernel is latency-bound)
constexpr int kFullHits = 20;                 // hits of a (ray, model) that k_emu_full keeps in shared memory (46 KB per CTA with the stack)
constexpr int kReplayBlock = 128, kReplayBatch = 32;   // k_emu_tail: threads per CTA, queue entries per cursor fetch
constexpr int kSetupBlock = 128;                      // k_emu_setup
#ifndef PTAP_EMU_SETUP_STEPS
#define PTAP_EMU_SETUP_STEPS 2
#endif
#ifndef PTAP_EMU_BURST
#define PTAP_EMU_BURST 8
#endif
constexpr int kBurst = PTAP_EMU_BURST;                // voxels outside the hits' box that one step call may take in a row
#ifndef PTAP_EMU_SETUP_BURST
#define PTAP_EMU_SETUP_BURST PTAP_EMU_BURST
#endif
constexpr int kSetupBurst = PTAP_EMU_SETUP_BURST;    // the same inside the set-up kernel (its threads wait for the longest burst of their warp)
constexpr int kSetupSteps = PTAP_EMU_SETUP_STEPS;     // voxel steps a replay takes in the set-up kernel before it is queued
constexpr unsigned kGuard = 0x20080200u;      // bits 9, 19, 29: one guard bit above each 9-bit voxel index of a packed (x | y << 10 | z << 20)

}  // namespace

// ---- launch 1: exact closest hit + all hits of the ray in the nearest model ------------------------------------------------------------
template <bool COUNT>
__global__ void __launch_bounds__(kTraceBlock, PTAP_EMU_MIN_CTAS)
k_trace_emu(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit,
            int4* __restrict__ counts, FrameState* st, int round, int n_fixed, unsigned long long* __restrict__ stamp, EmuBuf emu)
{
    const int n = n_fixed >= 0 ? n_fixed : st->n_active[round];
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_fixed < 0) st->rays_traced += (unsigned long long)n;
    if (stamp && threadIdx.x == 0) atomicMin(stamp, globalTimerNs());
    unsigned int* cursor = &st->fetch[round];
    unsigned long long tot_x = 0, tot_z = 0;
    int4 cnt = make_int4(0, 0, 0, 0);      // counting build: nodes visited, (voxels replayed: launch 2), triangles tested

    if (sc.tlas_root < 0) {                            // no instance has triangles: every ray misses
        for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
            hit[k] = make_float4(kFloatMax, __int_as_float(-1), __int_as_float(-1), 0.0f);
            emu.n[k] = 0;
            if (COUNT && counts) counts[k] = cnt;
        }
        return;
    }

    __shared__ int s_stack[kSmemStack * kTraceBlock];
    int l_stack[kBvhStack - kSmemStack];
    SplitStack stack(s_stack, l_stack);
    // the hits of the instance being traversed and of the nearest instance so far: two buffers [buffer][hit][thread] that swap roles
    __shared__ int s_id[2 * kEmuHits * kTraceBlock];
    __shared__ float s_t[2 * kEmuHits * kTraceBlock];
    int cur = 0, nh = 0, nh_best = 0;                // buffer being filled; hits of the current instance / of the nearest one (may exceed kEmuHits)
    // Fact 3 needs "no model answers nearer than its own closest hit".  A walk's answer t' >= t_min can only be nearer in DISTANCE |t'| when
    // t_min < 0 (the predicate accepts hits up to EPSILON behind the origin) and the model has a second hit: such an instance is
    // `ambiguous`.  As the nearest model it is settled by its replay; anywhere else it sends the ray to the walk.
    int n_amb = 0; bool best_amb = false;
    float c_t = kFloatMax; int c_tri = -1;           // closest hit of the current instance (Renderer.cpp:209 over every triangle: tier R1)

    int node = kDone, i = -1;
    V3 bo = v3(0, 0, 0), bd = v3(0, 0, 0);          // the ray as stored (Ray::base, Primitive.h:160-164)
    V3 winv = v3(0, 0, 0);                          // reciprocal of the normalised world direction (TLAS level)
    unsigned near_off = 0u, wnear_off = 0u;
    V3 ro = v3(0, 0, 0), rd = v3(0, 0, 1), rinv = v3(0, 0, 0);   // the ray of the current level: world, or model space of the entered instance (exact)
    float tmin = 0.0f, tmax = 0.0f;
    float g_dist = kFloatMax, g_t = 0.0f;
    int g_model = -1, g_tri = -1;
    WarpBatch work;
    const int vote_tri = sc.vote_tri, vote_inst = sc.vote_inst, vote_refill = sc.vote_refill;

    for (;;) {
        // ---- (1) inner nodes: as k_trace_bvh, except that inside an instance the interval never shrinks (every hit is wanted)
        if (node >= 0) {
            int key[4], lnk[4];
            nodeChildren<true>(reinterpret_cast<const char*>(&sc.nodes[node]), ro, rinv, near_off, tmin, tmax, key, lnk);
            if (COUNT) cnt.x++;
            node = stack.descend(key, lnk);
        }
        // ---- (2) who waits for what
        const LaneVote vt = laneVote(node, i >= 0 || !work.exhausted);
        if (vt.n_all == 0u) break;
        const unsigned code = vt.code;

        // ---- (3a) one triangle of the held leaf: the reference's predicate (Renderer.cpp:174-201), every hit recorded
        if (vt.tri && vt.n_tri >= min(vote_tri, vt.n_inner)) {
            const TriTest h = leafTriangle(sc, (int)(code >> 3), ro, rd);
            if (COUNT) cnt.z++;
            if (!h.reject) {
                const int id = h.id; const float t = h.t;
                if (nh < kEmuHits) {
                    const int slot = ((cur * kEmuHits + nh) * kTraceBlock) + threadIdx.x;
                    s_id[slot] = id; s_t[slot] = t;
                }
                ++nh;
                if (t < c_t || (t == c_t && c_tri >= 0 && id < c_tri)) { c_t = t; c_tri = id; }      // brute force in index order
            }
            if (code & 7u) node = (int)~(code + 7u); else node = stack.pop();
        }
        // ---- (3b) TLAS leaf: enter instance `im` (Renderer.cpp:381-384)
        if (vt.enter && vt.n_enter >= min(vote_inst, vt.n_inner)) {
            const int im = (int)(code & kIndexMask);
            const InstanceTrace* __restrict__ inst = &sc.inst[im];
            const float mscale = enterInstance(inst, bo, bd, ro, rd, rinv, near_off);
            tmin = kModelTmin;
            tmax = 3.0e38f;                                                     // all hits: a far one can keep the walk going until it meets a near one
            nh = 0; c_t = kFloatMax; c_tri = -1;
            stack.push(__float_as_int(__fdividef(1.0f, mscale)));                  // world distance per unit of model-space t, for the exit step
            stack.push((int)~(kExitBit | (unsigned)im));
            node = __float_as_int(__ldg(&inst->grid.z));                        // BLAS root of the instance's mesh
        }
        // ---- (3c) marker popped: leave instance `im`; nearest-model decision (Renderer.cpp:388-398) exactly as k_trace_bvh makes it
        if (vt.exit && vt.n_exit >= min(vote_inst, vt.n_inner)) {
            const int im = (int)(code & kIndexMask);
            const float ascale = __int_as_float(stack.pop());
            const float cb = rankSlack(sc, bo);
            const bool amb = c_tri >= 0 && c_t < 0.0f && nh >= 2;
            if (amb) ++n_amb;
            if (c_tri >= 0 && takeInstance<false>(sc, bo, bd, cb, im, c_t, ascale, g_model, g_t, g_dist)) {
                g_model = im; g_tri = c_tri; g_t = c_t;
                nh_best = nh; cur ^= 1;                                          // the buffer just filled is kept; the next instance fills the other
                best_amb = amb;
            }
            nh = 0; c_t = kFloatMax; c_tri = -1;
            ro = bo; rinv = winv; near_off = wnear_off;
            tmin = sc.tmin_world; tmax = worldBound(g_dist, sc.prune, cb);
            node = stack.pop();
        }
        // ---- (3d) retire finished rays, refill the lanes from the warp's batch
        if (vt.n_done > 0 && vt.n_done >= min(vote_refill, vt.n_inner)) {
            const unsigned m_done = __ballot_sync(kFull, vt.done && vt.live);
            if (vt.done && i >= 0) {
                const bool found = g_model >= 0;
                hit[i] = make_float4(found ? -1.0f : kFloatMax, __int_as_float(found ? g_tri : -1), __int_as_float(found ? g_model : -1), g_t);
                emu.n[i] = !found ? 0 : n_amb > (best_amb ? 1 : 0) ? kEmuHits + 1 : nh_best;      // > kEmuHits: not replayed, the walk answers
                if (found && nh_best > 1) {                                      // a single hit is the one in the hit record
                    const int kept = min(nh_best, kEmuHits), base = (cur ^ 1) * kEmuHits;
                    for (int j = 0; j < kept; ++j) {
                        const int slot = (base + j) * kTraceBlock + threadIdx.x;
                        emu.id[(size_t)j * emu.stride + i] = s_id[slot]; emu.t[(size_t)j * emu.stride + i] = s_t[slot];
                    }
                }
                if (COUNT) { if (counts) counts[i] = cnt; tot_x += cnt.x; tot_z += cnt.z; }
                i = -1;
            }
            work.fetch(cursor, sc.batch, n);
            int next;
            if (work.claim(m_done, vt.done && vt.live, next)) {
                i = next;
                const float4 o4 = O[i], d4 = D[i];
                bo = v3(o4); bd = v3(d4);
                const float il = rsqrtf(bd.x * bd.x + bd.y * bd.y + bd.z * bd.z);
                winv = v3(safeInv(bd.x * il), safeInv(bd.y * il), safeInv(bd.z * il));
                wnear_off = nearOffsets(bd);
                ro = bo; rinv = winv; near_off = wnear_off;
                tmin = sc.tmin_world; tmax = 3.0e38f;
                g_dist = kFloatMax; g_model = -1; g_tri = -1; g_t = 0.0f;
                nh = 0; nh_best = 0; c_t = kFloatMax; c_tri = -1; n_amb = 0; best_amb = false;
                if (COUNT) cnt = make_int4(0, 0, 0, 0);
                stack.sp = 0; stack.push(kDone);
                node = sc.tlas_root;
            }
            work.advance(m_done);
        }
    }
    if (stamp && (threadIdx.x & 31) == 0) atomicMax(stamp + 1, globalTimerNs());
    if (COUNT) { warpTotalAdd(&st->count_nodes, tot_x); warpTotalAdd(&st->count_tris, tot_z); }
}

// ---- launches 2 and 3: replay the walk of the nearest model over its hits (Renderer.cpp:238-360) -----------------------------------------
// Most replays end in the entry voxel (a ray that meets a wall enters the wall's box at the hit), a few take 30-70 steps (a ray that leaves
// a scaled-up sphere starts its walk at the far side of the sphere's box).  One thread per slot for the whole replay ran at 6 of 32 lanes
// (profiles/r02/ncu_emu_bundled.txt); one persistent kernel that sets up new slots for the lanes that finished ran either the set-up or the
// steps at a quarter of the warp.  So the two parts get a kernel each:
//   k_emu_setup  one thread per slot, full width: the reference's ray transform, slab test, entry voxel and DDA increments (~600
//                instructions of un-contracted divides and square roots), then up to kSetupSteps voxel steps; a replay that is not over by
//                then is written to a queue (80 bytes of DDA state);
//   k_emu_tail   persistent warps: a lane owns one queued replay at a time, every round all lanes take ONE voxel step, and when enough
//                lanes are free they load the next queue entries (cheap: no arithmetic to redo).
namespace {

struct Replay {
    int i, nh, ix, iy, iz, cx, cy, cz, k, best_k, w_tri, steps;
    unsigned ulo, uhi, gpos, seen;
    float tmx, tmy, tmz, dx, dy, dz, w_t, t_star;
    bool inter, passed;
};

// the walk leaves the model: more than two voxels past the last voxel that listed a hit triangle (Renderer.cpp:326-329)
__device__ __forceinline__ bool pastLastHit(const Replay& r)
{
    return r.inter && (abs(r.cx - r.ix) > 2 || abs(r.cy - r.iy) > 2 || abs(r.cz - r.iz) > 2);
}

// one DDA step to the next voxel (Renderer.cpp:331-357, without branches); true when the walk leaves the grid
__device__ __forceinline__ bool ddaStep(Replay& r, int GX, int GY, int GZ)
{
    const bool px = r.gpos & (1u << 9), py = r.gpos & (1u << 19), pz = r.gpos & (1u << 29);
    const bool sx = r.tmx < r.tmy && r.tmx < r.tmz, sy = !sx && r.tmy < r.tmz;
    r.ix += sx ? (px ? 1 : -1) : 0; r.iy += sy ? (py ? 1 : -1) : 0; r.iz += (sx || sy) ? 0 : (pz ? 1 : -1);
    const float tsel = sx ? r.tmx : sy ? r.tmy : r.tmz;
    const int isel = sx ? r.ix : sy ? r.iy : r.iz, lim = sx ? (px ? GX : -1) : sy ? (py ? GY : -1) : (pz ? GZ : -1);
    if (isel == lim || tsel >= kFloatMax) return true;
    r.tmx = sx ? xadd(r.tmx, r.dx) : r.tmx; r.tmy = sy ? xadd(r.tmy, r.dy) : r.tmy; r.tmz = (sx || sy) ? r.tmz : xadd(r.tmz, r.dz);
    return false;
}

// the box (ulo, uhi) around the voxel boxes of a replay's hits: start empty, then add each hit's box [lj, hj]
constexpr unsigned kEmptyLo = 0x1ffu | (0x1ffu << 10) | (0x1ffu << 20), kEmptyHi = 0u;
__device__ __forceinline__ void unionBox(unsigned& ulo, unsigned& uhi, unsigned lj, unsigned hj)
{
    if ((((hj | kGuard) - lj) & kGuard) == kGuard) {                    // listed somewhere (lo <= hi on every axis)
        ulo = min(ulo & 0x1ffu, lj & 0x1ffu) | min(ulo & (0x1ffu << 10), lj & (0x1ffu << 10)) | min(ulo & (0x1ffu << 20), lj & (0x1ffu << 20));
        uhi = max(uhi & 0x1ffu, hj & 0x1ffu) | max(uhi & (0x1ffu << 10), hj & (0x1ffu << 10)) | max(uhi & (0x1ffu << 20), hj & (0x1ffu << 20));
    }
}

// one voxel of the walk; true when the replay is over (r.w_tri / r.w_t hold the walk's answer so far)
template <int BURST = kBurst>
__device__ __forceinline__ bool replayStep(Replay& r, int GX, int GY, int GZ, const unsigned* s_lo, const unsigned* s_hi, const float* s_ts, const int* s_ids, int stride)
{
    ++r.steps;
    const unsigned gneg = kGuard ^ r.gpos;
    const unsigned v = (unsigned)r.ix | ((unsigned)r.iy << 10) | ((unsigned)r.iz << 20);
    bool any = false, finished = false;
    const unsigned u1 = (v | kGuard) - r.ulo, u2 = (r.uhi | kGuard) - v;      // per axis: guard bit set <=> lo <= index / index <= hi
    if ((u1 & u2 & kGuard) == kGuard) {                                       // inside the box around all hits: look at them one by one
#pragma unroll 1
        for (int j = 0; j < r.nh; ++j) {
            const int slot = j * stride + threadIdx.x;
            const unsigned d1 = (v | kGuard) - s_lo[slot], d2 = (s_hi[slot] | kGuard) - v;
            if ((d1 & d2 & kGuard) == kGuard) {
                any = true;                                        // the voxel lists a triangle the ray hits (Renderer.cpp:217-236)
                if (!((r.seen >> j) & 1u)) {                       // its first test: the only one that can update the nearest hit
                    r.seen |= 1u << j;
                    const float tj = s_ts[slot]; const int idj = s_ids[slot];
                    if (r.w_t > tj || (r.w_t == tj && r.best_k == r.k && idj < r.w_tri)) { r.w_t = tj; r.w_tri = idj; r.best_k = r.k; }   // Renderer.cpp:209
                }
            }
        }
    } else if ((~u2 & r.gpos) | (~u1 & gneg)) r.passed = true;               // indices move one way only
    // t* is the smallest t of ALL the model's hits: once the walk has met a hit with that t nothing it does later can change
    // its answer's t, and a tie for the triangle is settled inside the voxel just closed - the rest of the walk is not needed
    if (r.w_t == r.t_star) finished = true;
    else {
        if (any) { r.cx = r.ix; r.cy = r.iy; r.cz = r.iz; r.inter = true; }
        if (pastLastHit(r)) finished = true;
        else if (r.passed) finished = true;         // no voxel ahead lists a hit triangle: the walk ends with what it has
        else finished = ddaStep(r, GX, GY, GZ);
    }
    ++r.k;
    // Voxels outside the box around the hits list no hit triangle: nothing but the walk's own exit tests and DDA arithmetic happens there,
    // so up to kBurst of them are taken at once (a ray that leaves a scaled-up mesh walks a dozen such voxels before it reaches the first hit).
#pragma unroll 1
    for (int b = 0; b < BURST && !finished; ++b) {
        const unsigned w = (unsigned)r.ix | ((unsigned)r.iy << 10) | ((unsigned)r.iz << 20);
        const unsigned q1 = (w | kGuard) - r.ulo, q2 = (r.uhi | kGuard) - w;
        if ((q1 & q2 & kGuard) == kGuard) break;                               // inside: the next call looks at the hits
        ++r.steps;
        if ((~q2 & r.gpos) | (~q1 & gneg)) finished = true;                     // passed for good (this voxel is visited, the walk ends after it)
        else if (pastLastHit(r)) finished = true;
        else finished = ddaStep(r, GX, GY, GZ);
        ++r.k;
    }
    return finished;
}

// the start of a model's walk (Renderer.cpp:150-170, 252-311): slab test against the mesh box, entry point, entry voxel, DDA increments.
// false: the reference does not enter the grid (its answer for the model is "no hit")
__device__ __forceinline__ bool replayEnter(const InstanceTrace* __restrict__ inst, const V3& ro, const V3& rd, int GX, int GY, int GZ, Replay& r)
{
    const float4 bbmin_wx = ldg4(&inst->bb_min), bbmax_wy = ldg4(&inst->bb_max), gridrec = ldg4(&inst->grid);
    const V3 mn = v3(bbmin_wx), mx = v3(bbmax_wy);
    const V3 inv = v3(xdiv(1.0f, rd.x), xdiv(1.0f, rd.y), xdiv(1.0f, rd.z));   // Renderer.cpp:383
    // Renderer.cpp:150-170
    const float t1 = rd.x == 0.0f ? kFloatMin : xmul(xsub(mn.x, ro.x), inv.x);
    const float t2 = rd.x == 0.0f ? kFloatMax : xmul(xsub(mx.x, ro.x), inv.x);
    const float t3 = rd.y == 0.0f ? kFloatMin : xmul(xsub(mn.y, ro.y), inv.y);
    const float t4 = rd.y == 0.0f ? kFloatMax : xmul(xsub(mx.y, ro.y), inv.y);
    const float t5 = rd.z == 0.0f ? kFloatMin : xmul(xsub(mn.z, ro.z), inv.z);
    const float t6 = rd.z == 0.0f ? kFloatMax : xmul(xsub(mx.z, ro.z), inv.z);
    const float sl_min = max_std(max_std(min_std(t1, t2), min_std(t3, t4)), min_std(t5, t6));
    const float sl_max = min_std(min_std(max_std(t1, t2), max_std(t3, t4)), max_std(t5, t6));
    const V3 p = xadd(ro, xscale(rd, sl_min));
    if ((sl_max < 0 || sl_min > sl_max) || (xsub(p.x, mn.x) < -kEpsilon || xsub(p.y, mn.y) < -kEpsilon || xsub(p.z, mn.z) < -kEpsilon)) return false;   // Renderer.cpp:252-259
    const float wx = bbmin_wx.w, wy = bbmax_wy.w, wz = gridrec.x;
    r.ix = f2i_x86(xdiv(xabs(xadd(xsub(p.x, mn.x), kEpsilon)), wx));
    r.iy = f2i_x86(xdiv(xabs(xadd(xsub(p.y, mn.y), kEpsilon)), wy));
    r.iz = f2i_x86(xdiv(xabs(xadd(xsub(p.z, mn.z), kEpsilon)), wz));
    r.ix = min(max(r.ix, 0), GX - 1); r.iy = min(max(r.iy, 0), GY - 1); r.iz = min(max(r.iz, 0), GZ - 1);
    r.tmx = kFloatMax; r.tmy = kFloatMax; r.tmz = kFloatMax; r.dx = kFloatMax; r.dy = kFloatMax; r.dz = kFloatMax;
    if (rd.x != 0) { const int nx = rd.x > 0.0f ? r.ix + 1 : r.ix; r.dx = xabs(xmul(wx, inv.x)); r.tmx = xmul(xsub(xadd(mn.x, xmul((float)nx, wx)), p.x), inv.x); }
    if (rd.y != 0) { const int ny = rd.y > 0.0f ? r.iy + 1 : r.iy; r.dy = xabs(xmul(wy, inv.y)); r.tmy = xmul(xsub(xadd(mn.y, xmul((float)ny, wy)), p.y), inv.y); }
    if (rd.z != 0) { const int nz = rd.z > 0.0f ? r.iz + 1 : r.iz; r.dz = xabs(xmul(wz, inv.z)); r.tmz = xmul(xsub(xadd(mn.z, xmul((float)nz, wz)), p.z), inv.z); }
    // guard bits of the axes along which the voxel index grows: "the walk has passed a box for good" is one mask test
    r.gpos = (rd.x > 0.0f ? 1u << 9 : 0u) | (rd.y > 0.0f ? 1u << 19 : 0u) | (rd.z > 0.0f ? 1u << 29 : 0u);
    r.seen = 0u; r.passed = false; r.cx = 0; r.cy = 0; r.cz = 0; r.best_k = -1; r.k = 0; r.inter = false;
    return true;
}

// the hits of slot i and their voxel boxes into the lane's shared-memory column; (ulo, uhi) = the box around all of them
__device__ __forceinline__ void replayLoadHits(const SceneDev& sc, const EmuBuf& emu, int i, int nh, int first_id, float t_star, unsigned& ulo, unsigned& uhi,
                                               unsigned* s_lo, unsigned* s_hi, float* s_ts, int* s_ids, int stride)
{
    ulo = kEmptyLo; uhi = kEmptyHi;
#pragma unroll 1
    for (int j = 0; j < nh; ++j) {
        const int slot = j * stride + threadIdx.x;
        const int idj = nh == 1 ? first_id : emu.id[(size_t)j * emu.stride + i];
        s_ids[slot] = idj; s_ts[slot] = nh == 1 ? t_star : emu.t[(size_t)j * emu.stride + i];
        const int2 bx = __ldg(&sc.tri_box[idj]);
        const unsigned lj = (unsigned)bx.x, hj = (unsigned)bx.y;
        s_lo[slot] = lj; s_hi[slot] = hj;
        unionBox(ulo, uhi, lj, hj);
    }
}

// the end of a replay: confirm the closest hit as the reference's answer, or hand the slot to the walk itself
template <bool UV>
__device__ __forceinline__ void replayFinish(const SceneDev& sc, const Replay& r, const float4& h, const float4* __restrict__ O, const float4* __restrict__ D,
                                             float4* __restrict__ hit, float2* __restrict__ uv, FrameState* st, int round, const EmuBuf& emu)
{
    if (r.w_tri >= 0 && r.w_t == r.t_star) {
        // the walk of the nearest model finds the closest hit: that is the reference's answer (the triangle is the WALK's: its tie rule)
        if (r.w_tri != __float_as_int(h.y)) hit[r.i] = make_float4(h.x, __int_as_float(r.w_tri), h.z, h.w);
        if (UV && uv) uv[r.i] = hitBarycentrics(sc, __float_as_int(h.z), v3(O[r.i]), v3(D[r.i]), r.w_tri);
    } else emu.list[atomicAdd(&st->n_replay[round], 1u)] = r.i;                 // the walk itself answers this one (last launch)
}

}  // namespace

template <bool UV, bool COUNT>
__global__ void __launch_bounds__(kSetupBlock)
k_emu_setup(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit, float2* __restrict__ uv,
            int4* __restrict__ counts, FrameState* st, int round, int n_fixed, EmuBuf emu)
{
    const int n = n_fixed >= 0 ? n_fixed : st->n_active[round];
    const int GX = sc.gx, GY = sc.gy, GZ = sc.gz;
    __shared__ int s_ids[kEmuHits * kSetupBlock];                  // [hit][thread]: the hits of the thread's replay
    __shared__ float s_ts[kEmuHits * kSetupBlock];
    __shared__ unsigned s_lo[kEmuHits * kSetupBlock], s_hi[kEmuHits * kSetupBlock];
    unsigned long long steps_total = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 h = hit[i];
        const int im = __float_as_int(h.z);
        if (im < 0) { if (UV && uv) uv[i] = make_float2(0.0f, 0.0f); continue; }      // no real hit: no walk finds one
        Replay r;
        r.i = i; r.nh = emu.n[i]; r.t_star = h.w; r.w_tri = -1; r.w_t = kFloatMax; r.steps = 0;
        bool walking = false;
        if (r.nh <= kEmuHits) {
            const V3 bo = v3(O[i]), bd = v3(D[i]);
            const InstanceTrace* __restrict__ inst = &sc.inst[im];
            const float4 w0 = ldg4(&inst->w2m[0]), w1 = ldg4(&inst->w2m[1]), w2 = ldg4(&inst->w2m[2]);
            const V3 ro = xmat4(w0, w1, w2, bo, 1.0f);                               // Renderer.cpp:381
            const V3 rd = xnormalize(xmat4(w0, w1, w2, bd, 0.0f));                   // Renderer.cpp:382
            if (replayEnter(inst, ro, rd, GX, GY, GZ, r)) {
                replayLoadHits(sc, emu, i, r.nh, __float_as_int(h.y), r.t_star, r.ulo, r.uhi, s_lo, s_hi, s_ts, s_ids, kSetupBlock);
                walking = true;
#pragma unroll 1
                for (int s = 0; s < kSetupSteps && walking; ++s) walking = !replayStep<kSetupBurst>(r, GX, GY, GZ, s_lo, s_hi, s_ts, s_ids, kSetupBlock);
            }
        }
        if (walking) {
            const unsigned q = atomicAdd(&st->n_cont[round], 1u);
            if (q < (unsigned)emu.cont_cap) {                       // the rest of this replay: k_emu_tail
                uint4* rec = emu.cont + (size_t)q * 5;
                rec[0] = make_uint4((unsigned)i, (unsigned)r.ix | ((unsigned)r.iy << 10) | ((unsigned)r.iz << 20), r.gpos | (r.inter ? 1u : 0u) | ((unsigned)r.nh << 1), r.seen);
                rec[1] = make_uint4(__float_as_uint(r.tmx), __float_as_uint(r.tmy), __float_as_uint(r.tmz), __float_as_uint(r.t_star));
                rec[2] = make_uint4(__float_as_uint(r.dx), __float_as_uint(r.dy), __float_as_uint(r.dz), __float_as_uint(r.w_t));
                rec[3] = make_uint4((unsigned)r.w_tri, (unsigned)r.best_k, (unsigned)r.k, (unsigned)r.cx | ((unsigned)r.cy << 10) | ((unsigned)r.cz << 20));
                rec[4] = make_uint4(r.ulo, r.uhi, (unsigned)r.steps, 0u);
                continue;
            }
            r.w_tri = -1;                                           // queue full (cannot happen with cont_cap = slots): the walk answers
        }
        if (COUNT) { if (counts) counts[i].y = r.steps; steps_total += r.steps; }
        replayFinish<UV>(sc, r, h, O, D, hit, uv, st, round, emu);
    }
    if (COUNT) warpTotalAdd(&st->count_cells, steps_total);
}

template <bool UV, bool COUNT>
__global__ void __launch_bounds__(kReplayBlock)
k_emu_tail(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit, float2* __restrict__ uv,
           int4* __restrict__ counts, FrameState* st, int round, EmuBuf emu)
{
    const int n = (int)min(st->n_cont[round], (unsigned)emu.cont_cap);
    unsigned int* cursor = &st->fetch_emu[round];
    const int GX = sc.gx, GY = sc.gy, GZ = sc.gz;
    __shared__ int s_ids[kEmuHits * kReplayBlock];
    __shared__ float s_ts[kEmuHits * kReplayBlock];
    __shared__ unsigned s_lo[kEmuHits * kReplayBlock], s_hi[kEmuHits * kReplayBlock];
    unsigned long long steps_total = 0;
    enum : int { R_IDLE = 0, R_STEP = 1, R_DONE = 2 };
    int state = R_IDLE;
    Replay r; r.i = -1; r.nh = 0; r.steps = 0;
    WarpBatch work;

    for (;;) {
        // ---- one voxel of every replay in progress
        if (state == R_STEP && replayStep(r, GX, GY, GZ, s_lo, s_hi, s_ts, s_ids, kReplayBlock)) state = R_DONE;
        // ---- who is where
        const unsigned m_step = __ballot_sync(kFull, state == R_STEP);
        if (m_step != 0u && 32 - __popc(m_step) < sc.emu_refill) continue;      // keep stepping until enough lanes are free (or none steps)
        // ---- results of the finished replays
        if (state == R_DONE) {
            if (COUNT) { if (counts) counts[r.i].y = r.steps; steps_total += r.steps; }
            replayFinish<UV>(sc, r, hit[r.i], O, D, hit, uv, st, round, emu);
            state = R_IDLE; r.i = -1;
        }
        // ---- the next queue entries for the free lanes
        work.fetch(cursor, kReplayBatch, n);
        const unsigned m_idle = __ballot_sync(kFull, state == R_IDLE);
        if (m_step == 0u && work.exhausted && work.w_next >= work.w_end) break;      // nothing in progress, nothing left (every lane is idle here)
        int next;
        if (work.claim(m_idle, state == R_IDLE, next)) {
            const uint4* rec = emu.cont + (size_t)next * 5;
            const uint4 a = rec[0], b = rec[1], c = rec[2], d = rec[3], e = rec[4];
            r.i = (int)a.x; r.ix = a.y & 0x3ff; r.iy = (a.y >> 10) & 0x3ff; r.iz = a.y >> 20;
            r.gpos = a.z & kGuard; r.inter = a.z & 1u; r.nh = (a.z >> 1) & 0xf; r.seen = a.w; r.passed = false;
            r.tmx = __uint_as_float(b.x); r.tmy = __uint_as_float(b.y); r.tmz = __uint_as_float(b.z); r.t_star = __uint_as_float(b.w);
            r.dx = __uint_as_float(c.x); r.dy = __uint_as_float(c.y); r.dz = __uint_as_float(c.z); r.w_t = __uint_as_float(c.w);
            r.w_tri = (int)d.x; r.best_k = (int)d.y; r.k = (int)d.z; r.cx = d.w & 0x3ff; r.cy = (d.w >> 10) & 0x3ff; r.cz = d.w >> 20;
            r.steps = (int)e.z;
            const float4 h = hit[r.i];
            replayLoadHits(sc, emu, r.i, r.nh, __float_as_int(h.y), r.t_star, r.ulo, r.uhi, s_lo, s_hi, s_ts, s_ids, kReplayBlock);
            state = R_STEP;
        }
        work.advance(m_idle);
    }
    if (COUNT) warpTotalAdd(&st->count_cells, steps_total);
}

// ---- launch 4: the rays the replay could not confirm, emulated in FULL -----------------------------------------------------------------
// For a ray on the list the walk of the nearest model does not return the closest hit, so the reference's answer may come from any model.
// This kernel answers it without the voxel lists all the same: every instance the ray's line meets is traversed for ALL its hits (no
// pruning by distance: a farther model may hold the answer), every such model's walk is replayed on the spot, and the models' answers are
// combined exactly as Renderer.cpp:388-398 does (exact world distances, ties to the lower model index).  It runs for ~0.5 % of the rays;
// walking the grids for them instead (k_trace_grid in list mode) cost 0.4 ms per bounce on the reference's scene and milliseconds on a
// dense mesh (one lane testing the hundreds of triangles of every voxel), for any number of rays.  It keeps kFullHits + kBigHits hits
// per model (rays with more than kEmuHits in their nearest model come here too: a ray that grazes a finely tessellated surface crosses
// it dozens of times); what still goes to the walk is a ray with more than that.
template <bool UV>
__global__ void __launch_bounds__(kTraceBlock, 4)
k_emu_full(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit, float2* __restrict__ uv,
           FrameState* st, int round, EmuBuf emu)
{
    // hits beyond the kFullHits kept in shared memory: kBigHits more per thread in global memory, (id, t, lo | seen flag, hi) each
    uint4* __restrict__ big = emu.big + (size_t)(blockIdx.x * blockDim.x + threadIdx.x) * kBigHits;
    const int n = (int)st->n_replay[round];
    if (blockIdx.x == 0 && threadIdx.x == 0) st->rays_reemulated += (unsigned long long)n;
    unsigned int* cursor = &st->fetch_replay[round];
    const int GX = sc.gx, GY = sc.gy, GZ = sc.gz;
    if (n == 0 || sc.tlas_root < 0) return;

    __shared__ int s_stack[kSmemStack * kTraceBlock];
    int l_stack[kBvhStack - kSmemStack];
    SplitStack stack(s_stack, l_stack);
    __shared__ int s_ids[kFullHits * kTraceBlock];                  // [hit][thread]: the hits of the instance being traversed
    __shared__ float s_ts[kFullHits * kTraceBlock];
    __shared__ unsigned s_lo[kFullHits * kTraceBlock], s_hi[kFullHits * kTraceBlock];
    int nh = 0;
    float c_t = kFloatMax;                          // smallest t of the instance's hits: the replay may stop when the walk meets it
    bool overflow = false;

    int node = kDone, i = -1;
    V3 bo = v3(0, 0, 0), bd = v3(0, 0, 0), winv = v3(0, 0, 0);
    unsigned near_off = 0u, wnear_off = 0u;
    V3 ro = v3(0, 0, 0), rd = v3(0, 0, 1), rinv = v3(0, 0, 0);
    float tmin = 0.0f, tmax = 0.0f;
    float g_dist = kFloatMax, g_t = 0.0f;
    int g_model = -1, g_tri = -1;
    WarpBatch work;
    const int vote_tri = sc.vote_tri, vote_inst = sc.vote_inst, vote_refill = sc.vote_refill;

    for (;;) {
        if (node >= 0) {
            int key[4], lnk[4];
            nodeChildren<true>(reinterpret_cast<const char*>(&sc.nodes[node]), ro, rinv, near_off, tmin, tmax, key, lnk);
            node = stack.descend(key, lnk);
        }
        const LaneVote vt = laneVote(node, i >= 0 || !work.exhausted);
        if (vt.n_all == 0u) break;
        const unsigned code = vt.code;

        // ---- one triangle of the held leaf: the reference's predicate (Renderer.cpp:174-201), every hit recorded with its voxel box
        if (vt.tri && vt.n_tri >= min(vote_tri, vt.n_inner)) {
            const TriTest h = leafTriangle(sc, (int)(code >> 3), ro, rd);
            if (!h.reject) {
                const float t = h.t;
                if (nh < kFullHits + kBigHits) {
                    const int id = h.id;
                    const int2 bx = __ldg(&sc.tri_box[id]);
                    if (nh < kFullHits) {
                        const int slot = nh * kTraceBlock + threadIdx.x;
                        s_ids[slot] = id; s_ts[slot] = t; s_lo[slot] = (unsigned)bx.x; s_hi[slot] = (unsigned)bx.y;
                    } else big[nh - kFullHits] = make_uint4((unsigned)id, __float_as_uint(t), (unsigned)bx.x, (unsigned)bx.y);
                }
                ++nh;
                if (t < c_t) c_t = t;
            }
            if (code & 7u) node = (int)~(code + 7u); else node = stack.pop();
        }
        // ---- enter instance `im` (Renderer.cpp:381-384)
        if (vt.enter && vt.n_enter >= min(vote_inst, vt.n_inner)) {
            const int im = (int)(code & kIndexMask);
            const InstanceTrace* __restrict__ inst = &sc.inst[im];
            enterInstance(inst, bo, bd, ro, rd, rinv, near_off);
            tmin = kModelTmin; tmax = 3.0e38f;
            nh = 0; c_t = kFloatMax;
            stack.push((int)~(kExitBit | (unsigned)im));
            node = __float_as_int(__ldg(&inst->grid.z));
        }
        // ---- leave instance `im`: replay its walk over the hits found, then the reference's nearest-model rule (Renderer.cpp:388-398)
        if (vt.exit && vt.n_exit >= min(vote_inst, vt.n_inner)) {
            const int im = (int)(code & kIndexMask);
            if (nh > kFullHits + kBigHits) overflow = true;
            else if (nh > kFullHits) {
                // a ray that grazes a finely tessellated surface: the same replay with the further hits read from global memory (no box
                // around all hits, no burst: rare)
                Replay r;
                r.i = i; r.nh = nh; r.t_star = c_t; r.w_tri = -1; r.w_t = kFloatMax; r.steps = 0;
                if (replayEnter(&sc.inst[im], ro, rd, GX, GY, GZ, r)) {
                    for (;;) {
                        const unsigned v = (unsigned)r.ix | ((unsigned)r.iy << 10) | ((unsigned)r.iz << 20);
                        bool any = false;
#pragma unroll 1
                        for (int j = 0; j < nh; ++j) {
                            unsigned lj, hj; float tj; int idj; bool was_seen;
                            if (j < kFullHits) {
                                const int slot = j * kTraceBlock + threadIdx.x;
                                lj = s_lo[slot]; hj = s_hi[slot]; tj = s_ts[slot]; idj = s_ids[slot]; was_seen = (r.seen >> j) & 1u;
                            } else {
                                const uint4 e = big[j - kFullHits];
                                idj = (int)e.x; tj = __uint_as_float(e.y); lj = e.z & 0x7fffffffu; hj = e.w; was_seen = e.z >> 31;
                            }
                            const unsigned d1 = (v | kGuard) - lj, d2 = (hj | kGuard) - v;
                            if ((d1 & d2 & kGuard) != kGuard) continue;
                            any = true;
                            if (was_seen) continue;
                            if (j < kFullHits) r.seen |= 1u << j; else big[j - kFullHits].z = lj | 0x80000000u;
                            if (r.w_t > tj || (r.w_t == tj && r.best_k == r.k && idj < r.w_tri)) { r.w_t = tj; r.w_tri = idj; r.best_k = r.k; }
                        }
                        if (r.w_t == r.t_star) break;
                        if (any) { r.cx = r.ix; r.cy = r.iy; r.cz = r.iz; r.inter = true; }
                        if (pastLastHit(r) || ddaStep(r, GX, GY, GZ)) break;
                        ++r.k;
                    }
                    if (r.w_tri >= 0) {
                        const float dn = exactHitDistance(sc, bo, bd, im, r.w_t);
                        if (g_dist > dn || (g_dist == dn && g_model >= 0 && im < g_model)) { g_dist = dn; g_model = im; g_tri = r.w_tri; g_t = r.w_t; }
                    }
                }
            }
            else if (nh > 0) {
                Replay r;
                r.i = i; r.nh = nh; r.t_star = c_t; r.w_tri = -1; r.w_t = kFloatMax; r.steps = 0;
                if (replayEnter(&sc.inst[im], ro, rd, GX, GY, GZ, r)) {
                    r.ulo = kEmptyLo; r.uhi = kEmptyHi;
#pragma unroll 1
                    for (int j = 0; j < nh; ++j) unionBox(r.ulo, r.uhi, s_lo[j * kTraceBlock + threadIdx.x], s_hi[j * kTraceBlock + threadIdx.x]);
#pragma unroll 1
                    while (!replayStep(r, GX, GY, GZ, s_lo, s_hi, s_ts, s_ids, kTraceBlock)) { }
                    if (r.w_tri >= 0) {
                        const float dn = exactHitDistance(sc, bo, bd, im, r.w_t);
                        if (g_dist > dn || (g_dist == dn && g_model >= 0 && im < g_model)) { g_dist = dn; g_model = im; g_tri = r.w_tri; g_t = r.w_t; }   // Renderer.cpp:393 in model order
                    }
                }
            }
            nh = 0; c_t = kFloatMax;
            ro = bo; rinv = winv; near_off = wnear_off;
            tmin = sc.tmin_world; tmax = 3.0e38f;                                // no pruning by distance: a farther model may hold the answer
            node = stack.pop();
        }
        // ---- retire finished rays, refill the lanes from the warp's batch of the list
        if (vt.n_done > 0 && vt.n_done >= min(vote_refill, vt.n_inner)) {
            const unsigned m_done = __ballot_sync(kFull, vt.done && vt.live);
            if (vt.done && i >= 0) {
                if (overflow) emu.list2[atomicAdd(&st->n_walk[round], 1u)] = i;      // more hits in one model than are kept: the walk itself
                else {
                    const bool found = g_dist < kFloatMax;
                    hit[i] = make_float4(found ? g_dist : kFloatMax, __int_as_float(found ? g_tri : -1), __int_as_float(found ? g_model : -1), found ? g_t : 0.0f);
                    if (UV && uv) uv[i] = found ? hitBarycentrics(sc, g_model, bo, bd, g_tri) : make_float2(0.0f, 0.0f);
                }
                i = -1;
            }
            work.fetch(cursor, kFullBatch, n);
            int next;
            if (work.claim(m_done, vt.done && vt.live, next)) {
                i = __ldg(&emu.list[next]);
                const float4 o4 = O[i], d4 = D[i];
                bo = v3(o4); bd = v3(d4);
                const float il = rsqrtf(bd.x * bd.x + bd.y * bd.y + bd.z * bd.z);
                winv = v3(safeInv(bd.x * il), safeInv(bd.y * il), safeInv(bd.z * il));
                wnear_off = nearOffsets(bd);
                ro = bo; rinv = winv; near_off = wnear_off;
                tmin = sc.tmin_world; tmax = 3.0e38f;
                g_dist = kFloatMax; g_model = -1; g_tri = -1; g_t = 0.0f;
                nh = 0; c_t = kFloatMax; overflow = false;
                stack.sp = 0; stack.push(kDone);
                node = sc.tlas_root;
            }
            work.advance(m_done);
        }
    }
}

void launchTraceEmu(const SceneDev& sc, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, bool count_totals,
                    FrameState* st, int round, int n_fixed, int grid, int grid_replay, int grid_full, cudaStream_t stream, unsigned long long* stamp, const EmuBuf& emu)
{
    const bool count = counts || count_totals;
    const int grid_setup = grid_replay * 2;
    if (count) k_trace_emu<true><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, counts, st, round, n_fixed, stamp, emu);
    else k_trace_emu<false><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, counts, st, round, n_fixed, stamp, emu);
    if (count) {
        k_emu_setup<true, true><<<grid_setup, kSetupBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, emu);
        k_emu_tail<true, true><<<grid_replay, kReplayBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, emu);
    } else if (uv) {
        k_emu_setup<true, false><<<grid_setup, kSetupBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, emu);
        k_emu_tail<true, false><<<grid_replay, kReplayBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, emu);
    } else {
        k_emu_setup<false, false><<<grid_setup, kSetupBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, emu);
        k_emu_tail<false, false><<<grid_replay, kReplayBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, emu);
    }
    if (uv) k_emu_full<true><<<grid_full, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, st, round, emu);
    else k_emu_full<false><<<grid_full, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, st, round, emu);
}

int traceEmuOccupancy()
{
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_trace_emu<false>, kTraceBlock, 0);
    return nb;
}

}  // namespace ptap
