// trace_bvh.cu - closest hit through a two-level BVH (PTAP_ACCEL_BVH).
//
// New design; the reference has no BVH.  Semantics = oracle tier R1: for every model, the reference's own per-model
// ray set-up (Renderer.cpp:381-384) and its tolerant Moller-Trumbore predicate (Renderer.cpp:174-215) applied to
// every triangle of the model's mesh, nearest model-space t wins (ties: lowest triangle index), converted to a world
// distance as Renderer.cpp:388-391, nearest world distance wins (ties: lowest model index).  The BVH only decides
// WHICH triangles get tested: node bounds are conservative for the predicate's tolerance band (bvh_build.cpp), the
// slab test is evaluated with outward rounding slack, pruning bounds carry relative slack, and the triangle
// arithmetic is the un-contracted exact one, so the winner is bit-identical to brute force.
//
// Execution model (DESIGN.md "Closest hit"): a persistent grid of warps, each lane owning one ray at a time, scheduled as a
// warp-wide state machine.  A lane is in one of five states, encoded in its `node` register: at an inner node, holding
// a triangle leaf, about to enter an instance, about to leave one, or finished.  Every iteration of the ONE loop
//  (1) advances all lanes that are at inner nodes by one node (TLAS and BLAS share the 64-byte node format),
//  (2) counts the lanes waiting in each other state with warp ballots, and
//  (3) runs a state's step only when enough lanes wait for it (or when it is at least as popular as descending):
//      one Moller-Trumbore test per lane, the instance entry (the reference's world->model ray set-up), the instance
//      exit (model t -> world distance, nearest-model bookkeeping), retire + refill from the work-stealing cursor.
// Lanes never wait for a slower warp-mate's whole descent (the while-while form of this kernel measured 6 active
// lanes of 32 in its node loop, and the v1 per-model loop 7 of 32): they only wait until their state's queue fills.
//  * work stealing: each warp takes batches of consecutive rays from a device-side cursor (one atomic per batch).
//  * cross-instance pruning: once some instance reported a hit at world distance g, TLAS nodes beyond g are skipped and
//    the next instance is entered with the model-space bound t <= (g + |M o_m - o_w|) / |M3 d_m|.
//  * ANY (ptap_query_occluded, DESIGN.md 4.8): every ray starts as if a winner at its segment length L = D[i].w existed, and retires
//    as occluded at the first accepted triangle whose model's winner is provably nearer than L; the record it leaves otherwise is a
//    closest-hit candidate that k_resolve_occluded compares with L.
//
// Node = 128 B = one L1 line: a node-local origin, four links, and four child boxes as binary32 offsets from that origin
// (device_types.h: BvhNode); leaf-order triangle = 64 B with its global id (2 x LDG.E.256).  The node step costs one FMA per plane:
//   t = offset * inv + (p - o) * inv,
// with the (p - o) * inv term evaluated once per node.  Because it is taken RELATIVE TO THE NODE, the cancellation error of the FMA
// form is bounded by the node's own extent (the builder's outward margin covers it); the textbook form plane * inv - o * inv is
// unbounded for axis-parallel rays, which is why round 1's kernel spent a subtract and a multiply per plane.  Two children share one
// FFMA2 (packed binary32 FMA, new on sm_100), and the near / far planes of an axis are picked by ADDRESS from the direction's sign
// bits (they lie 16 bytes apart) instead of by a min / max pair per child and axis.
#include "bvh_traverse.cuh"

namespace ptap {

using namespace bvh;

#ifndef PTAP_TRACE_MIN_CTAS
#define PTAP_TRACE_MIN_CTAS 8     // 64 registers: 8 CTAs of 128 threads per SM, as round 1's kernel
#endif

// The triangle step's acceptance on top of the predicate: `tmax` is the model-space bound of the traversal AND the best t so far (they are
// the same number once best_tri >= 0); t must not exceed it, and !(t <= tmax) also rejects NaN (a degenerate det passes none of the
// predicate's rejections as true).  Then brute force's tie rule in index order: strictly nearer, or equal t and lower global id.
template <bool UV>
__device__ __forceinline__ void keepNearest(const TriTest& h, float& tmax, int& best_tri, float& best_u, float& best_v)
{
    if ((h.reject | (h.t > tmax)) || !(h.t <= tmax)) return;
    if (h.t < tmax || (best_tri >= 0 && h.id < best_tri)) { tmax = h.t; best_tri = h.id; if (UV) { best_u = h.u; best_v = h.v; } }
}

template <bool UV, bool COUNT, bool ANY = false>
__global__ void __launch_bounds__(kTraceBlock, PTAP_TRACE_MIN_CTAS)
k_trace_bvh(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit,
            float2* __restrict__ uv, int4* __restrict__ counts, FrameState* st, int round, int n_fixed, unsigned long long* __restrict__ stamp)
{
    const int n = n_fixed >= 0 ? n_fixed : st->n_active[round];
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_fixed < 0) st->rays_traced += (unsigned long long)n;
    if (stamp && threadIdx.x == 0) atomicMin(stamp, globalTimerNs());
    unsigned int* cursor = &st->fetch[round];
    unsigned long long tot_x = 0, tot_z = 0;
    int4 cnt = make_int4(0, 0, 0, 0);

    if (sc.tlas_root < 0) {                            // no instance has triangles: every ray misses
        for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
            hit[k] = make_float4(kFloatMax, __int_as_float(-1), __int_as_float(-1), 0.0f);
            if (UV && uv) uv[k] = make_float2(0.0f, 0.0f);
            if (COUNT && counts) counts[k] = cnt;
        }
        return;
    }

    __shared__ int s_stack[kSmemStack * kTraceBlock];
    int l_stack[kBvhStack - kSmemStack];
    SplitStack stack(s_stack, l_stack);
    int node = kDone, i = -1;
    // What only the instance enter / exit and the retire / refill steps touch: the ray as stored (bo, bd: Ray::base, Primitive.h:160-164),
    // the reciprocal of its normalised direction and its near-plane offsets (TLAS level), the nearest model so far (g_*; model and triangle
    // as float bit patterns).  A lane sets all of them when it takes a ray, before any step reads them.  Left uninitialised and with the ids
    // in float registers, the kernel compiles to the spill figures it had when these lived in one float array; as initialised ints, ptxas
    // spills up to 16 more bytes per instantiation at the 64-register bound.
    V3 bo, bd, winv;
    unsigned wnear_off;
    float g_dist, g_t, g_u, g_v;
    float g_model_f, g_tri_f;
    unsigned near_off = 0u;                         // byte offsets of the near planes inside a node for the current level
    V3 ro = v3(0, 0, 0), rd = v3(0, 0, 1), rinv = v3(0, 0, 0);   // the ray of the current level: world, or model space of the entered instance
    float tmin = 0.0f, tmax = 0.0f;
    int best_tri = -1; float best_u = 0.0f, best_v = 0.0f;
    WarpBatch work;
    const int vote_tri = sc.vote_tri, vote_inst = sc.vote_inst, vote_refill = sc.vote_refill;
    // ANY only: the segment length L, the absolute slack cb of the exit step for this ray, world units per model-space t of the entered instance
    float any_len = 0.0f, any_cb = 0.0f, any_scale = 0.0f;

    for (;;) {
        // ---- (1) inner nodes (TLAS and BLAS share the 4-wide format): test the four child boxes, continue with the nearest hit child,
        // push the other hit children farthest first.  An any-hit traversal takes the hit children in node order: 3 % faster than nearest
        // first (DESIGN 4.8).
        if (node >= 0) {
            int key[4], lnk[4];
            nodeChildren<!ANY>(reinterpret_cast<const char*>(&sc.nodes[node]), ro, rinv, near_off, tmin, tmax, key, lnk);
            if (COUNT) cnt.x++;
            node = stack.descend(key, lnk);
        }
        // ---- (2) who waits for what
        const LaneVote vt = laneVote(node, i >= 0 || !work.exhausted);
        if (vt.n_all == 0u) break;                              // every ray of the launch is retired
        const unsigned code = vt.code;

        // ---- (3a) one triangle of the held leaf (Renderer.cpp:174-215)
        if (vt.tri && vt.n_tri >= min(vote_tri, vt.n_inner)) {
            const TriTest h = leafTriangle(sc, (int)(code >> 3), ro, rd);
            if (COUNT) cnt.z++;
            keepNearest<UV>(h, tmax, best_tri, best_u, best_v);
            if constexpr (ANY) {
                // The model's true winner has t in [-EPSILON, tmax] (the best accepted t so far), so its world distance is at most
                // m = max(|tmax|, EPSILON) * ascale up to the exit step's slack m * tie + cb: when that is below L (at most kFloatMax), so
                // is the closest hit.
                bool occluded = false;
                if (best_tri >= 0) {
                    const float m = fmaxf(fabsf(tmax), kEpsilon) * any_scale;
                    occluded = m + (m * sc.tie + any_cb) < any_len;
                }
                if (occluded) { stack.sp = 0; node = kDone; g_model_f = __int_as_float(kAnyOccluded); }     // retire: empty stack, done state
                else if (code & 7u) node = (int)~(code + 7u); else node = stack.pop();
            } else {
                if (code & 7u) node = (int)~(code + 7u); else node = stack.pop();   // (first + 1, count - 1), or pop when the leaf is finished
            }
        }
        // ---- (3b) TLAS leaf: enter instance `im` (Renderer.cpp:381-384)
        if (vt.enter && vt.n_enter >= min(vote_inst, vt.n_inner)) {
            const int im = (int)(code & kIndexMask);
            const InstanceTrace* __restrict__ inst = &sc.inst[im];
            const float mscale = enterInstance(inst, bo, bd, ro, rd, rinv, near_off);
            tmin = kModelTmin;
            tmax = kFloatMax; best_tri = -1;                                    // Renderer.cpp:384
            if (g_dist < kFloatMax) {
                // World distance of a model-space t along this ray is t * |d_w| / |W3 d_w| when model_to_world inverts world_to_model
                // (checked at upload, else sc.prune = inf): a winner needs t <= g * |W3 d_w| / |d_w|, plus slack for the matrices' residual.
                const float tb = (g_dist * sc.prune + sc.c_pad + 1e-4f * (fabsf(bo.x) + fabsf(bo.y) + fabsf(bo.z))) * mscale * 1.0001f;
                if (tb < kFloatMax) tmax = tb;                                  // false for NaN / inf: no bound
            }
            if constexpr (ANY) any_scale = __fdividef(1.0f, mscale);           // the triangle step's copy of what is pushed next
            stack.push(__float_as_int(__fdividef(1.0f, mscale)));              // world distance per unit of model-space t, for the exit step
            stack.push((int)~(kExitBit | (unsigned)im));
            node = __float_as_int(__ldg(&inst->grid.z));                        // BLAS root of the instance's mesh
        }
        // ---- (3c) marker popped: leave instance `im` (Renderer.cpp:388-398)
        if (vt.exit && vt.n_exit >= min(vote_inst, vt.n_inner)) {
            const int im = (int)(code & kIndexMask);
            const float ascale = __int_as_float(stack.pop());                   // pushed under the marker at entry
            const float cb = rankSlack(sc, bo);
            if (best_tri >= 0 && takeInstance<ANY>(sc, bo, bd, cb, im, tmax, ascale, __float_as_int(g_model_f), g_t, g_dist)) {
                g_model_f = __int_as_float(im); g_tri_f = __int_as_float(best_tri); g_t = tmax;
                if (UV) { g_u = best_u; g_v = best_v; }
            }
            ro = bo; rinv = winv; near_off = wnear_off;
            tmin = sc.tmin_world; tmax = worldBound(g_dist, sc.prune, cb);
            node = stack.pop();
        }
        // ---- (3d) retire finished rays, refill the lanes from the warp's batch
        if (vt.n_done > 0 && vt.n_done >= min(vote_refill, vt.n_inner)) {
            const unsigned m_done = __ballot_sync(kFull, vt.done && vt.live);
            if (vt.done && i >= 0) {
                const bool found = g_dist < kFloatMax;
                // hit.x < 0 (a constant: the consumers only test the sign) tells the consumer to evaluate the exact world distance
                // from (model, t) (kernels.cuh: exactHitDistance)
                if constexpr (ANY) {
                    // g_dist starts at L here, so a candidate is a taken model; model kAnyOccluded = retired early, -1 = no candidate
                    const bool cand = __float_as_int(g_model_f) >= 0;
                    hit[i] = make_float4(cand ? -1.0f : kFloatMax, cand ? g_tri_f : __int_as_float(-1), g_model_f, g_t);
                } else {
                    hit[i] = make_float4(found ? -1.0f : kFloatMax, found ? g_tri_f : __int_as_float(-1), found ? g_model_f : __int_as_float(-1), g_t);
                }
                if (UV && uv) uv[i] = make_float2(g_u, g_v);
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
                wnear_off = nearOffsets(bd);                         // the normalisation keeps the sign bits
                ro = bo; rinv = winv; near_off = wnear_off;
                tmin = sc.tmin_world; tmax = 3.0e38f;
                g_dist = kFloatMax; g_model_f = __int_as_float(-1); g_tri_f = __int_as_float(-1); g_t = 0.0f; g_u = 0.0f; g_v = 0.0f;
                best_tri = -1;
                if (COUNT) cnt = make_int4(0, 0, 0, 0);
                stack.sp = 0; stack.push(kDone);
                node = sc.tlas_root;
                if constexpr (ANY) {
                    // Hits at world distance >= kFloatMax are misses of the closest hit (the reference starts min_dist there), so
                    // L >= kFloatMax (inf: "any hit") asks the same as L = kFloatMax; the comparison keeps NaN, which retires below.
                    any_len = d4.w > kFloatMax ? kFloatMax : d4.w;
                    any_cb = rankSlack(sc, bo);                                  // the exit step's cb for this ray
                    if (any_len < kFloatMax) { g_dist = any_len; tmax = worldBound(any_len, sc.prune, any_cb); }   // a virtual winner at L
                    if (!(any_len > 0.0f)) node = stack.pop();                   // L <= 0 or NaN: nothing can be nearer; retire (kDone)
                }
            }
            work.advance(m_done);
        }
    }
    if (stamp && (threadIdx.x & 31) == 0) atomicMax(stamp + 1, globalTimerNs());
    if (COUNT) { warpTotalAdd(&st->count_nodes, tot_x); warpTotalAdd(&st->count_tris, tot_z); }   // never used for timing
}

void launchTraceBvhAny(const SceneDev& sc, const float4* O, const float4* D, float4* hit, FrameState* st, int n, int grid, cudaStream_t stream)
{
    k_trace_bvh<false, false, true><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, nullptr, nullptr, st, 0, n, nullptr);
}

void launchTraceBvh(const SceneDev& sc, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, bool count_totals,
                     FrameState* st, int round, int n_fixed, int grid, cudaStream_t stream, unsigned long long* stamp)
{
    if (counts || count_totals) k_trace_bvh<true, true><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, stamp);
    else if (uv) k_trace_bvh<true, false><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, stamp);
    else k_trace_bvh<false, false><<<grid, kTraceBlock, 0, stream>>>(sc, O, D, hit, uv, counts, st, round, n_fixed, stamp);
}

int traceBvhOccupancy()
{
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_trace_bvh<false, false>, kTraceBlock, 0);
    return nb;
}

}  // namespace ptap
