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

namespace {

#ifndef PTAP_TRACE_MIN_CTAS
#define PTAP_TRACE_MIN_CTAS 8     // 64 registers: 8 CTAs of 128 threads per SM, as round 1's kernel
#endif
#ifndef PTAP_NODE_LDG256
#define PTAP_NODE_LDG256 0
#endif
#ifndef PTAP_COLD_SMEM
#define PTAP_COLD_SMEM 0
#endif
#ifndef PTAP_SMEM_STACK
#define PTAP_SMEM_STACK 12
#endif
constexpr int kSmemStack = PTAP_SMEM_STACK;   // stack entries per ray kept in shared memory (0: all in local memory)
#ifndef PTAP_NODE_STEPS
#define PTAP_NODE_STEPS 1
#endif
constexpr int kNodeSteps = PTAP_NODE_STEPS;    // inner nodes a lane may take per scheduling round

// Renderer.cpp:174-215; tie rule of brute force in index order: strictly nearer, or equal t and lower global id.
// `tmax` is the model-space bound of the traversal AND the best t so far (they are the same number once best_tri >= 0).
template <bool UV, bool COUNT>
__device__ __forceinline__ void leafTriangle(const SceneDev& sc, const V3& o, const V3& d, float& tmax, int& best_tri, float& best_u, float& best_v,
                                             int k, int4& cnt)
{
    const F8 ta = ldg8(&sc.bvh_tris[k]), tb = ldg8(reinterpret_cast<const char*>(&sc.bvh_tris[k]) + 32);
    if (COUNT) cnt.z++;
    // Straight-line evaluation: the reference's early returns (Renderer.cpp:188-201) have no side effects, so testing all of its
    // rejection conditions at the end gives the same verdict, and the handful of lanes in a triangle step do not diverge further.
    const V3 v0 = v3(ta.v[0], ta.v[1], ta.v[2]), v0v1 = v3(ta.v[3], ta.v[4], ta.v[5]), v0v2 = v3(ta.v[6], ta.v[7], tb.v[0]);
    const V3 pvec = xcross(d, v0v2);
    const float det = xdot(v0v1, pvec);
    const float invDet = xdiv(1.0f, det);
    const V3 tvec = xsub(o, v0);
    const float u = xmul(xdot(tvec, pvec), invDet);
    const V3 qvec = xcross(tvec, v0v1);
    const float v = xmul(xdot(d, qvec), invDet);
    const float t = xmul(xdot(v0v2, qvec), invDet);
    const bool reject = (xabs(xsub(det, 0.0f)) < kEpsilon) | (u < (0.0f - kEpsilon)) | (u > (1.0f + kEpsilon)) |
                        (v < (0.0f - kEpsilon)) | (xadd(u, v) > (1.0f + kEpsilon)) | (t < (0.0f - kEpsilon)) | (t > tmax);
    if (reject || !(t <= tmax)) return;                        // the second test only catches NaN (a degenerate det passes none of the above as true)
    const int id = __float_as_int(tb.v[1]);
    if (t < tmax || (best_tri >= 0 && id < best_tri)) { tmax = t; best_tri = id; if (UV) { best_u = u; best_v = v; } }
}

}  // namespace

template <bool UV, bool COUNT, bool ANY = false>
__global__ void __launch_bounds__(kTraceBlock, PTAP_TRACE_MIN_CTAS)
k_trace_bvh(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, float4* __restrict__ hit,
            float2* __restrict__ uv, int4* __restrict__ counts, FrameState* st, int round, int n_fixed, unsigned long long* __restrict__ stamp)
{
    const int n = n_fixed >= 0 ? n_fixed : st->n_active[round];
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_fixed < 0) st->rays_traced += (unsigned long long)n;
    if (stamp && threadIdx.x == 0) atomicMin(stamp, globalTimerNs());
    unsigned int* cursor = &st->fetch[round];
    const int lane = threadIdx.x & 31;
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

    int sp = 0;
    // Traversal stack.  Entries 0 .. kSmemStack - 1 of every lane live in shared memory, laid out [entry][thread]: whatever entry each lane
    // touches, lane l hits bank l, so a warp-wide push or pop is ONE L1 wavefront.  In local memory the same access costs one 32-byte
    // sector per lane (the lanes' stack pointers differ), and the stack was 25 % of the kernel's L1 sector traffic - the unit that
    // limits it (profiles/r02).  Deeper entries spill to local memory.
    __shared__ int s_stack[kSmemStack > 0 ? kSmemStack * kTraceBlock : 1];
    int l_stack[kBvhStack > kSmemStack ? kBvhStack - kSmemStack : 1];
    auto push = [&](int v) {
        if (kSmemStack > 0 && sp < kSmemStack) s_stack[sp * kTraceBlock + threadIdx.x] = v; else l_stack[sp - kSmemStack] = v;
        ++sp;
    };
    auto pop = [&]() {
        --sp;
        return (kSmemStack > 0 && sp < kSmemStack) ? s_stack[sp * kTraceBlock + threadIdx.x] : l_stack[sp - kSmemStack];
    };
    int node = kDone, i = -1;
    // What only the instance enter / exit and the retire / refill steps touch - the ray as stored (bo, bd: Ray::base, Primitive.h:160-164),
    // the reciprocal of its normalised direction and its near-plane offsets (TLAS level), the nearest model so far (g_*) - lives in
    // shared memory, [word][thread] like the stack, when PTAP_COLD_SMEM is set: 16 registers fewer are live across the node and triangle
    // steps, so that more warps fit an SM (the kernel waits on dependent node loads; `profiles/r02`).
#if PTAP_COLD_SMEM
    __shared__ float s_cold[16 * kTraceBlock];
    float* const cold = s_cold + threadIdx.x;
#define CF(k) cold[(k) * kTraceBlock]
#else
    float cold_regs[16];
#define CF(k) cold_regs[k]
#endif
#define C_BO v3(CF(0), CF(1), CF(2))
#define C_BD v3(CF(3), CF(4), CF(5))
#define C_WINV v3(CF(6), CF(7), CF(8))
#define C_WNEAR CF(9)
#define g_dist CF(10)
#define g_t CF(11)
#define g_model_f CF(12)
#define g_tri_f CF(13)
#define g_u CF(14)
#define g_v CF(15)
    unsigned near_off = 0u;                         // byte offsets of the near planes inside a node for the current level
    V3 ro = v3(0, 0, 0), rd = v3(0, 0, 1), rinv = v3(0, 0, 0);   // the ray of the current level: world, or model space of the entered instance
    float tmin = 0.0f, tmax = 0.0f;
    int best_tri = -1; float best_u = 0.0f, best_v = 0.0f;
    int w_next = 0, w_end = 0;
    bool exhausted = false;
    const int vote_tri = sc.vote_tri, vote_inst = sc.vote_inst, vote_refill = sc.vote_refill;
    // ANY only: the segment length L, the absolute slack cb of the exit step for this ray, world units per model-space t of the entered instance
    float any_len = 0.0f, any_cb = 0.0f, any_scale = 0.0f;

    for (;;) {
        // ---- (1) inner nodes (TLAS and BLAS share the 4-wide format): test the four child boxes, continue with the nearest hit child,
        // push the other hit children farthest first
#pragma unroll
        for (int rep = 0; rep < kNodeSteps; ++rep) {
            if (node >= 0) {
                const char* __restrict__ np = reinterpret_cast<const char*>(&sc.nodes[node]);
                const F8 hd = ldg8(np);                                           // origin, four links
#if PTAP_NODE_LDG256
                // variant: the whole node in four 32-byte loads, near / far planes picked per child and axis by min / max
                const F8 px8 = ldg8(np + 32), py8 = ldg8(np + 64), pz8 = ldg8(np + 96);
                if (COUNT) cnt.x++;
                const float cx = (hd.v[0] - ro.x) * rinv.x, cy = (hd.v[1] - ro.y) * rinv.y, cz = (hd.v[2] - ro.z) * rinv.z;
                const float2 ix = make_float2(rinv.x, rinv.x), iy = make_float2(rinv.y, rinv.y), iz = make_float2(rinv.z, rinv.z);
                const float2 ccx = make_float2(cx, cx), ccy = make_float2(cy, cy), ccz = make_float2(cz, cz);
                const float2 lxa = fma2(make_float2(px8.v[0], px8.v[1]), ix, ccx), lxb = fma2(make_float2(px8.v[2], px8.v[3]), ix, ccx), hxa = fma2(make_float2(px8.v[4], px8.v[5]), ix, ccx), hxb = fma2(make_float2(px8.v[6], px8.v[7]), ix, ccx);
                const float2 lya = fma2(make_float2(py8.v[0], py8.v[1]), iy, ccy), lyb = fma2(make_float2(py8.v[2], py8.v[3]), iy, ccy), hya = fma2(make_float2(py8.v[4], py8.v[5]), iy, ccy), hyb = fma2(make_float2(py8.v[6], py8.v[7]), iy, ccy);
                const float2 lza = fma2(make_float2(pz8.v[0], pz8.v[1]), iz, ccz), lzb = fma2(make_float2(pz8.v[2], pz8.v[3]), iz, ccz), hza = fma2(make_float2(pz8.v[4], pz8.v[5]), iz, ccz), hzb = fma2(make_float2(pz8.v[6], pz8.v[7]), iz, ccz);
#define PTAP_MM(l, h, c) fminf(l.c, h.c), fmaxf(l.c, h.c)
                const float2 nxa = make_float2(fminf(lxa.x, hxa.x), fminf(lxa.y, hxa.y)), fxa = make_float2(fmaxf(lxa.x, hxa.x), fmaxf(lxa.y, hxa.y));
                const float2 nxb = make_float2(fminf(lxb.x, hxb.x), fminf(lxb.y, hxb.y)), fxb = make_float2(fmaxf(lxb.x, hxb.x), fmaxf(lxb.y, hxb.y));
                const float2 nya = make_float2(fminf(lya.x, hya.x), fminf(lya.y, hya.y)), fya = make_float2(fmaxf(lya.x, hya.x), fmaxf(lya.y, hya.y));
                const float2 nyb = make_float2(fminf(lyb.x, hyb.x), fminf(lyb.y, hyb.y)), fyb = make_float2(fmaxf(lyb.x, hyb.x), fmaxf(lyb.y, hyb.y));
                const float2 nza = make_float2(fminf(lza.x, hza.x), fminf(lza.y, hza.y)), fza = make_float2(fmaxf(lza.x, hza.x), fmaxf(lza.y, hza.y));
                const float2 nzb = make_float2(fminf(lzb.x, hzb.x), fminf(lzb.y, hzb.y)), fzb = make_float2(fmaxf(lzb.x, hzb.x), fmaxf(lzb.y, hzb.y));
#undef PTAP_MM
#else
                const unsigned nox = near_off & 0xffu, noy = (near_off >> 8) & 0xffu, noz = near_off >> 16;
                const uint4 NX = ldg4u(np + nox), FX = ldg4u(np + (nox ^ 16u));   // near / far planes by address
                const uint4 NY = ldg4u(np + noy), FY = ldg4u(np + (noy ^ 16u));
                const uint4 NZ = ldg4u(np + noz), FZ = ldg4u(np + (noz ^ 16u));
                if (COUNT) cnt.x++;
                const float cx = (hd.v[0] - ro.x) * rinv.x, cy = (hd.v[1] - ro.y) * rinv.y, cz = (hd.v[2] - ro.z) * rinv.z;
                const float2 ix = make_float2(rinv.x, rinv.x), iy = make_float2(rinv.y, rinv.y), iz = make_float2(rinv.z, rinv.z);
                const float2 ccx = make_float2(cx, cx), ccy = make_float2(cy, cy), ccz = make_float2(cz, cz);
                const float2 nxa = fma2(make_float2(__uint_as_float(NX.x), __uint_as_float(NX.y)), ix, ccx), nxb = fma2(make_float2(__uint_as_float(NX.z), __uint_as_float(NX.w)), ix, ccx);
                const float2 nya = fma2(make_float2(__uint_as_float(NY.x), __uint_as_float(NY.y)), iy, ccy), nyb = fma2(make_float2(__uint_as_float(NY.z), __uint_as_float(NY.w)), iy, ccy);
                const float2 nza = fma2(make_float2(__uint_as_float(NZ.x), __uint_as_float(NZ.y)), iz, ccz), nzb = fma2(make_float2(__uint_as_float(NZ.z), __uint_as_float(NZ.w)), iz, ccz);
                const float2 fxa = fma2(make_float2(__uint_as_float(FX.x), __uint_as_float(FX.y)), ix, ccx), fxb = fma2(make_float2(__uint_as_float(FX.z), __uint_as_float(FX.w)), ix, ccx);
                const float2 fya = fma2(make_float2(__uint_as_float(FY.x), __uint_as_float(FY.y)), iy, ccy), fyb = fma2(make_float2(__uint_as_float(FY.z), __uint_as_float(FY.w)), iy, ccy);
                const float2 fza = fma2(make_float2(__uint_as_float(FZ.x), __uint_as_float(FZ.y)), iz, ccz), fzb = fma2(make_float2(__uint_as_float(FZ.z), __uint_as_float(FZ.w)), iz, ccz);
#endif
                int key[4], lnk[4];
                key[0] = childKey(nxa.x, nya.x, nza.x, fxa.x, fya.x, fza.x, tmin, tmax);
                key[1] = childKey(nxa.y, nya.y, nza.y, fxa.y, fya.y, fza.y, tmin, tmax);
                key[2] = childKey(nxb.x, nyb.x, nzb.x, fxb.x, fyb.x, fzb.x, tmin, tmax);
                key[3] = childKey(nxb.y, nyb.y, nzb.y, fxb.y, fyb.y, fzb.y, tmin, tmax);
#pragma unroll
                for (int c = 0; c < 4; ++c) lnk[c] = __float_as_int(hd.v[4 + c]);
                if (!ANY) {     // an any-hit traversal takes the hit children in node order: 3 % faster than nearest first (DESIGN 4.8)
#define PTAP_CSWAP(a, b) { const bool sw = key[b] < key[a]; const int ka = sw ? key[b] : key[a], kb = sw ? key[a] : key[b]; \
                           const int la = sw ? lnk[b] : lnk[a], lb = sw ? lnk[a] : lnk[b]; key[a] = ka; key[b] = kb; lnk[a] = la; lnk[b] = lb; }
                    PTAP_CSWAP(0, 1) PTAP_CSWAP(2, 3) PTAP_CSWAP(0, 2) PTAP_CSWAP(1, 3) PTAP_CSWAP(1, 2)
#undef PTAP_CSWAP
                }
                if (key[3] != 0x7f800000) push(lnk[3]);
                if (key[2] != 0x7f800000) push(lnk[2]);
                if (key[1] != 0x7f800000) push(lnk[1]);
                if (key[0] != 0x7f800000) node = lnk[0]; else node = pop();
            }
        }
        // ---- (2) who waits for what: one warp reduction over 6-bit counters, one per state
        const unsigned code = ~(unsigned)node;
        const unsigned state = min(code >> 29, 4u);             // 0 tri, 1 enter, 2 exit, 3 done, 4 inner
        const bool live = state != 3u || i >= 0 || !exhausted;  // a retired lane with nothing left to fetch takes no part
        const unsigned sum = __reduce_add_sync(kFull, live ? 1u << (6u * state) : 0u);
        if (sum == 0u) break;                                   // every ray of the launch is retired
        const int n_tri = sum & 63u, n_enter = (sum >> 6) & 63u, n_exit = (sum >> 12) & 63u, n_done = (sum >> 18) & 63u, n_inner = (sum >> 24) & 63u;
        const bool s_tri = state == 0u, s_enter = state == 1u, s_exit = state == 2u, s_done = state == 3u;

        // ---- (3a) one triangle of the held leaf (Renderer.cpp:174-215)
        if (s_tri && n_tri >= min(vote_tri, n_inner)) {
            leafTriangle<UV, COUNT>(sc, ro, rd, tmax, best_tri, best_u, best_v, (int)(code >> 3), cnt);
            if constexpr (ANY) {
                // The model's true winner has t in [-EPSILON, tmax] (the best accepted t so far), so its world distance is at most
                // m = max(|tmax|, EPSILON) * ascale up to the exit step's slack m * tie + cb: when that is below L (at most kFloatMax), so
                // is the closest hit.
                bool occluded = false;
                if (best_tri >= 0) {
                    const float m = fmaxf(fabsf(tmax), kEpsilon) * any_scale;
                    occluded = m + (m * sc.tie + any_cb) < any_len;
                }
                if (occluded) { sp = 0; node = kDone; g_model_f = __int_as_float(kAnyOccluded); }     // retire: empty stack, done state
                else if (code & 7u) node = (int)~(code + 7u); else node = pop();
            } else {
                if (code & 7u) node = (int)~(code + 7u); else node = pop();   // (first + 1, count - 1), or pop when the leaf is finished
            }
        }
        // ---- (3b) TLAS leaf: enter instance `im` (Renderer.cpp:381-384)
        if (s_enter && n_enter >= min(vote_inst, n_inner)) {
            const int im = (int)(code & kIndexMask);
            const InstanceTrace* __restrict__ inst = &sc.inst[im];
            const float4 w0 = ldg4(&inst->w2m[0]), w1 = ldg4(&inst->w2m[1]), w2 = ldg4(&inst->w2m[2]);
            const V3 bo = C_BO, bd = C_BD;
            ro = xmat4(w0, w1, w2, bo, 1.0f);                                   // Renderer.cpp:381
            const V3 dm = xmat4(w0, w1, w2, bd, 0.0f);
            const float mlen = xsqrt(xdot(dm, dm));
            rd = xscale(dm, xdiv(1.0f, mlen));                                  // glm::normalize, Renderer.cpp:382
            rinv = v3(safeInv(rd.x), safeInv(rd.y), safeInv(rd.z));
            near_off = nearOffsets(rd);
            const float wil = rsqrtf(bd.x * bd.x + bd.y * bd.y + bd.z * bd.z);
            tmin = -(kEpsilon + 1e-4f);                                         // the predicate accepts t >= -EPSILON
            tmax = kFloatMax; best_tri = -1;                                    // Renderer.cpp:384
            if (g_dist < kFloatMax) {
                // World distance of a model-space t along this ray is t * |d_w| / |W3 d_w| when model_to_world inverts world_to_model
                // (checked at upload, else sc.prune = inf): a winner needs t <= g * |W3 d_w| / |d_w|, plus slack for the matrices' residual.
                const float tb = (g_dist * sc.prune + sc.c_pad + 1e-4f * (fabsf(bo.x) + fabsf(bo.y) + fabsf(bo.z))) * (mlen * wil) * 1.0001f;
                if (tb < kFloatMax) tmax = tb;                                  // false for NaN / inf: no bound
            }
            if constexpr (ANY) any_scale = __fdividef(1.0f, mlen * wil);      // the triangle step's copy of what is pushed next
            push(__float_as_int(__fdividef(1.0f, mlen * wil)));                  // world distance per unit of model-space t, for the exit step
            push((int)~(kExitBit | (unsigned)im));
            node = __float_as_int(__ldg(&inst->grid.z));                        // BLAS root of the instance's mesh
        }
        // ---- (3c) marker popped: leave instance `im` (Renderer.cpp:388-398).  The nearest-model decision of the reference compares exact
        // world distances; here the instance's winner is ranked by t * |d_w| / |W3 d_w| (its world distance up to `tie`), and the
        // exact distances are evaluated only when two candidates are closer than that slack, or when pruning is off.
        if (s_exit && n_exit >= min(vote_inst, n_inner)) {
            const int im = (int)(code & kIndexMask);
            const float ascale = __int_as_float(pop());                          // pushed under the marker at entry
            const V3 bo = C_BO, bd = C_BD;
            const int g_model = __float_as_int(g_model_f);
            const float cb = sc.c_pad + 1e-4f * (fabsf(bo.x) + fabsf(bo.y) + fabsf(bo.z));
            if (best_tri >= 0) {
                // |t|: the reference ranks instances by length(hit - origin) >= 0 (Renderer.cpp:391-393), and the predicate accepts
                // t down to -EPSILON, which is up to EPSILON * (world units per model unit) behind the origin
                const float a = fabsf(tmax * ascale);
                const float a_lo = a - (fabsf(a) * sc.tie + cb), a_hi = a + (fabsf(a) * sc.tie + cb);
                const float g_lo = g_dist - (g_dist * sc.tie + cb), g_hi = g_dist + (g_dist * sc.tie + cb);
                bool take;
                float nd = a;
                if (a_hi < g_lo && a_hi < 0.99f * kFloatMax) take = true;        // clearly nearer than the current winner (or the first one)
                else if ((ANY || g_model >= 0) && a_lo > g_hi) take = false;     // clearly farther (ANY: than L as well, so L keeps bounding)
                else {                                                           // near-tie, or no usable bound: the reference's comparison
                    const float dn = exactHitDistance(sc, bo, bd, im, tmax);
                    // ANY: a candidate must be nearer than the virtual winner at L (at kFloatMax when L is not below it) to be taken
                    const float dg = g_model >= 0 ? exactHitDistance(sc, bo, bd, g_model, g_t) : ANY ? g_dist : kFloatMax;
                    take = dg > dn || (dg == dn && g_model >= 0 && im < g_model);   // Renderer.cpp:393 in model order
                    nd = dn;
                    if (!take && g_model >= 0) g_dist = dg;
                }
                if (take) {
                    g_dist = nd; g_model_f = __int_as_float(im); g_tri_f = __int_as_float(best_tri); g_t = tmax;
                    if (UV) { g_u = best_u; g_v = best_v; }
                }
            }
            ro = bo; rinv = C_WINV; near_off = __float_as_uint(C_WNEAR);
            tmin = sc.tmin_world; tmax = worldBound(g_dist, sc.prune, cb);
            node = pop();
        }
        // ---- (3d) retire finished rays, refill the lanes from the warp's batch
        if (n_done > 0 && n_done >= min(vote_refill, n_inner)) {
            const unsigned m_done = __ballot_sync(kFull, s_done && live);
            if (s_done && i >= 0) {
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
            if (w_next >= w_end && !exhausted) {      // the warp's batch is used up: take the next one
                unsigned b = 0;
                if (lane == 0) b = atomicAdd(cursor, (unsigned)sc.batch);
                b = __shfl_sync(kFull, b, 0);
                if (b >= (unsigned)n) { exhausted = true; w_next = w_end = n; }
                else { w_next = (int)b; w_end = min((int)b + sc.batch, n); }
            }
            const int avail = w_end - w_next;
            const int rank = __popc(m_done & ((1u << lane) - 1u));
            if (s_done && live && rank < avail) {
                i = w_next + rank;
                const float4 o4 = O[i], d4 = D[i];
                const V3 bo = v3(o4), bd = v3(d4);
                const float il = rsqrtf(bd.x * bd.x + bd.y * bd.y + bd.z * bd.z);
                const V3 winv = v3(safeInv(bd.x * il), safeInv(bd.y * il), safeInv(bd.z * il));
                const unsigned wnear_off = nearOffsets(bd);          // the normalisation keeps the sign bits
                CF(0) = bo.x; CF(1) = bo.y; CF(2) = bo.z; CF(3) = bd.x; CF(4) = bd.y; CF(5) = bd.z;
                CF(6) = winv.x; CF(7) = winv.y; CF(8) = winv.z; C_WNEAR = __uint_as_float(wnear_off);
                ro = bo; rinv = winv; near_off = wnear_off;
                tmin = sc.tmin_world; tmax = 3.0e38f;
                g_dist = kFloatMax; g_model_f = __int_as_float(-1); g_tri_f = __int_as_float(-1); g_t = 0.0f; g_u = 0.0f; g_v = 0.0f;
                best_tri = -1;
                if (COUNT) cnt = make_int4(0, 0, 0, 0);
                sp = 0; push(kDone);
                node = sc.tlas_root;
                if constexpr (ANY) {
                    // Hits at world distance >= kFloatMax are misses of the closest hit (the reference starts min_dist there), so
                    // L >= kFloatMax (inf: "any hit") asks the same as L = kFloatMax; the comparison keeps NaN, which retires below.
                    any_len = d4.w > kFloatMax ? kFloatMax : d4.w;
                    any_cb = sc.c_pad + 1e-4f * (fabsf(bo.x) + fabsf(bo.y) + fabsf(bo.z));    // the exit step's cb for this ray
                    if (any_len < kFloatMax) { g_dist = any_len; tmax = worldBound(any_len, sc.prune, any_cb); }   // a virtual winner at L
                    if (!(any_len > 0.0f)) node = pop();                         // L <= 0 or NaN: nothing can be nearer; retire (kDone)
                }
            }
            w_next += min(__popc(m_done), avail);
        }
    }
    if (stamp && (threadIdx.x & 31) == 0) atomicMax(stamp + 1, globalTimerNs());
    if (COUNT) {        // counting build: per-warp totals into the frame state (never used for timing)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { tot_x += __shfl_xor_sync(kFull, tot_x, d); tot_z += __shfl_xor_sync(kFull, tot_z, d); }
        if (lane == 0) { atomicAdd(&st->count_nodes, tot_x); atomicAdd(&st->count_tris, tot_z); }
    }
}

#undef CF
#undef C_BO
#undef C_BD
#undef C_WINV
#undef C_WNEAR
#undef g_dist
#undef g_t
#undef g_model_f
#undef g_tri_f
#undef g_u
#undef g_v

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
