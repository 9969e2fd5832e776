// bvh_traverse.cuh - the steps that the kernels walking the two-level BVH share (k_trace_bvh in trace_bvh.cu; k_trace_emu and k_emu_full in
// trace_emu.cu): the encoding of a lane's state in its `node` register and the per-state vote, the reference's triangle predicate, the
// one-FMA-per-plane child test on node-local offsets, the split traversal stack, instance entry and the nearest-instance ranking at exit.
// Each kernel keeps its own loop, per-ray state and result records; see trace_bvh.cu for the design.
#pragma once
#include "kernels.cuh"

namespace ptap {
namespace bvh {

constexpr int kDone = (int)0x80000000u;        // ~0x7fffffff: bottom-of-stack sentinel
// A negative `node` is ~code with the lane's state in code >> 29:
//   0: triangle leaf (first << 3 | count - 1), 1: TLAS leaf = enter instance (code & kIndexMask), 2: marker = leave instance, 3: done
constexpr unsigned kEnterBit = 0x20000000u, kExitBit = 0x40000000u, kIndexMask = 0x1fffffffu;
constexpr int kMissKey = 0x7f800000;           // childKey of a missed child
constexpr float kModelTmin = -(kEpsilon + 1e-4f);   // traversal interval start inside an instance: the predicate accepts t >= -EPSILON

__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c)          // FFMA2 (sm_100): two binary32 FMAs per issue slot
{
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}

__device__ __forceinline__ uint4 ldg4u(const void* p)
{
    uint4 r;
    asm("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// Entry distance of a child as an order-preserving integer key (a missed child sorts last): interval test with relative slack on the
// entry / exit parameters of the six planes (near / far already selected by the ray's direction signs).
__device__ __forceinline__ int childKey(float nx, float ny, float nz, float fx, float fy, float fz, float tmin, float tmax)
{
    const float tn = fmaxf(fmaxf(fmaxf(nx, ny), nz), tmin);
    const float tf = fminf(fminf(fminf(fx, fy), fz), tmax);
    const bool h = tn <= tf + __fmaf_rn(fabsf(tf), 2e-6f, 1e-6f);
    return h ? __float_as_int(fmaxf(tn, 0.0f)) : kMissKey;
}

// direction-sign bits, taken from the SIGN BIT (not d < 0) so that they agree with safeInv for -0.0f: they decide which plane of a pair
// is the near one, and a near / far swap against the sign of the reciprocal would turn every box into a miss.
// Result: byte offsets (x | y << 8 | z << 16) of the near planes inside a node: lower planes at 32 / 64 / 96, upper planes 16 further.
__device__ __forceinline__ unsigned nearOffsets(const V3& d)
{
    const unsigned sx = __float_as_uint(d.x) >> 31, sy = __float_as_uint(d.y) >> 31, sz = __float_as_uint(d.z) >> 31;
    return (32u + (sx << 4)) | ((64u + (sy << 4)) << 8) | ((96u + (sz << 4)) << 16);
}

// traversal-only reciprocal: guarded against 0 (the exact predicate never uses it)
__device__ __forceinline__ float safeInv(float d)
{
    const float ooeps = 1e-30f;
    return __fdividef(1.0f, fabsf(d) > ooeps ? d : copysignf(ooeps, d));     // 1-ulp reciprocal: inside the slab test's 2e-6 slack
}

// TLAS pruning bound once some instance reported world distance g_dist: g_dist may be the approximation t * |d_w| / |W3 d_w| of the exact
// distance (off by at most g_dist * tie + cb, tie < prune - 1), so the bound carries the same absolute slack cb as the instance-entry bound
__device__ __forceinline__ float worldBound(float g_dist, float prune, float cb)
{
    return g_dist < kFloatMax ? g_dist * prune + cb + 1e-3f : 3.0e38f;
}

// The absolute slack of the exit step's ranking and of the pruning bounds for the stored ray origin bo
__device__ __forceinline__ float rankSlack(const SceneDev& sc, const V3& bo)
{
    return sc.c_pad + 1e-4f * (fabsf(bo.x) + fabsf(bo.y) + fabsf(bo.z));
}

// ---- the lane states and the per-state vote ---------------------------------------------------------------------------------------------
// One warp reduction over 6-bit counters, one per state.  `busy`: the lane holds a ray or may still fetch one; a retired lane with nothing
// left to fetch takes no part.  n_all == 0: every ray of the launch is retired.
struct LaneVote {
    unsigned code;                               // ~node: the index fields of the tri / enter / exit states
    bool tri, enter, exit, done, live;
    int n_tri, n_enter, n_exit, n_done, n_inner;
    unsigned n_all;
};
__device__ __forceinline__ LaneVote laneVote(int node, bool busy)
{
    LaneVote v;
    v.code = ~(unsigned)node;
    const unsigned state = min(v.code >> 29, 4u);           // 0 tri, 1 enter, 2 exit, 3 done, 4 inner
    v.live = state != 3u || busy;
    const unsigned sum = __reduce_add_sync(kFull, v.live ? 1u << (6u * state) : 0u);
    v.n_all = sum;
    v.n_tri = sum & 63u; v.n_enter = (sum >> 6) & 63u; v.n_exit = (sum >> 12) & 63u; v.n_done = (sum >> 18) & 63u; v.n_inner = (sum >> 24) & 63u;
    v.tri = state == 0u; v.enter = state == 1u; v.exit = state == 2u; v.done = state == 3u;
    return v;
}

// ---- the split traversal stack --------------------------------------------------------------------------------------------------------
// Entries 0 .. kSmemStack - 1 of every lane live in shared memory, laid out [entry][thread]: whatever entry each lane touches, lane l hits
// bank l, so a warp-wide push or pop is ONE L1 wavefront.  In local memory the same access costs one 32-byte sector per lane (the lanes'
// stack pointers differ), and the stack was 25 % of k_trace_bvh's L1 sector traffic - the unit that limits it (profiles/r02).  Deeper
// entries spill to local memory.  The kernel declares both arrays (kept out of this type, whose `sp` would otherwise live in local memory
// with the array: +40 bytes of stack frame and more spills in k_trace_bvh).
constexpr int kSmemStack = 12;
struct SplitStack {
    int* smem;                                   // the kernel's __shared__ int[kSmemStack * kTraceBlock]
    int* local;                                  // the kernel's int[kBvhStack - kSmemStack]
    int sp;
    __device__ __forceinline__ SplitStack(int* s, int* l) : smem(s), local(l), sp(0) {}
    __device__ __forceinline__ void push(int v) { if (sp < kSmemStack) smem[sp * kTraceBlock + threadIdx.x] = v; else local[sp - kSmemStack] = v; ++sp; }
    __device__ __forceinline__ int pop() { --sp; return sp < kSmemStack ? smem[sp * kTraceBlock + threadIdx.x] : local[sp - kSmemStack]; }
    // after the node step: push the other hit children farthest first, return the next node (the nearest hit child, or the popped entry)
    __device__ __forceinline__ int descend(const int key[4], const int lnk[4])
    {
        if (key[3] != kMissKey) push(lnk[3]);
        if (key[2] != kMissKey) push(lnk[2]);
        if (key[1] != kMissKey) push(lnk[1]);
        return key[0] != kMissKey ? lnk[0] : pop();
    }
};

// ---- the node step --------------------------------------------------------------------------------------------------------------------
// The four children of an inner node, tested against the ray interval [tmin, tmax]: key[c] = order-preserving integer key of child c's
// entry distance (kMissKey: missed), lnk[c] its link; SORT: sorted by entry distance, else in node order.  One FMA per plane on node-local
// offsets (two children per FFMA2), near / far planes picked by address from the direction's sign bits (near_off: nearOffsets()).
template <bool SORT>
__device__ __forceinline__ void nodeChildren(const char* __restrict__ np, const V3& ro, const V3& rinv, unsigned near_off, float tmin, float tmax, int key[4], int lnk[4])
{
    const F8 hd = ldg8(np);                                           // origin, four links
    const unsigned nox = near_off & 0xffu, noy = (near_off >> 8) & 0xffu, noz = near_off >> 16;
    const uint4 NX = ldg4u(np + nox), FX = ldg4u(np + (nox ^ 16u));   // near / far planes by address
    const uint4 NY = ldg4u(np + noy), FY = ldg4u(np + (noy ^ 16u));
    const uint4 NZ = ldg4u(np + noz), FZ = ldg4u(np + (noz ^ 16u));
    const float cx = (hd.v[0] - ro.x) * rinv.x, cy = (hd.v[1] - ro.y) * rinv.y, cz = (hd.v[2] - ro.z) * rinv.z;
    const float2 ix = make_float2(rinv.x, rinv.x), iy = make_float2(rinv.y, rinv.y), iz = make_float2(rinv.z, rinv.z);
    const float2 ccx = make_float2(cx, cx), ccy = make_float2(cy, cy), ccz = make_float2(cz, cz);
    const float2 nxa = fma2(make_float2(__uint_as_float(NX.x), __uint_as_float(NX.y)), ix, ccx), nxb = fma2(make_float2(__uint_as_float(NX.z), __uint_as_float(NX.w)), ix, ccx);
    const float2 nya = fma2(make_float2(__uint_as_float(NY.x), __uint_as_float(NY.y)), iy, ccy), nyb = fma2(make_float2(__uint_as_float(NY.z), __uint_as_float(NY.w)), iy, ccy);
    const float2 nza = fma2(make_float2(__uint_as_float(NZ.x), __uint_as_float(NZ.y)), iz, ccz), nzb = fma2(make_float2(__uint_as_float(NZ.z), __uint_as_float(NZ.w)), iz, ccz);
    const float2 fxa = fma2(make_float2(__uint_as_float(FX.x), __uint_as_float(FX.y)), ix, ccx), fxb = fma2(make_float2(__uint_as_float(FX.z), __uint_as_float(FX.w)), ix, ccx);
    const float2 fya = fma2(make_float2(__uint_as_float(FY.x), __uint_as_float(FY.y)), iy, ccy), fyb = fma2(make_float2(__uint_as_float(FY.z), __uint_as_float(FY.w)), iy, ccy);
    const float2 fza = fma2(make_float2(__uint_as_float(FZ.x), __uint_as_float(FZ.y)), iz, ccz), fzb = fma2(make_float2(__uint_as_float(FZ.z), __uint_as_float(FZ.w)), iz, ccz);
    key[0] = childKey(nxa.x, nya.x, nza.x, fxa.x, fya.x, fza.x, tmin, tmax);
    key[1] = childKey(nxa.y, nya.y, nza.y, fxa.y, fya.y, fza.y, tmin, tmax);
    key[2] = childKey(nxb.x, nyb.x, nzb.x, fxb.x, fyb.x, fzb.x, tmin, tmax);
    key[3] = childKey(nxb.y, nyb.y, nzb.y, fxb.y, fyb.y, fzb.y, tmin, tmax);
#pragma unroll
    for (int c = 0; c < 4; ++c) lnk[c] = __float_as_int(hd.v[4 + c]);
    if (SORT) {
#define PTAP_CSWAP(a, b) { const bool sw = key[b] < key[a]; const int ka = sw ? key[b] : key[a], kb = sw ? key[a] : key[b]; \
                           const int la = sw ? lnk[b] : lnk[a], lb = sw ? lnk[a] : lnk[b]; key[a] = ka; key[b] = kb; lnk[a] = la; lnk[b] = lb; }
        PTAP_CSWAP(0, 1) PTAP_CSWAP(2, 3) PTAP_CSWAP(0, 2) PTAP_CSWAP(1, 3) PTAP_CSWAP(1, 2)
#undef PTAP_CSWAP
    }
}

// ---- the triangle step ----------------------------------------------------------------------------------------------------------------
// The reference's tolerant Moller-Trumbore predicate (Renderer.cpp:174-201) on leaf-order triangle k (64 B: v0, v0v1, v0v2, global id).
// Straight-line evaluation: the reference's early returns have no side effects, so testing all of its rejection conditions at the end
// gives the same verdict, and the handful of lanes in a triangle step do not diverge further.  Every operation is the un-contracted one.
struct TriTest {
    bool reject;
    float u, v, t;
    int id;                                      // global triangle id
};
__device__ __forceinline__ TriTest leafTriangle(const SceneDev& sc, int k, const V3& o, const V3& d)
{
    const F8 ta = ldg8(&sc.bvh_tris[k]), tb = ldg8(reinterpret_cast<const char*>(&sc.bvh_tris[k]) + 32);
    const V3 v0 = v3(ta.v[0], ta.v[1], ta.v[2]), v0v1 = v3(ta.v[3], ta.v[4], ta.v[5]), v0v2 = v3(ta.v[6], ta.v[7], tb.v[0]);
    TriTest h;
    const V3 pvec = xcross(d, v0v2);
    const float det = xdot(v0v1, pvec);
    const float invDet = xdiv(1.0f, det);
    const V3 tvec = xsub(o, v0);
    h.u = xmul(xdot(tvec, pvec), invDet);
    const V3 qvec = xcross(tvec, v0v1);
    h.v = xmul(xdot(d, qvec), invDet);
    h.t = xmul(xdot(v0v2, qvec), invDet);
    h.reject = (xabs(xsub(det, 0.0f)) < kEpsilon) | (h.u < (0.0f - kEpsilon)) | (h.u > (1.0f + kEpsilon)) |
               (h.v < (0.0f - kEpsilon)) | (xadd(h.u, h.v) > (1.0f + kEpsilon)) | (h.t < (0.0f - kEpsilon));
    h.id = __float_as_int(tb.v[1]);
    return h;
}

// Barycentrics of triangle `tri` for the stored ray (bo, bd) in model `im`, as the predicate computes them (Renderer.cpp:174-201)
__device__ __forceinline__ float2 hitBarycentrics(const SceneDev& sc, int im, const V3& bo, const V3& bd, int tri)
{
    const InstanceTrace* __restrict__ inst = &sc.inst[im];
    const float4 w0 = ldg4(&inst->w2m[0]), w1 = ldg4(&inst->w2m[1]), w2 = ldg4(&inst->w2m[2]);
    const V3 ro = xmat4(w0, w1, w2, bo, 1.0f), rd = xnormalize(xmat4(w0, w1, w2, bd, 0.0f));
    const float4 a = ldg4(&sc.tris[tri].v0), b = ldg4(&sc.tris[tri].e1), c = ldg4(&sc.tris[tri].e2);
    const V3 pvec = xcross(rd, v3(c));
    const float invDet = xdiv(1.0f, xdot(v3(b), pvec));
    const V3 tvec = xsub(ro, v3(a));
    return make_float2(xmul(xdot(tvec, pvec), invDet), xmul(xdot(rd, xcross(tvec, v3(b))), invDet));
}

// ---- instance entry and exit ----------------------------------------------------------------------------------------------------------
// Enter instance `inst` with the stored ray (bo, bd) (Renderer.cpp:381-382): the model-space ray (ro, rd) exactly as the reference sets it
// up, with the traversal's reciprocal and near-plane offsets.  Returns |W3 d_w| / |d_w|, model-space t per unit of world distance.
__device__ __forceinline__ float enterInstance(const InstanceTrace* __restrict__ inst, const V3& bo, const V3& bd, V3& ro, V3& rd, V3& rinv, unsigned& near_off)
{
    const float4 w0 = ldg4(&inst->w2m[0]), w1 = ldg4(&inst->w2m[1]), w2 = ldg4(&inst->w2m[2]);
    ro = xmat4(w0, w1, w2, bo, 1.0f);                                   // Renderer.cpp:381
    const V3 dm = xmat4(w0, w1, w2, bd, 0.0f);
    const float mlen = xsqrt(xdot(dm, dm));
    rd = xscale(dm, xdiv(1.0f, mlen));                                  // glm::normalize, Renderer.cpp:382
    rinv = v3(safeInv(rd.x), safeInv(rd.y), safeInv(rd.z));
    near_off = nearOffsets(rd);
    const float wil = rsqrtf(bd.x * bd.x + bd.y * bd.y + bd.z * bd.z);
    return mlen * wil;
}

// Leaving instance `im` whose winner is at model-space t (ascale: world distance per unit of t, the reciprocal of enterInstance's result):
// the nearest-model decision of the reference (Renderer.cpp:388-398) against the nearest model so far (g_model at g_t, world distance
// g_dist), true when `im` becomes the nearest.  The reference compares exact world distances; here the instance's winner is ranked by
// t * ascale (its world distance up to `tie`), and the exact distances are evaluated only when two candidates are closer than that slack,
// or when pruning is off.  g_dist receives the new winner's distance, or the exact distance of the old one when that was evaluated.
// ANY: g_dist starts at the segment length L as a virtual winner (g_model < 0), which a candidate must be nearer than to be taken.
template <bool ANY>
__device__ __forceinline__ bool takeInstance(const SceneDev& sc, const V3& bo, const V3& bd, float cb, int im, float t, float ascale,
                                             int g_model, float g_t, float& g_dist)
{
    // |t|: the reference ranks instances by length(hit - origin) >= 0 (Renderer.cpp:391-393), and the predicate accepts t down to
    // -EPSILON, which is up to EPSILON * (world units per model unit) behind the origin
    const float a = fabsf(t * ascale);
    const float a_lo = a - (fabsf(a) * sc.tie + cb), a_hi = a + (fabsf(a) * sc.tie + cb);
    const float g_lo = g_dist - (g_dist * sc.tie + cb), g_hi = g_dist + (g_dist * sc.tie + cb);
    bool take;
    float nd = a;
    if (a_hi < g_lo && a_hi < 0.99f * kFloatMax) take = true;        // clearly nearer than the current winner (or the first one)
    else if ((ANY || g_model >= 0) && a_lo > g_hi) take = false;     // clearly farther (ANY: than L as well, so L keeps bounding)
    else {                                                           // near-tie, or no usable bound: the reference's comparison
        const float dn = exactHitDistance(sc, bo, bd, im, t);
        // ANY: a candidate must be nearer than the virtual winner at L (at kFloatMax when L is not below it) to be taken
        const float dg = g_model >= 0 ? exactHitDistance(sc, bo, bd, g_model, g_t) : ANY ? g_dist : kFloatMax;
        take = dg > dn || (dg == dn && g_model >= 0 && im < g_model);   // Renderer.cpp:393 in model order
        nd = dn;
        if (!take && g_model >= 0) g_dist = dg;
    }
    if (take) g_dist = nd;
    return take;
}

}  // namespace bvh
}  // namespace ptap
