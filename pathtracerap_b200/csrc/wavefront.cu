// wavefront.cu - ray generation, shading + stable compaction + film accumulation, hit resolve.
//
// Replaces generateRaysKernel (Renderer.cpp:521-555), shadeRayKernel (:411-479), compactStencilKernel +
// thrust::stable_partition (:506-519, :628-630), gatherImageDataKernel (:481-496) and initImageKernel (:557-565).
//
// Design (DESIGN.md 4.3, 4.5): path state is SoA float4 (origin+pixel, direction, throughput) in ping-pong queues.
// Per bounce, k_scan reads the hit records once and produces, for every 32-slot tile, the number of surviving paths in
// all earlier slots (one pass, decoupled look-back over 2048-slot blocks); k_shade then shades a slot and writes a
// survivor straight to its compacted position in the other queue, while a terminated path adds sqrt(throughput) to the
// film on the spot - or, when several lanes are in flight, stores it in the lane's contribution buffer, which one
// k_film_add per iteration adds to the film in iteration order (each pixel owns exactly one path per iteration, so both
// equal the reference's end-of-iteration gather).  The compaction is ORDER-PRESERVING, as thrust::stable_partition is,
// because the reference seeds its RNG with the slot index after compaction (Renderer.cpp:435, utility.h:57-62): same
// slots => same random streams => the same image, sample for sample.  No 80-byte struct is moved twice, no temporary
// is allocated, no count is read back by the host.
#include "kernels.cuh"

namespace ptap {

namespace {

constexpr float kTwoPi = 6.2831853071795864769252867665590057683943f;          // utility.h:20
constexpr float kSqrtOneThird = 0.5773502691896257645091487805019574556476f;   // utility.h:21

// utility.h:43-53
__device__ __forceinline__ unsigned utilHash(unsigned a)
{
    a = (a + 0x7ed55d16u) + (a << 12);
    a = (a ^ 0xc761c23cu) ^ (a >> 19);
    a = (a + 0x165667b1u) + (a << 5);
    a = (a + 0xd3a2646cu) ^ (a << 9);
    a = (a + 0xfd7046c5u) + (a << 3);
    a = (a ^ 0xb55a4f09u) ^ (a >> 16);
    return a;
}

// thrust::minstd_rand seeded as utility.h:57-62 does; uniform_real_distribution<float>(0,1) draws (SURVEY.md 8a a8).
struct Lcg {
    unsigned x;
    __device__ __forceinline__ Lcg(int iter, int index, int depth)
    {
        const unsigned h = utilHash(0x80000000u | ((unsigned)depth << 22) | (unsigned)iter) ^ utilHash((unsigned)index);
        x = h % 2147483647u;
        if (x == 0u) x = 1u;
    }
    __device__ __forceinline__ float u01()
    {
        x = (unsigned)(((unsigned long long)x * 48271ull) % 2147483647ull);
        return xdiv((float)(x - 1u), 2147483648.0f);
    }
};

// utility.h:64-69: n - 2 (i.n) n  (the reference's "mirror" keeps the normal as base vector)
__device__ __forceinline__ V3 reflectRay(V3 i, V3 n) { return xsub(n, xscale(n, xmul(2.0f, xdot(i, n)))); }

// utility.h:91-123
__device__ __forceinline__ V3 hemisphere(V3 n, Lcg& rng)
{
    const float up = xsqrt(rng.u01());
    const float over = xsqrt(xsub(1.0f, xmul(up, up)));
    const float around = xmul(rng.u01(), kTwoPi);
    V3 nn;
    if (xabs(n.x) < kSqrtOneThird) nn = v3(1, 0, 0);
    else if (xabs(n.y) < kSqrtOneThird) nn = v3(0, 1, 0);
    else nn = v3(0, 0, 1);
    const V3 p1 = xnormalize(xcross(n, nn));
    const V3 p2 = xnormalize(xcross(n, p1));
    float s, c;
    s = sinf(around); c = cosf(around);
    return xadd(xadd(xscale(n, up), xscale(p1, xmul(c, over))), xscale(p2, xmul(s, over)));
}

// utility.h:145-170
__device__ __forceinline__ V3 metal(V3 n, V3 dir, Lcg& rng)
{
    rng.u01(); rng.u01();                                   // `up`/`around` are drawn but unused (utility.h:150-152)
    const float phi = xmul(kTwoPi, rng.u01());
    const float r2 = rng.u01();
    const float cosTheta = powf(xsub(1.0f, r2), xdiv(1.0f, xadd(30.0f, 1.0f)));
    const float sinTheta = xsqrt(xsub(1.0f, xmul(cosTheta, cosTheta)));
    const V3 w = xnormalize(xsub(dir, xscale(xscale(n, 2.0f), xdot(n, dir))));
    const V3 a = ((double)xabs(w.x) > .1) ? v3(0, 1, 0) : v3(1, 0, 0);
    const V3 u = xnormalize(xcross(a, w));
    const V3 v = xcross(w, u);
    return xadd(xadd(xscale(xscale(u, cosf(phi)), sinTheta), xscale(xscale(v, sinf(phi)), sinTheta)), xscale(w, cosTheta));
}

// utility.h:125-143
__device__ __forceinline__ V3 coat(V3 n, V3 dir, Lcg& rng)
{
    if (rng.u01() < 0.5f) return reflectRay(dir, n);
    return hemisphere(n, rng);
}

// world-space shading normal of (model, tri): normalize(transpose(inverse(mat3(M))) * flat_normal)
// (Renderer.cpp:203,397; utility.h:82-88); matrix rows and flat normal are precomputed at upload with the same arithmetic.
__device__ __forceinline__ V3 worldNormal(const SceneDev& sc, int model, int tri, float4& nm0, float4& nm1, float4& nm2)
{
    const V3 n = v3(ldg4(&sc.normals[tri]));
    nm0 = ldg4(&sc.shade[model].nm0); nm1 = ldg4(&sc.shade[model].nm1); nm2 = ldg4(&sc.shade[model].nm2);
    const V3 r = v3(xadd(xadd(xmul(nm0.x, n.x), xmul(nm0.y, n.y)), xmul(nm0.z, n.z)),
                    xadd(xadd(xmul(nm1.x, n.x), xmul(nm1.y, n.y)), xmul(nm1.z, n.z)),
                    xadd(xadd(xmul(nm2.x, n.x), xmul(nm2.y, n.y)), xmul(nm2.z, n.z)));
    return xnormalize(r);
}

constexpr unsigned long long kFlagAgg = 1ull << 62, kFlagPrefix = 2ull << 62, kValueMask = 0xFFFFFFFFull;

__device__ __forceinline__ unsigned long long ldVolatile(const unsigned long long* p)
{
    return *reinterpret_cast<const volatile unsigned long long*>(p);
}
__device__ __forceinline__ void stVolatile(unsigned long long* p, unsigned long long v)
{
    *reinterpret_cast<volatile unsigned long long*>(p) = v;
}

}  // namespace

// generateRaysKernel (Renderer.cpp:521-555) + per-iteration reset of the device-side frame state.
__global__ void __launch_bounds__(kGenBlock) k_generate(WaveDev wv, int iter_now)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int stride = gridDim.x * blockDim.x;
    FrameState* st = wv.st;
    if (tid == 0) {
        st->iter_cur = st->iter_next; st->iter_next = st->iter_cur + wv.iter_stride;
        st->n_active[0] = wv.N;
        st->paths += (unsigned long long)wv.N;
    }
    if (tid >= 1 && tid <= kMaxDepth + 1) st->n_active[tid] = 0;
    if (tid < kMaxDepth + 2) { st->ticket[tid] = 0u; st->fetch[tid] = 0u; st->n_replay[tid] = 0u; st->fetch_replay[tid] = 0u; st->fetch_emu[tid] = 0u; st->n_cont[tid] = 0u; st->n_walk[tid] = 0u; st->fetch_walk[tid] = 0u; }
    const int nwords = wv.nscan * wv.depth;
    for (int i = tid; i < nwords; i += stride) wv.tile_status[i] = 0ull;      // one look-back word per 2048-slot scan block and round
    for (int i = tid; i < wv.N; i += stride) {
        const int y = i / wv.W, x = i % wv.W;
        // float world_x = -10.0 + x * step_x  (double add of a float product, Renderer.cpp:541-542); the camera's numbers are parameters
        // (ptap_set_camera), the arithmetic is the reference's: with its own camera the rays are bit-identical
        float fx = (float)x, fy = (float)y;
        if (wv.jitter) {        // sub-pixel offset in [0, 1)^2, a hash of (seed, iteration, pixel): the reference has no jitter (Renderer.cpp:527-548)
            const unsigned h = utilHash(wv.jitter_seed ^ utilHash((unsigned)iter_now + 0x9e3779b9u)) ^ utilHash((unsigned)i);
            fx = xadd(fx, xmul((float)(utilHash(h) >> 8), 5.9604644775390625e-8f));
            fy = xadd(fy, xmul((float)(utilHash(h ^ 0x85ebca6bu) >> 8), 5.9604644775390625e-8f));
        }
        const float wx = (float)((double)wv.cam_p[0] + (double)xmul(fx, wv.step_x));
        const float wy = (float)((double)wv.cam_p[1] + (double)xmul(fy, wv.step_y));
        wv.O[0][i] = make_float4(wv.cam_o[0], wv.cam_o[1], wv.cam_o[2], __int_as_float(i));
        wv.D[0][i] = make_float4(xsub(wx, wv.cam_o[0]), xsub(wy, wv.cam_o[1]), xsub(wv.cam_p[2], wv.cam_o[2]), 0.0f);
        wv.C[0][i] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
    }
}

// Survival of slot i after this bounce: bounces-- leaves > 0 (Renderer.cpp:478, 512); EMISSIVE zeroes the count (Renderer.cpp:459),
// a miss too (Renderer.cpp:476).  It depends only on the hit record, the material type and the round.
__device__ __forceinline__ bool survives(const SceneDev& sc, const float4& h, int remaining, int& type)
{
    const bool is_hit = h.x < kFloatMax;                                         // Renderer.cpp:426
    type = is_hit ? __ldg(&sc.shade[__float_as_int(h.z)].mat.x) : -1;
    return is_hit && remaining > 1 && type != PTAP_EMISSIVE;
}

// compactStencilKernel + the scan half of thrust::stable_partition (Renderer.cpp:506-519, 628-630), as ONE pass over the hit records:
// for every 32-slot tile of the round's wavefront, the number of surviving paths in all earlier slots (tile_offset), and the new
// active count.  A CTA takes a 2048-slot block by ticket (8 coalesced slots per thread), scans its 64 tile counts in shared
// memory, and obtains its own base by decoupled look-back over the earlier CTAs' status words (flag | count in one 64-bit word).
// k_shade then writes survivors to tile_offset[tile] + rank: the same order-preserving placement, with no dependency between tiles.
__global__ void __launch_bounds__(kScanBlock)
k_scan(SceneDev sc, WaveDev wv, int round, const float4* __restrict__ hit, int remaining, int n_fixed)
{
    __shared__ int s_cnt[kScanTiles];
    __shared__ unsigned s_ticket;
    constexpr int kSub = kScanSlots / kScanBlock, kWarps = kScanBlock / 32, kClasses = 8;      // 256-slot shade blocks per scan block
    __shared__ unsigned short s_wcnt[kSub][kWarps][kClasses];       // slots of material class c in tile (k, w) ...
    __shared__ unsigned short s_wbase[kSub][kWarps][kClasses];      // ... and where they start in the regrouped order of shade block k
    FrameState* st = wv.st;
    const int n = n_fixed >= 0 ? n_fixed : st->n_active[round];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long* status = wv.tile_status + (size_t)round * wv.nscan;
    if (threadIdx.x == 0) s_ticket = atomicAdd(&st->ticket[round], 1u);
    __syncthreads();
    const int blk = (int)s_ticket;
    const int base = blk * kScanSlots;
    if (base >= n) return;
    const bool sort = sc.shade_sort != 0;
    unsigned packed[kSub / 4] = {};                                               // (class << 5 | rank in the tile's class) per k, one byte each
#pragma unroll
    for (int k = 0; k < kScanSlots / kScanBlock; ++k) {
        const int i = base + k * kScanBlock + threadIdx.x;
        bool alive = false;
        int type = -1;
        float hx = kFloatMax;
        if (i < n) { const float4 h = hit[i]; hx = h.x; alive = survives(sc, h, remaining, type); }
        const unsigned ballot = __ballot_sync(0xffffffffu, alive);
        if (lane == 0) s_cnt[k * (kScanBlock / 32) + warp] = __popc(ballot);     // tile j = k * 8 + warp covers slots base + 32 j ..
        if (sort) {
            // material class of the slot: what k_shade will execute for it (survivors by scattering routine, terminated hits, misses)
            if (lane == 0 && base + k * kScanBlock + warp * 32 < n) wv.tile_ballot[base / 32 + k * kWarps + warp] = ballot;
            const int cls = i >= n ? 7 : !(hx < kFloatMax) ? 5 : !alive ? 4
                          : type == PTAP_DIFFUSE ? 0 : type == PTAP_METAL ? 1 : type == PTAP_COAT ? 2 : type == PTAP_REFLECTIVE ? 3 : 6;
            int r = 0;
#pragma unroll
            for (int c = 0; c < kClasses; ++c) {
                const unsigned m = __ballot_sync(0xffffffffu, cls == c);
                if (cls == c) r = __popc(m & ((1u << lane) - 1u));
                if (lane == c) s_wcnt[k][warp][c] = (unsigned short)__popc(m);
            }
            packed[k >> 2] |= (unsigned)(cls << 5 | r) << (8 * (k & 3));
        }
    }
    __syncthreads();
    if (sort) {
        // start of (tile w, class c) within shade block k: class-major, tile-minor
        for (int e = threadIdx.x; e < kSub * kWarps * kClasses; e += kScanBlock) {
            const int k = e / (kWarps * kClasses), w = (e / kClasses) % kWarps, c = e % kClasses;
            int acc = 0;
            for (int cc = 0; cc <= c; ++cc)
                for (int ww = 0; ww < (cc < c ? kWarps : w); ++ww) acc += s_wcnt[k][ww][cc];
            s_wbase[k][w][c] = (unsigned short)acc;
        }
    }
    if (warp == 0) {
        // exclusive scan of the 64 tile counts (two per lane), block total, look-back
        const int c0 = s_cnt[2 * lane], c1 = s_cnt[2 * lane + 1];
        int incl = c0 + c1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int up = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += up; }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        const int ex = incl - (c0 + c1);
        int excl = 0;
        if (blk == 0) {
            if (lane == 0) stVolatile(&status[0], kFlagPrefix | (unsigned long long)total);
        } else {
            if (lane == 0) stVolatile(&status[blk], kFlagAgg | (unsigned long long)total);
            int look = blk - 1;
            for (;;) {
                const int idx = look - lane;
                const unsigned long long w = idx >= 0 ? ldVolatile(&status[idx]) : kFlagPrefix;
                const unsigned has_prefix = __ballot_sync(0xffffffffu, (w >> 62) == 2ull);
                const unsigned is_empty = __ballot_sync(0xffffffffu, (w >> 62) == 0ull);
                const int p = has_prefix ? __ffs(has_prefix) - 1 : 32;           // nearest block with an inclusive prefix
                const unsigned need = p >= 31 ? 0xffffffffu : ((2u << p) - 1u);
                if (is_empty & need) continue;                                   // a needed predecessor has not published yet
                int v = (lane <= p) ? (int)(w & kValueMask) : 0;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                excl += v;
                if (p < 32) break;
                look -= 32;
            }
            if (lane == 0) stVolatile(&status[blk], kFlagPrefix | (unsigned long long)(excl + total));
        }
        s_cnt[2 * lane] = excl + ex; s_cnt[2 * lane + 1] = excl + ex + c0;
        if (lane == 0 && base + kScanSlots >= n) st->n_active[n_fixed < 0 ? round + 1 : kMaxDepth + 1] = excl + total;
    }
    __syncthreads();
    if (threadIdx.x < kScanTiles && base + threadIdx.x * 32 < n) wv.tile_offset[base / 32 + threadIdx.x] = s_cnt[threadIdx.x];
    if (sort) {
#pragma unroll
        for (int k = 0; k < kSub; ++k) {
            if (base + k * kScanBlock >= n) break;
            const unsigned pk = (packed[k >> 2] >> (8 * (k & 3))) & 0xffu;
            wv.perm[base + k * kScanBlock + s_wbase[k][warp][pk >> 5] + (pk & 31u)] = (unsigned char)threadIdx.x;
        }
    }
}

// shadeRayKernel + the move half of stable_partition + film accumulation for one bounce (Renderer.cpp:411-479, 481-496, 628).
// Slot i of queue `in` holds a path with `remaining` bounces left (every live path of a round has the same count).
// A CTA takes kShadeBlock consecutive slots (kShadeBlock / 32 compaction tiles).  Results are placement-independent: a survivor of slot i
// goes to tile_offset[tile(i)] + (survivors before i in its tile) in queue `in ^ 1`, its random stream is seeded with i, and a terminated
// path adds sqrt(throughput) to its own pixel (each pixel owns exactly one path per iteration).  So WHICH thread shades a slot is free,
// and with SORT the threads of a block take its slots regrouped by material class (DIFFUSE / METAL / COAT / REFLECTIVE survivors,
// terminated hits, misses: a counting sort per 256-slot block that k_scan makes while it reads the hit records anyway), so that a warp
// runs one scattering routine instead of up to four in turn.  The reference's per-slot semantics (RNG seed by slot, stable order) are
// untouched; only the SIMT schedule changes.  No shared memory, no barrier.
template <bool SORT>
__global__ void __launch_bounds__(kShadeBlock)
k_shade(SceneDev sc, WaveDev wv, int round, int in, const float4* __restrict__ hit, int remaining, int n_fixed, int iter_fixed,
        int* __restrict__ slot_pos)
{
    const FrameState* st = wv.st;
    const int n = n_fixed >= 0 ? n_fixed : st->n_active[round];
    const int iter = n_fixed >= 0 ? iter_fixed : st->iter_cur;
    const float4* __restrict__ Oi = wv.O[in]; const float4* __restrict__ Di = wv.D[in]; const float4* __restrict__ Ci = wv.C[in];
    float4* __restrict__ Oo = wv.O[in ^ 1]; float4* __restrict__ Do = wv.D[in ^ 1]; float4* __restrict__ Co = wv.C[in ^ 1];
    const int nblocks = (n + kShadeBlock - 1) / kShadeBlock;

    int s_next = threadIdx.x;
    if (SORT && (int)blockIdx.x < nblocks) s_next = wv.perm[(size_t)blockIdx.x * kShadeBlock + threadIdx.x];
    for (int blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const int base = blk * kShadeBlock;
        const int s = s_next;                                // the slot (within the block) this thread shades: regrouped by material class (k_scan)
        if (SORT && blk + (int)gridDim.x < nblocks) s_next = wv.perm[(size_t)(blk + gridDim.x) * kShadeBlock + threadIdx.x];   // one block ahead
        const int i = base + s;
        const bool in_range = i < n;
        float4 h = make_float4(kFloatMax, 0, 0, 0);
        if (in_range) h = hit[i];
        int type;
        const bool alive = survives(sc, h, remaining, type) && in_range;
        // survivors of the slot's tile: k_scan's ballot when the slots are regrouped, else this warp holds exactly that tile
        const unsigned tile_ballot = SORT ? (in_range ? __ldg(&wv.tile_ballot[(base >> 5) + (s >> 5)]) : 0u) : __ballot_sync(0xffffffffu, alive);
        if (in_range) {
            // queue traffic is read once and written once per bounce: streaming (evict-first) loads and stores keep it from displacing
            // the scene's nodes and triangles in L2 (+0.8 % per frame, profiles/r01/README.md)
            float4 o4 = __ldcs(&Oi[i]), d4 = __ldcs(&Di[i]), c4 = __ldcs(&Ci[i]);
            const int excl = __ldg(&wv.tile_offset[(base >> 5) + (s >> 5)]);
            const bool is_hit = h.x < kFloatMax;
            const int tri = __float_as_int(h.y), model = __float_as_int(h.z);
            const int rank = __popc(tile_ballot & ((1u << (s & 31)) - 1u));

            V3 col = v3(c4);
            if (is_hit) {
                float4 nm0, nm1, nm2;
                const V3 nrm = worldNormal(sc, model, tri, nm0, nm1, nm2);
                const V3 albedo = v3(nm0.w, nm1.w, nm2.w);
                const V3 dir = xnormalize(v3(d4));                               // Renderer.cpp:428
                // IntersectionData::impact_distance (Renderer.cpp:391): k_trace_bvh leaves it to be evaluated here (hit.x < 0)
                const float dist = h.x >= 0.0f ? h.x : exactHitDistance(sc, v3(o4), v3(d4), model, h.w);
                const V3 pt = xadd(v3(o4), xscale(dir, dist));                   // Renderer.cpp:429
                if (type == PTAP_DIFFUSE || type == PTAP_METAL || type == PTAP_COAT) {   // Renderer.cpp:433-453
                    if (alive) {
                        Lcg rng(iter, i, remaining);
                        const V3 nd = type == PTAP_DIFFUSE ? hemisphere(nrm, rng) : type == PTAP_METAL ? metal(nrm, dir, rng) : coat(nrm, dir, rng);
                        const V3 no = xadd(pt, xscale(nrm, 0.1f));
                        o4.x = no.x; o4.y = no.y; o4.z = no.z; d4.x = nd.x; d4.y = nd.y; d4.z = nd.z;
                    }
                    col = xmul(col, albedo);
                } else if (type == PTAP_EMISSIVE) {                              // Renderer.cpp:454-460
                    col = xmul(col, albedo);
                } else if (type == PTAP_REFLECTIVE) {                            // Renderer.cpp:461-467
                    col = xmul(col, albedo);
                    const V3 nd = reflectRay(dir, nrm);
                    const V3 no = xadd(pt, xscale(nrm, 0.1f));
                    o4.x = no.x; o4.y = no.y; o4.z = no.z; d4.x = nd.x; d4.y = nd.y; d4.z = nd.z;
                }                                                                // SPECULAR / REFRACTIVE: no branch, ray unchanged
            } else {                                                             // Renderer.cpp:471-477
                col = xmul(col, v3(0.01f, 0.01f, 0.01f));
            }
            c4.x = col.x; c4.y = col.y; c4.z = col.z;
            const int pos = alive ? excl + rank : -1;
            if (alive) { __stcs(&Oo[pos], o4); __stcs(&Do[pos], d4); __stcs(&Co[pos], c4); }
            else if (wv.contrib) {                                               // several lanes: the add happens in iteration order (k_film_add)
                float* px = wv.contrib + 3 * (size_t)__float_as_int(o4.w);
                px[0] = xsqrt(col.x); px[1] = xsqrt(col.y); px[2] = xsqrt(col.z);
            } else {                                                             // gatherImageDataKernel, Renderer.cpp:481-496
                float* px = wv.film + 3 * (size_t)__float_as_int(o4.w);
                px[0] = xadd(px[0], xsqrt(col.x)); px[1] = xadd(px[1], xsqrt(col.y)); px[2] = xadd(px[2], xsqrt(col.z));
            }
            if (slot_pos) slot_pos[i] = pos;
        }
    }
}

// (dist, tri, model, t) + (u, v) -> PtapHit with the world normal and material the reference would have stored
__global__ void k_resolve_hits(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, const float4* __restrict__ hit,
                               const float2* __restrict__ uv, int n, PtapHit* __restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 h = hit[i];
    PtapHit r;
    r.tri = __float_as_int(h.y); r.model = __float_as_int(h.z); r.t_model = h.w; r.dist = h.x;
    r.u = 0.0f; r.v = 0.0f; r.normal[0] = r.normal[1] = r.normal[2] = 0.0f; r.mat_type = -1;
    if (h.x < kFloatMax && r.model >= 0) {
        float4 a, b, c;
        const V3 nrm = worldNormal(sc, r.model, r.tri, a, b, c);
        r.normal[0] = nrm.x; r.normal[1] = nrm.y; r.normal[2] = nrm.z;
        r.mat_type = sc.shade[r.model].mat.x;
        if (h.x < 0.0f) r.dist = exactHitDistance(sc, v3(O[i]), v3(D[i]), r.model, h.w);      // deferred by k_trace_bvh
        if (uv) { r.u = uv[i].x; r.v = uv[i].y; }
    } else {
        r.model = -1; r.tri = -1; r.t_model = 0.0f;
    }
    out[i] = r;
}

// occlusion of a segment of world length L = D[i].w (ptap_query_occluded): the closest hit is nearer than L.  A record is a closest hit
// (launchTrace), or what the any-hit traversal left: retired as occluded (model kAnyOccluded), a candidate (model, t) to compare, or a miss.
__global__ void k_resolve_occluded(SceneDev sc, const float4* __restrict__ O, const float4* __restrict__ D, const float4* __restrict__ hit,
                                   int n, uint8_t* __restrict__ occluded)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 h = hit[i];
    const int model = __float_as_int(h.z);
    bool occ = model == kAnyOccluded;
    if (h.x < kFloatMax && model >= 0) {
        const float4 d4 = D[i];
        const float dist = h.x >= 0.0f ? h.x : exactHitDistance(sc, v3(O[i]), v3(d4), model, h.w);   // as k_resolve_hits
        occ = dist < d4.w;                                                                      // NaN L: false
    }
    occluded[i] = occ ? 1 : 0;
}

__global__ void k_set_iter(FrameState* st, int iter) { st->iter_next = iter; }

// normals[t] = flat normal of global triangle t (the .w lanes of its TriRec), one 16-byte record for the shade kernel's gather
__global__ void k_extract_normals(const TriRec* __restrict__ tris, int n, float4* __restrict__ normals)
{
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x)
        normals[t] = make_float4(tris[t].v0.w, tris[t].e1.w, tris[t].e2.w, 0.0f);
}

// bvh_tris[k] = tris[tri_id[k]]: triangle records in BVH leaf order, gathered on the device (the host uploads each record once)
__global__ void k_gather_tris(const TriRec* __restrict__ tris, const int* __restrict__ tri_id, int n, LeafTri* __restrict__ out)
{
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const int id = tri_id[k];
        const float4 a = tris[id].v0, b = tris[id].e1, c = tris[id].e2;
        float4* o = reinterpret_cast<float4*>(&out[k]);
        o[0] = make_float4(a.x, a.y, a.z, b.x);
        o[1] = make_float4(b.y, b.z, c.x, c.y);
        o[2] = make_float4(c.z, __int_as_float(id), 0.0f, 0.0f);
        o[3] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
}

// Renderer::renderImage's per-pixel arithmetic on the device (Renderer.cpp:42-53): byte = (char)(image * (1 / ITER) * 255), three bytes per
// pixel in (x, y, z) order, rows bottom-up as stored.  The host then copies 3 bytes per pixel instead of 12 and only writes the file.
__global__ void k_resolve_bmp(const float* __restrict__ film, size_t nvalues, float div, unsigned char* __restrict__ out)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvalues; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (unsigned char)(int)xmul(xmul(film[i], div), 255.0f);
}

// SAMPLESX x SAMPLESY box resolve (ptap.h: ptap_read_film_resolved): out(x, y) = sum over the pixel's lattice samples, row-major, of
// avg * film(sample), avg = 1.0f / (sx * sy) - the per-sample weight gatherImageDataKernel intends (Renderer.cpp:493).
__global__ void k_resolve_box(const float* __restrict__ film, int W, int H, int sx, int sy, float* __restrict__ out)
{
    const int Wp = W / sx, Hp = H / sy;
    const float avg = xdiv(1.0f, (float)(sx * sy));
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < (size_t)Wp * Hp * 3; e += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % 3), x = (int)((e / 3) % Wp), y = (int)(e / 3 / Wp);
        float acc = 0.0f;
        for (int j = 0; j < sy; ++j)
            for (int i = 0; i < sx; ++i) acc = xadd(acc, xmul(avg, film[((size_t)(y * sy + j) * W + (x * sx + i)) * 3 + c]));
        out[e] = acc;
    }
}

__global__ void k_film_add(float* __restrict__ film, const float* __restrict__ add, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) film[i] += add[i];
}

void launchGenerate(const WaveDev& wv, int iter, int grid, cudaStream_t stream) { k_generate<<<grid, kGenBlock, 0, stream>>>(wv, iter); }

void launchScan(const SceneDev& sc, const WaveDev& wv, int round, const float4* hit, int remaining, int n_fixed, cudaStream_t stream)
{
    if (wv.nscan > 0) k_scan<<<wv.nscan, kScanBlock, 0, stream>>>(sc, wv, round, hit, remaining, n_fixed);
}

void launchShade(const SceneDev& sc, const WaveDev& wv, int round, int in_buf, const float4* hit, int remaining, int n_fixed,
                 int iter_fixed, int* slot_pos, int grid, cudaStream_t stream)
{
    if (sc.shade_sort) k_shade<true><<<grid, kShadeBlock, 0, stream>>>(sc, wv, round, in_buf, hit, remaining, n_fixed, iter_fixed, slot_pos);
    else k_shade<false><<<grid, kShadeBlock, 0, stream>>>(sc, wv, round, in_buf, hit, remaining, n_fixed, iter_fixed, slot_pos);
}

int shadeOccupancy()
{
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_shade<true>, kShadeBlock, 0);
    return nb;
}

void launchResolveHits(const SceneDev& sc, const float4* O, const float4* D, const float4* hit, const float2* uv, int n, PtapHit* out, cudaStream_t stream)
{
    if (n > 0) k_resolve_hits<<<(n + 255) / 256, 256, 0, stream>>>(sc, O, D, hit, uv, n, out);
}

void launchResolveOccluded(const SceneDev& sc, const float4* O, const float4* D, const float4* hit, int n, uint8_t* occluded, cudaStream_t stream)
{
    if (n > 0) k_resolve_occluded<<<(n + 255) / 256, 256, 0, stream>>>(sc, O, D, hit, n, occluded);
}

void launchSetIter(FrameState* st, int iter, cudaStream_t stream) { k_set_iter<<<1, 1, 0, stream>>>(st, iter); }

void launchExtractNormals(const TriRec* tris, int n, float4* normals, cudaStream_t stream)
{
    if (n > 0) k_extract_normals<<<148 * 4, 256, 0, stream>>>(tris, n, normals);
}

void launchGatherTris(const TriRec* tris, const int* tri_id, int n, LeafTri* out, cudaStream_t stream)
{
    if (n > 0) k_gather_tris<<<148 * 4, 256, 0, stream>>>(tris, tri_id, n, out);
}

void launchResolveBox(const float* film, int W, int H, int sx, int sy, float* out, cudaStream_t stream)
{
    k_resolve_box<<<148 * 8, 256, 0, stream>>>(film, W, H, sx, sy, out);
}

void launchResolveBmp(const float* film, size_t nvalues, float div, unsigned char* out, cudaStream_t stream)
{
    if (nvalues) k_resolve_bmp<<<148 * 8, 256, 0, stream>>>(film, nvalues, div, out);
}

void launchFilmAdd(float* film, const float* add, size_t n, cudaStream_t stream)
{
    if (n) k_film_add<<<148 * 4, 256, 0, stream>>>(film, add, n);
}

}  // namespace ptap
