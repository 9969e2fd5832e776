// bvh_device.cu - builds the per-mesh 4-wide BVH on the GPU (PTAP_ACCEL_BVH_DEVICE): an LBVH in milliseconds instead of the host's
// binned-SAH build in seconds (SURVEY.md 8f row 2; the reference builds its only structure, the 25^3 grid, on the host: Scene.cpp:318-396).
//
//   1  k_lbvh_keys      per triangle: box of the FATTENED triangle (the predicate's tolerance band, as bvh_build.cpp) and the 30-bit Morton
//                       code of its centroid inside the mesh bounds
//   2  cub radix sort   (key, triangle id) pairs                                        [library call: not on the render path]
//   3  k_lbvh_leaves    every sorted triangle (or cluster of kCluster consecutive ones) becomes a leaf: LeafTri records in leaf order, leaf boxes
//   4  k_lbvh_topology  Karras 2012: every internal node of the binary radix tree over the leaves finds its range and split independently
//   5  k_lbvh_refit     bottom-up box fit, the second child to arrive at a node continues upwards (one atomic counter per node)
//   6  k_lbvh_collapse  breadth-first, one launch per level: a binary node and its two children become one 4-wide BvhNode, its child boxes
//                       encoded as outward-rounded offsets from a node-local origin exactly as the host builder does (bvh_build.cpp: encodeNode)
//
// PTAP_DEVICE_BUILDER=ploc (default) replaces steps 4-5 by PLOC (Meister & Bittner 2018, "Parallel locally-ordered clustering"): the
// Morton-sorted leaves are merged bottom-up, every cluster pairing with the neighbour (within kPlocRadius positions) whose union with it
// has the smallest surface area whenever the choice is mutual; the surviving clusters are compacted and the round repeats until one is
// left.  Boxes are made at the merges, no refit pass is needed, and the tree is close to a SAH tree where the radix tree is not.
// PTAP_DEVICE_BUILDER=lbvh keeps the radix tree.  PLOC stops at kPlocTop clusters; the levels above them come from a binned-SAH build on the
// host over the cluster boxes (buildTopSah: under a millisecond), because merges that are local in Morton order are arbitrary near the root.
//
// The tree is a different one than the host builder's, so rays visit different boxes; hits are bit-identical all the same, because the
// boxes are conservative for the reference's predicate and the triangle arithmetic is the exact one (tests/test_gpu_device_bvh.py).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "host_math.h"
#include "instance_math.h"
#include "kernels.cuh"

namespace ptap {

namespace {

constexpr float kBandEpsF = 0.0056f;          // > EPSILON (Config.h:4), as bvh_build.cpp
#ifndef PTAP_LBVH_CLUSTER
#define PTAP_LBVH_CLUSTER 1
#endif
constexpr int kCluster = PTAP_LBVH_CLUSTER;    // consecutive Morton-sorted triangles per leaf

__device__ __forceinline__ unsigned expandBits(unsigned v)
{
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

struct Box6 { float lo[3], hi[3]; };

__device__ __forceinline__ Box6 fatBox(const TriRec& r, float slack)
{
    // corners of the fattened triangle at (u, v) = (-e, -e), (1 + 2e, -e), (-e, 1 + 2e); the slack dwarfs the rounding of this arithmetic
    Box6 b;
    const float uv[3][2] = {{-kBandEpsF, -kBandEpsF}, {1.0f + 2.0f * kBandEpsF, -kBandEpsF}, {-kBandEpsF, 1.0f + 2.0f * kBandEpsF}};
    const float v0[3] = {r.v0.x, r.v0.y, r.v0.z}, e1[3] = {r.e1.x, r.e1.y, r.e1.z}, e2[3] = {r.e2.x, r.e2.y, r.e2.z};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float lo = 3e38f, hi = -3e38f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float p = v0[k] + uv[c][0] * e1[k] + uv[c][1] * e2[k];
            lo = fminf(lo, p); hi = fmaxf(hi, p);
        }
        const float pad = slack + 2e-6f * fmaxf(fabsf(lo), fabsf(hi));
        b.lo[k] = lo - pad; b.hi[k] = hi + pad;
    }
    return b;
}

__global__ void k_lbvh_keys(const TriRec* __restrict__ tris, int t0, int n, float3 mlo, float3 minv, unsigned* __restrict__ keys, int* __restrict__ ids)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const TriRec r = tris[t0 + i];
    const float cx = r.v0.x + (r.e1.x + r.e2.x) * (1.0f / 3.0f), cy = r.v0.y + (r.e1.y + r.e2.y) * (1.0f / 3.0f), cz = r.v0.z + (r.e1.z + r.e2.z) * (1.0f / 3.0f);
    const unsigned qx = (unsigned)fminf(fmaxf((cx - mlo.x) * minv.x, 0.0f), 1023.0f);
    const unsigned qy = (unsigned)fminf(fmaxf((cy - mlo.y) * minv.y, 0.0f), 1023.0f);
    const unsigned qz = (unsigned)fminf(fmaxf((cz - mlo.z) * minv.z, 0.0f), 1023.0f);
    keys[i] = (expandBits(qx) << 2) | (expandBits(qy) << 1) | expandBits(qz);
    ids[i] = t0 + i;
}

// leaf c = sorted triangles [kCluster c, min(kCluster (c + 1), n)): LeafTri records at leaf_base + k, global ids, the cluster's box and its 64-bit key
__global__ void k_lbvh_leaves(const TriRec* __restrict__ tris, const unsigned* __restrict__ keys, const int* __restrict__ ids, int n, int nleaves,
                              float slack, int leaf_base, LeafTri* __restrict__ btris, int* __restrict__ btid, Box6* __restrict__ leaf_box,
                              unsigned long long* __restrict__ leaf_key)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nleaves) return;
    Box6 box;
#pragma unroll
    for (int k = 0; k < 3; ++k) { box.lo[k] = 3e38f; box.hi[k] = -3e38f; }
    const int first = kCluster * c, last = min(first + kCluster, n);
    for (int s = first; s < last; ++s) {
        const int id = ids[s];
        const TriRec r = tris[id];
        const Box6 b = fatBox(r, slack);
#pragma unroll
        for (int k = 0; k < 3; ++k) { box.lo[k] = fminf(box.lo[k], b.lo[k]); box.hi[k] = fmaxf(box.hi[k], b.hi[k]); }
        float4* o = reinterpret_cast<float4*>(&btris[leaf_base + s]);
        o[0] = make_float4(r.v0.x, r.v0.y, r.v0.z, r.e1.x);
        o[1] = make_float4(r.e1.y, r.e1.z, r.e2.x, r.e2.y);
        o[2] = make_float4(r.e2.z, __int_as_float(id), 0.0f, 0.0f);
        o[3] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        btid[leaf_base + s] = id;
    }
    leaf_box[c] = box;
    leaf_key[c] = ((unsigned long long)keys[first] << 32) | (unsigned)c;          // the index makes equal Morton codes distinct
}

__device__ __forceinline__ int delta(const unsigned long long* __restrict__ k, int n, int i, int j)
{
    return (j < 0 || j >= n) ? -1 : __clzll(k[i] ^ k[j]);
}

// Karras, "Maximizing parallelism in the construction of BVHs, octrees and k-d trees" (2012): internal node i of n - 1.
// child >= 0: internal node; child < 0: leaf ~index.
__global__ void k_lbvh_topology(const unsigned long long* __restrict__ key, int nleaves, int2* __restrict__ child, int* __restrict__ parent_internal,
                                int* __restrict__ parent_leaf)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nleaves - 1) return;
    const int d = delta(key, nleaves, i, i + 1) - delta(key, nleaves, i, i - 1) >= 0 ? 1 : -1;
    const int dmin = delta(key, nleaves, i, i - d);
    int lmax = 2;
    while (delta(key, nleaves, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(key, nleaves, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(key, nleaves, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (delta(key, nleaves, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int left = lo == gamma ? ~gamma : gamma, right = hi == gamma + 1 ? ~(gamma + 1) : gamma + 1;
    child[i] = make_int2(left, right);
    if (left >= 0) parent_internal[left] = i; else parent_leaf[~left] = i;
    if (right >= 0) parent_internal[right] = i; else parent_leaf[~right] = i;
    if (i == 0) parent_internal[0] = -1;
}

__device__ __forceinline__ Box6 loadBoxL2(const Box6* p)
{
    Box6 b;
    const float* f = reinterpret_cast<const float*>(p);
#pragma unroll
    for (int k = 0; k < 3; ++k) { b.lo[k] = __ldcg(f + k); b.hi[k] = __ldcg(f + 3 + k); }
    return b;
}

__global__ void k_lbvh_refit(const int2* __restrict__ child, const int* __restrict__ parent_internal, const int* __restrict__ parent_leaf,
                             const Box6* __restrict__ leaf_box, int nleaves, Box6* __restrict__ node_box, int* __restrict__ arrived)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nleaves) return;
    int node = parent_leaf[c];
    while (node >= 0) {
        if (atomicAdd(&arrived[node], 1) == 0) return;              // the first child to arrive stops; the second one owns the node
        __threadfence();
        const int2 ch = child[node];
        // boxes written by other SMs during this launch: read through L2 (an L1 line may predate the sibling's store)
        const Box6 a = ch.x >= 0 ? loadBoxL2(&node_box[ch.x]) : leaf_box[~ch.x], b = ch.y >= 0 ? loadBoxL2(&node_box[ch.y]) : leaf_box[~ch.y];
        Box6 u;
#pragma unroll
        for (int k = 0; k < 3; ++k) { u.lo[k] = fminf(a.lo[k], b.lo[k]); u.hi[k] = fmaxf(a.hi[k], b.hi[k]); }
        node_box[node] = u;
        __threadfence();
        node = parent_internal[node];
    }
}

__device__ __forceinline__ int leafLink(int c, int n, int leaf_base)
{
    const int first = kCluster * c, count = min(kCluster, n - first);
    return ~(((leaf_base + first) << 3) | (count - 1));
}

// Child boxes of `nd` from up to four boxes (`ne` of them, slots 0 .. ne - 1), as bvh_build.cpp: encodeNode does on the host: local origin
// just below the node's lower corner, binary32 offsets rounded outward after a margin of 2^-20 of the largest coordinate; unused slots
// get an inverted box.
__device__ void encodeNodeDevice(BvhNode& nd, const Box6* boxes, int ne)
{
    float lo[3] = {3e38f, 3e38f, 3e38f}, mag = 0.0f;
    for (int c = 0; c < ne; ++c)
        for (int k = 0; k < 3; ++k) {
            lo[k] = fminf(lo[k], boxes[c].lo[k]);
            mag = fmaxf(mag, fmaxf(fabsf(boxes[c].lo[k]), fabsf(boxes[c].hi[k])));
        }
    const float margin = __fmul_ru(mag, 9.5367431640625e-7f) + 1e-30f;       // 2^-20
    float p[3];
    for (int k = 0; k < 3; ++k) p[k] = nextafterf(__fsub_rd(lo[k], margin), -3e38f);
    nd.px = p[0]; nd.py = p[1]; nd.pz = p[2]; nd.pad = 0;
    for (int c = 0; c < 4; ++c)
        for (int k = 0; k < 3; ++k) {
            if (c < ne) {
                nd.planes[k][0][c] = nextafterf(__fsub_rd(__fsub_rd(boxes[c].lo[k], margin), p[k]), -3e38f);
                nd.planes[k][1][c] = nextafterf(__fsub_ru(__fadd_ru(boxes[c].hi[k], margin), p[k]), 3e38f);
            } else { nd.planes[k][0][c] = 1e15f; nd.planes[k][1][c] = -1e15f; }
        }
}

// Leaf c of a TLAS (INST): instance leaf ~(0x20000000 | model), the model being leaf_model[c]
__device__ __forceinline__ int instLeafLink(const int* __restrict__ leaf_model, int c) { return ~(0x20000000 | leaf_model[c]); }

// One breadth-first level: frontier item = (binary internal node, index of the 4-wide node that represents it).  INST: the leaves are
// instances (a TLAS, leaf_model), else triangle clusters.
template <bool INST = false>
__global__ void k_lbvh_collapse(const int2* __restrict__ child, const Box6* __restrict__ node_box, const Box6* __restrict__ leaf_box, int n, int leaf_base,
                                const int2* __restrict__ frontier, int nfrontier, int2* __restrict__ next, int* __restrict__ counters /* [0] nodes, [1] next size */,
                                int node_base, BvhNode* __restrict__ out, const int* __restrict__ leaf_model = nullptr)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nfrontier) return;
    const int2 item = frontier[f];
    // up to four entries (>= 0: binary internal node, < 0: leaf ~index): starting from the node's two children, the internal entry with
    // the largest box is replaced by its own two children - the same greedy rule as the host collapse (bvh_build.cpp), which keeps big,
    // often-hit boxes out of the wide node instead of always taking the four grandchildren
    int ent[4]; Box6 ebox[4]; int ne = 2;
    { const int2 ch = child[item.x]; ent[0] = ch.x; ent[1] = ch.y; }
    for (int k = 0; k < 2; ++k) ebox[k] = ent[k] >= 0 ? node_box[ent[k]] : leaf_box[~ent[k]];
    while (ne < 4) {
        int best = -1; float best_area = -1.0f;
        for (int k = 0; k < ne; ++k) {
            if (ent[k] < 0) continue;
            const float dx = ebox[k].hi[0] - ebox[k].lo[0], dy = ebox[k].hi[1] - ebox[k].lo[1], dz = ebox[k].hi[2] - ebox[k].lo[2];
            const float a = dx * dy + dy * dz + dz * dx;
            if (a > best_area) { best_area = a; best = k; }
        }
        if (best < 0) break;
        const int2 g = child[ent[best]];
        ent[best] = g.x; ebox[best] = g.x >= 0 ? node_box[g.x] : leaf_box[~g.x];
        ent[ne] = g.y; ebox[ne] = g.y >= 0 ? node_box[g.y] : leaf_box[~g.y];
        ++ne;
    }
    BvhNode nd;
    Box6 boxes[4];
    for (int k = 0; k < 4; ++k) {
        if (k < ne) {
            const int e = ent[k];
            boxes[k] = ebox[k];
            if (e >= 0) {
                const int idx = atomicAdd(&counters[0], 1);
                next[atomicAdd(&counters[1], 1)] = make_int2(e, idx);
                nd.link[k] = node_base + idx;
            } else nd.link[k] = INST ? instLeafLink(leaf_model, ~e) : leafLink(~e, n, leaf_base);
        } else nd.link[k] = nd.link[0];
    }
    encodeNodeDevice(nd, boxes, ne);
    out[item.y] = nd;
}

// a mesh whose triangles fit one leaf (a scene with one instance): a root with a single child
template <bool INST = false>
__global__ void k_lbvh_single(const Box6* __restrict__ leaf_box, int n, int leaf_base, BvhNode* __restrict__ out, const int* __restrict__ leaf_model = nullptr)
{
    BvhNode nd;
    const Box6 b = leaf_box[0];
    for (int k = 0; k < 4; ++k) nd.link[k] = INST ? instLeafLink(leaf_model, 0) : leafLink(0, n, leaf_base);
    encodeNodeDevice(nd, &b, 1);
    out[0] = nd;
}

// ---- PLOC ------------------------------------------------------------------------------------------------------------------------

#ifndef PTAP_PLOC_RADIUS
#define PTAP_PLOC_RADIUS 16
#endif
constexpr int kPlocRadius = PTAP_PLOC_RADIUS;
#ifndef PTAP_PLOC_TOP
#define PTAP_PLOC_TOP 4096
#endif
constexpr int kPlocTop = PTAP_PLOC_TOP;

__device__ __forceinline__ float unionArea(const Box6& a, const Box6& b)
{
    const float dx = fmaxf(a.hi[0], b.hi[0]) - fminf(a.lo[0], b.lo[0]), dy = fmaxf(a.hi[1], b.hi[1]) - fminf(a.lo[1], b.lo[1]), dz = fmaxf(a.hi[2], b.hi[2]) - fminf(a.lo[2], b.lo[2]);
    return dx * dy + dy * dz + dz * dx;
}

__global__ void k_ploc_init(const Box6* __restrict__ leaf_box, int n, Box6* __restrict__ cbox, int* __restrict__ cnode)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { cbox[i] = leaf_box[i]; cnode[i] = ~i; }
}

// Tie key of the pair {i, j}, the same from either end: the partner in the same aligned pair (i >> 1 == j >> 1) first, then the nearer
// position, then the lower one.  A rule that is not symmetric (such as "the lower position") lets tied clusters point along a chain, i -> i - 1,
// in which only the first pair is mutual: coincident triangles or a long ribbon of equal quads then merge one pair per round.
__device__ __forceinline__ unsigned long long plocTieKey(int i, int j)
{
    return ((unsigned long long)((i >> 1) != (j >> 1)) << 63) | ((unsigned long long)abs(i - j) << 32) | (unsigned)min(i, j);
}

// nearest[i] = the position within the radius whose union with cluster i has the smallest area, ties broken by plocTieKey.  The order on
// (area, key) is the same for both ends of every pair, so the globally smallest pair is mutual and every round merges.
__global__ void k_ploc_nearest(const Box6* __restrict__ cbox, int n, int* __restrict__ nearest)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Box6 me = cbox[i];
    float best = 3e38f; int bj = -1; unsigned long long bkey = ~0ull;
    const int j0 = max(0, i - kPlocRadius), j1 = min(n - 1, i + kPlocRadius);
    for (int j = j0; j <= j1; ++j) {
        if (j == i) continue;
        const float a = unionArea(me, cbox[j]);
        const unsigned long long key = plocTieKey(i, j);
        if (a < best || (a == best && key < bkey)) { best = a; bj = j; bkey = key; }
    }
    nearest[i] = bj;
}

// mutual nearest neighbours merge into a new binary node (stored at the lower position); the partner's slot is dropped
__global__ void k_ploc_merge(Box6* __restrict__ cbox, int* __restrict__ cnode, const int* __restrict__ nearest, int n, int2* __restrict__ child,
                             Box6* __restrict__ node_box, int* __restrict__ counter, int* __restrict__ keep)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = nearest[i];
    if (j >= 0 && nearest[j] == i) {
        if (i < j) {
            const Box6 a = cbox[i], b = cbox[j];
            Box6 u;
#pragma unroll
            for (int k = 0; k < 3; ++k) { u.lo[k] = fminf(a.lo[k], b.lo[k]); u.hi[k] = fmaxf(a.hi[k], b.hi[k]); }
            const int id = atomicAdd(counter, 1);
            child[id] = make_int2(cnode[i], cnode[j]);
            node_box[id] = u;
            cbox[i] = u; cnode[i] = id;      // nobody else reads slot i in this launch: its only reader is its partner, which reads nothing
            keep[i] = 1;
        } else keep[i] = 0;
    } else keep[i] = 1;
}

__global__ void k_ploc_compact(const Box6* __restrict__ cbox, const int* __restrict__ cnode, const int* __restrict__ keep, const int* __restrict__ pos, int n,
                               Box6* __restrict__ obox, int* __restrict__ onode)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && keep[i]) { obox[pos[i]] = cbox[i]; onode[pos[i]] = cnode[i]; }
}

// Top of the tree: once PLOC has merged the leaves down to a few thousand clusters, the levels above them are built on the HOST by the
// same binned SAH as bvh_build.cpp uses (16 bins on the centroid axis with the lowest cost), over the cluster boxes - a few thousand items,
// well under a millisecond.  PLOC's merges are local in Morton order (radius 16): good near the leaves, arbitrary near the root, where a
// bad split costs every ray; this puts the surface-area heuristic where it matters and leaves the bulk of the work on the device.
struct TopItem { Box6 box; float c[3]; int link; };

int buildTopSah(std::vector<TopItem>& it, int begin, int end, int base, std::vector<int2>& out_child, std::vector<Box6>& out_box, Box6& bounds)
{
    auto grow = [](Box6& a, const Box6& b) { for (int k = 0; k < 3; ++k) { a.lo[k] = std::min(a.lo[k], b.lo[k]); a.hi[k] = std::max(a.hi[k], b.hi[k]); } };
    auto area = [](const Box6& b) { const float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2]; return dx < 0 ? 0.0f : dx * dy + dy * dz + dz * dx; };
    auto empty = []() { Box6 b; for (int k = 0; k < 3; ++k) { b.lo[k] = 3e38f; b.hi[k] = -3e38f; } return b; };
    bounds = empty();
    float clo[3] = {3e38f, 3e38f, 3e38f}, chi[3] = {-3e38f, -3e38f, -3e38f};
    for (int i = begin; i < end; ++i) { grow(bounds, it[i].box); for (int k = 0; k < 3; ++k) { clo[k] = std::min(clo[k], it[i].c[k]); chi[k] = std::max(chi[k], it[i].c[k]); } }
    if (end - begin == 1) return it[begin].link;
    constexpr int kBins = 16;
    int best_axis = -1, best_bin = -1; float best_cost = 3e38f;
    for (int axis = 0; axis < 3; ++axis) {
        const float ext = chi[axis] - clo[axis];
        if (!(ext > 0.0f)) continue;
        Box6 bb[kBins]; int cnt[kBins];
        for (int b = 0; b < kBins; ++b) { bb[b] = empty(); cnt[b] = 0; }
        const float scale = kBins / ext;
        for (int i = begin; i < end; ++i) { const int b = std::min(kBins - 1, std::max(0, (int)((it[i].c[axis] - clo[axis]) * scale))); grow(bb[b], it[i].box); cnt[b]++; }
        float right_area[kBins]; int right_cnt[kBins];
        Box6 acc = empty(); int c = 0;
        for (int b = kBins - 1; b > 0; --b) { grow(acc, bb[b]); c += cnt[b]; right_area[b] = area(acc); right_cnt[b] = c; }
        acc = empty(); c = 0;
        for (int b = 0; b < kBins - 1; ++b) {
            grow(acc, bb[b]); c += cnt[b];
            if (c == 0 || right_cnt[b + 1] == 0) continue;
            const float cost = area(acc) * c + right_area[b + 1] * right_cnt[b + 1];
            if (cost < best_cost) { best_cost = cost; best_axis = axis; best_bin = b; }
        }
    }
    int mid = begin + (end - begin) / 2;
    if (best_axis >= 0) {
        const float lo = clo[best_axis], scale = kBins / (chi[best_axis] - clo[best_axis]);
        auto m = std::partition(it.begin() + begin, it.begin() + end, [&](const TopItem& t) { return std::min(kBins - 1, std::max(0, (int)((t.c[best_axis] - lo) * scale))) <= best_bin; });
        const int k = (int)(m - it.begin());
        if (k > begin && k < end) mid = k;
    }
    const int me = (int)out_child.size();
    out_child.push_back(make_int2(0, 0)); out_box.push_back(bounds);
    Box6 b0, b1;
    const int l0 = buildTopSah(it, begin, mid, base, out_child, out_box, b0);
    const int l1 = buildTopSah(it, mid, end, base, out_child, out_box, b1);
    out_child[me] = make_int2(l0, l1);
    return base + me;
}

template <typename T> T* carve(char*& p, size_t count)
{
    T* r = reinterpret_cast<T*>(p);
    p += (count * sizeof(T) + 255) & ~size_t(255);
    return r;
}

size_t cubBytes(int n, int end_bit)
{
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned*)nullptr, (unsigned*)nullptr, (const int*)nullptr, (int*)nullptr, n, 0, end_bit);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int*)nullptr, (int*)nullptr, n);
    return std::max(sort_bytes, scan_bytes);
}

// carveBuild's bytes for `count` primitives in `leaves` leaves
size_t scratchBytes(int count, int leaves, int end_bit)
{
    const size_t n = (size_t)std::max(count, 1), L = (size_t)std::max(leaves, 1);
    return 4 * ((n * 4 + 255) & ~size_t(255)) + cubBytes((int)n, end_bit) + 256 + 4 * ((L * sizeof(Box6) + 255) & ~size_t(255)) + ((L * 8 + 255) & ~size_t(255)) * 4 +
           ((L * 4 + 255) & ~size_t(255)) * 3 + 4096;
}

// Scratch of one build over n primitives grouped into L leaves: the sort of the front, then the leaves and the clusters / binary nodes of
// the back.  The back reuses the front's unsorted keys and ids.
struct BuildScratch {
    unsigned *keys, *keys2; int *ids, *ids2;
    void* cub_tmp; size_t cub_bytes;
    Box6 *leaf_box, *node_box, *cbox_a, *cbox_b;
    unsigned long long* leaf_key;
    int2 *child, *fr_a, *fr_b;
    int *parent_internal, *parent_leaf, *arrived, *counters;
};

BuildScratch carveBuild(char*& p, int n, int L, int end_bit)
{
    BuildScratch s;
    s.keys = carve<unsigned>(p, n); s.keys2 = carve<unsigned>(p, n);
    s.ids = carve<int>(p, n); s.ids2 = carve<int>(p, n);
    s.cub_bytes = cubBytes(n, end_bit);
    s.cub_tmp = carve<char>(p, s.cub_bytes + 1);
    s.leaf_box = carve<Box6>(p, L); s.node_box = carve<Box6>(p, L);
    s.cbox_a = carve<Box6>(p, L); s.cbox_b = carve<Box6>(p, L);
    s.leaf_key = carve<unsigned long long>(p, L);
    s.child = carve<int2>(p, L); s.fr_a = carve<int2>(p, L); s.fr_b = carve<int2>(p, L);
    s.parent_internal = carve<int>(p, L); s.parent_leaf = carve<int>(p, L); s.arrived = carve<int>(p, L);
    s.counters = carve<int>(p, 64);
    return s;
}

// The back of both builds, from L leaf boxes and keys in Morton order (s.leaf_box, s.leaf_key): PLOC (or the radix tree) to kPlocTop
// clusters, the binned SAH on the host above them, and the breadth-first collapse into out_nodes[0 .. *nnodes) with links relative to
// node_base.  Triangle leaves (leaf_model null) are the clusters of n triangles at leaf_base; a TLAS's leaf c is instance leaf_model[c].
int buildTreeDevice(const BuildScratch& s, int L, int n, int leaf_base, const int* leaf_model, int node_base, BvhNode* out_nodes, cudaStream_t stream,
                    int* nnodes, int* depth, std::string* why)
{
    const int B = 256;
    cudaError_t e = cudaSuccess;
    size_t cub_bytes = s.cub_bytes;
    if (L == 1) {
        if (leaf_model) k_lbvh_single<true><<<1, 1, 0, stream>>>(s.leaf_box, n, leaf_base, out_nodes, leaf_model);
        else k_lbvh_single<<<1, 1, 0, stream>>>(s.leaf_box, n, leaf_base, out_nodes);
        *nnodes = 1; *depth = 1;
        return cudaGetLastError();
    }
    int root_node = 0;
    const char* which = getenv("PTAP_DEVICE_BUILDER");
    if (which && std::string(which) == "lbvh") {
        k_lbvh_topology<<<(L - 1 + B - 1) / B, B, 0, stream>>>(s.leaf_key, L, s.child, s.parent_internal, s.parent_leaf);
        e = cudaMemsetAsync(s.arrived, 0, (size_t)L * sizeof(int), stream);
        if (e != cudaSuccess) return e;
        k_lbvh_refit<<<(L + B - 1) / B, B, 0, stream>>>(s.child, s.parent_internal, s.parent_leaf, s.leaf_box, L, s.node_box, s.arrived);
    } else {
        // PLOC: clusters (box, node) in Morton order, double-buffered across the compaction; scratch arrays of the radix-tree path are reused
        Box6 *cb = s.cbox_a, *cb2 = s.cbox_b;
        int *cn = s.parent_internal, *cn2 = s.parent_leaf, *nearest = s.arrived, *keep = reinterpret_cast<int*>(s.keys), *pos = s.ids;
        int2* child = s.child;
        Box6* node_box = s.node_box;
        int* counters = s.counters;
        e = cudaMemsetAsync(counters + 8, 0, sizeof(int), stream);
        if (e != cudaSuccess) return e;
        k_ploc_init<<<(L + B - 1) / B, B, 0, stream>>>(s.leaf_box, L, cb, cn);
        int m = L, rounds = 0;
        const char* top_env = getenv("PTAP_PLOC_TOP");
        const int top = top_env ? atoi(top_env) : kPlocTop;       // clusters handed to the host's SAH build of the upper levels (0: PLOC to the root)
        while (m > 1 && !(top > 1 && m <= top)) {
            const int g = (m + B - 1) / B;
            k_ploc_nearest<<<g, B, 0, stream>>>(cb, m, nearest);
            k_ploc_merge<<<g, B, 0, stream>>>(cb, cn, nearest, m, child, node_box, counters + 8, keep);
            e = cub::DeviceScan::ExclusiveSum(s.cub_tmp, cub_bytes, keep, pos, m, stream);
            if (e != cudaSuccess) return e;
            k_ploc_compact<<<g, B, 0, stream>>>(cb, cn, keep, pos, m, cb2, cn2);
            int last[2];
            e = cudaMemcpyAsync(&last[0], pos + m - 1, sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(&last[1], keep + m - 1, sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            if (e != cudaSuccess) return e;
            const int m2 = last[0] + last[1];
            if (m2 >= m || ++rounds > 4096) {                              // every round merges at least the globally best pair
                if (why) *why = "PLOC merging stalled at " + std::to_string(m2) + " of " + std::to_string(L) + " clusters after " + std::to_string(rounds) + " rounds";
                return cudaErrorUnknown;
            }
            m = m2;
            std::swap(cb, cb2); std::swap(cn, cn2);
        }
        if (m > 1) {
            // the upper levels on the host: cluster boxes and links down, new binary nodes back up (appended after PLOC's)
            std::vector<Box6> hb(m); std::vector<int> hl(m);
            int made = 0;
            e = cudaMemcpyAsync(hb.data(), cb, (size_t)m * sizeof(Box6), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(hl.data(), cn, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(&made, counters + 8, sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            if (e != cudaSuccess) return e;
            if (made + m - 1 > L) return cudaErrorUnknown;                 // L leaves have L - 1 internal nodes
            std::vector<TopItem> items(m);
            for (int k = 0; k < m; ++k) { items[k].box = hb[k]; items[k].link = hl[k]; for (int a = 0; a < 3; ++a) items[k].c[a] = 0.5f * (hb[k].lo[a] + hb[k].hi[a]); }
            std::vector<int2> tc; std::vector<Box6> tb;
            tc.reserve(m); tb.reserve(m);
            Box6 bounds;
            root_node = buildTopSah(items, 0, m, made, tc, tb, bounds);
            e = cudaMemcpyAsync(child + made, tc.data(), tc.size() * sizeof(int2), cudaMemcpyHostToDevice, stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(node_box + made, tb.data(), tb.size() * sizeof(Box6), cudaMemcpyHostToDevice, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);       // tc / tb are stack-owned
            if (e != cudaSuccess) return e;
        } else {
            e = cudaMemcpyAsync(&root_node, cn, sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            if (e != cudaSuccess) return e;
        }
        if (root_node < 0) return cudaErrorUnknown;
    }
    // breadth-first collapse from the binary root: it becomes 4-wide node 0
    const int2 root = make_int2(root_node, 0);
    const int init[2] = {1, 0};
    e = cudaMemcpyAsync(s.fr_a, &root, sizeof root, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s.counters, init, sizeof init, cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;
    int nfrontier = 1, levels = 0;
    int2 *cur = s.fr_a, *nxt = s.fr_b;
    while (nfrontier > 0) {
        ++levels;
        const int g = (nfrontier + B - 1) / B;
        if (leaf_model) k_lbvh_collapse<true><<<g, B, 0, stream>>>(s.child, s.node_box, s.leaf_box, n, leaf_base, cur, nfrontier, nxt, s.counters, node_base, out_nodes, leaf_model);
        else k_lbvh_collapse<<<g, B, 0, stream>>>(s.child, s.node_box, s.leaf_box, n, leaf_base, cur, nfrontier, nxt, s.counters, node_base, out_nodes);
        int host_counters[2];
        e = cudaMemcpyAsync(host_counters, s.counters, sizeof host_counters, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return e;
        nfrontier = host_counters[1];
        *nnodes = host_counters[0];
        const int zero = 0;
        e = cudaMemcpyAsync(s.counters + 1, &zero, sizeof zero, cudaMemcpyHostToDevice, stream);
        if (e != cudaSuccess) return e;
        std::swap(cur, nxt);
        if (levels > 200) { if (why) *why = "the 4-wide collapse exceeded 200 levels"; return cudaErrorUnknown; }
    }
    *depth = levels;
    return cudaGetLastError();
}

// ---- TLAS front: the instances of ptap_update_models -----------------------------------------------------------------------------

// What k_update_instances reduces over the instances that have triangles (atomics on order-preserving bit patterns: the maxima of
// non-negative doubles, the minimum index, the centre bounds as ordered floats).  The same values in any order of the atomics.
struct InstanceReduce {
    unsigned long long max_scale, max_pad, max_trans;   // bits of non-negative doubles
    int first_bad;                                      // first model whose matrices are not inverses (INT_MAX: none)
    unsigned clo[3], chi[3];                            // bounds of the world-box centres (orderedBits)
};

__device__ __forceinline__ unsigned orderedBits(float f)
{
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fromOrderedBits(unsigned u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

template <typename T> __device__ __forceinline__ T warpMax(T v) { for (int o = 16; o; o >>= 1) { const T w = __shfl_xor_sync(~0u, v, o); v = w > v ? w : v; } return v; }
template <typename T> __device__ __forceinline__ T warpMin(T v) { for (int o = 16; o; o >>= 1) { const T w = __shfl_xor_sync(~0u, v, o); v = w < v ? w : v; } return v; }

// bits of a non-negative double for an atomic maximum; NaN (which std::max skips on the host) becomes 0
__device__ __forceinline__ unsigned long long maxBits(double v) { return v == v ? (unsigned long long)__double_as_longlong(v) : 0ull; }

// One thread per model.  Models [first, first + count) take their staged record: InstanceTrace.w2m / m2w (grid fields kept) and
// InstanceShade; the others keep theirs.  With a BVH (nodes), every model that has triangles then gets its world box and its terms of
// the scene constants from instanceBox (instance_math.h), the function finishBvh evaluates on the host; box / trans of a model without
// triangles are an empty box and -1.
__global__ void k_update_instances(InstanceTrace* __restrict__ inst, InstanceShade* __restrict__ shade, int nm, const PtapModel* __restrict__ staged,
                                   int first, int count, const BvhNode* __restrict__ nodes, Box6* __restrict__ box, double* __restrict__ trans,
                                   InstanceReduce* __restrict__ red)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double scale = 0.0, pad = 0.0;
    int bad = INT_MAX;
    unsigned clo[3] = {~0u, ~0u, ~0u}, chi[3] = {0u, 0u, 0u};
    if (i < nm) {
        float W[16], M[16];
        InstanceTrace& it = inst[i];
        if (i >= first && i < first + count) {
            const PtapModel& m = staged[i - first];
            for (int k = 0; k < 16; ++k) { W[k] = m.world_to_model[k]; M[k] = m.model_to_world[k]; }
            for (int r = 0; r < 3; ++r) { it.w2m[r] = make_float4(W[r], W[4 + r], W[8 + r], W[12 + r]); it.m2w[r] = make_float4(M[r], M[4 + r], M[8 + r], M[12 + r]); }
            float nmx[9];
            hm::normal_matrix(M, nmx);
            InstanceShade sh;
            sh.nm0 = make_float4(nmx[0], nmx[1], nmx[2], m.mat.color[0]);
            sh.nm1 = make_float4(nmx[3], nmx[4], nmx[5], m.mat.color[1]);
            sh.nm2 = make_float4(nmx[6], nmx[7], nmx[8], m.mat.color[2]);
            sh.mat = make_int4(m.mat.type, 0, 0, 0);
            shade[i] = sh;
        } else {
            for (int r = 0; r < 3; ++r) {
                const float4 w = it.w2m[r], v = it.m2w[r];
                W[r] = w.x; W[4 + r] = w.y; W[8 + r] = w.z; W[12 + r] = w.w;
                M[r] = v.x; M[4 + r] = v.y; M[8 + r] = v.z; M[12 + r] = v.w;
            }
            W[3] = W[7] = W[11] = M[3] = M[7] = M[11] = 0.0f; W[15] = M[15] = 1.0f;
        }
        if (nodes) {
            const int root = __float_as_int(it.grid.z);
            Box6 b;
            for (int k = 0; k < 3; ++k) { b.lo[k] = 3e38f; b.hi[k] = -3e38f; }
            double t = -1.0;
            InstanceBox ib;
            if (root >= 0 && instanceBox(W, M, nodes[root], ib)) {
                for (int k = 0; k < 3; ++k) {
                    b.lo[k] = ib.lo[k]; b.hi[k] = ib.hi[k];
                    clo[k] = chi[k] = orderedBits(0.5f * (ib.lo[k] + ib.hi[k]));
                }
                t = ib.trans; scale = ib.scale; pad = ib.pad;
                if (!ib.consistent) bad = i;
            }
            box[i] = b; trans[i] = t;
        }
    }
    if (!nodes) return;
    const unsigned long long s = warpMax(maxBits(scale)), p = warpMax(maxBits(pad));
    bad = warpMin(bad);
    for (int k = 0; k < 3; ++k) { clo[k] = warpMin(clo[k]); chi[k] = warpMax(chi[k]); }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(&red->max_scale, s); atomicMax(&red->max_pad, p); atomicMin(&red->first_bad, bad);
        for (int k = 0; k < 3; ++k) { atomicMin(&red->clo[k], clo[k]); atomicMax(&red->chi[k], chi[k]); }
    }
}

// Morton key of every instance's box centre inside the centre bounds (0xffffffff for instances without triangles: sorted last), and
// max_trans over the models up to the first inconsistent one
__global__ void k_instance_keys(const Box6* __restrict__ box, const double* __restrict__ trans, int nm, InstanceReduce* __restrict__ red,
                                unsigned* __restrict__ keys, int* __restrict__ ids)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long t = 0ull;
    if (i < nm) {
        unsigned key = 0xffffffffu;
        if (trans[i] >= 1.0) {
            const Box6 b = box[i];
            unsigned q[3];
            for (int k = 0; k < 3; ++k) {
                const float lo = fromOrderedBits(red->clo[k]), hi = fromOrderedBits(red->chi[k]);
                const float inv = hi > lo ? 1023.999f / (hi - lo) : 0.0f;
                q[k] = (unsigned)fminf(fmaxf((0.5f * (b.lo[k] + b.hi[k]) - lo) * inv, 0.0f), 1023.0f);
            }
            key = (expandBits(q[0]) << 2) | (expandBits(q[1]) << 1) | expandBits(q[2]);
            if (i <= red->first_bad) t = maxBits(trans[i]);
        }
        keys[i] = key; ids[i] = i;
    }
    t = warpMax(t);
    if ((threadIdx.x & 31) == 0) atomicMax(&red->max_trans, t);
}

__global__ void k_instance_leaves(const Box6* __restrict__ box, const unsigned* __restrict__ keys, const int* __restrict__ ids, int L,
                                  Box6* __restrict__ leaf_box, unsigned long long* __restrict__ leaf_key)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= L) return;
    leaf_box[c] = box[ids[c]];
    leaf_key[c] = ((unsigned long long)keys[c] << 32) | (unsigned)c;
}

}  // namespace

size_t deviceBvhScratchBytes(int ntris) { return scratchBytes(ntris, (std::max(ntris, 1) + kCluster - 1) / kCluster, 30); }

size_t instanceUpdateScratchBytes(int nmodels)
{
    const size_t n = (size_t)std::max(nmodels, 1);
    return scratchBytes(nmodels, nmodels, 32) +                       // one leaf per instance, whatever kCluster is
           ((n * sizeof(Box6) + 255) & ~size_t(255)) + ((n * sizeof(double) + 255) & ~size_t(255)) + 256;
}

// Builds the BLAS of one mesh (triangles [t0, t1) of the global table) into out_nodes[0 .. *nnodes) with links relative to node_base,
// leaf-order triangles into btris / btid at [leaf_base, leaf_base + n).  Returns a cudaError_t; *depth = levels of 4-wide nodes.  When the
// build itself gives up (not a CUDA call), *why says why.
int buildMeshBvhDevice(const TriRec* d_tris, int t0, int t1, const float* bb_min, const float* bb_max, int node_base, BvhNode* out_nodes, int leaf_base,
                       LeafTri* btris, int* btid, char* scratch, size_t scratch_bytes, cudaStream_t stream, int* nnodes, int* depth, std::string* why)
{
    const int n = t1 - t0, L = (n + kCluster - 1) / kCluster;
    *nnodes = 0; *depth = 0;
    if (n <= 0) return cudaSuccess;
    if (deviceBvhScratchBytes(n) > scratch_bytes) return cudaErrorMemoryAllocation;
    char* p = scratch;
    const BuildScratch s = carveBuild(p, n, L, 30);

    double ext = 0.0;
    float3 mlo, minv;
    {
        const float lo[3] = {bb_min[0], bb_min[1], bb_min[2]}, hi[3] = {bb_max[0], bb_max[1], bb_max[2]};
        for (int k = 0; k < 3; ++k) ext = std::max(ext, (double)std::max(std::fabs(lo[k]), std::fabs(hi[k])));
        mlo = make_float3(lo[0], lo[1], lo[2]);
        auto inv = [](float a, float b) { return b > a ? 1023.999f / (b - a) : 0.0f; };
        minv = make_float3(inv(lo[0], hi[0]), inv(lo[1], hi[1]), inv(lo[2], hi[2]));
    }
    const float slack = (float)(ext * 4e-6 + 1e-6);
    const int B = 256;
    k_lbvh_keys<<<(n + B - 1) / B, B, 0, stream>>>(d_tris, t0, n, mlo, minv, s.keys, s.ids);
    size_t cub_bytes = s.cub_bytes;
    const cudaError_t e = cub::DeviceRadixSort::SortPairs(s.cub_tmp, cub_bytes, (const unsigned*)s.keys, s.keys2, (const int*)s.ids, s.ids2, n, 0, 30, stream);
    if (e != cudaSuccess) return e;
    k_lbvh_leaves<<<(L + B - 1) / B, B, 0, stream>>>(d_tris, s.keys2, s.ids2, n, L, slack, leaf_base, btris, btid, s.leaf_box, s.leaf_key);
    return buildTreeDevice(s, L, n, leaf_base, nullptr, node_base, out_nodes, stream, nnodes, depth, why);
}

int updateInstancesDevice(InstanceTrace* inst, InstanceShade* shade, int nmodels, const PtapModel* staged, int first, int count, BvhNode* nodes,
                          int node_base, int ninst, char* scratch, size_t scratch_bytes, cudaStream_t stream, TlasBuild* out, std::string* why)
{
    const int B = 256, g = (nmodels + B - 1) / B;
    *out = TlasBuild{};
    if (!nodes) {
        k_update_instances<<<g, B, 0, stream>>>(inst, shade, nmodels, staged, first, count, nullptr, nullptr, nullptr, nullptr);
        return cudaGetLastError();
    }
    if (instanceUpdateScratchBytes(nmodels) > scratch_bytes) return cudaErrorMemoryAllocation;
    char* p = scratch;
    const BuildScratch s = carveBuild(p, nmodels, nmodels, 32);
    Box6* box = carve<Box6>(p, nmodels);
    double* trans = carve<double>(p, nmodels);
    InstanceReduce* red = carve<InstanceReduce>(p, 1);
    InstanceReduce init;
    init.max_scale = init.max_pad = 0ull;
    { const double one = 1.0; memcpy(&init.max_trans, &one, sizeof one); }
    init.first_bad = INT_MAX;
    for (int k = 0; k < 3; ++k) { init.clo[k] = ~0u; init.chi[k] = 0u; }
    cudaError_t e = cudaMemcpyAsync(red, &init, sizeof init, cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;
    k_update_instances<<<g, B, 0, stream>>>(inst, shade, nmodels, staged, first, count, nodes, box, trans, red);
    k_instance_keys<<<g, B, 0, stream>>>(box, trans, nmodels, red, s.keys, s.ids);
    size_t cub_bytes = s.cub_bytes;
    e = cub::DeviceRadixSort::SortPairs(s.cub_tmp, cub_bytes, (const unsigned*)s.keys, s.keys2, (const int*)s.ids, s.ids2, nmodels, 0, 32, stream);
    if (e != cudaSuccess) return e;
    InstanceReduce r;
    e = cudaMemcpyAsync(&r, red, sizeof r, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return e;
    memcpy(&out->max_scale, &r.max_scale, sizeof(double)); memcpy(&out->max_pad, &r.max_pad, sizeof(double)); memcpy(&out->max_trans, &r.max_trans, sizeof(double));
    out->consistent = r.first_bad == INT_MAX;
    out->root = -1;
    if (ninst == 0) return cudaSuccess;
    k_instance_leaves<<<(ninst + B - 1) / B, B, 0, stream>>>(box, s.keys2, s.ids2, ninst, s.leaf_box, s.leaf_key);
    e = (cudaError_t)buildTreeDevice(s, ninst, ninst, 0, s.ids2, node_base, nodes + node_base, stream, &out->nnodes, &out->depth, why);
    if (e == cudaSuccess) out->root = node_base;
    return e;
}

}  // namespace ptap
