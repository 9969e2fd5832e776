// bvh_build.cpp - binned-SAH BVH2 builder, one BLAS per mesh (instances share it, as they share the reference's grid).
//
// Leaf bounds are CONSERVATIVE FOR THE REFERENCE'S PREDICATE, not for the exact triangle: computeRayTriangleIntersection
// (Renderer.cpp:188-201) accepts u,v >= -0.005, u+v <= 1.005 in barycentric units, i.e. hits up to 0.5 % of an edge
// length outside the triangle.  Each triangle is therefore bounded by its fattened version with corners at
// (u,v) = (-e,-e), (1+2e,-e), (-e,1+2e), e slightly above 0.005, plus a floating-point slack proportional to the
// mesh extent.  With exact bounds a BVH silently drops the hits the reference finds in the tolerance band
// (SURVEY.md 0.5 third hazard / hard part 2).
#include "bvh_build.h"
#include "host_math.h"

#include <algorithm>
#include <cfloat>
#include <functional>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <thread>

namespace ptap {

namespace {

constexpr int kBins = 16;
int gMaxLeaf = 4;                    // SAH may stop earlier; hard cap 8 by the link encoding (PTAP_BVH_LEAF, tuning only)
float gNodeCost = 1.0f;              // cost of one inner node in units of one triangle test (PTAP_BVH_CI, tuning only)
constexpr double kBandEps = 0.0056;  // > EPSILON (Config.h:4) to absorb rounding of u, v

struct Box {
    float lo[3], hi[3];
    void reset() { for (int k = 0; k < 3; ++k) { lo[k] = FLT_MAX; hi[k] = -FLT_MAX; } }
    void grow(const Box& b) { for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], b.lo[k]); hi[k] = std::max(hi[k], b.hi[k]); } }
    void grow(const float* p) { for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], p[k]); hi[k] = std::max(hi[k], p[k]); } }
    float area() const
    {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        return dx < 0 ? 0.f : 2.f * (dx * dy + dy * dz + dz * dx);
    }
};

struct Prim { Box box; float c[3]; int id; };

// A subtree the top-level (serial) pass leaves to a worker thread: primitives [begin, end), to be linked at child `slot` of `parent`.
struct Task { int begin, end, parent, slot, depth; };

struct Builder {
    std::vector<Prim>& prims;
    std::vector<Bvh2Node>& nodes;
    std::vector<int>& order;      // leaf-order list of prim ids (local to the mesh), appended
    int leaf_base;                // leaf-order offset of this mesh in the global arrays
    int max_depth = 0;
    std::vector<Task>* tasks = nullptr;   // non-null: the top pass; subtrees of at most task_size primitives are deferred
    int task_size = 0;
    static constexpr int kDeferred = 0x7fffffff;   // placeholder link of a deferred subtree

    static int leafLink(int first, int count) { return ~((first << 3) | (count - 1)); }

    // returns link (node index >= 0 or leaf < 0) and the bounds of the subtree
    int build(int begin, int end, Box& bounds, int depth)
    {
        max_depth = std::max(max_depth, depth);
        bounds.reset();
        Box cb; cb.reset();
        for (int i = begin; i < end; ++i) { bounds.grow(prims[i].box); cb.grow(prims[i].c); }
        const int n = end - begin;
        if (tasks && n <= task_size && depth > 0) return kDeferred;      // bounds are set; the caller records the task
        auto makeLeaf = [&]() {
            int first = leaf_base + (int)order.size();
            for (int i = begin; i < end; ++i) order.push_back(prims[i].id);
            return leafLink(first, n);
        };
        if (n <= 1) return makeLeaf();
        // binned SAH over the largest centroid axis first, then the others if it fails
        int best_axis = -1, best_bin = -1; float best_cost = FLT_MAX;
        for (int axis = 0; axis < 3; ++axis) {
            const float lo = cb.lo[axis], ext = cb.hi[axis] - cb.lo[axis];
            if (!(ext > 0.f)) continue;
            Box bb[kBins]; int cnt[kBins];
            for (int b = 0; b < kBins; ++b) { bb[b].reset(); cnt[b] = 0; }
            const float scale = kBins / ext;
            for (int i = begin; i < end; ++i) {
                int b = std::min(kBins - 1, std::max(0, (int)((prims[i].c[axis] - lo) * scale)));
                bb[b].grow(prims[i].box); cnt[b]++;
            }
            float rightArea[kBins]; int rightCnt[kBins];
            Box acc; acc.reset(); int c = 0;
            for (int b = kBins - 1; b > 0; --b) { acc.grow(bb[b]); c += cnt[b]; rightArea[b] = acc.area(); rightCnt[b] = c; }
            acc.reset(); c = 0;
            for (int b = 0; b < kBins - 1; ++b) {
                acc.grow(bb[b]); c += cnt[b];
                if (c == 0 || rightCnt[b + 1] == 0) continue;
                float cost = acc.area() * c + rightArea[b + 1] * rightCnt[b + 1];
                if (cost < best_cost) { best_cost = cost; best_axis = axis; best_bin = b; }
            }
        }
        const float leaf_cost = bounds.area() * n;
        if (n <= gMaxLeaf && (best_axis < 0 || best_cost + bounds.area() * gNodeCost >= leaf_cost)) return makeLeaf();
        int mid;
        if (best_axis < 0) {
            if (n <= 8) return makeLeaf();
            mid = begin + n / 2;         // identical centroids: split by count
        } else {
            const float lo = cb.lo[best_axis], scale = kBins / (cb.hi[best_axis] - cb.lo[best_axis]);
            auto it = std::partition(prims.begin() + begin, prims.begin() + end, [&](const Prim& p) {
                int b = std::min(kBins - 1, std::max(0, (int)((p.c[best_axis] - lo) * scale)));
                return b <= best_bin;
            });
            mid = (int)(it - prims.begin());
            if (mid == begin || mid == end) mid = begin + n / 2;
        }
        const int me = (int)nodes.size();
        nodes.emplace_back();
        Box b0, b1;
        const int l0 = build(begin, mid, b0, depth + 1);
        if (l0 == kDeferred) tasks->push_back(Task{begin, mid, me, 0, depth + 1});
        const int l1 = build(mid, end, b1, depth + 1);
        if (l1 == kDeferred) tasks->push_back(Task{mid, end, me, 1, depth + 1});
        Bvh2Node& nd = nodes[me];
        nd.xy0 = make_float4(b0.lo[0], b0.hi[0], b0.lo[1], b0.hi[1]);
        nd.xy1 = make_float4(b1.lo[0], b1.hi[0], b1.lo[1], b1.hi[1]);
        nd.z01 = make_float4(b0.lo[2], b0.hi[2], b1.lo[2], b1.hi[2]);
        nd.link = make_int4(l0, l1, 0, 0);
        return me;
    }
};

}  // namespace

void encodeNode(BvhNode& nd, const ChildBox boxes[4], unsigned used)
{
    double lo[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, mag = 0.0;
    for (int c = 0; c < 4; ++c) {
        if (!(used >> c & 1)) continue;
        for (int k = 0; k < 3; ++k) {
            lo[k] = std::min(lo[k], (double)boxes[c].lo[k]);
            mag = std::max(mag, std::max(std::fabs((double)boxes[c].lo[k]), std::fabs((double)boxes[c].hi[k])));
        }
    }
    if (!used) { for (int k = 0; k < 3; ++k) lo[k] = 0.0; }
    // Margin for the traversal's own arithmetic: it evaluates (p - o) * inv and one FMA per plane in binary32, which perturbs a plane by
    // a few 2^-24 of the coordinates involved; 2^-20 of the largest coordinate of the node covers it many times over.
    const double margin = std::ldexp(mag, -20) + 1e-30;
    const float p[3] = {std::nextafter((float)(lo[0] - margin), -FLT_MAX), std::nextafter((float)(lo[1] - margin), -FLT_MAX), std::nextafter((float)(lo[2] - margin), -FLT_MAX)};
    nd.px = p[0]; nd.py = p[1]; nd.pz = p[2]; nd.pad = 0;
    for (int c = 0; c < 4; ++c)
        for (int k = 0; k < 3; ++k) {
            if (used >> c & 1) {
                // rounded outward: p + offset (in real arithmetic) lies beyond the builder's plane by at least the margin
                nd.planes[k][0][c] = std::nextafter((float)((double)boxes[c].lo[k] - margin - (double)p[k]), -FLT_MAX);
                nd.planes[k][1][c] = std::nextafter((float)((double)boxes[c].hi[k] + margin - (double)p[k]), FLT_MAX);
            } else { nd.planes[k][0][c] = 1e15f; nd.planes[k][1][c] = -1e15f; }       // inverted: near > far on every axis, never entered
        }
}

long long validateBvh(const BvhNode* nodes, int nnodes, int root, int nleafprims, const std::function<ChildBox(int)>& prim_box, int* depth)
{
    // A ray that must reach a primitive has to enter EVERY child box on the path from the root, so each primitive's box is checked against
    // the intersection of all decoded boxes above it.
    long long bad = 0;
    struct Item { int node, depth; double lo[3], hi[3]; };
    std::vector<Item> todo;
    Item r{}; r.node = root; r.depth = 1;
    for (int k = 0; k < 3; ++k) { r.lo[k] = -DBL_MAX; r.hi[k] = DBL_MAX; }
    todo.push_back(r);
    std::vector<char> seen(std::max(nnodes, 0), 0);
    int maxd = 0;
    while (!todo.empty()) {
        const Item it = todo.back(); todo.pop_back();
        if (it.node < 0 || it.node >= nnodes || seen[it.node]) { ++bad; continue; }
        seen[it.node] = 1;
        maxd = std::max(maxd, it.depth);
        const BvhNode& nd = nodes[it.node];
        for (int c = 0; c < 4; ++c) {
            if (!slotUsed(nd, c)) continue;
            double lo[3], hi[3];
            decodeChild(nd, c, lo, hi);
            for (int k = 0; k < 3; ++k) { lo[k] = std::max(lo[k], it.lo[k]); hi[k] = std::min(hi[k], it.hi[k]); }
            const int l = nd.link[c];
            if (l >= 0) {
                Item ch{}; ch.node = l; ch.depth = it.depth + 1;
                for (int k = 0; k < 3; ++k) { ch.lo[k] = lo[k]; ch.hi[k] = hi[k]; }
                todo.push_back(ch);
            } else {
                const int code = ~l, first = code >> 3, cnt = (code & 7) + 1;
                if (code >= 0x20000000) { ++bad; continue; }
                for (int j = 0; j < cnt; ++j) {
                    const int pos = first + j;
                    if (pos < 0 || pos >= nleafprims) { ++bad; continue; }
                    const ChildBox pb = prim_box(pos);
                    for (int k = 0; k < 3; ++k) if (!(lo[k] <= (double)pb.lo[k] && hi[k] >= (double)pb.hi[k])) ++bad;
                }
            }
        }
    }
    if (depth) *depth = maxd;
    return bad;
}

int collapseBvh2(const Bvh2Node* n2, int root2, std::vector<BvhNode>& out, int base, int depth, int& max_depth)
{
    struct Child { float lo[3], hi[3]; int link; };
    auto childrenOf = [&](int n, Child* dst) {
        const Bvh2Node& nd = n2[n];
        dst[0] = Child{{nd.xy0.x, nd.xy0.z, nd.z01.x}, {nd.xy0.y, nd.xy0.w, nd.z01.y}, nd.link.x};
        if (nd.link.x == nd.link.y) return 1;
        dst[1] = Child{{nd.xy1.x, nd.xy1.z, nd.z01.z}, {nd.xy1.y, nd.xy1.w, nd.z01.w}, nd.link.y};
        return 2;
    };
    max_depth = std::max(max_depth, depth);
    Child ch[5];
    int n = childrenOf(root2, ch);
    while (n < 4) {
        int best = -1; float best_area = -1.f;
        for (int i = 0; i < n; ++i) {
            if (ch[i].link < 0) continue;
            Box bx; for (int k = 0; k < 3; ++k) { bx.lo[k] = ch[i].lo[k]; bx.hi[k] = ch[i].hi[k]; }
            const float a = bx.area();
            if (a > best_area) { best_area = a; best = i; }
        }
        if (best < 0) break;
        Child two[2];
        const int m = childrenOf(ch[best].link, two);
        ch[best] = two[0];
        if (m == 2) ch[n++] = two[1];
    }
    const int me = (int)out.size();
    out.emplace_back();
    int links[4];
    for (int i = 0; i < n; ++i) links[i] = ch[i].link >= 0 ? collapseBvh2(n2, ch[i].link, out, base, depth + 1, max_depth) : ch[i].link;
    BvhNode& nd = out[me];
    memset(&nd, 0, sizeof nd);
    ChildBox boxes[4];
    unsigned used = 0u;
    for (int i = 0; i < 4; ++i) {
        if (i < n) {
            for (int k = 0; k < 3; ++k) { boxes[i].lo[k] = ch[i].lo[k]; boxes[i].hi[k] = ch[i].hi[k]; }
            used |= 1u << i;
            nd.link[i] = links[i];
        } else nd.link[i] = links[0];
    }
    encodeNode(nd, boxes, used);
    return base + me;
}

void makeTriRecs(const PtapVertex* vertices, const PtapTriangle* triangles, int ntris, TriRec* out)
{
    for (int t = 0; t < ntris; ++t) {
        const PtapVertex& a = vertices[triangles[t].v[0]];
        const PtapVertex& b = vertices[triangles[t].v[1]];
        const PtapVertex& c = vertices[triangles[t].v[2]];
        const hm::V3 v0 = hm::v3(a.position);
        const hm::V3 e1 = hm::sub(hm::v3(b.position), v0), e2 = hm::sub(hm::v3(c.position), v0);     // Renderer.cpp:183-184
        const hm::V3 n = hm::normalize(hm::scale(hm::add(hm::add(hm::v3(a.normal), hm::v3(b.normal)), hm::v3(c.normal)), 1 / 3.0f));   // :203
        out[t].v0 = make_float4(v0.x, v0.y, v0.z, n.x);
        out[t].e1 = make_float4(e1.x, e1.y, e1.z, n.y);
        out[t].e2 = make_float4(e2.x, e2.y, e2.z, n.z);
    }
}

void buildSceneBvh(const TriRec* tris, int ntris, const PtapMesh* meshes, int nmeshes, BvhBuildResult& out)
{
    out.nodes.clear(); out.tri_id.clear();
    if (const char* e = getenv("PTAP_BVH_LEAF")) gMaxLeaf = std::min(8, std::max(1, atoi(e)));
    if (const char* e = getenv("PTAP_BVH_CI")) gNodeCost = (float)atof(e);
    out.mesh_root.assign(nmeshes, -1);
    out.max_depth = 0;
    for (int mi = 0; mi < nmeshes; ++mi) {
        const PtapMesh& mesh = meshes[mi];
        const int t0 = mesh.t_start, t1 = mesh.t_end;
        if (t1 <= t0 || t0 < 0 || t1 > ntris) continue;
        // extent of the mesh for the floating-point slack
        double ext = 0;
        for (int t = t0; t < t1; ++t) {
            const TriRec& r = tris[t];
            const double v[3][3] = {{r.v0.x, r.v0.y, r.v0.z}, {(double)r.v0.x + r.e1.x, (double)r.v0.y + r.e1.y, (double)r.v0.z + r.e1.z},
                                    {(double)r.v0.x + r.e2.x, (double)r.v0.y + r.e2.y, (double)r.v0.z + r.e2.z}};
            for (auto& p : v) for (double c : p) ext = std::max(ext, std::fabs(c));
        }
        const float slack = (float)(ext * 4e-6 + 1e-6);
        std::vector<Prim> prims((size_t)(t1 - t0));
        for (int t = t0; t < t1; ++t) {
            const TriRec& r = tris[t];
            Prim& p = prims[t - t0];
            p.id = t; p.box.reset();
            const double uv[3][2] = {{-kBandEps, -kBandEps}, {1 + 2 * kBandEps, -kBandEps}, {-kBandEps, 1 + 2 * kBandEps}};
            double cx = 0, cy = 0, cz = 0;
            for (auto& c : uv) {
                const double x = r.v0.x + c[0] * r.e1.x + c[1] * r.e2.x, y = r.v0.y + c[0] * r.e1.y + c[1] * r.e2.y, z = r.v0.z + c[0] * r.e1.z + c[1] * r.e2.z;
                const float lo[3] = {std::nextafter((float)x, -FLT_MAX) - slack, std::nextafter((float)y, -FLT_MAX) - slack, std::nextafter((float)z, -FLT_MAX) - slack};
                const float hi[3] = {std::nextafter((float)x, FLT_MAX) + slack, std::nextafter((float)y, FLT_MAX) + slack, std::nextafter((float)z, FLT_MAX) + slack};
                p.box.grow(lo); p.box.grow(hi);
                cx += x; cy += y; cz += z;
            }
            p.c[0] = (float)(cx / 3); p.c[1] = (float)(cy / 3); p.c[2] = (float)(cz / 3);
        }
        std::vector<int> order; order.reserve(prims.size());
        std::vector<Bvh2Node> n2;
        n2.reserve(prims.size());
        const int leaf_base = (int)out.tri_id.size();
        Builder b{prims, n2, order, leaf_base};
        Box bounds;
        // Large meshes: the top of the tree is built here, subtrees of <= n/64 primitives on worker threads into private arrays, which are
        // then appended (node indices and leaf positions shifted).  The tree is the one the serial build produces; only node numbering differs.
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        std::vector<Task> tasks;
        if (prims.size() >= 65536 && hw > 1) { b.tasks = &tasks; b.task_size = std::max<int>(1024, (int)prims.size() / 64); }
        const int link = b.build(0, (int)prims.size(), bounds, 0);
        if (!tasks.empty()) {
            struct Sub { std::vector<Bvh2Node> nodes; std::vector<int> order; int link = 0, depth = 0; };
            std::vector<Sub> subs(tasks.size());
            std::atomic<size_t> next{0};
            auto work = [&]() {
                for (size_t k; (k = next.fetch_add(1)) < tasks.size();) {
                    Builder sb{prims, subs[k].nodes, subs[k].order, 0};
                    Box bb;
                    subs[k].link = sb.build(tasks[k].begin, tasks[k].end, bb, tasks[k].depth);
                    subs[k].depth = sb.max_depth;
                }
            };
            std::vector<std::thread> pool;
            for (unsigned t = 0; t + 1 < std::min<unsigned>(hw, (unsigned)tasks.size()); ++t) pool.emplace_back(work);
            work();
            for (std::thread& t : pool) t.join();
            for (size_t k = 0; k < tasks.size(); ++k) {          // tasks were recorded in depth-first order: so is the leaf order
                const int node_off = (int)n2.size(), leaf_off = leaf_base + (int)order.size();
                auto shift = [&](int l) { return l >= 0 ? l + node_off : ~(~l + (leaf_off << 3)); };
                for (Bvh2Node nd : subs[k].nodes) { nd.link.x = shift(nd.link.x); nd.link.y = shift(nd.link.y); n2.push_back(nd); }
                order.insert(order.end(), subs[k].order.begin(), subs[k].order.end());
                const int l = shift(subs[k].link);
                if (tasks[k].slot == 0) n2[tasks[k].parent].link.x = l; else n2[tasks[k].parent].link.y = l;
                b.max_depth = std::max(b.max_depth, subs[k].depth);
            }
        }
        if (link < 0) {
            // the whole mesh fits one leaf: a root with a single child
            Bvh2Node nd;
            nd.xy0 = make_float4(bounds.lo[0], bounds.hi[0], bounds.lo[1], bounds.hi[1]);
            nd.xy1 = nd.xy0;
            nd.z01 = make_float4(bounds.lo[2], bounds.hi[2], bounds.lo[2], bounds.hi[2]);
            nd.link = make_int4(link, link, 0, 0);
            n2.push_back(nd);
        }
        int depth4 = 0;
        out.mesh_root[mi] = collapseBvh2(n2.data(), link < 0 ? (int)n2.size() - 1 : link, out.nodes, 0, 1, depth4);
        out.max_depth = std::max(out.max_depth, depth4);
        for (int id : order) out.tri_id.push_back(id);
    }
}

}  // namespace ptap
