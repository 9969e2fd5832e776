// bvh_build.h - host builder of the two-level BVH (PTAP_ACCEL_BVH).
// New design: the reference has only the fixed 25^3 grid of Scene::addMeshesToGrid (Scene.cpp:318-396).
#pragma once
#include <functional>
#include <vector>

#include "../../include/ptap.h"
#include "device_types.h"

namespace ptap {

struct BvhBuildResult {
    std::vector<BvhNode> nodes;      // all BLASes back to back (4-wide nodes)
    std::vector<int> tri_id;         // leaf-order position -> global triangle id
    std::vector<int> mesh_root;      // per mesh: index of its BLAS root node, -1 if the mesh has no triangles
    int max_depth = 0;
};

struct ChildBox { float lo[3], hi[3]; };
// Fills the boxes of node `nd` from up to four (slot, box) pairs: local origin, binary32 offsets rounded outward after a margin that
// covers the traversal's own arithmetic; unused slots get an inverted box.  `boxes[c]` is read only when bit c of `used` is set.
void encodeNode(BvhNode& nd, const ChildBox boxes[4], unsigned used);
// Decoded box of slot c (what the traversal kernel tests), in double: p + offset.  Host and device (instance_math.h).
__host__ __device__ inline void decodeChild(const BvhNode& nd, int c, double lo[3], double hi[3])
{
    const double p[3] = {nd.px, nd.py, nd.pz};
    for (int k = 0; k < 3; ++k) { lo[k] = p[k] + (double)nd.planes[k][0][c]; hi[k] = p[k] + (double)nd.planes[k][1][c]; }
}
__host__ __device__ inline bool slotUsed(const BvhNode& nd, int c) { return nd.planes[0][0][c] <= nd.planes[0][1][c]; }

// Collapses the binary subtree rooted at node `root2` of `n2` into 4-wide nodes appended to `out` (absolute index = base + position in
// `out`): a child is replaced by its own two children, largest box first, until the node has four.  Returns the new root's index.
int collapseBvh2(const Bvh2Node* n2, int root2, std::vector<BvhNode>& out, int base, int depth, int& max_depth);

// tris: global triangle table (v0, e1, e2 in .xyz).  One BLAS per mesh over [t_start, t_end).
void buildSceneBvh(const TriRec* tris, int ntris, const PtapMesh* meshes, int nmeshes, BvhBuildResult& out);
// (v0, e1 = v1 - v0, e2 = v2 - v0, flat normal in .w lanes) with the reference's arithmetic (Renderer.cpp:183-184, 203)
void makeTriRecs(const PtapVertex* vertices, const PtapTriangle* triangles, int ntris, TriRec* out);
// Walks the nodes from `root` and returns the number of violations of the structure's contract: every primitive's box (`prim_box(leaf
// position)`) must lie inside EVERY decoded child box on its path from the root; links in range, leaf counts 1..8, no node reachable twice.
long long validateBvh(const BvhNode* nodes, int nnodes, int root, int nleafprims, const std::function<ChildBox(int)>& prim_box, int* depth);

}  // namespace ptap
