// device_types.h - layouts of everything libptap keeps in HBM (see DESIGN.md "Data layout").
// All records are multiples of 16 B and fetched with 16-byte vector loads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ptap {

constexpr float kEpsilon = 0.005f;          // Config.h:4
constexpr float kFloatMax = 9999999.0f;     // Config.h:5
constexpr float kFloatMin = -9999990.0f;    // Config.h:6
constexpr int kAnyOccluded = -2;            // model field of an any-hit record whose ray retired as occluded (k_trace_bvh<.., ANY>)
constexpr int kMaxDepth = 16;               // rounds per iteration the context reserves state for
constexpr int kBigHits = 108;               // k_emu_full: further hits of a (ray, model) kept per thread in global memory (128 with the 20 in shared memory)
constexpr int kEmuHits = 8;                 // PTAP_ACCEL_GRID_EMULATED: hits of a (ray, model) that are kept for the replay of the walk
constexpr int kBvhStack = 160;              // traversal stack entries per ray (upload fails for deeper trees)

// Per-model record read by the closest-hit kernels: 9 x float4 = 144 B.
// Rows 0..2 of the reference's column-major mat4s (the w row is never used by
// transformPosition/transformDirection, utility.h:71-80).
struct InstanceTrace {
    float4 w2m[3];      // w2m[r] = (m[0][r], m[1][r], m[2][r], m[3][r]) of world_to_model
    float4 m2w[3];      // same for model_to_world
    float4 bb_min;      // mesh bbox min (through the grid's creating model, Renderer.cpp:245-249); .w = voxel width x
    float4 bb_max;      // mesh bbox max; .w = voxel width y
    float4 grid;        // .x = voxel width z, .y = bits(first voxel of the grid), .z = bits(BLAS root node), .w = bits(first BVH triangle)
};

// Per-model record read by the shade kernel: 4 x float4 = 64 B.
struct InstanceShade {
    float4 nm0;         // rows of transpose(inverse(mat3(model_to_world))) (utility.h:82-88): nm0 = (r0.x, r0.y, r0.z, color.r)
    float4 nm1;         // (r1.x, r1.y, r1.z, color.g)
    float4 nm2;         // (r2.x, r2.y, r2.z, color.b)
    int4 mat;           // .x = material type (Primitive.h:70-79)
};

// Triangle, model space: 3 x float4 = 48 B.  e1 = v1 - v0 and e2 = v2 - v0 are the same fp32 subtractions the
// reference performs per test (Renderer.cpp:183-184); the .w lanes carry the flat shading normal
// normalize((n0+n1+n2)*(1/3.0f)) (Renderer.cpp:203), read only by the shade kernel.
struct TriRec {
    float4 v0;          // (v0.xyz, n.x)
    float4 e1;          // (e1.xyz, n.y)
    float4 e2;          // (e2.xyz, n.z)
};

// Triangle in BVH leaf order, 64 B = two 32-byte vector loads (LDG.E.256 on sm_100): the three edge-form vectors of the TriRec and
// the GLOBAL triangle id, so that accepting a hit needs no second gather.
struct __align__(32) LeafTri {
    float v0[3], e1[3], e2[3];
    int id;
    int pad[6];
};

// Binary node of the builder (host only): both children's bounds and links.  The device format is the 4-wide BvhNode below.
struct Bvh2Node {
    float4 xy0;         // child0: (lo.x, hi.x, lo.y, hi.y)
    float4 xy1;         // child1: (lo.x, hi.x, lo.y, hi.y)
    float4 z01;         // (c0.lo.z, c0.hi.z, c1.lo.z, c1.hi.z)
    int4 link;          // (child0, child1, 0, 0); >= 0: node index, < 0: leaf; link.x == link.y: only child0 exists
};

// BVH4 node, 128 B = one L1 line: up to four children, their boxes as binary32 OFFSETS in a node-local frame, and their links.
//   plane = p + offset, every lower plane rounded down and every upper plane rounded up after an outward margin (bvh_build.cpp:
//   encodeNode), so a child box always CONTAINS the builder's box, which itself bounds the reference predicate's +-0.005 tolerance band:
//   the structure only decides which triangles are tested, the exact predicate decides hits.  The node-local frame is what makes a
//   one-FMA-per-plane slab test safe (trace_bvh.cu); the lower and upper planes of an axis sit 16 bytes apart so that the traversal
//   picks the near / far ones by address from the ray's direction signs.
// link >= 0: node index; link < 0: triangle leaf ~((first << 3) | (count - 1)) or (TLAS only) instance leaf ~(0x20000000 | model index).
// An unused slot holds an inverted box (lower offsets +1e15, upper offsets -1e15) that no ray interval enters.
struct __align__(32) BvhNode {
    float px, py, pz;           // node-local origin (just below the lower corner of the node)
    int pad;
    int link[4];
    float planes[3][2][4];      // [axis][0 = lower, 1 = upper][slot]
};
static_assert(sizeof(BvhNode) == 128, "BvhNode must be one 128-byte line");

// Device-resident frame state: lets a whole iteration run without a host round trip.
struct FrameState {
    int n_active[kMaxDepth + 2];        // rays entering round r
    unsigned int ticket[kMaxDepth + 2]; // tile tickets of the shade kernel, per round
    unsigned int fetch[kMaxDepth + 2];  // work-stealing cursors of the trace kernel, per round
    unsigned int n_replay[kMaxDepth + 2];      // PTAP_ACCEL_GRID_EMULATED: slots of the round whose replay did not confirm the closest hit (-> k_emu_full)
    unsigned int fetch_replay[kMaxDepth + 2];  // work-stealing cursors of k_emu_full
    unsigned int n_walk[kMaxDepth + 2];        // slots that only the grid walk itself can answer (-> k_trace_grid in list mode)
    unsigned int fetch_walk[kMaxDepth + 2];    // work-stealing cursors of that launch
    unsigned int fetch_emu[kMaxDepth + 2];     // work-stealing cursors of k_emu_tail
    unsigned int n_cont[kMaxDepth + 2];        // replays that k_emu_setup queued for k_emu_tail
    int iter_cur, iter_next;
    int cache_valid;                    // first-hit cache holds round-0 hits
    int pad;
    unsigned long long rays_traced;
    unsigned long long rays_walked;     // PTAP_ACCEL_GRID_EMULATED: rays handed to k_trace_grid in list mode
    unsigned long long rays_reemulated; // PTAP_ACCEL_GRID_EMULATED: rays handed to k_emu_full
    unsigned long long paths;
    unsigned long long count_nodes, count_tris, count_cells, count_refs;   // counting build only
};

struct SceneDev {
    const InstanceTrace* inst;
    const InstanceShade* shade;
    const TriRec* tris;         // indexed by GLOBAL triangle id (reference order)
    const float4* normals;      // flat shading normal per GLOBAL triangle id (copy of the TriRec .w lanes, 16-byte gather for k_shade)
    const int2* cells;          // grid voxels: (start, end) into refs
    const int* refs;            // global triangle ids
    const int2* tri_box;        // per GLOBAL triangle id: the box of voxels that list it, (lo, hi) packed x | y << 10 | z << 20, indices < 512 (trace_emu.cu)
    const BvhNode* nodes;       // all BLAS nodes, then the TLAS nodes
    const LeafTri* bvh_tris;    // triangles in BVH leaf order
    const int* bvh_tri_id;      // leaf-order position -> global triangle id (build-time input of k_gather_tris; the kernels read LeafTri::id)
    int nmodels;
    int gx, gy, gz;
    int tlas_root;              // node index of the TLAS root, -1 when no instance has triangles
    float tmin_world;           // lower end of the world-space ray interval: -(EPSILON band mapped to world units + box padding)
    int batch;                  // rays a warp takes from the work-stealing cursor per atomic (PTAP_BATCH)
    int shade_sort;             // k_shade regroups each block's slots by material class before shading (PTAP_SHADE_SORT=1; default off)
    int vote_grid;              // k_trace_grid: lanes that must wait in a state before its step runs (the most popular state always runs)
    int emu_refill;             // k_emu_tail: free lanes of a warp that trigger the loading of the next queued replays (PTAP_EMU_REFILL)
    int vote_tri, vote_inst, vote_refill;   // lanes that must wait in a state before the warp runs that state's step (PTAP_VOTE_*)
    float c_pad;                // slack of the pruning bound for the residual of model_to_world * world_to_model - I
    float tie;                  // two instances' winners whose approximate world distances differ by less than this relative slack are compared exactly
    float prune;                // relative slack of cross-instance pruning (1.0001), +inf when some model's matrices are not inverses
};

// PTAP_ACCEL_GRID_EMULATED (trace_emu.cu): what k_trace_emu hands to the replay kernels for every wavefront slot, their queue, and the lists
struct EmuBuf {
    int* n;                     // [slot] hits of the ray in its nearest model (> kEmuHits: not all kept - the walk answers that ray)
    int* id;                    // [hit][slot] their global triangle ids (stride slots per hit)
    float* t;                   // [hit][slot] their model-space t
    int* list;                  // slots that k_emu_full must answer (FrameState::n_replay of them)
    int* list2;                 // slots that k_trace_grid must answer (FrameState::n_walk of them)
    uint4* cont;                // queue of replays in progress, 5 x uint4 each (k_emu_setup -> k_emu_tail)
    uint4* big;                 // k_emu_full: kBigHits x uint4 per thread of its grid (one CTA per SM)
    int stride;
    int cont_cap;               // entries the queue holds
};

struct WaveDev {
    float4* O[2];               // (orig.xyz, bits(ipixel)) ping-pong
    float4* D[2];               // (dir.xyz, unused)
    float4* C[2];               // (throughput rgb, unused)
    float4* hit;                // (dist, bits(tri), bits(model), t_model) per slot; dist < 0: hit whose exact distance the consumer evaluates
    float4* hit_cache;          // round-0 hits (first-hit cache, Renderer.cpp:594-613)
    float2* uv;                 // parity entry only
    EmuBuf emu;                 // PTAP_ACCEL_GRID_EMULATED only (api.cu: ensureEmuBuffers), else null pointers
    float* film;                // W*H*3 running sum (Pixel, Primitive.h:145-148)
    float* contrib;             // multi-lane rendering: this iteration's sqrt(throughput) per pixel, added to the film in iteration order; else null
    unsigned long long* tile_status;   // k_scan look-back words: rounds x 2048-slot scan blocks
    int* tile_offset;           // survivors before each 32-slot tile of the current round (k_scan -> k_shade)
    unsigned* tile_ballot;      // survival bits of each 32-slot tile, in slot order (k_scan -> k_shade<SORT>)
    unsigned char* perm;        // per 256-slot shade block: regrouped position -> slot within the block (k_scan -> k_shade<SORT>)
    FrameState* st;
    int W, H, N, depth, ntiles, nscan;   // ntiles = ceil(N / 32), nscan = ceil(N / 2048)
    float step_x, step_y;
    float cam_o[3], cam_p[3];   // camera origin and lower-left corner of the image plane (Renderer.cpp:541-545: (0, 0, 920) and (-10, -4, 900))
    int jitter; unsigned jitter_seed;   // sub-pixel jitter per iteration (an extension; 0 = the reference's fixed pixel corners)
    int iter_stride;            // iterations between two consecutive iterations of this lane (= lanes in use)
};

}  // namespace ptap
