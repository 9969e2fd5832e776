// kernels.cuh - launch wrappers of the wavefront kernels (one translation unit per kernel family).
#pragma once
#include <string>

#include "device_types.h"
#include "exact_math.cuh"
#include "../../include/ptap.h"

namespace ptap {

#ifndef PTAP_TRACE_BLOCK
#define PTAP_TRACE_BLOCK 128
#endif
constexpr int kTraceBlock = PTAP_TRACE_BLOCK;
constexpr int kShadeBlock = 256;     // slots a CTA of k_shade regroups by material class and shades
constexpr int kShadeTile = 32;       // one compaction tile = one warp = 32 consecutive slots
constexpr int kScanBlock = 256, kScanSlots = 2048, kScanTiles = kScanSlots / kShadeTile;   // k_scan: slots per CTA, tiles per CTA
constexpr int kGenBlock = 256;
constexpr int kMaxLanes = 8, kDefaultLanes = 4, kSmallFrameLanes = 8;   // wavefronts in flight per context (api.cu: multi-lane rendering)
constexpr int kTraceBatch = 32;      // rays a warp takes from the work-stealing cursor per atomic
constexpr int kVoteTri = 8, kVoteInst = 6, kVoteRefill = 8;   // state-machine thresholds of k_trace_bvh (trace_bvh.cu)
constexpr int kVoteGrid = 5;         // same for k_trace_grid (one threshold for all of its states)
constexpr unsigned kFull = 0xffffffffu;   // every lane of a warp

__device__ __forceinline__ unsigned long long globalTimerNs()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// A warp's share of a work-stealing cursor: the items [w_next, w_end) of the batch it took last.  Every lane of the warp calls both steps.
struct WarpBatch {
    int w_next = 0, w_end = 0;
    bool exhausted = false;                      // the cursor has passed n: nothing left to fetch
    // the warp's batch is used up: take the next `batch` items (one atomic per warp)
    __device__ __forceinline__ void fetch(unsigned int* cursor, int batch, int n)
    {
        if (w_next >= w_end && !exhausted) {
            unsigned b = 0;
            if ((threadIdx.x & 31) == 0) b = atomicAdd(cursor, (unsigned)batch);
            b = __shfl_sync(kFull, b, 0);
            if (b >= (unsigned)n) { exhausted = true; w_next = w_end = n; }
            else { w_next = (int)b; w_end = min((int)b + batch, n); }
        }
    }
    // the lanes of `free` (ballot of `mine`) take the next items in lane order: true when this lane gets one (`item`); then every lane calls
    // advance() past the items taken
    __device__ __forceinline__ bool claim(unsigned free, bool mine, int& item) const
    {
        const int rank = __popc(free & ((1u << (threadIdx.x & 31)) - 1u));
        item = w_next + rank;
        return mine && rank < w_end - w_next;
    }
    __device__ __forceinline__ void advance(unsigned free) { w_next += min(__popc(free), w_end - w_next); }
};

// counting builds: the warp's sum of v added to *total by lane 0
__device__ __forceinline__ void warpTotalAdd(unsigned long long* total, unsigned long long v)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
    if ((threadIdx.x & 31) == 0) atomicAdd(total, v);
}

// World distance of the hit at model-space parameter t of model `im` along the stored ray (bo, bd), exactly as the reference computes
// it (Renderer.cpp:381-382 ray set-up, :388-391 conversion).  k_trace_bvh only carries an approximate distance while traversing
// (it needs the exact one just to break near-ties); the consumers of a hit record (k_shade, k_resolve_hits) evaluate this function,
// at full SIMT efficiency, instead of the traversal doing it with a handful of active lanes.
__device__ __forceinline__ float exactHitDistance(const SceneDev& sc, V3 bo, V3 bd, int im, float t)
{
    const InstanceTrace* __restrict__ inst = &sc.inst[im];
    const float4 w0 = ldg4(&inst->w2m[0]), w1 = ldg4(&inst->w2m[1]), w2 = ldg4(&inst->w2m[2]);
    const V3 ro = xmat4(w0, w1, w2, bo, 1.0f);                                   // Renderer.cpp:381
    const V3 rd = xnormalize(xmat4(w0, w1, w2, bd, 0.0f));                       // Renderer.cpp:382
    const V3 nd = xnormalize(rd);                                                // Renderer.cpp:388
    const V3 pm = xadd(ro, xscale(nd, t));                                       // Renderer.cpp:389
    const V3 pw = xmat4(ldg4(&inst->m2w[0]), ldg4(&inst->m2w[1]), ldg4(&inst->m2w[2]), pm, 1.0f);   // :390
    return xlength(xsub(pw, bo));                                                // Renderer.cpp:391
}

// closest hit, grid-compat (trace_grid.cu) and BVH (trace_bvh.cu).  n_fixed < 0: read the count from st->n_active[round].
// stamp (may be null): two 64-bit words that receive the earliest start and the latest end of the launch in %globaltimer nanoseconds
// (atomicMin / atomicMax by every CTA), so that bench.py can time the closest-hit kernel inside the real multi-lane schedule.
// list (may be null): walk only the slots list[0 .. st->n_walk[round]) - the last launch of PTAP_ACCEL_GRID_EMULATED.
void launchTraceGrid(const SceneDev& sc, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, bool count_totals,
                     FrameState* st, int round, int n_fixed, int grid, cudaStream_t stream, unsigned long long* stamp = nullptr, const int* list = nullptr);
// trace_emu.cu: the results of the grid walk (tier R0) through the BVH, in two launches: nearest model + all of the ray's hits in it,
// then the replay of the walk over those hits; slots the replay cannot confirm are appended to emu.list for launchTraceGrid(list)
void launchTraceEmu(const SceneDev& sc, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, bool count_totals,
                    FrameState* st, int round, int n_fixed, int grid, int grid_replay, int grid_full, cudaStream_t stream, unsigned long long* stamp, const EmuBuf& emu);
int traceEmuOccupancy();
// grid_device.cu: per-triangle voxel boxes of the grids on the device + the checks that make the emulation exact; *ok = 0 when some list is
// not what a box-shaped registration produces (the caller then keeps the walk).  grid_tri_range: 2 ints per grid (lowest / highest listed id).
int gridTriBoxes(const int2* cells, const int* refs, int ngrids, const int* grid_first_cell, int gx, int gy, int gz, int ntris, int2* tri_box,
                 int* grid_tri_range_host, int* ok, cudaStream_t stream);
int traceGridOccupancy();
void launchTraceBvh(const SceneDev& sc, const float4* O, const float4* D, float4* hit, float2* uv, int4* counts, bool count_totals,
                    FrameState* st, int round, int n_fixed, int grid, cudaStream_t stream, unsigned long long* stamp = nullptr);
int traceBvhOccupancy();
// the any-hit traversal of ptap_query_occluded over rays [0, n): L = D[i].w; records for launchResolveOccluded
void launchTraceBvhAny(const SceneDev& sc, const float4* O, const float4* D, float4* hit, FrameState* st, int n, int grid, cudaStream_t stream);

// bvh_device.cu
size_t deviceBvhScratchBytes(int ntris);
int buildMeshBvhDevice(const TriRec* d_tris, int t0, int t1, const float* bb_min, const float* bb_max, int node_base, BvhNode* out_nodes, int leaf_base,
                       LeafTri* btris, int* btid, char* scratch, size_t scratch_bytes, cudaStream_t stream, int* nnodes, int* depth,
                       std::string* why);
// ptap_update_models: models [first, first + count) take the staged records (device copies) in their InstanceTrace (grid fields kept) and
// InstanceShade.  With a BVH (nodes non-null), the TLAS over the instances' world boxes is then built at nodes + node_base (ninst = models
// with triangles) and the scene-constant terms are reduced (TlasBuild), all from the same per-instance function as finishBvh.
struct TlasBuild {
    int root = -1, nnodes = 0, depth = 0;       // root node index (-1: no instance has triangles), 4-wide nodes and levels of the TLAS
    double max_scale = 0.0, max_pad = 0.0, max_trans = 1.0;
    bool consistent = true;
};
size_t instanceUpdateScratchBytes(int nmodels);
int updateInstancesDevice(InstanceTrace* inst, InstanceShade* shade, int nmodels, const PtapModel* staged, int first, int count, BvhNode* nodes,
                          int node_base, int ninst, char* scratch, size_t scratch_bytes, cudaStream_t stream, TlasBuild* out, std::string* why);

// grid_device.cu: Scene::addMeshesToGrid on the device, one mesh's grid at a time
int gridDeviceCount(const float* d_pos, int t0, int n, const float bb_min[3], const float width[3], const int gd[3], int* d_count, int* d_offset,
                    long long* d_sum, void* d_tmp, size_t tmp_bytes, cudaStream_t stream, long long* npairs);
int gridDeviceFill(const float* d_pos, int t0, int n, const float bb_min[3], const float width[3], const int gd[3], const int* d_offset, int npairs,
                   int* d_keys, int* d_vals, int* d_keys2, void* d_tmp, size_t tmp_bytes, int ref_base, int* d_refs, int2* d_cells, cudaStream_t stream);
size_t gridDeviceTempBytes(int ntris, long long npairs);

// wavefront.cu
void launchGenerate(const WaveDev& wv, int iter /* the iteration being generated: seeds the camera jitter */, int grid, cudaStream_t stream);
void launchScan(const SceneDev& sc, const WaveDev& wv, int round, const float4* hit, int remaining, int n_fixed, cudaStream_t stream);
void launchShade(const SceneDev& sc, const WaveDev& wv, int round, int in_buf, const float4* hit, int remaining, int n_fixed,
                 int iter_fixed, int* slot_pos, int grid, cudaStream_t stream);
int shadeOccupancy();
void launchResolveHits(const SceneDev& sc, const float4* O, const float4* D, const float4* hit, const float2* uv, int n, PtapHit* out, cudaStream_t stream);
// occluded[i] = closest hit of ray i nearer than L = D[i].w, from closest-hit records or any-hit ones (model kAnyOccluded: occluded)
void launchResolveOccluded(const SceneDev& sc, const float4* O, const float4* D, const float4* hit, int n, uint8_t* occluded, cudaStream_t stream);
void launchSetIter(FrameState* st, int iter, cudaStream_t stream);
void launchFilmAdd(float* film, const float* add, size_t n, cudaStream_t stream);
void launchResolveBmp(const float* film, size_t nvalues, float div, unsigned char* out, cudaStream_t stream);
void launchResolveBox(const float* film, int W, int H, int sx, int sy, float* out, cudaStream_t stream);
void launchExtractNormals(const TriRec* tris, int n, float4* normals, cudaStream_t stream);
void launchGatherTris(const TriRec* tris, const int* tri_id, int n, LeafTri* out, cudaStream_t stream);

}  // namespace ptap
