// grid_device.cu - Scene::addMeshesToGrid + computeVoxelIndex (Scene.cpp:293-396) on the GPU: the per-mesh uniform grids of the
// bit-compatible closest-hit path (PTAP_ACCEL_GRID_COMPAT) built by SORTING instead of the reference's vector-of-vectors push_back
// (SURVEY.md 8f row 2).  At 160^3 on a 1.3 M-triangle mesh the host build is the whole set-up cost of a "BVH vs grid" comparison.
//
//   1  k_grid_ranges  per triangle: the voxel range it covers, with the reference's own arithmetic - floor(abs(bbox.min - tri.{min,max}) /
//                     width) clamped to the grid (Scene.cpp:300-315), every operation an IEEE binary32 one - and the number of cells
//   2  sum of the counts in 64 bits, then their exclusive scan in 32 (cub)                    [library call, off the render path]
//   3  k_grid_pairs   per triangle: one (cell, triangle) pair per covered cell, written at the triangle's offset; triangles are
//                     processed in ascending order, so the pair list is ordered by triangle
//   4  stable radix sort of the pairs by cell (cub): inside a cell the triangles stay ascending, exactly the order the reference's
//                     per-voxel push_back produces (Scene.cpp:366-374)
//   5  k_grid_cells   cell c = [lower_bound(c), lower_bound(c + 1)) of the sorted keys
// The output (cells, reference list) is bit-identical to the host builder's (scene_host.cpp: buildGrids), which tests/test_host.py pins to
// the reference's own output.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "kernels.cuh"

namespace ptap {

namespace {

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// positions: 9 floats per triangle (v0, v1, v2 as the reference stores them: no edge form, the min / max must see the original vertices)
__device__ __forceinline__ void voxelRange(const float* __restrict__ p, const float bb_min[3], const float width[3], const int gd[3], int lo[3], int hi[3])
{
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float mn = kFloatMax, mx = kFloatMin;                      // BoundingBox(), Primitive.h:38-47
#pragma unroll
        for (int v = 0; v < 3; ++v) { const float x = p[3 * v + k]; mn = mn > x ? x : mn; mx = mx < x ? x : mx; }
        lo[k] = clampi(f2i_x86(floorf(xdiv(fabsf(xsub(bb_min[k], mn)), width[k]))), 0, gd[k] - 1);      // Scene.cpp:300-315
        hi[k] = clampi(f2i_x86(floorf(xdiv(fabsf(xsub(bb_min[k], mx)), width[k]))), 0, gd[k] - 1);
    }
}

struct GridParams { float bb_min[3], width[3]; int gd[3]; int t0, n; };

__global__ void k_grid_ranges(const float* __restrict__ pos, GridParams g, int* __restrict__ count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n) return;
    int lo[3], hi[3];
    voxelRange(pos + 9 * (size_t)i, g.bb_min, g.width, g.gd, lo, hi);
    count[i] = (hi[0] - lo[0] + 1) * (hi[1] - lo[1] + 1) * (hi[2] - lo[2] + 1);
}

__global__ void k_grid_pairs(const float* __restrict__ pos, GridParams g, const int* __restrict__ offset, int* __restrict__ keys, int* __restrict__ vals)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n) return;
    int lo[3], hi[3];
    voxelRange(pos + 9 * (size_t)i, g.bb_min, g.width, g.gd, lo, hi);
    int o = offset[i];
    for (int z = lo[2]; z <= hi[2]; ++z)
        for (int y = lo[1]; y <= hi[1]; ++y)
            for (int x = lo[0]; x <= hi[0]; ++x) { keys[o] = x + y * g.gd[0] + g.gd[0] * g.gd[1] * z; vals[o] = g.t0 + i; ++o; }
}

__global__ void k_grid_cells(const int* __restrict__ keys, int npairs, int ncell, int ref_base, int2* __restrict__ cells)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    auto lower = [&](int key) { int a = 0, b = npairs; while (a < b) { const int m = a + ((b - a) >> 1); if (keys[m] < key) a = m + 1; else b = m; } return a; };
    cells[c] = make_int2(ref_base + lower(c), ref_base + lower(c + 1));
}

struct Widen { __host__ __device__ long long operator()(int x) const { return x; } };
using WideCounts = thrust::transform_iterator<Widen, const int*, long long>;

}  // namespace

// Counts the references of one mesh's grid: *npairs, summed in 64 bits (synchronises the stream).  d_count / d_offset: n ints each,
// d_sum: one long long.  The offsets are scanned only when *npairs fits an int; above INT32_MAX the caller refuses the mesh.
int gridDeviceCount(const float* d_pos, int t0, int n, const float bb_min[3], const float width[3], const int gd[3], int* d_count, int* d_offset,
                    long long* d_sum, void* d_tmp, size_t tmp_bytes, cudaStream_t stream, long long* npairs)
{
    GridParams g;
    for (int k = 0; k < 3; ++k) { g.bb_min[k] = bb_min[k]; g.width[k] = width[k]; g.gd[k] = gd[k]; }
    g.t0 = t0; g.n = n;
    *npairs = 0;
    if (n <= 0) return cudaSuccess;
    k_grid_ranges<<<(n + 255) / 256, 256, 0, stream>>>(d_pos, g, d_count);
    cudaError_t e = cub::DeviceReduce::Sum(d_tmp, tmp_bytes, WideCounts((const int*)d_count, Widen()), d_sum, n, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(npairs, d_sum, sizeof(long long), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return e;
    if (*npairs <= INT32_MAX) e = cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_count, d_offset, n, stream);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

// Emits, sorts and indexes the pairs of one grid: d_refs[0 .. npairs) and cells[0 .. ncell) with reference positions offset by ref_base.
int gridDeviceFill(const float* d_pos, int t0, int n, const float bb_min[3], const float width[3], const int gd[3], const int* d_offset, int npairs,
                   int* d_keys, int* d_vals, int* d_keys2, void* d_tmp, size_t tmp_bytes, int ref_base, int* d_refs, int2* d_cells, cudaStream_t stream)
{
    GridParams g;
    for (int k = 0; k < 3; ++k) { g.bb_min[k] = bb_min[k]; g.width[k] = width[k]; g.gd[k] = gd[k]; }
    g.t0 = t0; g.n = n;
    const int ncell = gd[0] * gd[1] * gd[2];
    if (n > 0 && npairs > 0) {
        k_grid_pairs<<<(n + 255) / 256, 256, 0, stream>>>(d_pos, g, d_offset, d_keys, d_vals);
        int bits = 1;
        while ((1ll << bits) < ncell) ++bits;
        cudaError_t e = cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, (const int*)d_keys, d_keys2, (const int*)d_vals, d_refs, npairs, 0, bits, stream);
        if (e != cudaSuccess) return e;
    }
    k_grid_cells<<<(ncell + 255) / 256, 256, 0, stream>>>(d_keys2, n > 0 ? npairs : 0, ncell, ref_base, d_cells);
    return cudaGetLastError();
}

// ---- per-triangle voxel boxes (PTAP_ACCEL_GRID_EMULATED, trace_emu.cu) ------------------------------------------------------------------
// Scene::addMeshesToGrid lists a triangle in every voxel of the index box its bounds cover (Scene.cpp:357-374), so "is triangle T listed
// in voxel v" is a box test - IF the lists on the device really have that shape.  They may come from anywhere (the reference's own
// Scene.cpp in the integration build, ptap_scene_build_grids, the device builder, a caller's arrays), so the boxes are DERIVED from the
// lists and the shape is VERIFIED: per triangle the bounding index box of the voxels that list it, the number of listings (must equal
// the box volume), the grid that lists it (must be one), and per voxel an ascending list (the order the walk tests in decides exact-t ties).
namespace {

struct TriAcc { int lo[3], hi[3], cnt, gid; };

__global__ void k_tribox_init(TriAcc* acc, int ntris, int* grange, int ngrids)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ntris) { TriAcc a; a.lo[0] = a.lo[1] = a.lo[2] = 0x7fffffff; a.hi[0] = a.hi[1] = a.hi[2] = -1; a.cnt = 0; a.gid = -1; acc[t] = a; }
    if (t < ngrids) { grange[2 * t] = 0x7fffffff; grange[2 * t + 1] = -1; }
}

__global__ void k_tribox_cells(const int2* __restrict__ cells, const int* __restrict__ refs, const int* __restrict__ first_cell, int ngrids, int gx, int gy, int gz,
                               int ntris, TriAcc* acc, int* grange, int* bad)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int ncell = gx * gy * gz;
    if (idx >= (long long)ngrids * ncell) return;
    const int g = (int)(idx / ncell), l = (int)(idx % ncell);
    const int x = l % gx, y = (l / gx) % gy, z = l / (gx * gy);
    const int2 cell = cells[first_cell[g] + l];
    int prev = -1;
    for (int r = cell.x; r < cell.y; ++r) {
        const int t = refs[r];
        if (t < 0 || t >= ntris || t <= prev) { *bad = 1; continue; }
        prev = t;
        atomicMin(&acc[t].lo[0], x); atomicMin(&acc[t].lo[1], y); atomicMin(&acc[t].lo[2], z);
        atomicMax(&acc[t].hi[0], x); atomicMax(&acc[t].hi[1], y); atomicMax(&acc[t].hi[2], z);
        atomicAdd(&acc[t].cnt, 1);
        const int old = atomicCAS(&acc[t].gid, -1, g);
        if (old != -1 && old != g) *bad = 1;
        atomicMin(&grange[2 * g], t); atomicMax(&grange[2 * g + 1], t);
    }
}

__global__ void k_tribox_finish(const TriAcc* __restrict__ acc, int ntris, int2* __restrict__ tri_box, int* bad)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntris) return;
    const TriAcc a = acc[t];
    if (a.cnt == 0) { tri_box[t] = make_int2(511 | (511 << 10) | (511 << 20), 0); return; }   // listed nowhere: lo > hi on every axis, no voxel is inside
    const long long vol = (long long)(a.hi[0] - a.lo[0] + 1) * (a.hi[1] - a.lo[1] + 1) * (a.hi[2] - a.lo[2] + 1);
    if (vol != (long long)a.cnt) *bad = 1;
    tri_box[t] = make_int2(a.lo[0] | (a.lo[1] << 10) | (a.lo[2] << 20), a.hi[0] | (a.hi[1] << 10) | (a.hi[2] << 20));
}

}  // namespace

int gridTriBoxes(const int2* cells, const int* refs, int ngrids, const int* grid_first_cell, int gx, int gy, int gz, int ntris, int2* tri_box,
                 int* grid_tri_range_host, int* ok, cudaStream_t stream)
{
    *ok = 0;
    if (ngrids <= 0 || ntris <= 0 || gx > 512 || gy > 512 || gz > 512) return cudaSuccess;      // 9 bits per packed index + a guard bit (trace_emu.cu)
    TriAcc* acc = nullptr; int* d_small = nullptr;       // d_small: first cells, grid ranges, the flag
    cudaError_t e = cudaMalloc(&acc, (size_t)ntris * sizeof(TriAcc));
    if (e == cudaSuccess) e = cudaMalloc(&d_small, ((size_t)3 * ngrids + 1) * sizeof(int));
    if (e != cudaSuccess) { cudaFree(acc); cudaFree(d_small); return e; }
    int* d_first = d_small, *d_range = d_small + ngrids, *d_bad = d_small + 3 * ngrids;
    cudaMemcpyAsync(d_first, grid_first_cell, ngrids * sizeof(int), cudaMemcpyHostToDevice, stream);
    cudaMemsetAsync(d_bad, 0, sizeof(int), stream);
    const int nmax = std::max(ntris, ngrids);
    k_tribox_init<<<(nmax + 255) / 256, 256, 0, stream>>>(acc, ntris, d_range, ngrids);
    const long long total = (long long)ngrids * gx * gy * gz;
    k_tribox_cells<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(cells, refs, d_first, ngrids, gx, gy, gz, ntris, acc, d_range, d_bad);
    k_tribox_finish<<<(ntris + 255) / 256, 256, 0, stream>>>(acc, ntris, tri_box, d_bad);
    int bad = 1;
    e = cudaMemcpyAsync(grid_tri_range_host, d_range, 2 * ngrids * sizeof(int), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    cudaFree(acc); cudaFree(d_small);
    if (e != cudaSuccess) return e;
    *ok = bad ? 0 : 1;
    return cudaGetLastError();
}

size_t gridDeviceTempBytes(int ntris, long long npairs)
{
    size_t a = 0, b = 0, c = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, a, (const int*)nullptr, (int*)nullptr, std::max(ntris, 1));
    cub::DeviceRadixSort::SortPairs(nullptr, b, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, (int)std::max(npairs, 1ll), 0, 30);
    cub::DeviceReduce::Sum(nullptr, c, WideCounts((const int*)nullptr, Widen()), (long long*)nullptr, std::max(ntris, 1));
    return std::max(std::max(a, b), c) + 256;
}

}  // namespace ptap
