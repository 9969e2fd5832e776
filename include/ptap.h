/* ptap.h - C ABI of libptap.so, the B200-native render core behind PathTracerAP's API.
 *
 * The reference (purvakulkarni15/PathTracerAP) has no FFI: its boundary is the C++ surface
 * main.cpp:8-22 uses (Scene.h:21-39, Renderer.h:46-55, GPUMemoryPool.h:10-46).  Every entry
 * point below names the reference interface it replaces; the headers under include/PathTracerAP/ wrap
 * this ABI back into those C++ classes so that the reference's main.cpp compiles unchanged
 * (INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; every call returns 0 on success, a negative
 * PTAP_E_* code or a positive cudaError_t otherwise, with text in ptap_last_error().
 * One context per GPU; a context is not thread-safe; no global state; the caller owns all
 * host buffers, the library owns the device arena.  There is no CPU fallback: every compute
 * entry fails with PTAP_E_NO_DEVICE when no sm_100 device is usable.
 *
 * Streams: all work of a context is ordered on ONE stream, ptap_stream().  ptap_render pipelines its iterations over several
 * internal streams ("lanes"), which fork from and join that stream inside the call, so anything the caller orders on
 * ptap_stream() (an NCCL reduce of the film, a timer event) is ordered with the whole render.
 *
 * Environment (read once, in ptap_create; none of them changes a result bit):
 *   PTAP_LANES=1..8        wavefronts in flight per context (default: 4, or 8 for frames of at most 2^20 pixels; 130 B of device
 *                          memory per pixel and lane)
 *   PTAP_TRACE_CTAS=n      CTAs per SM of the closest-hit kernels (default: occupancy query)
 *   PTAP_VOTE_TRI / PTAP_VOTE_INST / PTAP_VOTE_REFILL / PTAP_VOTE_GRID, PTAP_BATCH   scheduling thresholds of the closest-hit kernels
 *   PTAP_SHADE_SORT=1      k_shade takes each 256-slot block regrouped by material class (measured slower; off)
 *   PTAP_BVH_LEAF, PTAP_BVH_CI   leaf size and node cost of the host SAH builder
 */
#ifndef PTAP_H
#define PTAP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTAP_VERSION 4      /* 2: PtapBvhNode carries node-local offsets; ptap_render_probe, ptap_reduce*, stamps
                               3: ray queries on device buffers, ptap_query_closest / ptap_query_occluded
                               4: ptap_update_models */

enum {
    PTAP_OK = 0,
    PTAP_E_INVALID = -1,      /* bad argument / call order */
    PTAP_E_NO_DEVICE = -2,    /* no usable CUDA device (never falls back to the CPU) */
    PTAP_E_NOMEM = -3,        /* device arena exhausted */
    PTAP_E_IO = -4,           /* file could not be read / written */
    PTAP_E_PARSE = -5,        /* malformed OBJ / Config.txt */
    PTAP_E_STATE = -6,        /* scene / accel / render parameters missing */
    PTAP_E_UNSUPPORTED = -7   /* the request is valid but this input cannot take the fast path asked for; the message names the alternative */
};

/* ---- PODs with the reference's exact layouts (Primitive.h:10-179) ----------------------- */

typedef struct { int32_t type; float refractive_index, reflectivity; float color[3]; } PtapMaterial;   /* Primitive.h:68-83, 24 B */
typedef struct { int32_t grid_index, mesh_index; float model_to_world[16], world_to_model[16]; PtapMaterial mat; } PtapModel; /* :93-100, 160 B, column-major */
typedef struct { int32_t v_start, v_end, t_start, t_end; float bb_min[3], bb_max[3]; } PtapMesh;       /* :85-90, 40 B */
typedef struct { float position[3], normal[3], uv[2]; } PtapVertex;                                    /* :23-28, 32 B */
typedef struct { int32_t v[3]; } PtapTriangle;                                                         /* :30-33, 12 B */
typedef struct { int32_t v_start, v_end; float width[3]; int32_t entity_type, entity_index; } PtapGrid;/* :126-137, 28 B */
typedef struct { int32_t start, end, entity_type; } PtapVoxel;                                         /* :120-124, 12 B */

enum { PTAP_DIFFUSE = 0, PTAP_SPECULAR, PTAP_REFLECTIVE, PTAP_REFRACTIVE, PTAP_EMISSIVE, PTAP_COAT, PTAP_METAL }; /* Primitive.h:70-79 */

/* BVH4 node (new; the reference has no BVH), 128 bytes: a node-local origin, the links of up to four children, and their boxes as
 * binary32 OFFSETS from that origin: plane = p + planes[axis][0 lower | 1 upper][slot], lower planes rounded down and upper planes rounded
 * up, so every child box contains the builder's box (which bounds the reference predicate's tolerance band).
 * link >= 0: child node index; link < 0: leaf, ~link = (first_leaf_triangle << 3) | (count - 1).
 * An unused slot holds an inverted box (lower offsets 1e15, upper offsets -1e15). */
typedef struct {
    float p[3];
    int32_t pad;
    int32_t link[4];
    float planes[3][2][4];
} PtapBvhNode;

/* The seven public vectors of the reference's Scene (Scene.h:26-32) as raw arrays. */
typedef struct {
    const PtapModel* models; int32_t nmodels;
    const PtapMesh* meshes; int32_t nmeshes;
    const PtapVertex* vertices; int32_t nvertices;
    const PtapTriangle* triangles; int32_t ntriangles;
    const PtapGrid* grids; int32_t ngrids;            /* may be NULL/0 when only the BVH is used */
    const PtapVoxel* voxels; int32_t nvoxels;
    const int32_t* refs; int32_t nrefs;               /* Scene::per_voxel_data_pool */
    int32_t grid_dim[3];                              /* GRID_X/Y/Z (Config.h:8-10) */
    /* optional prebuilt BVH (ptap_scene_build_bvh); NULL/0: ptap_build_accel(PTAP_ACCEL_BVH) builds it from the triangles */
    const PtapBvhNode* bvh_nodes; int32_t n_bvh_nodes;
    const int32_t* bvh_tri_id; int32_t n_bvh_tris;    /* leaf-order position -> global triangle index */
    const int32_t* bvh_mesh_root; int32_t n_bvh_roots;/* per mesh: root node, -1 if empty */
    int32_t bvh_depth;                                /* deepest BLAS level (a hint: upload always recomputes it from the nodes) */
    /* optional triangle records prepared by ptap_scene_build_bvh / ptap_scene_pack_triangles (48 B per triangle: v0, v1-v0, v2-v0, flat normal in the .w lanes,
     * reference arithmetic); NULL/0: ptap_upload_scene derives them from vertices + triangles.  ptap_scene keeps its upload-bound
     * arrays (these, the BVH nodes, the leaf order) in page-locked host memory when a CUDA device is present. */
    const void* tri_recs; int32_t n_tri_recs;
} PtapSceneView;

/* Closest-hit record of the parity entry point.  The reference's IntersectionData (Primitive.h:150-156)
 * has no primitive id; these fields are what BASELINE.json's parity contract compares. */
typedef struct {
    int32_t model, tri;       /* winning model, GLOBAL triangle index; -1 = miss */
    float t_model, dist;      /* model-space t; world distance (9999999.0f = miss) */
    float u, v;
    float normal[3];          /* world-space flat shading normal */
    int32_t mat_type;
} PtapHit;                    /* 40 B */

/* One path of a caller-supplied wavefront (parity entry point for the shade kernel). */
typedef struct {
    float orig[3], dir[3], color[3];
    int32_t ipixel;
    int32_t model, tri;       /* closest hit of this ray (-1, -1 = miss) */
    float dist;
} PtapPathIn;                 /* 52 B */
typedef struct {
    float orig[3], dir[3], color[3];
    int32_t ipixel;
    int32_t alive;            /* 1: continues to the next bounce */
} PtapPathOut;                /* 44 B */

typedef struct {
    int64_t rays_traced;          /* sum of active rays over closest-hit launches (BASELINE.md metric) */
    int64_t paths;                /* camera paths started */
    int64_t kernel_launches;      /* this library's kernels launched by render calls */
    int64_t active_per_round[16]; /* last iteration: active rays entering each round */
    float ms_render;              /* device time of the last ptap_render call (CUDA events on the context stream) */
    float ms_trace, ms_shade, ms_generate;  /* per-kernel split of that call when profiling is enabled, else 0 */
    float avg_nodes, avg_tris, avg_cells, avg_refs;  /* per traced ray, PTAP_FLAG_COUNT renders only */
    int64_t trace_launches;       /* closest-hit launches inside the last ptap_render call */
    int64_t scene_bytes;          /* bytes copied host->device by the last ptap_upload_scene */
    float ms_build;               /* device time of the last PTAP_ACCEL_BVH_DEVICE build */
    int32_t bvh_nodes, bvh_depth; /* 4-wide nodes and levels of that build */
    int32_t lanes;                /* wavefronts in flight of the current render parameters (PTAP_LANES, or 4 / 8 by frame size) */
    float ms_trace_inflight;      /* PTAP_FLAG_STAMP: time of the last ptap_render call during which at least one closest-hit kernel was resident */
    float ms_trace_sum;           /* PTAP_FLAG_STAMP: summed residency of its closest-hit launches (lanes overlap: may exceed ms_render) */
    int64_t rays_walked;          /* PTAP_ACCEL_GRID_EMULATED: rays (of rays_traced) that the grid walk itself had to answer */
    int64_t rays_reemulated;      /* PTAP_ACCEL_GRID_EMULATED: rays whose nearest model's walk does not return the closest hit (emulated in full) */
} PtapStats;

/* Camera of generateRaysKernel (Renderer.cpp:527-548), whose numbers the reference hard-codes: rays start at `origin` and pass through
 * pixel (x, y)'s lower-left corner plane_min + (x * span[0] / W, y * span[1] / H, 0) of an axis-aligned image plane (un-normalised
 * directions, non-square pixels unless span matches the aspect ratio - as the reference).  jitter != 0 adds a per-iteration sub-pixel
 * offset in [0, 1)^2 (a hash of jitter_seed, iteration and pixel); camera rays then differ between iterations, so the first-hit cache
 * (Renderer.cpp:594-613) is not used whatever PTAP_FLAG_FIRST_HIT_CACHE says.  Parity: with the default values the rays are bit-identical
 * to the reference's; everything else is an extension with no reference behaviour (tested against a numpy restatement). */
typedef struct {
    float origin[3];          /* (0, 0, 920) */
    float plane_min[3];       /* (-10, -4, 900) */
    float span[2];            /* (20, 16) */
    int32_t jitter;
    uint32_t jitter_seed;
} PtapCamera;

typedef struct ptap_scene ptap_scene;   /* host-side scene: replaces class Scene (Scene.h:21-39) */
typedef struct ptap_ctx ptap_ctx;       /* per-GPU render context: replaces class Renderer + RenderData (Renderer.h:19-55) */

/* ---- host scene: replaces Scene (Scene.h:21-39, Scene.cpp) ------------------------------ */

/* Scene::Scene as coded at Scene.cpp:3-224 (its `config` argument is ignored there): the 3 bundled meshes, 11 models.
 * `root` is the directory containing "Input data/". */
int ptap_scene_create_builtin(const char* root, ptap_scene** out);
/* Scene(config) for the schema sketched in Config.txt:1-31 (the reference never parses it; see DESIGN.md). */
int ptap_scene_create_from_config(const char* config_path, ptap_scene** out);
int ptap_scene_create_empty(ptap_scene** out);
int ptap_scene_create_from_view(const PtapSceneView* view, ptap_scene** out);
/* Scene::loadAndProcessMeshFile (Scene.cpp:226-291) with an in-repo Wavefront reader (Assimp is not vendored):
 * one vertex per face corner, positions and normals scaled by BASE_MODEL_SCALE (Config.h:17). */
int ptap_scene_add_obj(ptap_scene* s, const char* path, int32_t* mesh_index);
int ptap_scene_add_mesh(ptap_scene* s, const PtapVertex* vertices, int32_t nvertices, const int32_t* indices, int32_t ntriangles, int32_t* mesh_index);
/* synthetic displaced icosphere (SURVEY.md 8d, configs 2 and 4): 20*4^level triangles, radius `radius` model units */
int ptap_scene_add_icosphere(ptap_scene* s, int32_t level, float radius, float displacement, uint32_t seed, int32_t* mesh_index);
/* models.push_back(Model{...}) (Scene.cpp:32-221): world_to_model is computed from model_to_world when NULL */
int ptap_scene_add_model(ptap_scene* s, int32_t mesh_index, const float model_to_world[16], const float* world_to_model, const PtapMaterial* mat, int32_t* model_index);
/* glm::translate * glm::rotate(Y) * glm::scale as every model of Scene.cpp composes it; writes model_to_world, world_to_model */
void ptap_compose_trs(const float translate[3], float rotate_y_degrees, const float scale[3], float model_to_world[16], float world_to_model[16]);
/* Scene::addMeshesToGrid (Scene.cpp:318-396) */
int ptap_scene_build_grids(ptap_scene* s, int32_t gx, int32_t gy, int32_t gz);
/* Builds one BVH per mesh on the host (binned SAH); part of scene construction like addMeshesToGrid, so that
 * Renderer::allocateOnGPU only uploads.  Bounds are conservative for the reference's tolerance band (DESIGN.md). */
int ptap_scene_build_bvh(ptap_scene* s);
/* Only the upload-bound triangle records (page-locked), without a host BVH: for PTAP_ACCEL_BVH_DEVICE and the grid modes, so that
 * ptap_upload_scene copies instead of repacking every triangle on every call.  ptap_scene_build_bvh implies it. */
int ptap_scene_pack_triangles(ptap_scene* s);
/* Host-side check of that BVH: the number of triangles whose tolerance band (what the reference's predicate can accept) sticks out of a
 * compressed child box on its path from the root, plus structural errors; 0 for a correct tree. */
int ptap_scene_validate_bvh(const ptap_scene* s, int64_t* violations, int32_t* depth);
int ptap_scene_view(const ptap_scene* s, PtapSceneView* out);     /* pointers stay owned by the scene */
PtapModel* ptap_scene_models(ptap_scene* s);                      /* mutable, like the public vector */
void ptap_scene_destroy(ptap_scene* s);
const char* ptap_scene_last_error(const ptap_scene* s);
/* RESOLUTION / ITER / DEPTH keys of a parsed Config.txt (0 when absent): out4 = {W, H, iters, depth} */
int ptap_scene_config_params(const ptap_scene* s, int32_t out4[4]);
/* CAMERA_ORIGIN / CAMERA_PLANE / CAMERA_SPAN / JITTER keys of a parsed Config.txt: returns 1 and fills *out when any of them was given
 * (missing ones keep the reference's values), 0 otherwise */
int ptap_scene_config_camera(const ptap_scene* s, PtapCamera* out);

/* ---- device context: replaces Renderer (Renderer.h:46-55) -------------------------------- */

enum { PTAP_ACCEL_GRID_COMPAT = 0,  /* the reference's per-mesh uniform grid walked exactly as Renderer.cpp:238-360 (oracle tier R0) */
       PTAP_ACCEL_BVH = 1,          /* two-level BVH, exact closest hit under the reference's triangle predicate (oracle tier R1);
                                       the per-mesh trees are the host's binned-SAH ones (ptap_scene_build_bvh, or built at this call) */
       PTAP_ACCEL_BVH_DEVICE = 2,   /* same traversal and results, per-mesh trees built on the GPU (PLOC) in milliseconds */
       PTAP_ACCEL_GRID_EMULATED = 3 };
                                    /* the RESULTS of PTAP_ACCEL_GRID_COMPAT (tier R0, bit for bit: the walk's misses and early exits
                                       included) computed through the BVH: all hits of a model, then a replay of the walk's voxel sequence
                                       over the voxel boxes of the hit triangles (trace_emu.cu).  Needs the grids (their lists define the
                                       result) and builds a BVH on the device if none is there.  ptap_build_accel fails with
                                       PTAP_E_UNSUPPORTED when the lists on the device do not have the shape Scene::addMeshesToGrid
                                       produces (Scene.cpp:357-374); PTAP_ACCEL_GRID_COMPAT then remains available. */

enum { PTAP_FLAG_FIRST_HIT_CACHE = 1,   /* Renderer.cpp:580,594-613 */
       PTAP_FLAG_PROFILE = 2,           /* per-kernel CUDA-event split in PtapStats (adds event records) */
       PTAP_FLAG_COUNT = 4,             /* counting build of the closest-hit kernel: avg_* in PtapStats (slower; not for timing) */
       PTAP_FLAG_STAMP = 8,
       PTAP_FLAG_ITER_TIMES = 16 };     /* one event per iteration: ptap_get_iteration_times (the "Iteration k: ..." lines of Renderer.cpp:641-643) */           /* every closest-hit launch records its first start / last end on the device's nanosecond clock
                                           (two atomics per CTA): ms_trace_inflight / ms_trace_sum in PtapStats, measured inside the real
                                           multi-lane schedule */

int ptap_create(int device, size_t arena_bytes /* 0 = sized on demand */, ptap_ctx** out);
void ptap_destroy(ptap_ctx* ctx);                                   /* Renderer::free (Renderer.cpp:132-148) */
const char* ptap_last_error(const ptap_ctx* ctx);

/* Renderer::allocateOnGPU (Renderer.cpp:65-130): copies the scene into the device arena (repacked, see DESIGN.md). */
int ptap_upload_scene(ptap_ctx* ctx, const PtapSceneView* view);
int ptap_build_accel(ptap_ctx* ctx, int kind);
/* Replace the records of models [first, first + count) of the uploaded scene: transforms and material.  mesh_index and grid_index must
 * equal the uploaded ones (anything else needs ptap_upload_scene).  The instance records and, when a BVH is on the device, the TLAS are
 * rebuilt on the GPU; BLAS, triangles and grids are untouched.  Ordered after everything already enqueued on ptap_stream(ctx); returns when
 * the device work is done.  Afterwards every entry point behaves exactly as after ptap_upload_scene + ptap_build_accel(current accel) of
 * the scene with these models: hits, films and query answers bit for bit (the TLAS is a different tree, so traversal counts and
 * PTAP_FLAG_COUNT averages may differ).  The first-hit cache is forgotten.  count == 0 is a no-op.
 * Errors: PTAP_E_STATE without an uploaded scene; PTAP_E_INVALID for a bad range, a changed mesh_index or grid_index or a singular
 * world_to_model, checked before anything changes (the context then traces exactly as before the call).  A failure after these checks (a
 * CUDA error, a TLAS too deep for the traversal stack) keeps the new models but drops the BVH: ptap_build_accel builds it again. */
int ptap_update_models(ptap_ctx* ctx, const PtapModel* models, int32_t first, int32_t count);
/* Scene::addMeshesToGrid (Scene.cpp:318-396) on the DEVICE for the scene last uploaded (`view` must be that scene's view: vertices and
 * triangles are read again): one gx x gy x gz grid per distinct mesh in model order, built by sorting (cell, triangle) pairs; cells and
 * reference lists are bit-identical to the host builder's / the reference's (ascending triangle order per cell).  Selects
 * PTAP_ACCEL_GRID_COMPAT; PtapStats::ms_build reports the device time.  ptap_read_grids copies the result back in the reference's layout
 * (voxels / refs NULL: counts only; counts = {voxels, references}). */
int ptap_build_grids_device(ptap_ctx* ctx, const PtapSceneView* view, int32_t gx, int32_t gy, int32_t gz);
int ptap_read_grids(ptap_ctx* ctx, PtapVoxel* voxels, int32_t* refs, int32_t counts[2]);
int ptap_set_render_params(ptap_ctx* ctx, int32_t W, int32_t H, int32_t depth, uint32_t flags);
/* NULL restores the reference's camera.  May be called before or after ptap_set_render_params. */
int ptap_set_camera(ptap_ctx* ctx, const PtapCamera* camera);
/* Renderer::renderLoop (Renderer.cpp:567-648) for iterations [iter_begin, iter_end); the film accumulates.
 * Asynchronous on the context stream; ptap_sync / ptap_read_film / ptap_get_stats wait for it. */
int ptap_render(ptap_ctx* ctx, int32_t iter_begin, int32_t iter_end);
/* start of a new renderLoop: zero film (initImageKernel), forget the first-hit cache, zero the stats counters */
int ptap_frame_begin(ptap_ctx* ctx);
int ptap_film_reset(ptap_ctx* ctx);                                /* initImageKernel (Renderer.cpp:557-565) */
int ptap_sync(ptap_ctx* ctx);
/* CUDA-event timer on the context stream (device time of everything enqueued between the two calls) */
int ptap_timer_start(ptap_ctx* ctx);
int ptap_timer_stop(ptap_ctx* ctx, float* ms);
/* render_data.dev_image_data->pool (Renderer.cpp:49): the un-normalised sum over iterations, W*H*3 floats */
int ptap_read_film(ptap_ctx* ctx, float* rgb);
int ptap_film_device_ptr(ptap_ctx* ctx, void** dev_ptr, size_t* nfloats);   /* for the NCCL reduce (SURVEY.md 8e) */
int ptap_film_add(ptap_ctx* ctx, const float* rgb);                /* host film += (multi-rank emulation / resume) */
/* Renderer::renderImage (Renderer.cpp:15-63): 24-bpp BMP, bottom-up, bytes (uint8)(sum/iters*255) */
int ptap_write_bmp(ptap_ctx* ctx, const char* path, int32_t iters);
/* Supersampled output: SAMPLESX x SAMPLESY (Config.h:14-15).  generateRaysKernel lays RX*SX x RY*SY camera rays on ONE lattice
 * (Renderer.cpp:527-542), which is exactly what ptap_set_render_params(RX*SX, RY*SY) renders.  The reference's gather is broken for
 * SAMPLES > 1: avg = 1 / (SAMPLESX * SAMPLESY) is an integer division (= 0) and ipixel = iray (Renderer.cpp:493, 530-533), so its image
 * stays black; these two calls implement the evident intent (the commented-out mapping at Renderer.cpp:530-532): pixel (x, y) =
 * sum of avg * sample over its sx * sy lattice samples, avg = 1.0f / (sx * sy), in row-major sample order.  The film must have been
 * rendered at (W, H) divisible by (sx, sy); rgb receives (W / sx) * (H / sy) * 3 floats.  sx = sy = 1 equals the plain calls.
 * Parity unpinned: no reference behaviour exists for this row (SURVEY.md 8f row 4). */
int ptap_read_film_resolved(ptap_ctx* ctx, int32_t sx, int32_t sy, float* rgb);
int ptap_write_bmp_resolved(ptap_ctx* ctx, const char* path, int32_t iters, int32_t sx, int32_t sy);
int ptap_get_stats(ptap_ctx* ctx, PtapStats* out);
/* PTAP_FLAG_ITER_TIMES: device time from the start of the last ptap_render call to the completion of each of its iterations, in order
 * (*n = iterations recorded; at most `cap` values are written).  Renderer::renderLoop prints the differences (Renderer.cpp:641-643). */
int ptap_get_iteration_times(ptap_ctx* ctx, float* ms_since_start, int32_t cap, int32_t* n);

/* ---- multi-GPU: sample partitioning (SURVEY.md 8e) -------------------------------------------------------------------------------
 * Every GPU renders its own range of iterations [iter_begin, iter_end) of the same frame into its own film (the reference seeds its RNG
 * with the iteration number, Renderer.cpp:435, so the union is exactly the one-GPU sample set); the films are then summed.
 * The reference has no multi-GPU path; these calls replace nothing, they extend Renderer::renderLoop. */
/* One process, several contexts (main.cpp's process-global Renderer on N devices): film(dst) += film(src) over a peer copy (NVLink),
 * ordered after the renders enqueued on both contexts.  Calling it for src = rank 1, 2, ... gives a fixed order of float additions:
 * the reduced film is bit-reproducible. */
int ptap_reduce_peer(ptap_ctx* dst, ptap_ctx* src);
/* One process per GPU: NCCL (libnccl.so.2 is loaded at run time; PTAP_NCCL_LIB overrides the name).  Rank 0 makes the 128-byte id, the
 * host side distributes it by whatever means it has (MPI, torch.distributed, a file), every rank joins, and ptap_reduce issues
 * ncclReduce(sum) of the film onto `root` in place on the context stream - ordered after the render without a host synchronisation. */
int ptap_nccl_unique_id(void* id128);
int ptap_nccl_init(ptap_ctx* ctx, const void* id128, int32_t nranks, int32_t rank);
int ptap_reduce(ptap_ctx* ctx, int32_t root);
int ptap_nccl_finalize(ptap_ctx* ctx);
void* ptap_stream(ptap_ctx* ctx);                                  /* cudaStream_t of the context */

/* ---- ray queries on device buffers (DESIGN.md 4.8) ----------------------------------------------------------------------------------
 * Embree's rtcIntersect / rtcOccluded for rays already in GPU memory.  Every pointer is a DEVICE (or managed) pointer on the context's
 * device; org and dir each hold n x 4 floats, 16-byte aligned: org[i] = (ox, oy, oz, unused), dir[i] = (dx, dy, dz, L_i).  Origin and
 * direction are in world space, d need not be normalised, and distances are WORLD distances, length(hit - o) (Renderer.cpp:388-391).
 *   ptap_query_closest:  hits[i] = what ptap_trace returns for (o, d) under the current accel, bit for bit (tier R0 for the grid modes,
 *                        R1 for the BVH modes); dir[i].w is not read.
 *   ptap_query_occluded: occluded[i] = (closest.model >= 0 && closest.dist < L_i) in binary32 (1 / 0): L = +inf is "any hit", a NaN L
 *                        gives 0.  Under PTAP_ACCEL_BVH / BVH_DEVICE an any-hit traversal stops at the first hit that provably decides
 *                        the answer; the grid modes compute the closest hit (their walk can miss hits, so no early exit is exact) and compare.
 * stream: NULL = ptap_stream(ctx); otherwise the work is ordered after everything already enqueued on `stream`, and `stream` is ordered
 * after the query (event record + wait both ways).  The call returns after enqueueing: no host synchronisation.  Work already enqueued on
 * ptap_stream(ctx) (a render) runs first; the queries use scratch of their own and never change the film.  Rays are processed in chunks
 * of 2^22; the scratch (one chunk: 16 B per ray, 24 B for closest, plus 156 B per ray + 33 MB under PTAP_ACCEL_GRID_EMULATED) is kept
 * for later calls.  Bad pointers (host memory, another device, misaligned) give PTAP_E_INVALID naming the argument; n == 0 is a no-op. */
int ptap_query_closest(ptap_ctx* ctx, const float* org, const float* dir, int32_t n, PtapHit* hits, void* stream);
int ptap_query_occluded(ptap_ctx* ctx, const float* org, const float* dir, int32_t n, uint8_t* occluded, void* stream);

/* ---- parity entry points (what BASELINE.json's contract measures) ------------------------- */

/* computeRaySceneIntersectionKernel (Renderer.cpp:363-409) on a caller ray set: n x 6 host floats (origin, direction). */
int ptap_trace(ptap_ctx* ctx, const float* rays_od, int32_t n, PtapHit* out);
/* same, also returning per-ray traversal counts (nodes or cells, refs, triangle tests): n x 4 int32 */
int ptap_trace_count(ptap_ctx* ctx, const float* rays_od, int32_t n, PtapHit* out, int32_t* counts);
/* shadeRayKernel + compaction (Renderer.cpp:411-479, 506-519, 628-630) on a caller wavefront whose slot i is paths[i];
 * `remaining` is Ray::meta_data.remaining_bounces of every path.  out[i] is the post-shade state of slot i;
 * order[k] is the slot that the stable compaction moved to position k (k < *n_alive). */
int ptap_shade(ptap_ctx* ctx, const PtapPathIn* paths, int32_t n, int32_t iter, int32_t remaining, PtapPathOut* out, int32_t* order, int32_t* n_alive);

/* The PRODUCTION closest-hit path under test.  ptap_trace above launches the barycentric-recording instantiations of the closest-hit
 * kernels; Renderer::renderLoop's replacement (ptap_render) launches the plain ones and defers BVH hit distances to the shade kernel.
 * This call enqueues iteration `iter` exactly as ptap_render does (one lane) up to and including the closest-hit launch
 * (computeRaySceneIntersectionKernel, Renderer.cpp:617) of round `round`, and returns that round's wavefront: n_out active rays, their
 * (origin, direction) as the kernel read them (rays_od, n x 6), their pixels (Ray::meta_data.ipixel), and the hit records the kernel wrote
 * (u = v = 0).  Buffers hold `cap` entries; any of them may be NULL.  Leaves film and first-hit cache unspecified: ptap_frame_begin next. */
int ptap_render_probe(ptap_ctx* ctx, int32_t iter, int32_t round, float* rays_od, int32_t* pixels, PtapHit* hits, int32_t cap, int32_t* n_out);

/* device-resident timing helpers for bench.py (inputs already in HBM): trace the active queue of a primed wavefront `reps` times */
int ptap_bench_trace(ptap_ctx* ctx, const float* rays_od, int32_t n, int32_t reps, float* ms_per_launch);

#ifdef __cplusplus
}
#endif
#endif
