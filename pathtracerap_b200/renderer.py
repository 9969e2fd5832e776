"""Device-side renderer: the Python mirror of the reference's `Renderer` (Renderer.h:46-55) over the C ABI.

`allocateOnGPU / renderLoop / renderImage / free` keep the reference's names and meaning; the remaining
methods expose what the reference hard-codes (resolution, iterations, depth) and the parity entry points.
"""
from __future__ import annotations

import ctypes as C
import numbers

import numpy as np

from . import _native as N
from .scene import Scene


class Renderer:
    # Config.h:12-13,19 and Renderer.cpp:550
    RESOLUTION_X, RESOLUTION_Y, ITER, DEPTH = 1000, 800, 500, 5

    def __init__(self, device: int = 0, width: int | None = None, height: int | None = None, iters: int | None = None,
                 depth: int | None = None, accel: int = N.ACCEL_GRID_EMULATED, first_hit_cache: bool = True, profile: bool = False,
                 arena_bytes: int = 0):
        self.device = device
        self.W = width or self.RESOLUTION_X; self.H = height or self.RESOLUTION_Y
        self.iters = iters or self.ITER; self.depth = depth or self.DEPTH
        self.accel = accel
        self.flags = (N.FLAG_FIRST_HIT_CACHE if first_hit_cache else 0) | (N.FLAG_PROFILE if profile else 0)
        self._iters_done = 0
        h = C.c_void_p()
        rc = N.lib().ptap_create(device, arena_bytes, C.byref(h))
        if rc != 0:
            raise N.PtapError(f"ptap_create(device={device}) failed with {rc}: a CUDA sm_100 device is required (no CPU fallback)")
        self.h = h

    def _check(self, rc, what):
        if rc != 0:
            raise N.PtapError(f"{what}: error {rc}: {N.lib().ptap_last_error(self.h).decode()}")

    # -- the reference's four methods ----------------------------------------------------------------------------
    def allocateOnGPU(self, scene: Scene):
        v = scene.view()
        self._check(N.lib().ptap_upload_scene(self.h, C.byref(v)), "allocateOnGPU/upload_scene")
        rc = N.lib().ptap_build_accel(self.h, self.accel)
        if rc == N.E_UNSUPPORTED and self.accel == N.ACCEL_GRID_EMULATED:
            # grids whose lists are not the box-shaped registrations of Scene.cpp:357-374: the same results by walking them
            self.accel = N.ACCEL_GRID_COMPAT
            rc = N.lib().ptap_build_accel(self.h, self.accel)
        self._check(rc, "allocateOnGPU/build_accel")
        self._check(N.lib().ptap_set_render_params(self.h, self.W, self.H, self.depth, self.flags), "allocateOnGPU/set_render_params")
        self._iters_done = 0

    def renderLoop(self):
        self.render(0, self.iters)
        self.sync()

    def renderImage(self, path: str = "Render.bmp", samples: tuple[int, int] = (1, 1)):
        """Renderer::renderImage; `samples` = (SAMPLESX, SAMPLESY) of Config.h:14-15 when the film was rendered on the W*SX x H*SY lattice."""
        self._check(N.lib().ptap_write_bmp_resolved(self.h, path.encode(), max(self._iters_done, 1), samples[0], samples[1]), "renderImage")

    def free(self):
        if getattr(self, "h", None):
            N.lib().ptap_destroy(self.h)
            self.h = None

    # -- finer control -------------------------------------------------------------------------------------------
    def set_accel(self, accel: int):
        self.accel = accel
        self._check(N.lib().ptap_build_accel(self.h, accel), "build_accel")

    def set_params(self, width, height, depth, first_hit_cache=True, profile=False, count=False, stamp=False, iter_times=False):
        self.W, self.H, self.depth = width, height, depth
        self.flags = (N.FLAG_FIRST_HIT_CACHE if first_hit_cache else 0) | (N.FLAG_PROFILE if profile else 0) | (N.FLAG_COUNT if count else 0) | (N.FLAG_STAMP if stamp else 0) | (N.FLAG_ITER_TIMES if iter_times else 0)
        self._check(N.lib().ptap_set_render_params(self.h, width, height, depth, self.flags), "set_render_params")
        self._iters_done = 0

    def set_camera(self, origin=(0.0, 0.0, 920.0), plane_min=(-10.0, -4.0, 900.0), span=(20.0, 16.0), jitter=False, jitter_seed=0):
        """generateRaysKernel's camera (Renderer.cpp:527-548) as parameters; the defaults are the reference's hard-coded numbers."""
        cam = N.Camera((C.c_float * 3)(*origin), (C.c_float * 3)(*plane_min), (C.c_float * 2)(*span), int(bool(jitter)), int(jitter_seed))
        self._check(N.lib().ptap_set_camera(self.h, C.byref(cam)), "set_camera")

    def build_grids_device(self, scene: Scene, gx=25, gy=25, gz=25):
        """Scene::addMeshesToGrid on the GPU for the scene last uploaded (`scene` must be that scene); selects the grid walk."""
        v = scene.view()
        self._check(N.lib().ptap_build_grids_device(self.h, C.byref(v), gx, gy, gz), "build_grids_device")
        self.accel = N.ACCEL_GRID_COMPAT

    def read_grids(self):
        """(voxels, refs) of the device-built grids in the reference's layout."""
        cnt = (C.c_int32 * 2)()
        self._check(N.lib().ptap_read_grids(self.h, None, None, cnt), "read_grids")
        vox = np.zeros(cnt[0], N.VOXEL); refs = np.zeros(max(cnt[1], 1), np.int32)
        self._check(N.lib().ptap_read_grids(self.h, N.ptr(vox), N.ptr(refs), cnt), "read_grids")
        return vox, refs[:cnt[1]]

    def build_stats(self) -> dict:
        """Device time, node count and depth of the last PTAP_ACCEL_BVH_DEVICE build."""
        st = self.stats()
        return {"ms_build": st["ms_build"], "bvh_nodes": st["bvh_nodes"], "bvh_depth": st["bvh_depth"]}

    def render(self, iter_begin: int, iter_end: int):
        """Enqueue iterations [iter_begin, iter_end) (asynchronous)."""
        self._check(N.lib().ptap_render(self.h, iter_begin, iter_end), "render")
        self._iters_done += iter_end - iter_begin

    def sync(self):
        self._check(N.lib().ptap_sync(self.h), "sync")

    def upload(self, scene: Scene):
        """ptap_upload_scene only (host -> device copy of the scene arrays, including a prebuilt BVH when the scene has one)."""
        v = scene.view()
        self._check(N.lib().ptap_upload_scene(self.h, C.byref(v)), "upload_scene")
        self._check(N.lib().ptap_build_accel(self.h, self.accel), "build_accel")

    def update_models(self, models, first: int = 0):
        """Replace models [first, first + len(models)) of the uploaded scene (transforms and material; ptap_update_models): the
        instance records and the TLAS are rebuilt on the GPU, the meshes' BVHs stay.  `models` is an N.MODEL array, or a Scene for all
        of its models.  Afterwards the renderer traces and renders exactly as one that uploaded the scene with these models."""
        if isinstance(models, Scene):
            models = models.models
        if not isinstance(models, np.ndarray) or models.dtype != N.MODEL:
            raise N.PtapError(f"update_models: models must be an array of dtype MODEL, got {getattr(models, 'dtype', type(models).__name__)}")
        models = np.ascontiguousarray(models.reshape(-1))
        self._check(N.lib().ptap_update_models(self.h, N.ptr(models), int(first), len(models)), "update_models")

    def frame_begin(self):
        """Start of a renderLoop: zero film, forget the first-hit cache, zero the counters."""
        self._check(N.lib().ptap_frame_begin(self.h), "frame_begin")
        self._iters_done = 0

    def timer_start(self):
        self._check(N.lib().ptap_timer_start(self.h), "timer_start")

    def timer_stop(self) -> float:
        ms = C.c_float(0)
        self._check(N.lib().ptap_timer_stop(self.h, C.byref(ms)), "timer_stop")
        return ms.value

    def film_reset(self):
        self._check(N.lib().ptap_film_reset(self.h), "film_reset")
        self._iters_done = 0

    def film(self) -> np.ndarray:
        """Un-normalised running sum, H x W x 3 (render_data.dev_image_data->pool, Renderer.cpp:49)."""
        out = np.zeros((self.H, self.W, 3), np.float32)
        self._check(N.lib().ptap_read_film(self.h, N.ptr(out)), "read_film")
        return out

    def film_resolved(self, samples: tuple[int, int]) -> np.ndarray:
        """Box-resolved film for SAMPLESX x SAMPLESY supersampling (ptap.h: ptap_read_film_resolved), (H / sy) x (W / sx) x 3."""
        sx, sy = samples
        out = np.zeros((self.H // max(sy, 1), self.W // max(sx, 1), 3), np.float32)
        self._check(N.lib().ptap_read_film_resolved(self.h, sx, sy, N.ptr(out)), "read_film_resolved")
        return out

    def film_add(self, rgb: np.ndarray):
        rgb = np.ascontiguousarray(rgb, np.float32)
        assert rgb.size == self.W * self.H * 3
        self._check(N.lib().ptap_film_add(self.h, N.ptr(rgb)), "film_add")

    # -- multi-GPU through the C ABI (ptap.h: ptap_nccl_*, ptap_reduce, ptap_reduce_peer) ----------------------------------------
    def nccl_init(self, unique_id: bytes, nranks: int, rank: int):
        buf = (C.c_char * 128).from_buffer_copy(unique_id)
        self._check(N.lib().ptap_nccl_init(self.h, C.cast(buf, C.c_void_p), nranks, rank), "nccl_init")

    def reduce(self, root: int = 0):
        """ncclReduce(sum) of the film onto `root`, in place, on the renderer's own stream (asynchronous)."""
        self._check(N.lib().ptap_reduce(self.h, root), "reduce")

    def reduce_peer(self, src: "Renderer"):
        """film(self) += film(src) for two renderers of this process (peer copy + add, fixed order: bit-reproducible)."""
        self._check(N.lib().ptap_reduce_peer(self.h, src.h), "reduce_peer")

    def nccl_finalize(self):
        N.lib().ptap_nccl_finalize(self.h)

    def iteration_times(self) -> np.ndarray:
        """Device time (ms since the start of the last render call) at which each of its iterations completed (needs iter_times=True)."""
        n = C.c_int32(0)
        self._check(N.lib().ptap_get_iteration_times(self.h, None, 0, C.byref(n)), "get_iteration_times")
        out = np.zeros(max(n.value, 1), np.float32)
        self._check(N.lib().ptap_get_iteration_times(self.h, N.ptr(out), n.value, C.byref(n)), "get_iteration_times")
        return out[:n.value]

    def stream_ptr(self) -> int:
        """cudaStream_t of the context (every kernel and copy of this renderer is ordered on it)."""
        return int(N.lib().ptap_stream(self.h))

    def film_device_ptr(self):
        p = C.c_void_p(); n = C.c_size_t()
        self._check(N.lib().ptap_film_device_ptr(self.h, C.byref(p), C.byref(n)), "film_device_ptr")
        return p.value, n.value

    def stats(self) -> dict:
        s = N.Stats()
        self._check(N.lib().ptap_get_stats(self.h, C.byref(s)), "get_stats")
        d = {k: getattr(s, k) for k, _ in N.Stats._fields_ if k != "active_per_round"}
        d["active_per_round"] = [int(x) for x in s.active_per_round]
        return d

    # -- ray queries on device tensors (ptap.h: ptap_query_closest / ptap_query_occluded) -----------------------------------------
    def _check_rays(self, org, dir):
        import torch
        for name, x in (("org", org), ("dir", dir)):
            if not isinstance(x, torch.Tensor):
                raise TypeError(f"{name} must be a torch tensor, got {type(x).__name__}")
            if x.dtype != torch.float32:
                raise TypeError(f"{name} must be float32, got {x.dtype}")
            if x.device.type != "cuda":
                raise ValueError(f"{name} is on {x.device}: the queries read device memory")
            if x.device.index != self.device:
                raise ValueError(f"{name} is on {x.device}, the renderer on cuda:{self.device}")
            if x.dim() != 2 or x.shape[1] not in (3, 4):
                raise ValueError(f"{name} must have shape (n, 3) or (n, 4), got {tuple(x.shape)}")
            if not x.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
        if org.shape[0] != dir.shape[0]:
            raise ValueError(f"org has {org.shape[0]} rays, dir {dir.shape[0]}")

    @staticmethod
    def _pack_rays(org, dir, length=None):
        """(n, 4) float32 origins and directions in the ABI's layout, dir[:, 3] = length when given (a copy only where needed)."""
        import torch
        n = org.shape[0]
        o4 = org if org.shape[1] == 4 else torch.cat([org, org.new_zeros((n, 1))], dim=1)
        if length is None:
            d4 = dir if dir.shape[1] == 4 else torch.cat([dir, dir.new_zeros((n, 1))], dim=1)
        else:
            d4 = torch.empty((n, 4), dtype=torch.float32, device=dir.device)
            d4[:, :3] = dir[:, :3]
            d4[:, 3] = length
        return o4, d4

    def _stream_handle(self):
        import torch
        # torch's default stream is the legacy NULL stream: name it (cudaStreamLegacy) so that the query is ordered with it, since NULL
        # would mean the renderer's own stream
        return torch.cuda.current_stream(self.device).cuda_stream or 1

    def query_closest(self, org, dir) -> dict:
        """Closest hit of every ray (o, d) of two (n, 3) or (n, 4) float32 CUDA tensors, on the current torch stream, without a host
        synchronisation: what trace() returns for the same rays, bit for bit.  A dict of views of one (n, 10) int32 tensor holding the
        PtapHit records: model, tri, t_model, dist, u, v, normal (n, 3), mat_type (model = -1: miss)."""
        import torch
        self._check_rays(org, dir)
        o4, d4 = self._pack_rays(org, dir)
        n = o4.shape[0]
        rec = torch.empty((n, 10), dtype=torch.int32, device=o4.device)
        self._check(N.lib().ptap_query_closest(self.h, o4.data_ptr(), d4.data_ptr(), n, rec.data_ptr(), self._stream_handle()), "query_closest")
        f = rec.view(torch.float32)
        return {"model": rec[:, 0], "tri": rec[:, 1], "t_model": f[:, 2], "dist": f[:, 3], "u": f[:, 4], "v": f[:, 5],
                "normal": f[:, 6:9], "mat_type": rec[:, 9]}

    def query_occluded(self, org, dir, tmax):
        """Is the segment from o along d of world length tmax blocked: closest.model >= 0 and closest.dist < tmax (binary32; inf = any
        hit, NaN = False).  tmax is a float or an (n,) float32 tensor on the same device.  A torch.bool tensor (n,), on the current stream."""
        import torch
        self._check_rays(org, dir)
        if isinstance(tmax, torch.Tensor):
            if tmax.dtype != torch.float32:
                raise TypeError(f"tmax must be float32, got {tmax.dtype}")
            if tmax.device != org.device:
                raise ValueError(f"tmax is on {tmax.device}, the rays on {org.device}")
            if tuple(tmax.shape) != (org.shape[0],):
                raise ValueError(f"tmax must have shape ({org.shape[0]},), got {tuple(tmax.shape)}")
        elif isinstance(tmax, numbers.Real) and not isinstance(tmax, (bool, np.bool_)):      # Python and numpy scalars
            tmax = float(tmax)
        else:
            raise TypeError(f"tmax must be a float or a tensor, got {type(tmax).__name__}")
        o4, d4 = self._pack_rays(org, dir, tmax)
        n = o4.shape[0]
        out = torch.empty(n, dtype=torch.bool, device=o4.device)
        self._check(N.lib().ptap_query_occluded(self.h, o4.data_ptr(), d4.data_ptr(), n, out.data_ptr(), self._stream_handle()), "query_occluded")
        return out

    # -- parity entry points -------------------------------------------------------------------------------------
    def trace(self, rays_od, counts: bool = False):
        rays_od = np.ascontiguousarray(rays_od, np.float32).reshape(-1, 6)
        out = np.zeros(len(rays_od), N.HIT)
        if counts:
            cnt = np.zeros((len(rays_od), 4), np.int32)
            self._check(N.lib().ptap_trace_count(self.h, N.ptr(rays_od), len(rays_od), N.ptr(out), N.ptr(cnt)), "trace_count")
            return out, cnt
        self._check(N.lib().ptap_trace(self.h, N.ptr(rays_od), len(rays_od), N.ptr(out)), "trace")
        return out

    def shade(self, paths, it: int, remaining: int):
        paths = np.ascontiguousarray(paths, N.PATH_IN)
        out = np.zeros(len(paths), N.PATH_OUT); order = np.full(len(paths), -1, np.int32); n_alive = C.c_int32(0)
        self._check(N.lib().ptap_shade(self.h, N.ptr(paths), len(paths), it, remaining, N.ptr(out), N.ptr(order), C.byref(n_alive)), "shade")
        return out, order[:n_alive.value]

    def render_probe(self, it: int, round_: int):
        """The wavefront of round `round_` of iteration `it` as ptap_render enqueues it (production kernel instantiations, one lane):
        returns (rays n x 6, pixels n, hits n).  Leaves the film unspecified; call frame_begin() before rendering again."""
        cap = self.W * self.H
        rays = np.zeros((cap, 6), np.float32); pix = np.zeros(cap, np.int32); hits = np.zeros(cap, N.HIT); n = C.c_int32(0)
        self._check(N.lib().ptap_render_probe(self.h, it, round_, N.ptr(rays), N.ptr(pix), N.ptr(hits), cap, C.byref(n)), "render_probe")
        return rays[:n.value], pix[:n.value], hits[:n.value]

    def bench_trace(self, rays_od, reps: int = 10) -> float:
        rays_od = np.ascontiguousarray(rays_od, np.float32).reshape(-1, 6)
        ms = C.c_float(0)
        self._check(N.lib().ptap_bench_trace(self.h, N.ptr(rays_od), len(rays_od), reps, C.byref(ms)), "bench_trace")
        return ms.value

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
