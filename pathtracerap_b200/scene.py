"""Host-side scene: the Python mirror of the reference's `Scene` (Scene.h:21-39) over the C ABI."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _native as N

_ARRAYS = [("models", N.MODEL), ("meshes", N.MESH), ("vertices", N.VERTEX), ("triangles", N.TRIANGLE),
           ("grids", N.GRID), ("voxels", N.VOXEL), ("refs", np.dtype("<i4"))]


class Scene:
    """`Scene(config)` as main.cpp:14-15 constructs it.

    The reference ignores `config` and always builds its hard-coded scene (Scene.cpp:3); here `config` selects:
    a path to a Config.txt-style file (schema of Config.txt:1-31) is parsed; anything else - including the
    reference's own "Input data\\\\lucy.obj" - builds the hard-coded scene, loading the three bundled OBJ files
    from `root` (default: the current directory, like the reference).
    """

    def __init__(self, config: str | None = None, root: str | None = None, _handle=None):
        L = N.lib()
        self._keep = None
        if _handle is not None:
            self.h = _handle
            return
        h = C.c_void_p()
        if config is not None and os.path.isfile(config) and not config.lower().endswith(".obj"):
            rc = L.ptap_scene_create_from_config(config.encode(), C.byref(h))
            if rc != 0:
                raise N.PtapError(f"Scene({config!r}): error {rc}")
        else:
            rc = L.ptap_scene_create_builtin((root or os.getcwd()).encode(), C.byref(h))
            if rc != 0:
                raise N.PtapError(f"Scene builtin: error {rc}")
        self.h = h

    # -- alternative constructors -------------------------------------------------------------------------
    @classmethod
    def empty(cls) -> "Scene":
        h = C.c_void_p()
        N.lib().ptap_scene_create_empty(C.byref(h))
        return cls(_handle=h)

    @classmethod
    def from_arrays(cls, models, meshes, vertices, triangles, grids=None, voxels=None, refs=None, grid_dim=(25, 25, 25)) -> "Scene":
        keep = {
            "models": np.ascontiguousarray(models, N.MODEL), "meshes": np.ascontiguousarray(meshes, N.MESH),
            "vertices": np.ascontiguousarray(vertices, N.VERTEX), "triangles": np.ascontiguousarray(triangles, N.TRIANGLE),
        }
        v = N.SceneView()
        v.models, v.nmodels = N.ptr(keep["models"]), len(keep["models"])
        v.meshes, v.nmeshes = N.ptr(keep["meshes"]), len(keep["meshes"])
        v.vertices, v.nvertices = N.ptr(keep["vertices"]), len(keep["vertices"])
        v.triangles, v.ntriangles = N.ptr(keep["triangles"]), len(keep["triangles"])
        if grids is not None and len(grids):
            keep["grids"] = np.ascontiguousarray(grids, N.GRID); keep["voxels"] = np.ascontiguousarray(voxels, N.VOXEL)
            keep["refs"] = np.ascontiguousarray(refs, np.int32)
            v.grids, v.ngrids = N.ptr(keep["grids"]), len(keep["grids"])
            v.voxels, v.nvoxels = N.ptr(keep["voxels"]), len(keep["voxels"])
            v.refs, v.nrefs = N.ptr(keep["refs"]), len(keep["refs"])
        v.grid_dim = (C.c_int32 * 3)(*grid_dim)
        h = C.c_void_p()
        rc = N.lib().ptap_scene_create_from_view(C.byref(v), C.byref(h))
        if rc != 0:
            raise N.PtapError(f"Scene.from_arrays: error {rc}")
        return cls(_handle=h)

    # -- building ------------------------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc != 0:
            raise N.PtapError(f"{what}: error {rc}: {N.lib().ptap_scene_last_error(self.h).decode()}")

    def add_obj(self, path: str) -> int:
        mi = C.c_int32(-1)
        self._check(N.lib().ptap_scene_add_obj(self.h, path.encode(), C.byref(mi)), f"add_obj({path})")
        return mi.value

    def add_mesh(self, vertices, indices) -> int:
        vertices = np.ascontiguousarray(vertices, N.VERTEX); indices = np.ascontiguousarray(indices, np.int32).reshape(-1, 3)
        mi = C.c_int32(-1)
        self._check(N.lib().ptap_scene_add_mesh(self.h, N.ptr(vertices), len(vertices), N.ptr(indices), len(indices), C.byref(mi)), "add_mesh")
        return mi.value

    def add_icosphere(self, level: int, radius: float = 1000.0, displacement: float = 0.05, seed: int = 1) -> int:
        mi = C.c_int32(-1)
        self._check(N.lib().ptap_scene_add_icosphere(self.h, level, radius, displacement, seed, C.byref(mi)), "add_icosphere")
        return mi.value

    @staticmethod
    def compose_trs(translate, rotate_y_degrees, scale):
        t = np.ascontiguousarray(translate, np.float32); s = np.ascontiguousarray(scale, np.float32)
        m2w = np.zeros(16, np.float32); w2m = np.zeros(16, np.float32)
        N.lib().ptap_compose_trs(N.ptr(t), float(rotate_y_degrees), N.ptr(s), N.ptr(m2w), N.ptr(w2m))
        return m2w, w2m

    def add_model(self, mesh_index: int, translate=(0, 0, 0), rotate_y_degrees=0.0, scale=(1, 1, 1), material=N.DIFFUSE,
                  color=(0.99, 0.99, 0.99), model_to_world=None, world_to_model=None) -> int:
        if model_to_world is None:
            model_to_world, world_to_model = self.compose_trs(translate, rotate_y_degrees, scale)
        m2w = np.ascontiguousarray(model_to_world, np.float32).reshape(16)
        w2m = None if world_to_model is None else np.ascontiguousarray(world_to_model, np.float32).reshape(16)
        mat = np.zeros(1, N.MATERIAL); mat["type"] = material; mat["color"] = color
        idx = C.c_int32(-1)
        self._check(N.lib().ptap_scene_add_model(self.h, mesh_index, N.ptr(m2w), None if w2m is None else N.ptr(w2m), N.ptr(mat), C.byref(idx)), "add_model")
        return idx.value

    def build_grids(self, gx=25, gy=25, gz=25):
        self._check(N.lib().ptap_scene_build_grids(self.h, gx, gy, gz), "build_grids")

    def build_bvh(self):
        """One BVH per mesh, built on the host as part of scene construction (like addMeshesToGrid for the grid)."""
        self._check(N.lib().ptap_scene_build_bvh(self.h), "build_bvh")

    def pack(self):
        """The upload-bound triangle records in page-locked memory, without a host BVH (for trees built on the GPU): uploads become copies."""
        self._check(N.lib().ptap_scene_pack_triangles(self.h), "pack_triangles")

    def validate_bvh(self) -> tuple[int, int]:
        """(violations, depth) of the host-built BVH: 0 violations = every triangle's tolerance band lies inside every compressed box above it."""
        bad = C.c_int64(-1); depth = C.c_int32(0)
        self._check(N.lib().ptap_scene_validate_bvh(self.h, C.byref(bad), C.byref(depth)), "validate_bvh")
        return bad.value, depth.value

    # -- the seven public vectors (Scene.h:26-32) as numpy copies -----------------------------------------------
    def view(self) -> N.SceneView:
        v = N.SceneView()
        self._check(N.lib().ptap_scene_view(self.h, C.byref(v)), "view")
        return v

    def arrays(self) -> dict:
        v = self.view()
        out = {}
        for name, dt in _ARRAYS:
            n = getattr(v, "n" + name)
            p = getattr(v, name)
            if n and p:
                buf = (C.c_char * (n * dt.itemsize)).from_address(p)
                out[name] = np.frombuffer(buf, dt, n).copy()
            else:
                out[name] = np.zeros(0, dt)
        out["grid_dim"] = tuple(v.grid_dim)
        return out

    def __getattr__(self, name):
        if name in {n for n, _ in _ARRAYS}:
            return self.arrays()[name]
        if name == "per_voxel_data_pool":
            return self.arrays()["refs"]
        raise AttributeError(name)

    def set_models(self, models):
        """Overwrite the models in place (material / transform edits, SURVEY.md A.3b).  A renderer that has uploaded the scene takes
        the edits through Renderer.update_models."""
        models = np.ascontiguousarray(models, N.MODEL)
        v = self.view()
        if len(models) != v.nmodels:
            raise ValueError("set_models: the number of models cannot change")
        C.memmove(N.lib().ptap_scene_models(self.h), N.ptr(models), models.nbytes)

    def config_params(self):
        out = np.zeros(4, np.int32)
        N.lib().ptap_scene_config_params(self.h, N.ptr(out))
        return {"W": int(out[0]), "H": int(out[1]), "iters": int(out[2]), "depth": int(out[3])}

    def config_camera(self):
        """CAMERA_* / JITTER keys of a parsed Config.txt as keyword arguments for Renderer.set_camera, or None when absent."""
        cam = N.Camera()
        if not N.lib().ptap_scene_config_camera(self.h, C.byref(cam)):
            return None
        return dict(origin=tuple(cam.origin), plane_min=tuple(cam.plane_min), span=tuple(cam.span), jitter=bool(cam.jitter), jitter_seed=int(cam.jitter_seed))

    def close(self):
        if getattr(self, "h", None):
            N.lib().ptap_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
