"""Inputs and outputs of the comparisons between the C restatement and the compiled reference on scenes the bundled fixtures
do not hold: random rotated / non-uniformly scaled instances with all five material branches, a dense displaced icosphere, and
the BMP writer.  tools/make_golden.py stores the outputs in tests/golden/live_scenes.npz; tests/test_oracle_golden.py computes
them again with the C restatement (and, where oracle/_ref is built, with the reference itself) and compares.

TEST INFRASTRUCTURE, like the rest of oracle/.
"""
from __future__ import annotations

import hashlib
import os
import tempfile

import numpy as np

from . import port, ref
from .ref import MODEL

INSTANCE_SCENES = ((24, 3), (7, 8))         # (instances, seed)
FRAME = (64, 48, 5, 2)                      # W, H, depth, iterations of the wavefront on the instance scenes
BMP = (96, 64, 5, 3)                        # W, H, depth, iterations of the film the BMP writers store


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def random_instances(golden_scene, n, seed):
    """n instances of the three bundled meshes under random rotations, non-uniform scales and translations (column-major matrices)."""
    rs = np.random.RandomState(seed)
    models = np.zeros(n, MODEL)
    for k in range(n):
        a = rs.randn(3); a /= np.linalg.norm(a)
        t = np.deg2rad(rs.uniform(0, 360)); c, s = np.cos(t), np.sin(t)
        K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        R = np.eye(3) * c + s * K + (1 - c) * np.outer(a, a)
        M = np.eye(4)
        M[:3, :3] = R @ np.diag(rs.uniform(0.02, 0.12, 3) * (0.3 if k % 3 == 0 else 1.0))
        M[:3, 3] = rs.uniform(-500, 500, 3) + [0, 0, 300]
        models[k]["mesh_index"] = k % 3
        models[k]["model_to_world"] = M.T.astype(np.float32).reshape(16)
        models[k]["world_to_model"] = np.linalg.inv(M.astype(np.float32).astype(np.float64)).T.astype(np.float32).reshape(16)
        models[k]["mat"]["type"] = [0, 6, 5, 2, 4][k % 5]          # DIFFUSE, METAL, COAT, REFLECTIVE, EMISSIVE
        models[k]["mat"]["color"] = rs.uniform(0.2, 0.99, 3)
    return models


def instance_scene(golden_scene, n, seed):
    """(scene arrays, rays) of one random-instance scene: 20,000 seeded rays, the first 200 with a zero x direction."""
    g = golden_scene
    arrays = {"models": random_instances(g, n, seed), "meshes": g["meshes"], "vertices": g["vertices"], "triangles": g["triangles"]}
    rs = np.random.RandomState(seed)
    o = rs.uniform(-700, 700, (20000, 3)) + [0, 0, 300]
    d = rs.uniform(-400, 400, (20000, 3)) + [0, 0, 300] - o
    d[:200, 0] = 0.0
    return arrays, np.concatenate([o, d], 1).astype(np.float32)


def dense_scene():
    """(scene arrays, rays): three instances of a displaced icosphere (5120 triangles, libptap's host-side generator, no GPU needed),
    so that voxels hold many references and the 3D-DDA early exit matters; 6,000 seeded rays."""
    from pathtracerap_b200 import DIFFUSE, Scene
    s = Scene.empty()
    mi = s.add_icosphere(4, radius=1000.0, displacement=0.05, seed=2)
    for k, (tr, sc) in enumerate([((0, 0, 0), 0.2), ((260, 40, -120), 0.12), ((-240, -60, 80), 0.3)]):
        s.add_model(mi, translate=tr, rotate_y_degrees=25.0 * k, scale=(sc, sc * (1 + 0.3 * k), sc), material=DIFFUSE, color=(0.7, 0.6, 0.5))
    a = s.arrays()
    assert len(a["triangles"]) == 5120
    rs = np.random.RandomState(4)
    o = rs.uniform(-600, 600, (6000, 3))
    d = rs.uniform(-250, 250, (6000, 3)) - o
    return {k: a[k] for k in ("models", "meshes", "vertices", "triangles")}, np.concatenate([o, d], 1).astype(np.float32)


class Port:
    """The C restatement (oracle/ptap_oracle.c)."""
    def scene(self, a): return port.OracleScene(a)
    def arrays(self, s): return s.arrays()
    def trace(self, s, rays, mode): return s.trace(rays, mode)

    def frame(self, s, W, H, depth, iters, mode):
        w = port.OracleWavefront(s, W, H, depth, mode=mode)
        w.init_image()
        counts = [w.run_iteration(it) for it in range(iters)]
        img = w.image(); w.close()
        return counts, img

    def close(self, s): pass


class Reference:
    """The reference's own Renderer.cpp / Scene.cpp compiled for the host (oracle/_ref)."""
    def scene(self, a): return ref.RefScene.from_arrays(a["models"], a["meshes"], a["vertices"], a["triangles"])
    def arrays(self, s): return s.arrays()

    def trace(self, s, rays, mode):
        rr = ref.RefRenderer(s, 32, 32, 5)
        out = rr.trace_rays(rays, mode); rr.close()
        return out

    def frame(self, s, W, H, depth, iters, mode):
        rr = ref.RefRenderer(s, W, H, depth)
        rr.init_image()
        counts = [rr.run_iteration(it, mode=mode) for it in range(iters)]
        img = rr.image(); rr.close()
        return counts, img

    def close(self, s): s.close()


def reference_bmp(golden_scene):
    """(film, file bytes) of Renderer::renderImage (Renderer.cpp:15-63) run by the compiled reference on its own BMP-sized film."""
    W, H, depth, iters = BMP
    g = golden_scene
    s = ref.RefScene.from_arrays(g["models"], g["meshes"], g["vertices"], g["triangles"])
    rr = ref.RefRenderer(s, W, H, depth)
    rr.init_image()
    for it in range(iters):
        rr.run_iteration(it)
    film = rr.image()
    with tempfile.TemporaryDirectory() as d:
        rr.write_bmp(d, iters)
        data = open(os.path.join(d, "Render.bmp"), "rb").read()
    rr.close(); s.close()
    return film, data


def scenes(golden_scene, which=("instances", "dense")):
    """(key, scene arrays, rays, whether whole wavefront iterations are compared) of every scene of the comparisons."""
    out = []
    if "instances" in which:
        out += [(f"inst{n}_{seed}", *instance_scene(golden_scene, n, seed), True) for n, seed in INSTANCE_SCENES]
    if "dense" in which:
        out.append(("dense", *dense_scene(), False))
    return out


def outputs(impl, scene_list) -> dict:
    """Everything the comparisons check, as a flat dict of arrays: per scene the grid build (grids bytes, voxel and reference hashes),
    both trace tiers on the seeded rays (ids in full; distance, u and v of the hits as hashes), and for the instance scenes two whole
    wavefront iterations at both tiers (active rays per bounce and the film)."""
    out = {}
    for key, arrays, rays, frames in scene_list:
        s = impl.scene(arrays)
        a = impl.arrays(s)
        out[f"{key}_grids"] = np.ascontiguousarray(a["grids"])
        out[f"{key}_voxels_sha"] = np.array(sha(a["voxels"])); out[f"{key}_refs_sha"] = np.array(sha(a["refs"]))
        for mode in (0, 1):
            h = impl.trace(s, rays, mode)
            hit = h["model"] >= 0
            out[f"{key}_r{mode}_model"] = h["model"].astype(np.int32); out[f"{key}_r{mode}_tri"] = h["tri"].astype(np.int32)
            for f in ("dist", "u", "v"):
                out[f"{key}_r{mode}_{f}_sha"] = np.array(sha(h[f][hit]))
            if frames:
                W, H, depth, iters = FRAME
                counts, film = impl.frame(s, W, H, depth, iters, mode)
                out[f"{key}_frame{mode}_counts"] = np.array([c + [0] * (depth - len(c)) for c in counts], np.int32)
                out[f"{key}_frame{mode}_film"] = film
        impl.close(s)
    return out
