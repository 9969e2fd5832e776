"""Host-side logic on the CPU: the C ABI surface, scene building (Config.txt, OBJ, TRS, grids), the BVH builder's invariants and
the multi-rank sample partition (gloo, world_size 2).  No compute entry point is called: those need a B200 and fail loudly."""
import ctypes as C
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import GOLDEN, ROOT


def test_library_exports_every_declared_symbol(libptap):
    hdr = open(os.path.join(ROOT, "include", "ptap.h")).read()
    declared = sorted(set(re.findall(r"\b(ptap_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 40
    for name in declared:
        assert hasattr(libptap, name), f"{name} is declared in include/ptap.h but not exported by libptap.so"
    from pathtracerap_b200 import _native
    assert sorted(_native.EXPORTS) == declared


def test_no_cpu_fallback(libptap):
    """Without a device every compute path fails with PTAP_E_NO_DEVICE (-2) instead of falling back."""
    from conftest import have_gpu
    if have_gpu():
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    assert libptap.ptap_create(0, 0, C.byref(h)) == -2 and not h.value
    from pathtracerap_b200 import PtapError, Renderer
    with pytest.raises(PtapError):
        Renderer()


def test_grid_builder_matches_reference_golden(libptap, golden_scene):
    """ptap_scene_build_grids = Scene::addMeshesToGrid (Scene.cpp:318-396): byte-equal grids, voxels and refs."""
    from pathtracerap_b200 import Scene
    g = golden_scene
    s = Scene.from_arrays(g["models"], g["meshes"], g["vertices"], g["triangles"])
    s.build_grids(25, 25, 25)
    a = s.arrays()
    import hashlib
    assert a["grids"].tobytes() == g["grids"].tobytes()
    assert len(a["voxels"]) == int(g["nvoxels"]) and len(a["refs"]) == int(g["nrefs"])
    assert hashlib.sha256(a["voxels"].tobytes()).hexdigest() == str(g["voxels_sha"])      # the reference's own arrays, hashed by tools/make_golden.py
    assert hashlib.sha256(a["refs"].tobytes()).hexdigest() == str(g["refs_sha"])
    assert np.array_equal(a["models"]["grid_index"], g["models"]["grid_index"])


def test_compose_trs_matches_reference_matrices(libptap, golden_scene):
    """translate * rotate(Y) * scale and its glm::inverse, bit-equal to the matrices the reference's Scene.cpp computes."""
    from pathtracerap_b200 import Scene
    m2w, w2m = Scene.compose_trs((-250.0, 0.0, 100.0), 30.0, (0.125, 0.125, 0.125))
    assert m2w.shape == (16,) and np.isfinite(m2w).all() and np.isfinite(w2m).all()
    prod = m2w.reshape(4, 4).T.astype(np.float64) @ w2m.reshape(4, 4).T.astype(np.float64)
    assert np.allclose(prod, np.eye(4), atol=1e-5)


NODE = np.dtype([("p", "<f4", 3), ("pad", "<i4"), ("link", "<i4", 4), ("planes", "<f4", (3, 2, 4))])          # PtapBvhNode, include/ptap.h


def _bvh_of(scene):
    scene.build_bvh()
    v = scene.view()
    assert NODE.itemsize == 128
    nodes = np.frombuffer((C.c_char * (v.n_bvh_nodes * 128)).from_address(v.bvh_nodes), NODE).copy()
    tri_id = np.frombuffer((C.c_char * (v.n_bvh_tris * 4)).from_address(v.bvh_tri_id), np.int32).copy()
    roots = np.frombuffer((C.c_char * (v.n_bvh_roots * 4)).from_address(v.bvh_mesh_root), np.int32).copy()
    assert v.bvh_depth >= 1 and v.n_tri_recs == v.n_bvh_tris
    return nodes, tri_id, roots


def _slots(nd):
    """(lo, hi, link) of the used child slots of a 4-wide node, decoded independently of the library: plane = p + offset in double
    (an unused slot holds an inverted box)."""
    out = []
    p, pl = nd["p"].astype(np.float64), nd["planes"].astype(np.float64)
    for k in range(4):
        if pl[0, 0, k] <= pl[0, 1, k]:
            out.append((p + pl[:, 0, k], p + pl[:, 1, k], int(nd["link"][k])))
    return out


def _check_bvh(nodes, tri_id, roots, arrays):
    verts, tris, meshes = arrays["vertices"]["position"].astype(np.float64), arrays["triangles"]["v"], arrays["meshes"]
    assert sorted(tri_id.tolist()) == list(range(len(tris)))            # a permutation: every triangle in exactly one leaf
    e = 0.0056                                                          # the predicate's band (bvh_build.cpp kBandEps)
    max_depth = 0
    visited = set()
    for mi, root in enumerate(roots):
        if root < 0:
            continue
        seen_leaf = []
        big = np.full(3, 1e300)
        stack = [(int(root), 1, -big, big)]
        while stack:
            n, d, alo, ahi = stack.pop()                                # (alo, ahi): intersection of every box above this node
            assert n not in visited                                     # a tree: no node is reachable twice
            visited.add(n)
            max_depth = max(max_depth, d)
            slots = _slots(nodes[n])
            assert 1 <= len(slots) <= 4
            for lo, hi, l in slots:
                lo, hi = np.maximum(lo, alo), np.minimum(hi, ahi)
                if l >= 0:
                    assert l > n                                        # parents precede their children
                    stack.append((l, d + 1, lo, hi))
                else:
                    code = ~l
                    first, cnt = code >> 3, (code & 7) + 1
                    assert 1 <= cnt <= 8 and code < 0x20000000
                    for k in range(first, first + cnt):
                        t = tris[tri_id[k]]
                        assert meshes[mi]["t_start"] <= tri_id[k] < meshes[mi]["t_end"]
                        p0, p1, p2 = verts[t[0]], verts[t[1]], verts[t[2]]
                        e1, e2 = p1 - p0, p2 - p0
                        for (u, v) in ((-e, -e), (1 + 2 * e, -e), (-e, 1 + 2 * e)):     # corners of the fattened triangle
                            q = p0 + u * e1 + v * e2
                            assert (q >= lo).all() and (q <= hi).all(), "a box above the leaf does not bound the predicate's tolerance band"
                        seen_leaf.append(k)
        assert len(seen_leaf) == meshes[mi]["t_end"] - meshes[mi]["t_start"]
    return max_depth


def test_bvh_builder_invariants_bundled(libptap, golden_scene):
    from pathtracerap_b200 import Scene
    g = golden_scene
    s = Scene.from_arrays(g["models"], g["meshes"], g["vertices"], g["triangles"])
    nodes, tri_id, roots = _bvh_of(s)
    depth = _check_bvh(nodes, tri_id, roots, g)
    assert 3 * depth + 12 <= 160                                         # kBvhStack (device_types.h): up to 3 pushes per level
    assert s.validate_bvh() == (0, depth)                                # the library's own checker agrees


def test_bvh_builder_invariants_icosphere(libptap):
    from pathtracerap_b200 import Scene
    s = Scene.empty()
    mi = s.add_icosphere(4, radius=1000.0, displacement=0.05, seed=3)    # 5120 triangles
    s.add_model(mi)
    nodes, tri_id, roots = _bvh_of(s)
    a = s.arrays()
    assert len(a["triangles"]) == 20 * 4 ** 4
    depth = _check_bvh(nodes, tri_id, roots, a)
    assert depth <= 20
    # degenerate input: many identical triangles (identical centroids force the split-by-count path)
    v = np.zeros(3, dtype=a["vertices"].dtype); v["position"] = [[0, 0, 0], [1000, 0, 0], [0, 1000, 0]]; v["normal"] = [[0, 0, 1000]] * 3
    s2 = Scene.empty()
    mi = s2.add_mesh(v, np.tile(np.array([[0, 1, 2]], np.int32), (37, 1)))
    s2.add_model(mi)
    nodes, tri_id, roots = _bvh_of(s2)
    _check_bvh(nodes, tri_id, roots, s2.arrays())


CONFIG = """
RESOLUTION
[320, 240]

ITER
7

DEPTH
6

DIFFUSE
white
[0.9, 0.8, 0.7]

EMISSIVE
lamp
[0.99, 0.99, 0.99]

BOX
room
[5.0, 5.0, 5.0]
[-5.0, -5.0, -5.0]
translate:[0, 1, 0]
rotateX:[0, 0, 0]
scale:[1, 1, 1]
material: white

SPHERE
ball
1.5
[0.5, 0, 0]
translate:[1, 2, 3]
scale:[2, 2, 2]
material: lamp

MESH
tri
one.obj
material: white
"""


def test_config_txt_parser(libptap, tmp_path):
    """Schema of the reference's Config.txt:1-31 (which no reference code reads; parity unpinned - DESIGN.md)."""
    from pathtracerap_b200 import DIFFUSE, EMISSIVE, PtapError, Scene
    (tmp_path / "one.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nv 1 1 0\nf 1 2 4 3\n")      # quad, no normals: fan + face normal
    cfg = tmp_path / "Config.txt"
    cfg.write_text(CONFIG)
    s = Scene(str(cfg))
    a = s.arrays()
    assert s.config_params() == {"W": 320, "H": 240, "iters": 7, "depth": 6}
    assert len(a["models"]) == 3 and len(a["meshes"]) == 3
    assert list(a["models"]["mat"]["type"]) == [DIFFUSE, EMISSIVE, DIFFUSE]
    assert np.allclose(a["models"]["mat"]["color"][0], [0.9, 0.8, 0.7])
    box, ball, quad = a["meshes"]
    assert box["t_end"] - box["t_start"] == 12 and np.allclose(box["bb_max"], 5000.0) and np.allclose(box["bb_min"], -5000.0)
    assert ball["t_end"] - ball["t_start"] == 20 * 4 ** 4
    assert np.allclose((ball["bb_min"] + ball["bb_max"]) / 2, [500.0, 0, 0], atol=20.0)       # the centre is folded into the vertices
    assert quad["t_end"] - quad["t_start"] == 2
    qn = a["vertices"]["normal"][quad["v_start"]:quad["v_end"]]
    assert np.allclose(qn, [[0, 0, 1000.0]] * 6)                                              # geometric normal, scaled like an import
    m = a["models"]["model_to_world"][1].reshape(4, 4).T
    assert np.allclose(m, [[2, 0, 0, 1], [0, 2, 0, 2], [0, 0, 2, 3], [0, 0, 0, 1]])
    assert len(a["grids"]) == 3 and len(a["voxels"]) == 3 * 25 ** 3
    assert s.config_camera() is None                                                          # no CAMERA_* key: the reference's camera
    cfg2 = tmp_path / "Config2.txt"
    cfg2.write_text(CONFIG + "\nCAMERA_ORIGIN\n[1, 2, 930]\n\nCAMERA_SPAN\n[16, 9]\n\nJITTER\n77\n")
    cam = Scene(str(cfg2)).config_camera()
    assert cam == dict(origin=(1.0, 2.0, 930.0), plane_min=(-10.0, -4.0, 900.0), span=(16.0, 9.0), jitter=True, jitter_seed=77)
    # errors are loud
    bad = tmp_path / "bad.txt"
    bad.write_text("TORUS\nx\n")
    with pytest.raises(PtapError):
        Scene(str(bad))
    bad.write_text("MESH\nm\nmissing.obj\n")
    with pytest.raises(PtapError):
        Scene(str(bad))


def test_reference_config_txt_parses(libptap, tmp_path):
    """The reference's own sample file (its MESH path points at a file that is not bundled).  The file belongs to the original
    PathTracerAP sources, which this repository does not carry: the test runs where PTAP_REFERENCE points at a checkout of them."""
    from oracle.ref import REFERENCE_ROOT
    src = os.path.join(REFERENCE_ROOT, "PathTracerAP", "Config.txt")
    if not os.path.exists(src):
        pytest.skip("needs the original PathTracerAP sources (PTAP_REFERENCE), which are not part of this repository")
    text = open(src).read()
    from pathtracerap_b200 import PtapError, Scene
    cfg = tmp_path / "Config.txt"
    cfg.write_text(text)
    try:
        s = Scene(str(cfg))
        assert len(s.arrays()["models"]) >= 2
    except PtapError:
        # only acceptable failure: the MESH block's OBJ file does not exist
        from pathtracerap_b200 import _native as N
        h = C.c_void_p()
        assert N.lib().ptap_scene_create_from_config(str(cfg).encode(), C.byref(h)) == -4


def test_obj_loader_edge_cases(libptap, tmp_path):
    from pathtracerap_b200 import PtapError, Scene
    s = Scene.empty()
    (tmp_path / "neg.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nvn 0 0 1\nf -3//-1 -2//-1 -1//-1\n# comment\n")
    mi = s.add_obj(str(tmp_path / "neg.obj"))
    a = s.arrays()
    assert mi == 0 and len(a["triangles"]) == 1 and np.allclose(a["vertices"]["position"][1], [1000, 0, 0])
    (tmp_path / "empty.obj").write_text("v 0 0 0\n")
    with pytest.raises(PtapError):
        s.add_obj(str(tmp_path / "empty.obj"))
    (tmp_path / "oob.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 9\n")
    with pytest.raises(PtapError):
        s.add_obj(str(tmp_path / "oob.obj"))
    with pytest.raises(PtapError):
        s.add_obj(str(tmp_path / "does_not_exist.obj"))


def test_obj_multi_object_quads_and_missing_normals(libptap, tmp_path):
    """Files beyond the bundled ones (SURVEY 8f row 1).  The reference keeps ONE Mesh per file and overwrites its index ranges for every
    aiMesh Assimp returns (Scene.cpp:240-252, 266, 277), so a multi-object file leaves only its LAST object reachable while the bounding
    box covers all of them - a bug, single-object files being the only ones it was run on.  This reader does the evident thing: `o` / `g`
    groups are concatenated into one mesh in file order, polygons are fan-triangulated (corner 0, k, k+1), corners without `vn` get the
    face's geometric normal scaled by BASE_MODEL_SCALE like imported normals (Scene.cpp:255-262), `vt` indices are skipped."""
    from pathtracerap_b200 import Scene
    (tmp_path / "multi.obj").write_text(
        "# two objects, a quad, a face without normals, texture indices\n"
        "o first\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvt 0 0\nvn 0 0 1\n"
        "f 1/1/1 2/1/1 3/1/1 4/1/1\n"
        "g second\no second\nv 0 0 2\nv 2 0 2\nv 0 2 2\n"
        "f 5 6 7\n"
        "f 5//1 7//1 6//1\n")
    s = Scene.empty()
    mi = s.add_obj(str(tmp_path / "multi.obj"))
    a = s.arrays()
    assert mi == 0 and len(a["meshes"]) == 1
    m = a["meshes"][0]
    assert (m["t_start"], m["t_end"], m["v_start"], m["v_end"]) == (0, 4, 0, 12)          # quad -> 2 triangles, + 2: every object is reachable
    P = a["vertices"]["position"] / 1000.0
    assert np.array_equal(a["triangles"]["v"], np.arange(12).reshape(4, 3))             # one vertex per face corner, in file order
    assert np.allclose(P[0:3], [[0, 0, 0], [1, 0, 0], [1, 1, 0]]) and np.allclose(P[3:6], [[0, 0, 0], [1, 1, 0], [0, 1, 0]])   # fan: (0,1,2), (0,2,3)
    assert np.allclose(P[6:9], [[0, 0, 2], [2, 0, 2], [0, 2, 2]])
    N = a["vertices"]["normal"]
    assert np.allclose(N[0:6], [[0, 0, 1000]] * 6)                                       # vn scaled by BASE_MODEL_SCALE
    assert np.allclose(N[6:9], [[0, 0, 1000]] * 3)                                       # no vn: geometric normal of (5,6,7), same scale
    assert np.allclose(N[9:12], [[0, 0, 1000]] * 3)                                      # explicit vn wins over the (opposite) winding
    assert np.allclose(m["bb_min"], [0, 0, 0]) and np.allclose(m["bb_max"], [2000, 2000, 2000])
    s.add_model(mi)
    s.build_grids(); s.build_bvh()
    assert s.validate_bvh()[0] == 0


def test_iteration_range_partition():
    from pathtracerap_b200.multi_gpu import iteration_range
    for iters in (0, 1, 7, 64, 1024):
        for world in (1, 2, 3, 8):
            spans = [iteration_range(r, world, iters) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == iters
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(e - b for b, e in spans) - min(e - b for b, e in spans) <= 1
    with pytest.raises(ValueError):
        iteration_range(2, 2, 8)


GLOO_WORKER = """
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
from pathtracerap_b200.multi_gpu import iteration_range, reduce_film
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
b, e = iteration_range(rank, world, 10)
# a stand-in "film": iteration k contributes the deterministic image k+1 (the real contribution depends only on k, Renderer.cpp:435)
film = torch.zeros(6 * 4 * 3)
for k in range(b, e):
    film += torch.full_like(film, float(k + 1))
reduce_film(film, 0)
if rank == 0:
    want = sum(range(1, 11))
    assert torch.equal(film, torch.full_like(film, float(want))), film[:4]
    print("REDUCE_OK", b, e)
dist.destroy_process_group()
"""


def test_two_rank_film_reduce_gloo(tmp_path):
    """N > 1 path on the CPU: two gloo ranks render disjoint iteration ranges and one reduce assembles the frame on rank 0."""
    w = tmp_path / "worker.py"
    w.write_text(textwrap.dedent(GLOO_WORKER.format(root=ROOT)))
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", str(w)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    assert "REDUCE_OK 0 5" in p.stdout


def test_bvh_builder_parallel_path(libptap):
    """Meshes of >= 65,536 triangles build their subtrees on worker threads (bvh_build.cpp); the stitched tree keeps every invariant."""
    from pathtracerap_b200 import Scene
    s = Scene.empty()
    mi = s.add_icosphere(6, radius=1000.0, displacement=0.05, seed=1)     # 81,920 triangles
    s.add_model(mi)
    nodes, tri_id, roots = _bvh_of(s)
    depth = _check_bvh(nodes, tri_id, roots, s.arrays())
    assert depth <= 16


def test_header_is_plain_c(tmp_path):
    """include/ptap.h is the drop-in boundary: it must compile as C99 (no C++ types, no CUDA headers) and keep the record sizes the
    reference's PODs have (SURVEY 8: Model 160, Mesh 40, Vertex 32, Triangle 12, Grid 28, Voxel 12, Material 24 bytes)."""
    import subprocess
    src = tmp_path / "abi.c"
    src.write_text('#include "ptap.h"\n#include <stdio.h>\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(PtapModel), sizeof(PtapMesh), sizeof(PtapVertex), '
                   'sizeof(PtapTriangle), sizeof(PtapGrid), sizeof(PtapVoxel), sizeof(PtapMaterial), sizeof(PtapBvhNode), sizeof(PtapStats)); return 0; }\n')
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert sizes[:8] == [160, 40, 32, 12, 28, 12, 24, 128]
    from pathtracerap_b200 import _native
    assert sizes[8] == C.sizeof(_native.Stats)


def test_reference_arm_arrays_equal_product_arrays(libptap, port):
    """bench.py's CPU arms build their scene WITHOUT the product library (oracle/synth.c); the arrays must be the product's, byte for byte:
    same synthetic mesh, same glm-composed model matrices, same bounding boxes - so that both arms time the same workload."""
    import bench
    for w in ("cornell", "mesh100k"):
        _, a = bench.build_scene(w)
        b = bench.reference_arrays(w)
        for k in ("models", "meshes", "vertices", "triangles"):
            assert np.ascontiguousarray(a[k]).tobytes() == np.ascontiguousarray(b[k]).tobytes(), f"{w}: {k} differ"
