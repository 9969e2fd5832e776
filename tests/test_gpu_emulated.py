"""PTAP_ACCEL_GRID_EMULATED (csrc/trace_emu.cu): the RESULTS of the reference's grid walk - oracle tier R0, its misses and early exits
included - computed through the BVH (all hits of a model, then a replay of the walk's voxel sequence over the voxel boxes of the hit
triangles).  The contract is bit equality with the walk on everything: ids, t, u, v, distance, whole films."""
import numpy as np
import pytest

from conftest import have_gpu
from test_gpu_trace import _random_rays, assert_hits_equal

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_gpu(), reason="no CUDA device")]


@pytest.fixture(scope="module")
def renderer(gpu_scene):
    from pathtracerap_b200 import ACCEL_GRID_EMULATED, Renderer
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_GRID_EMULATED)      # no BVH in the scene: built on the device at this call
    r.allocateOnGPU(gpu_scene)
    yield r
    r.free()


def test_emulated_vs_reference_golden(renderer, golden_trace):
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED
    renderer.set_accel(ACCEL_GRID_EMULATED)
    got = renderer.trace(golden_trace["rays"])
    assert_hits_equal(got, golden_trace["r0"], "emulated walk vs reference R0 (golden)")
    assert not np.array_equal(golden_trace["r0"]["tri"], golden_trace["r1"]["tri"])      # the fixture does hold rays the walk loses
    renderer.set_accel(ACCEL_GRID_COMPAT)
    assert_hits_equal(got, renderer.trace(golden_trace["rays"]), "emulated walk vs k_trace_grid")


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_emulated_random_rays_vs_oracle(renderer, oracle_scene, seed):
    """Origins anywhere in the room (inside mesh boxes too: the walk then starts BEHIND the origin), un-normalised directions,
    zero components and axis-parallel rays (the reference's slab test is not geometric there)."""
    from pathtracerap_b200 import ACCEL_GRID_EMULATED
    rays = _random_rays(300_000, seed)
    renderer.set_accel(ACCEL_GRID_EMULATED)
    got, cnt = renderer.trace(rays, counts=True)
    assert_hits_equal(got, oracle_scene.trace(rays, 0), "emulated walk vs oracle R0 (random rays)")
    assert_hits_equal(renderer.trace(rays), got, "UV build vs counting build")
    # nodes visited, voxels replayed (register arithmetic only: nothing is fetched), triangles tested per ray - against the walk's
    # ~40 voxel fetches and ~32 triangle tests
    assert cnt[:, 2].mean() < 12 and cnt[:, 1].mean() < 45


def test_emulated_with_host_bvh_and_device_grids(gpu_scene, oracle_scene, golden_trace):
    """Same answers whichever builder made the tree and the grids: host SAH tree + host grids, then the grids rebuilt on the device."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_EMULATED, Renderer
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(gpu_scene)
    rays = _random_rays(100_000, 7)
    want = oracle_scene.trace(rays, 0)
    r.set_accel(ACCEL_GRID_EMULATED)
    assert_hits_equal(r.trace(rays), want, "host SAH tree + host grids")
    r.build_grids_device(gpu_scene, 25, 25, 25)
    r.set_accel(ACCEL_GRID_EMULATED)
    assert_hits_equal(r.trace(rays), want, "host SAH tree + device grids")
    r.free()


def test_emulated_film_is_the_walks_film(gpu_scene):
    """Whole frames, multi-lane schedule, first-hit cache on and off: the film must equal k_trace_grid's bit for bit."""
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, Renderer
    W, H, depth, iters = 320, 240, 8, 6
    films = {}
    for accel in (ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED):
        r = Renderer(width=W, height=H, depth=depth, accel=accel, first_hit_cache=True)
        r.allocateOnGPU(gpu_scene)
        for cache in (True, False):
            r.set_params(W, H, depth, first_hit_cache=cache)
            r.frame_begin(); r.render(0, iters); r.sync()
            films[(accel, cache)] = (r.film().copy(), r.stats()["rays_traced"], list(r.stats()["active_per_round"]))
            if accel == ACCEL_GRID_EMULATED:
                st = r.stats()
                full, walked = st["rays_reemulated"] / st["rays_traced"], st["rays_walked"] / st["rays_traced"]
                print(f"emulated walk, cache={cache}: {full:.4%} of the rays emulated in full, {walked:.4%} answered by the walk itself")
                assert 0 < full < 0.05                       # the rays on which the walk is not a closest-hit query, and nothing like all of them
                assert walked < 0.001                        # only rays with more than 8 hits in one model are ever walked
        r.free()
    for cache in (True, False):
        a, b = films[(ACCEL_GRID_COMPAT, cache)], films[(ACCEL_GRID_EMULATED, cache)]
        assert a[1] == b[1] and a[2] == b[2]
        assert np.array_equal(a[0], b[0]), f"cache={cache}: {(a[0] != b[0]).any(axis=-1).sum()} pixels differ"


def _stacked_scene(copies):
    """One model whose mesh is `copies` coincident copies of two big triangles (plus a floor quad so that the grid has more than one
    layer): a ray through them hits `copies` triangles of ONE model, more than the emulation keeps per (ray, model)."""
    from pathtracerap_b200 import DIFFUSE, Scene, VERTEX
    quad = np.array([[-1, -1, 0], [1, -1, 0], [1, 1, 0], [-1, 1, 0]], np.float32)
    verts, idx = [], []
    for c in range(copies):
        base = len(verts)
        verts += [tuple(p) for p in quad]
        idx += [(base, base + 1, base + 2), (base, base + 2, base + 3)]
    base = len(verts)
    verts += [(-1, -1, -1), (1, -1, -1), (1, 1, -1), (-1, 1, -1)]
    idx += [(base, base + 1, base + 2), (base, base + 2, base + 3)]
    v = np.zeros(len(verts), VERTEX)
    v["position"] = np.array(verts, np.float32); v["normal"] = (0, 0, 1)
    s = Scene.empty()
    mi = s.add_mesh(v, np.array(idx, np.int32))
    s.add_model(mi, translate=(3, 2, 1), rotate_y_degrees=20.0, scale=(50, 40, 30), material=DIFFUSE)
    s.add_model(mi, translate=(-80, 10, -5), rotate_y_degrees=-35.0, scale=(20, 60, 10), material=DIFFUSE)
    s.build_grids(25, 25, 25)
    return s


@pytest.mark.parametrize("copies", [3, 12, 30])
def test_more_hits_than_slots_goes_to_the_walk(port, copies):
    """3 coincident copies stay inside the fast path; with 12, every ray through the quad has 12 (24 on the diagonal) hits in one model -
    beyond the 8 the replay keeps - and is emulated in full (k_emu_full keeps 20); with 30 it must be answered by the walk itself in the
    last launch.  All must equal the oracle's R0, exact-t ties included (coincident triangles have bit-equal t: the lowest id listed
    first wins, Renderer.cpp:209)."""
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, Renderer
    s = _stacked_scene(copies)
    a = s.arrays()
    osc = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    rs = np.random.RandomState(5)
    n = 60_000
    o = np.stack([rs.uniform(-150, 100, n), rs.uniform(-80, 80, n), rs.uniform(-100, 100, n)], 1)
    tgt = np.stack([rs.uniform(-120, 60, n), rs.uniform(-50, 50, n), rs.uniform(-40, 40, n)], 1)
    rays = np.concatenate([o, tgt - o], 1).astype(np.float32)
    want = osc.trace(rays, 0)
    assert (want["model"] >= 0).mean() > 0.2
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_GRID_EMULATED)
    r.allocateOnGPU(s)
    assert_hits_equal(r.trace(rays), want, f"{copies} coincident copies, emulated")
    r.set_accel(ACCEL_GRID_COMPAT)
    assert_hits_equal(r.trace(rays), want, f"{copies} coincident copies, walked")
    # the production instantiation too: one probed round of a frame whose camera looks at the models
    r.set_accel(ACCEL_GRID_EMULATED)
    r.set_params(96, 64, 3, first_hit_cache=False)
    r.set_camera(origin=(0.0, 0.0, 300.0), plane_min=(-120.0, -80.0, 100.0), span=(240.0, 160.0))
    rays_p, _, hits_p = r.render_probe(0, 0)
    want_p = osc.trace(rays_p, 0)
    for f in ("model", "tri", "t_model", "dist"):
        assert np.array_equal(hits_p[f], want_p[f]), f
    r.free()


def test_lists_that_are_not_boxes_are_refused(gpu_scene):
    """The emulation relies on box-shaped, ascending lists (Scene.cpp:357-374).  A grid whose lists were edited by hand is walked, not
    emulated: ptap_build_accel(PTAP_ACCEL_GRID_EMULATED) fails with PTAP_E_UNSUPPORTED and PTAP_ACCEL_GRID_COMPAT keeps working."""
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, PtapError, Renderer, Scene
    a = gpu_scene.arrays()
    vox, refs = a["voxels"].copy(), a["refs"].copy()
    # take a triangle listed in many voxels and drop it from the list of the middle one: its bounding box of voxels stays, one listing is gone
    tri = int(np.bincount(refs).argmax())
    listing = [c for c in np.flatnonzero(vox["end"] > vox["start"]) if tri in refs[vox["start"][c]:vox["end"][c]]]
    assert len(listing) >= 9
    k = int(listing[len(listing) // 2])
    s0, e0 = int(vox["start"][k]), int(vox["end"][k])
    keep = [t for t in refs[s0:e0] if t != tri]
    refs[s0:s0 + len(keep)] = keep
    vox["end"][k] = s0 + len(keep)
    s = Scene.from_arrays(a["models"], a["meshes"], a["vertices"], a["triangles"], a["grids"], vox, refs)
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_GRID_COMPAT)
    r.allocateOnGPU(s)
    with pytest.raises(PtapError, match="box-shaped"):
        r.set_accel(ACCEL_GRID_EMULATED)
    r.set_accel(ACCEL_GRID_COMPAT)
    assert len(r.trace(_random_rays(1000, 3))) == 1000
    # descending order inside one voxel: refused as well
    vox, refs = a["voxels"].copy(), a["refs"].copy()
    k = int(np.flatnonzero(vox["end"] - vox["start"] >= 2)[0])
    s0, e0 = int(vox["start"][k]), int(vox["end"][k])
    refs[s0:e0] = refs[s0:e0][::-1].copy()
    s2 = Scene.from_arrays(a["models"], a["meshes"], a["vertices"], a["triangles"], a["grids"], vox, refs)
    r.allocateOnGPU(s2)
    with pytest.raises(PtapError, match="box-shaped"):
        r.set_accel(ACCEL_GRID_EMULATED)
    r.free()


def test_emulated_on_the_million_triangle_mesh(libptap):
    """BASELINE configs[3]'s mesh (1.3 M triangles) through the reference's fixed 25^3 grid: ~84 triangles per voxel, and rays that graze the
    displaced surface cross it dozens of times (more hits in one model than the fast path or the shared-memory part of k_emu_full keep).
    GPU against GPU: the emulation must equal the walk on camera rays, bounce rays and rays aimed at the silhouette."""
    import bench
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_EMULATED, Renderer
    from test_gpu_large import _bounce_rays, _camera_rays
    scene, arrays = bench.build_scene("mesh1m")
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(scene)
    r.build_grids_device(scene, 25, 25, 25)
    cam = _camera_rays(320, 180)
    rs = np.random.RandomState(17)
    # tangent rays: from outside towards points at one displaced radius from the sphere's centre, perpendicular to the radius
    n = 20_000
    c = np.array([25.0, 230.0, -50.0]); radius = 250.0            # bench.ICO_MODEL: radius 1000 x scale 0.25, displaced by +-5 %
    u = rs.randn(n, 3); u /= np.linalg.norm(u, axis=1, keepdims=True)
    w = np.cross(u, rs.randn(n, 3)); w /= np.linalg.norm(w, axis=1, keepdims=True)
    p = c + u * (radius * rs.uniform(0.95, 1.05, (n, 1)))
    graze = np.concatenate([p - w * 400.0, w], 1).astype(np.float32)
    rays = np.concatenate([cam, _bounce_rays(40_000, 12), graze])
    walked = r.trace(rays)
    assert (walked["model"] == len(arrays["models"]) - 1).mean() > 0.2
    r.set_accel(ACCEL_GRID_EMULATED)
    assert_hits_equal(r.trace(rays), walked, "mesh1m 25^3: emulated vs walked")
    r.free()


DENSE_SHAPES = [(25, 25, 25), (64, 64, 64), (160, 160, 160), (96, 40, 160)]


@pytest.mark.parametrize("shape", DENSE_SHAPES, ids=[str(s[0]) if s[0] in (25, 64) else "x".join(map(str, s)) for s in DENSE_SHAPES])
def test_emulated_on_a_dense_mesh(libptap, port, shape):
    """An 82 k-triangle displaced icosphere in the room (BASELINE configs[1]) through grids built ON THE DEVICE: hundreds of triangles per
    voxel at 25^3, a handful at 64^3, less than one at the benchmarked 160^3, and a grid whose axes differ.  The emulation must equal the
    walk (GPU against GPU on 400 k camera + bounce rays, and a whole frame), and both the oracle's R0 on a subset."""
    import bench
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, Renderer
    from test_gpu_large import _bounce_rays, _camera_rays
    scene, arrays = bench.build_scene("mesh100k")
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)        # uploaded without grids; device-built tree
    r.allocateOnGPU(scene)
    r.build_grids_device(scene, *shape)
    cam = _camera_rays(640, 360)
    rays = np.concatenate([cam, _bounce_rays(170_000, 11)])
    walked = r.trace(rays)
    r.set_accel(ACCEL_GRID_EMULATED)
    emulated = r.trace(rays)
    assert_hits_equal(emulated, walked, f"mesh100k {shape}: emulated vs walked")
    assert (walked["model"] == len(arrays["models"]) - 1).mean() > 0.2
    sub = rays[:: len(rays) // 3000]
    oscene = port.OracleScene(arrays, grid_dim=shape)
    assert_hits_equal(r.trace(sub), oscene.trace(sub, 0), f"mesh100k {shape}: emulated vs oracle R0")
    W, H, depth, iters = 320, 180, 5, 4
    films = []
    for accel in (ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED):
        r.set_accel(accel)
        r.set_params(W, H, depth, first_hit_cache=True)
        r.frame_begin(); r.render(0, iters); r.sync()
        films.append(r.film().copy())
    assert np.array_equal(films[0], films[1])
    r.free()
