"""CPU model of PTAP_ACCEL_GRID_EMULATED (csrc/trace_emu.cu): the algorithm, not the kernels.

The GPU path claims that the reference's grid walk (oracle tier R0: Renderer.cpp:238-360, its misses and early exits included) follows
from three facts - only triangles the ray really hits influence a walk; a triangle is listed in a box of voxels, so a model's walk can be
replayed from the set of ALL its hits; and when the replayed walk of the model holding the exact closest hit returns that hit's t, the
reference's answer is that model with the walk's triangle.  This file states that algorithm in Python on top of three probes of the
oracle (all hits of one model under the reference's predicate, the voxel sequence of one model's walk when nothing is hit, the
model-t -> world-distance conversion) and requires bit equality with the oracle's own walk over the voxel LISTS, on the reference's
coded scene and on a scene of coincident meshes (exact-t ties).  It runs without a GPU; tests/test_gpu_emulated.py holds the kernels to
the same oracle."""
import numpy as np
import pytest

FLOAT_MAX = np.float32(9999999.0)


def voxel_boxes(scene):
    """Per global triangle the index box of the voxels that list it (csrc/grid_device.cu: gridTriBoxes), with the same shape checks:
    listings = box volume, one grid per triangle, ascending lists."""
    a = scene.arrays()
    gx, gy, gz = [int(v) for v in scene.c.grid_dim]
    ncell = gx * gy * gz
    nt = len(a["triangles"])
    lo = np.full((nt, 3), 1 << 30, np.int64); hi = np.full((nt, 3), -1, np.int64); cnt = np.zeros(nt, np.int64); gid = np.full(nt, -1, np.int64)
    for g, grid in enumerate(a["grids"]):
        v0 = int(grid["v_start"])
        vox = a["voxels"][v0:v0 + ncell]
        for l in np.flatnonzero(vox["end"] > vox["start"]):
            ids = a["refs"][vox["start"][l]:vox["end"][l]]
            assert (np.diff(ids) > 0).all(), "voxel lists must ascend"
            xyz = np.array([l % gx, (l // gx) % gy, l // (gx * gy)])
            lo[ids] = np.minimum(lo[ids], xyz); hi[ids] = np.maximum(hi[ids], xyz); cnt[ids] += 1
            assert ((gid[ids] == -1) | (gid[ids] == g)).all(), "a triangle listed by two grids"
            gid[ids] = g
    listed = cnt > 0
    assert (np.prod(hi[listed] - lo[listed] + 1, axis=1) == cnt[listed]).all(), "listings must fill the triangle's voxel box"
    return lo, hi, listed


def replay(path, hits_tri, hits_t, lo, hi, listed):
    """The walk of one model over its hits: (found, triangle, t).  `path` is the voxel sequence of the walk; a voxel "has a hit" when it
    lies in the voxel box of a hit triangle; the walk remembers the last such voxel and stops once it is more than two voxels away from it
    (Renderer.cpp:321-329); a hit takes effect at the first voxel that lists it, ascending triangle id inside a voxel (Renderer.cpp:209)."""
    best_t, best_tri, inter, last = FLOAT_MAX, -1, False, None
    seen = set()
    for v in path:
        inside = [k for k in range(len(hits_tri)) if listed[hits_tri[k]] and (lo[hits_tri[k]] <= v).all() and (v <= hi[hits_tri[k]]).all()]
        for k in sorted(inside, key=lambda k: hits_tri[k]):
            if k in seen:
                continue
            seen.add(k)
            if best_t > hits_t[k]:                       # strict: the first one tested keeps an exact tie
                best_t, best_tri = hits_t[k], int(hits_tri[k])
        if inside:
            last, inter = v, True
        if inter and (np.abs(last - v) > 2).any():
            break
    return inter and best_tri >= 0, best_tri, best_t


def emulate(scene, ray, lo, hi, listed):
    """(model, triangle, t) of the reference's answer for one ray, computed the way the GPU path does, plus which route it took."""
    nm = scene.c.nmodels
    hits = [scene.model_hits(ray, m) for m in range(nm)]
    # exact closest hit (tier R1): per model the smallest t (lowest id on ties), across models the smallest exact distance (lowest model on ties)
    star = None
    for m in range(nm):
        tri, t = hits[m]
        ok = t < FLOAT_MAX
        if not ok.any():
            continue
        k = np.lexsort((tri[ok], t[ok]))[0]
        d = scene.hit_distance(ray, m, t[ok][k])
        if star is None or d < star[0]:
            star = (d, m, int(tri[ok][k]), t[ok][k])
    if star is None:
        return (-1, -1, np.float32(0)), "miss"
    _, ms, _, ts = star
    # fact 3's exception: another model whose closest hit lies behind the origin and that has a second hit could answer nearer
    ambiguous = sum(1 for m in range(nm) if m != ms and len(hits[m][0]) >= 2 and hits[m][1].min() < 0)
    if not ambiguous:
        found, tri, t = replay(scene.grid_path(ray, ms), hits[ms][0], hits[ms][1], lo, hi, listed)
        if found and t == ts:
            return (ms, tri, t), "confirmed"
    # full emulation: every model's walk replayed, combined as Renderer.cpp:388-398 (exact distances, strict compare in model order)
    best = None
    for m in range(nm):
        if len(hits[m][0]) == 0:
            continue
        found, tri, t = replay(scene.grid_path(ray, m), hits[m][0], hits[m][1], lo, hi, listed)
        if not found:
            continue
        d = scene.hit_distance(ray, m, t)
        if best is None or d < best[0]:
            best = (d, m, tri, t)
    return ((best[1], best[2], best[3]) if best else (-1, -1, np.float32(0))), "full"


def _rays(n, seed):
    rs = np.random.RandomState(seed)
    o = np.stack([rs.uniform(-450, 500, n), rs.uniform(-100, 850, n), rs.uniform(-450, 900, n)], 1)
    d = rs.randn(n, 3)
    d[: n // 25, rs.randint(0, 3)] = 0.0
    d *= rs.uniform(0.1, 30.0, (n, 1))
    return np.concatenate([o, d], 1).astype(np.float32)


def _check(scene, rays):
    lo, hi, listed = voxel_boxes(scene)
    want = scene.trace(rays, 0)
    routes = {"miss": 0, "confirmed": 0, "full": 0}
    for i, ray in enumerate(rays):
        (m, tri, t), route = emulate(scene, ray, lo, hi, listed)
        routes[route] += 1
        assert (m, tri) == (int(want["model"][i]), int(want["tri"][i])), f"ray {i} ({route}): ({m}, {tri}) vs oracle R0 ({want['model'][i]}, {want['tri'][i]})"
        if m >= 0:
            assert np.float32(t) == want["t_model"][i], f"ray {i}: t"
    return routes, want


def test_emulation_algorithm_on_the_reference_scene(port, oracle_scene, golden_trace):
    """Random rays through the room, and the golden rays on which the walk is known to differ from brute force."""
    differ = np.flatnonzero(golden_trace["r0"]["tri"] != golden_trace["r1"]["tri"])
    assert len(differ) > 100
    rays = np.concatenate([_rays(20000, 31), golden_trace["rays"][differ]])
    routes, want = _check(oracle_scene, rays)
    assert routes["confirmed"] > 0.6 * len(rays) and routes["full"] >= len(differ)        # the fast route is the common one; the known deviations all take the full one
    assert (want["model"] >= 0).mean() > 0.5


@pytest.mark.parametrize("shape", [(7, 40, 3), (64, 1, 3)], ids=lambda s: "x".join(map(str, s)))
def test_emulation_algorithm_on_non_cubic_grids(port, golden_scene, shape):
    """The same algorithm on grids whose axes differ (and a thin one): voxel boxes, clamps and walk limits per axis."""
    scene = port.OracleScene({k: golden_scene[k] for k in ("models", "meshes", "vertices", "triangles")}, grid_dim=shape)
    routes, want = _check(scene, _rays(3000, 41))
    assert routes["confirmed"] > 0.5 * 3000 and routes["full"] > 0
    assert (want["model"] >= 0).mean() > 0.5


def test_emulation_algorithm_bounce_rays(port, oracle_scene):
    """Rays that start 0.1 above a surface, as the shade kernel restarts them (Renderer.cpp:471-476): the hit just left lies inside the
    predicate's -EPSILON band behind the origin, the case fact 3's exception is about."""
    w = port.OracleWavefront(oracle_scene, 160, 120, depth=3)
    w.init_image(); w.generate(); w.trace(); w.shade(0); n = w.compact()
    r = w.rays(n)
    rays = np.concatenate([r["orig"], r["dir"]], 1).astype(np.float32)
    w.close()
    routes, _ = _check(oracle_scene, rays)
    assert routes["confirmed"] > 0.5 * len(rays)


def test_emulation_algorithm_on_coincident_meshes(port):
    """Twelve coincident copies of a quad in two instances: 12-24 hits per model with bit-equal t; the lowest id listed first must win."""
    from test_gpu_emulated import _stacked_scene
    s = _stacked_scene(12)
    a = s.arrays()
    scene = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    rs = np.random.RandomState(5)
    n = 4000
    o = np.stack([rs.uniform(-150, 100, n), rs.uniform(-80, 80, n), rs.uniform(-100, 100, n)], 1)
    tgt = np.stack([rs.uniform(-120, 60, n), rs.uniform(-50, 50, n), rs.uniform(-40, 40, n)], 1)
    rays = np.concatenate([o, tgt - o], 1).astype(np.float32)
    routes, want = _check(scene, rays)
    assert (want["model"] >= 0).mean() > 0.3 and set(np.unique(want["tri"])) <= {-1, 0, 1, 24, 25}
