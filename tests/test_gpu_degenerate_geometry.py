"""Closest hit on meshes that stress the tree builders, held to brute force: coincident triangles, a long ribbon, a flat plane, meshes of a
handful of triangles, zero-area triangles, and coordinates around 1e6.

Every BVH tree - the host SAH tree and the three device builds (PLOC with the host SAH top, PLOC to the root, the Karras radix tree) - must
give the oracle's R1 hits bit for bit, and the device trees the very bytes of the host tree.  The grid walk and its emulation are held to
R0 on the same scenes.  The scene generators below are plain numpy; tests/test_ploc_model.py counts PLOC's merge rounds on the same meshes."""
import numpy as np
import pytest

from conftest import have_gpu

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_gpu(), reason="no CUDA device")]


# ---- meshes: (positions (nv, 3) float32, triangle indices (nt, 3) int32) ------------------------------------------------------------

def coincident_mesh(n):
    """n copies of one triangle: every PLOC merge cost is equal, every ray's hits tie exactly in t."""
    p = np.array([[-300.0, -250.0, 40.0], [420.0, -180.0, -60.0], [-90.0, 380.0, 20.0]], np.float32)
    return p, np.tile(np.array([[0, 1, 2]], np.int32), (n, 1))


def ribbon_mesh(nquads):
    """One row of nquads unit quads along x, in the plane z = 0."""
    x = np.arange(nquads + 1, dtype=np.float32)
    p = np.zeros((2 * (nquads + 1), 3), np.float32)
    p[0::2, 0] = x; p[1::2, 0] = x; p[1::2, 1] = 1.0
    k = np.arange(nquads, dtype=np.int32)[:, None]
    tri = np.concatenate([np.hstack([2 * k, 2 * k + 2, 2 * k + 3]), np.hstack([2 * k, 2 * k + 3, 2 * k + 1])])
    return p, tri


def tube_mesh(around, segments, radius=3.0):
    """A thin closed tube along x: `around` quads per ring, `segments` rings of unit length."""
    a = np.arange(around) * (2 * np.pi / around)
    x = np.arange(segments + 1, dtype=np.float64)
    p = np.zeros((segments + 1, around, 3))
    p[..., 0] = x[:, None]; p[..., 1] = radius * np.cos(a); p[..., 2] = radius * np.sin(a)
    s, j = np.meshgrid(np.arange(segments), np.arange(around), indexing="ij")
    i00, i01 = s * around + j, s * around + (j + 1) % around
    i10, i11 = i00 + around, i01 + around
    tri = np.concatenate([np.stack([i00, i10, i11], -1).reshape(-1, 3), np.stack([i00, i11, i01], -1).reshape(-1, 3)])
    return p.reshape(-1, 3).astype(np.float32), tri.astype(np.int32)


def plane_mesh(n, spacing=1.0):
    """n x n quads on [-n/2, n/2]^2 * spacing, z = 0 exactly: a mesh box of zero z extent."""
    c = (np.arange(n + 1, dtype=np.float64) - n / 2) * spacing
    X, Y = np.meshgrid(c, c, indexing="ij")
    p = np.stack([X, Y, np.zeros_like(X)], -1).reshape(-1, 3).astype(np.float32)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    v00 = (i * (n + 1) + j).ravel(); v10 = v00 + (n + 1); v01 = v00 + 1; v11 = v10 + 1
    tri = np.concatenate([np.stack([v00, v10, v11], 1), np.stack([v00, v11, v01], 1)]).astype(np.int32)
    return p, tri


def small_mesh(k, seed):
    """k random triangles of size ~40 in a box of side 120."""
    rs = np.random.RandomState(seed)
    c = rs.uniform(-60, 60, (k, 1, 3))
    p = (c + rs.uniform(-20, 20, (k, 3, 3))).reshape(-1, 3).astype(np.float32)
    return p, np.arange(3 * k, dtype=np.int32).reshape(k, 3)


def degenerate_mix_mesh(nx=80, ny=40):
    """2 nx ny > 4096 triangles of a bumpy surface: the first halves of the quads of plane_mesh(max(nx, ny)), a sawtooth of half-quads.  Every
    7th triangle repeats a vertex and every 11th has three collinear vertices (an edge midpoint is appended as a vertex): zero-area
    triangles, det = 0, mixed in with ordinary ones."""
    p, tri = plane_mesh(max(nx, ny), spacing=4.0)
    p = p.copy()
    p[:, 2] = (np.sin(p[:, 0] * 0.37) * np.cos(p[:, 1] * 0.23) * 3.0).astype(np.float32)
    tri = tri[: 2 * nx * ny].copy()
    tri[::7, 1] = tri[::7, 0]                                            # repeated vertex
    col = np.arange(3, len(tri), 11)
    mid = (0.5 * (p[tri[col, 0]].astype(np.float64) + p[tri[col, 1]])).astype(np.float32)
    tri[col, 2] = tri[col, 1]
    tri[col, 1] = len(p) + np.arange(len(col))                           # (a, midpoint(a, b), b): collinear
    return np.concatenate([p, mid]), tri


def far_mesh(n=3000, seed=5):
    """Unit triangles scattered over model-space coordinates 1e5 ... 1e6, plus one triangle spanning them all."""
    rs = np.random.RandomState(seed)
    c = np.stack([rs.uniform(1e5, 1e6, n), rs.uniform(1e5, 1e6, n), rs.uniform(1e5, 1.2e5, n)], 1)
    p = c[:, None, :] + rs.uniform(-0.7, 0.7, (n, 3, 3))
    span = np.array([[[1e5, 1e5, 1.1e5], [1e6, 1.5e5, 1.1e5], [1.2e5, 1e6, 1.15e5]]])
    p = np.concatenate([p, span]).reshape(-1, 3).astype(np.float32)
    return p, np.arange(len(p), dtype=np.int32).reshape(-1, 3)


def nested_mesh(n, r=1.05):
    """n right triangles in z = 0 sharing the corner at the origin, legs 3 r^k: every box lies inside the next one.  Each cluster's
    cheapest merge is with the smaller triangle below it, so PLOC to the root merges one pair per round into a chain, and its 4-wide
    collapse is about n / 3 levels deep.  (The host's binned SAH splits such a sequence in a few levels: see test_tree_at_the_stack_limit.)"""
    s = r ** np.arange(n, dtype=np.float64)
    p = np.zeros((n, 3, 3))
    p[:, 1, 0] = 3.0 * s; p[:, 2, 1] = 3.0 * s
    return p.reshape(-1, 3).astype(np.float32), np.arange(3 * n, dtype=np.int32).reshape(n, 3)


# ---- scenes ---------------------------------------------------------------------------------------------------------------------------

def _vertices(p):
    from pathtracerap_b200 import VERTEX
    v = np.zeros(len(p), VERTEX)
    v["position"] = p
    v["normal"] = (0.0, 0.0, 1.0)
    return v


def build_scene(meshes, instances):
    """meshes: [(positions, indices)]; instances: [(mesh, translate, rotate_y_degrees, scale)]."""
    from pathtracerap_b200 import Scene
    s = Scene.empty()
    ids = [s.add_mesh(_vertices(p), t) for p, t in meshes]
    for k, (m, tr, rot, sc) in enumerate(instances):
        s.add_model(ids[m], translate=tr, rotate_y_degrees=rot, scale=sc, color=(0.2 + 0.1 * (k % 7), 0.5, 0.7))
    return s


def world_triangles(a):
    """(n, 3, 3) float64 world positions of every instanced triangle of the scene arrays `a`."""
    out = []
    for m in a["models"]:
        M = m["model_to_world"].reshape(4, 4).T.astype(np.float64)
        mesh = a["meshes"][m["mesh_index"]]
        idx = a["triangles"]["v"][mesh["t_start"]:mesh["t_end"]]
        if len(idx) == 0:
            continue
        p = a["vertices"]["position"][idx].astype(np.float64)
        out.append(p @ M[:3, :3].T + M[:3, 3])
    return np.concatenate(out)


def make_rays(a, n, seed, scale_lo=0.2, scale_hi=5.0, far=0.0):
    """n rays (n, 6) float32 at the scene's triangles: random, aimed at points, vertices and edge midpoints, axis-parallel, with +0.0 and
    -0.0 direction components, and from origins on the surfaces.  far > 0 puts the random origins that far from the scene."""
    rs = np.random.RandomState(seed)
    W = world_triangles(a)
    lo, hi = W.reshape(-1, 3).min(0), W.reshape(-1, 3).max(0)
    ext = np.maximum(hi - lo, 1.0)
    pick = W[rs.randint(0, len(W), n)]
    b = rs.dirichlet((1.0, 1.0, 1.0), n)
    on = np.einsum("nk,nkd->nd", b, pick)                                 # a point on a triangle
    kind = rs.randint(0, 7, n)
    tgt = on.copy()
    tgt[kind == 1] = pick[kind == 1, rs.randint(0, 3)]                    # a vertex
    e = rs.randint(0, 3, n)
    edge = 0.5 * (pick[np.arange(n), e] + pick[np.arange(n), (e + 1) % 3])
    tgt[kind == 2] = edge[kind == 2]                                      # an edge midpoint
    tgt[kind == 3] = rs.uniform(lo - 0.2 * ext, hi + 0.2 * ext, (n, 3))[kind == 3]     # anywhere: many misses
    o = rs.uniform(lo - 0.5 * ext, hi + 0.5 * ext, (n, 3))
    if far > 0:
        u = rs.randn(n, 3); u /= np.linalg.norm(u, axis=1, keepdims=True)
        o[::2] = (0.5 * (lo + hi) + far * u)[::2]
    d = tgt - o
    ax = rs.randint(0, 3, n)                                              # axis-parallel: straight at the target along one axis
    par = kind == 4
    d[par] = 0.0
    d[par, ax[par]] = rs.choice([-1.0, 1.0], par.sum()) * rs.uniform(0.1, 1.0, par.sum()) * ext[ax[par]]
    o[par] = tgt[par] - d[par]
    surf = kind == 5                                                      # origin on the surface, any direction
    o[surf] = on[surf]
    d[surf] = rs.randn(surf.sum(), 3)
    d *= (rs.uniform(scale_lo, scale_hi, n) / np.maximum(np.linalg.norm(d, axis=1), 1e-30))[:, None]
    zc = kind == 6                                                        # one or two components exactly +0.0 or -0.0
    d[zc, ax[zc]] = rs.choice([0.0, -0.0], zc.sum())
    two = zc & (rs.rand(n) < 0.3)
    d[two, (ax[two] + 1) % 3] = rs.choice([0.0, -0.0], two.sum())
    return np.concatenate([o, d], 1).astype(np.float32)


# ---- checks ---------------------------------------------------------------------------------------------------------------------------

DEVICE_BUILDS = [("ploc", {}), ("ploc to the root", {"PTAP_PLOC_TOP": "0"}), ("lbvh", {"PTAP_DEVICE_BUILDER": "lbvh"})]


def _assert_equal(got, want, what):
    assert np.array_equal(got["model"], want["model"]), f"{what}: model ids differ on {(got['model'] != want['model']).sum()} rays"
    assert np.array_equal(got["tri"], want["tri"]), f"{what}: triangle ids differ on {(got['tri'] != want['tri']).sum()} rays"
    hit = want["model"] >= 0
    for f in ("t_model", "dist", "u", "v", "normal"):
        assert np.array_equal(got[f][hit], want[f][hit]), f"{what}: {f} not bit-equal"
    return hit


def _check_queries(r, rays, want, what):
    """query_closest is trace() bit for bit; query_occluded at L = dist and one ulp either side is (hit and dist < L)."""
    import torch
    from pathtracerap_b200 import HIT
    t = torch.from_numpy(rays).cuda()
    org, dir_ = t[:, :3].contiguous(), t[:, 3:].contiguous()
    q = r.query_closest(org, dir_)
    rec = np.zeros(len(rays), HIT)
    for f in ("model", "tri", "t_model", "dist", "u", "v", "normal", "mat_type"):
        rec[f] = q[f].cpu().numpy()
    assert rec.tobytes() == r.trace(rays).tobytes(), f"{what}: query_closest differs from trace"
    hit = want["model"] >= 0
    base = np.where(hit, want["dist"], np.float32(500.0)).astype(np.float32)
    for L, label in ((base, "L = dist"), (np.nextafter(base, np.float32(-np.inf)), "L one ulp below dist"),
                     (np.nextafter(base, np.float32(np.inf)), "L one ulp above dist")):
        got = r.query_occluded(org, dir_, torch.from_numpy(L).cuda()).cpu().numpy()
        truth = hit & (want["dist"] < L)
        assert np.array_equal(got, truth), f"{what}, {label}: occlusion differs on {(got != truth).sum()} rays"


def check_scene(s, rays, what, port, monkeypatch, emulated=True):
    """Every BVH tree against R1 (and the device trees against the host tree's bytes), then the grid walk and its emulation against R0.
    emulated=False: the scene's grids are expected to be refused by PTAP_ACCEL_GRID_EMULATED (PTAP_E_UNSUPPORTED)."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, ACCEL_GRID_EMULATED, Renderer
    from pathtracerap_b200 import _native as N
    a = s.arrays()
    o = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    want = o.trace(rays, 1)
    r = Renderer(width=32, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    host = r.trace(rays)
    hit = _assert_equal(host, want, f"{what}: host tree vs R1")
    assert 0.05 < hit.mean() < 0.98, f"{what}: {hit.mean():.3f} of the rays hit"
    _check_queries(r, rays, want, f"{what}: host tree")
    for name, env in DEVICE_BUILDS:
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            r.accel = ACCEL_BVH_DEVICE
            r.upload(s)                                  # a fresh upload: the device build runs under this environment
            got = r.trace(rays)
            _assert_equal(got, want, f"{what}: device tree ({name}) vs R1")
            assert got.tobytes() == host.tobytes(), f"{what}: device tree ({name}) differs from the host tree"
            _check_queries(r, rays, want, f"{what}: device tree ({name})")
            assert r.build_stats()["bvh_nodes"] > 0
    want0 = o.trace(rays, 0)
    r.build_grids_device(s, 25, 25, 25)
    _assert_equal(r.trace(rays), want0, f"{what}: grid walk vs R0")
    rc = N.lib().ptap_build_accel(r.h, ACCEL_GRID_EMULATED)
    if emulated:
        assert rc == 0, f"{what}: emulated walk refused: {N.lib().ptap_last_error(r.h).decode()}"
        r.accel = ACCEL_GRID_EMULATED
        _assert_equal(r.trace(rays), want0, f"{what}: emulated walk vs R0")
    else:
        assert rc == N.E_UNSUPPORTED, f"{what}: the emulated walk was expected to refuse these grids, got {rc}"
    r.free()
    return want


FLOOR = (np.array([[-3000.0, -3000.0, -800.0], [3000.0, -3000.0, -800.0], [3000.0, 3000.0, -800.0], [-3000.0, 3000.0, -800.0]], np.float32),
         np.array([[0, 1, 2], [0, 2, 3]], np.int32))


@pytest.mark.parametrize("n", [37, 5000, 12000])
def test_coincident_triangles(n, libptap, port, monkeypatch):
    """n identical triangles over a floor: every hit on them ties exactly in t and must go to the lowest triangle id; every PLOC merge
    cost is equal (before the symmetric tie key, 12000 of them stalled the default device build)."""
    s = build_scene([coincident_mesh(n), FLOOR], [(0, (0, 0, 0), 0.0, (1, 1, 1)), (1, (0, 0, 0), 0.0, (1, 1, 1))])
    rays = make_rays(s.arrays(), 30_000, n)
    want = check_scene(s, rays, f"{n} coincident triangles", port, monkeypatch)
    on = (want["model"] == 0)
    assert on.sum() > 3000 and (want["tri"][on] == 0).all()             # the lowest id wins every exact tie


def test_long_ribbon(libptap, port, monkeypatch):
    """1 x 20,000 unit quads: neighbouring merge costs tie along the whole ribbon (the default device build stalled on it)."""
    s = build_scene([ribbon_mesh(20_000)], [(0, (0, 0, 0), 0.0, (1, 1, 1))])
    rays = make_rays(s.arrays(), 30_000, 3, scale_lo=0.5, scale_hi=2.0)
    check_scene(s, rays, "1 x 20000 ribbon", port, monkeypatch)


def test_flat_plane(libptap, port, monkeypatch):
    """128 x 128 quads at z = 0: Morton minv.z = 0, grid width.z = 0; rays lying in the plane (o.z = 0, d.z = +-0.0) and rays through the
    shared edges and vertices, where both neighbours accept inside the tolerance band."""
    p, t = plane_mesh(128)
    s = build_scene([(p, t)], [(0, (0, 0, 0), 0.0, (1, 1, 1)), (0, (10, -5, 30), 30.0, (0.5, 0.5, 0.5))])
    a = s.arrays()
    rs = np.random.RandomState(9)
    rays = make_rays(a, 30_000, 9)
    # in the plane of the first instance: o.z = 0 and d.z = +0.0 / -0.0
    k = 4000
    inp = np.zeros((k, 6), np.float32)
    inp[:, :2] = rs.uniform(-80, 80, (k, 2))
    inp[:, 3:5] = rs.randn(k, 2)
    inp[:, 5] = np.where(rs.rand(k) < 0.5, 0.0, -0.0)
    # straight down (and up) through grid vertices and edge midpoints of the first instance, from both sides
    g = rs.randint(-64, 64, (k, 2)).astype(np.float32)
    g[k // 2:, 0] += 0.5
    down = np.zeros((k, 6), np.float32)
    down[:, :2] = g
    side = np.where(rs.rand(k) < 0.5, 1.0, -1.0).astype(np.float32)
    down[:, 2] = 5.0 * side; down[:, 5] = -side * rs.uniform(0.2, 3.0, k)
    down[::3, 3] = -0.0; down[1::3, 4] = -0.0
    rays = np.concatenate([rays, inp, down])
    want = check_scene(s, rays, "flat 128 x 128 plane", port, monkeypatch)
    assert (want["model"][-k:] == 0).mean() > 0.9


def test_tiny_meshes_instanced(libptap, port, monkeypatch):
    """Meshes of 1, 2, 3, 4, 5, 8, 9 and 17 triangles, three instances each: the single-leaf device tree and 4-wide nodes with unused slots."""
    counts = [1, 2, 3, 4, 5, 8, 9, 17]
    meshes = [small_mesh(k, k) for k in counts]
    inst = []
    for m in range(len(counts)):
        for j in range(3):
            inst.append((m, ((m - 4) * 150.0, (j - 1) * 160.0, 40.0 * j), 35.0 * j + 10 * m, (1.0 + 0.3 * j,) * 3))
    s = build_scene(meshes, inst)
    rays = make_rays(s.arrays(), 30_000, 21)
    want = check_scene(s, rays, "tiny meshes", port, monkeypatch)
    assert len(np.unique(want["model"][want["model"] >= 0])) == len(inst)


def test_zero_area_triangles(libptap, port, monkeypatch):
    """6400 triangles (above the 4096 clusters PLOC hands to the host) with repeated-vertex and collinear triangles mixed in: PLOC over
    degenerate boxes, and the predicate's det = 0 rejection."""
    p, t = degenerate_mix_mesh()
    s = build_scene([(p, t)], [(0, (0, 0, 0), 0.0, (1, 1, 1)), (0, (20, 10, -60), 15.0, (1, 1, 1))])
    rays = make_rays(s.arrays(), 30_000, 13)
    want = check_scene(s, rays, "zero-area triangles", port, monkeypatch)
    degenerate = np.zeros(len(t), bool)
    degenerate[::7] = True; degenerate[3::11] = True
    hit = want["model"] >= 0
    assert not degenerate[want["tri"][hit]].any()


def test_far_coordinates(libptap, port, monkeypatch):
    """Unit triangles at model coordinates 1e5 ... 1e6 and one triangle spanning them, instances translated to +-1e6, rays from near the
    surfaces and from 1e6 away: node-local offsets and their 2^-20 margin, the device builder's box slack, the TLAS pad."""
    p, t = far_mesh()
    s = build_scene([(p, t)], [(0, (-1e6, 0, 0), 0.0, (1, 1, 1)), (0, (1e6, -1e6, 2e5), 90.0, (1, 1, 1)), (0, (0, 1e6, -1e6), 0.0, (0.5, 2.0, 1.0))])
    a = s.arrays()
    near = make_rays(a, 20_000, 17, scale_lo=0.5, scale_hi=2.0)
    far = make_rays(a, 20_000, 18, scale_lo=0.5, scale_hi=2.0, far=1e6)
    check_scene(s, np.concatenate([near, far]), "coordinates around 1e6", port, monkeypatch)


N_AT_LIMIT, N_TOO_DEEP, DEPTH_AT_LIMIT = 148, 150, 49       # 3 (49 + 1) + 8 = 158 of kBvhStack = 160 entries; 50 levels need 161


def test_tree_at_the_stack_limit(libptap, port, monkeypatch):
    """A BLAS 49 levels deep under a one-level TLAS: the traversal stack of k_trace_bvh (closest hit and any-hit) and of the emulated walk
    two entries short of its end, bit-exact against R1 / R0.  One level deeper is refused with PTAP_E_INVALID, and a context whose tree
    was overwritten by the refused build traces nothing until a build succeeds.

    The deep tree comes from the device builder, PLOC to the root (PTAP_PLOC_TOP=0), over nested_mesh.  No geometry brings the host tree
    near the limit: its binned SAH over 16 bins splits a geometric sequence of positions or sizes several items at a time, box areas must
    stay finite in binary32 (coordinates below about 2^63), and below the fattening slack (4e-6 of the mesh extent) boxes are alike.  Such
    meshes reach 13 levels; the host tree of this one is checked to be shallow and exact instead."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, ACCEL_GRID_EMULATED, Renderer
    from pathtracerap_b200 import _native as N
    s = build_scene([nested_mesh(N_AT_LIMIT)], [(0, (0, 0, 0), 0.0, (1, 1, 1))])
    rays = make_rays(s.arrays(), 30_000, 31)
    want = check_scene(s, rays, "nested triangles", port, monkeypatch)           # host tree and the three device builds
    h = build_scene([nested_mesh(N_AT_LIMIT)], [(0, (0, 0, 0), 0.0, (1, 1, 1))])
    h.build_bvh()
    bad, host_depth = h.validate_bvh()
    assert bad == 0 and host_depth < 20
    a = s.arrays()
    o = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    monkeypatch.setenv("PTAP_PLOC_TOP", "0")
    r = Renderer(width=32, height=32, depth=5, accel=ACCEL_BVH_DEVICE)
    r.allocateOnGPU(s)
    assert r.build_stats()["bvh_depth"] == DEPTH_AT_LIMIT
    _assert_equal(r.trace(rays), want, "49-level tree vs R1")
    _check_queries(r, rays, want, "49-level tree")
    r.build_grids_device(s, 25, 25, 25)                   # the grids join the device tree, which the emulated walk traverses
    assert N.lib().ptap_build_accel(r.h, ACCEL_GRID_EMULATED) == 0, N.lib().ptap_last_error(r.h).decode()
    r.accel = ACCEL_GRID_EMULATED
    _assert_equal(r.trace(rays), o.trace(rays, 0), "49-level tree, emulated walk vs R0")
    r.free()

    deep = build_scene([nested_mesh(N_TOO_DEEP)], [(0, (0, 0, 0), 0.0, (1, 1, 1))])
    a = deep.arrays()
    o = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    rays = make_rays(a, 10_000, 32)
    r = Renderer(width=32, height=32, depth=5, accel=ACCEL_BVH_DEVICE)
    with pytest.raises(N.PtapError, match="error -1: BVH too deep"):
        r.allocateOnGPU(deep)
    with pytest.raises(N.PtapError, match="no BVH"):
        r.trace(rays)
    # a context holding a good host tree: the refused device build overwrites it, and nothing is traced through what is left
    r.set_accel(ACCEL_BVH)
    _assert_equal(r.trace(rays), o.trace(rays, 1), "host tree of the deeper mesh vs R1")
    with pytest.raises(N.PtapError, match="error -1: BVH too deep"):
        r.set_accel(ACCEL_BVH_DEVICE)
    import torch
    t = torch.from_numpy(rays).cuda()
    for call in (lambda: r.trace(rays), lambda: r.query_closest(t[:, :3].contiguous(), t[:, 3:].contiguous()),
                 lambda: r.query_occluded(t[:, :3].contiguous(), t[:, 3:].contiguous(), float("inf"))):
        with pytest.raises(N.PtapError, match="no BVH"):
            call()
    r.set_accel(ACCEL_BVH)
    _assert_equal(r.trace(rays), o.trace(rays, 1), "host tree rebuilt after the refusal vs R1")
    r.free()
