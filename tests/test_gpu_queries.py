"""Ray queries on device buffers (ptap_query_closest / ptap_query_occluded, Renderer.query_closest / query_occluded; DESIGN.md 4.8).

Closest hit equals ptap_trace bit for bit (and the oracle tier of the accel: R0 for the grid modes, R1 for the BVH modes).  Occlusion is
defined through that closest hit: occluded = model >= 0 and dist < L in binary32, whatever traversal answers it."""
import os
import sys

import numpy as np
import pytest

from test_gpu_emulated import _stacked_scene
from test_gpu_production import _sphere_scene
from test_query_model import far_rays

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
torch = pytest.importorskip("torch")
FIELDS = ("model", "tri", "t_model", "dist", "u", "v", "normal", "mat_type")


def _rays(n, seed, lo=-450.0, hi=850.0):
    rs = np.random.RandomState(seed)
    o = rs.uniform(lo, hi, (n, 3))
    d = rs.uniform(lo * 0.6, hi * 0.6, (n, 3)) - o
    d *= rs.uniform(0.2, 5.0, (n, 1)) / np.linalg.norm(d, axis=1, keepdims=True)
    d[: n // 40, 0] = 0.0
    return np.concatenate([o, d], 1).astype(np.float32)


def _dev(rays):
    t = torch.from_numpy(np.ascontiguousarray(rays)).cuda()
    return t[:, :3].contiguous(), t[:, 3:6].contiguous()


def _records(q):
    """query_closest's dict -> a HIT record array (bytes as ptap_trace writes them)."""
    from pathtracerap_b200 import HIT
    n = q["model"].shape[0]
    out = np.zeros(n, HIT)
    for f in FIELDS:
        out[f] = q[f].cpu().numpy()
    return out


def _assert_closest(got, want, what, oracle=False):
    if not oracle:
        assert got.tobytes() == want.tobytes(), f"{what}: records differ on {(got != want).sum()} rays"
        return
    assert np.array_equal(got["model"], want["model"]), f"{what}: model ids differ on {(got['model'] != want['model']).sum()} rays"
    assert np.array_equal(got["tri"], want["tri"]), f"{what}: triangle ids differ"
    hit = want["model"] >= 0
    for f in ("t_model", "dist", "u", "v"):
        assert np.array_equal(got[f][hit], want[f][hit]), f"{what}: {f} not bit-equal to the oracle"


def _lengths(dist, hit, rs):
    """Segment lengths per ray, every kind the contract names: uniform [0, 2 dist], dist itself (-> False), the next float up (-> True),
    tiny lengths, +inf, 0, negative, NaN (misses get the same menu with dist = 500)."""
    n = len(dist)
    base = np.where(hit, dist, np.float32(500.0)).astype(np.float32)
    kinds = rs.randint(0, 8, n)
    L = np.empty(n, np.float32)
    L[kinds == 0] = (rs.uniform(0, 2, n) * base)[kinds == 0]
    L[kinds == 1] = base[kinds == 1]
    L[kinds == 2] = np.nextafter(base, np.float32(np.inf))[kinds == 2]
    L[kinds == 3] = rs.choice([1e-6, 1e-4, 2e-3, 5e-3, 1e-2, 0.05], n).astype(np.float32)[kinds == 3]
    L[kinds == 4] = np.inf
    L[kinds == 5] = 0.0
    L[kinds == 6] = -rs.uniform(0, 10, n).astype(np.float32)[kinds == 6]
    L[kinds == 7] = np.nan
    return L


def _check_occluded(r, rays, want, what, seed):
    """query_occluded against (want.model >= 0) & (want.dist < L), `want` the closest hits of the accel's tier."""
    rs = np.random.RandomState(seed)
    hit = want["model"] >= 0
    L = _lengths(want["dist"], hit, rs)
    org, dir_ = _dev(rays)
    got = r.query_occluded(org, dir_, torch.from_numpy(L).cuda()).cpu().numpy()
    truth = hit & (want["dist"] < L)
    assert got.dtype == np.bool_
    assert np.array_equal(got, truth), f"{what}: occlusion differs on {(got != truth).sum()} of {len(L)} rays"
    assert truth.sum() > 0 and (~truth).sum() > 0
    # a scalar length: +inf is "any hit"
    assert np.array_equal(r.query_occluded(org, dir_, float("inf")).cpu().numpy(), hit), f"{what}: L = inf"
    return got


@pytest.fixture(scope="module")
def bundled(libptap, port, golden_scene):
    from pathtracerap_b200 import ACCEL_GRID_EMULATED, Renderer, Scene
    g = golden_scene
    s = Scene.from_arrays(g["models"], g["meshes"], g["vertices"], g["triangles"])
    s.build_grids(25, 25, 25)
    r = Renderer(width=64, height=48, depth=5, accel=ACCEL_GRID_EMULATED)
    r.allocateOnGPU(s)
    yield r, s
    r.free()


ACCELS = [("grid", 0, 0), ("emu", 3, 0), ("bvh", 1, 1), ("bvh_device", 2, 1)]     # name, accel, oracle tier


@pytest.mark.parametrize("name,accel,tier", ACCELS)
def test_query_closest_equals_trace_and_oracle(bundled, oracle_scene, golden_trace, name, accel, tier):
    r, _ = bundled
    r.set_accel(accel)
    golden = golden_trace["rays"]
    rnd = _rays(300_000, 17)
    for rays, what in ((golden, "golden rays"), (rnd, "300k random rays")):
        got = _records(r.query_closest(*_dev(rays)))
        _assert_closest(got, r.trace(rays), f"{name}, {what}")
        sub = rays if len(rays) < 50_000 else rays[::15]
        _assert_closest(got if len(rays) < 50_000 else got[::15], oracle_scene.trace(sub, tier), f"{name}, {what}, oracle R{tier}", oracle=True)
    # (n, 4) inputs are read as they are: the w lanes play no part in a closest-hit query
    t = torch.from_numpy(rnd).cuda()
    o4 = torch.cat([t[:, :3], torch.full_like(t[:, :1], 123.0)], 1)
    d4 = torch.cat([t[:, 3:], torch.full_like(t[:, :1], -1.0)], 1)
    assert _records(r.query_closest(o4, d4)).tobytes() == r.trace(rnd).tobytes()


@pytest.mark.parametrize("name,accel,tier", ACCELS)
def test_query_occluded_bundled(bundled, oracle_scene, golden_trace, name, accel, tier):
    r, _ = bundled
    r.set_accel(accel)
    rays = np.concatenate([golden_trace["rays"], _rays(200_000, 23)])
    _check_occluded(r, rays, r.trace(rays), name, 3)
    g = golden_trace["rays"]
    _check_occluded(r, g, oracle_scene.trace(g, tier), f"{name} vs oracle R{tier}", 4)


def test_query_occluded_large_instance_scale(libptap, port):
    """Instances scaled x500 ... x900, rays 0.1 world units off the surfaces at grazing angles: winners behind the origin, the EPSILON
    term of the early-exit rule, and lengths below EPSILON * scale."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, Renderer
    scales = [500.0, 650.0, 900.0, 520.0, 700.0]
    s, centres = _sphere_scene(scales, 11)
    a = s.arrays()
    s.build_bvh()
    rs = np.random.RandomState(12)
    rays = []
    for c, sc in centres:
        n = 6000
        p = rs.randn(n, 3); p /= np.linalg.norm(p, axis=1, keepdims=True)
        o = c + p * sc + p * rs.choice([-20.0, -3.0, -0.1, 0.1, 1.0, 3.0, 20.0], n)[:, None]
        t = rs.randn(n, 3); t -= p * np.sum(t * p, axis=1, keepdims=True); t /= np.linalg.norm(t, axis=1, keepdims=True)
        ang = rs.choice([0.0, 1e-3, 1e-2, 0.1, 0.5, 1.5], n)[:, None] * rs.choice([-1.0, 1.0], n)[:, None]
        rays.append(np.concatenate([o, (t * np.cos(ang) + p * np.sin(ang)) * rs.uniform(0.2, 40.0, (n, 1))], 1))
    rays = np.concatenate(rays).astype(np.float32)
    want = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")}).trace(rays, 1)
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    for accel in (ACCEL_BVH, ACCEL_BVH_DEVICE):
        r.set_accel(accel)
        _assert_closest(_records(r.query_closest(*_dev(rays))), want, "large scale", oracle=True)
        _check_occluded(r, rays, want, f"large scale, accel {accel}", 5)
        # lengths just above and below EPSILON * scale, where a self-hit behind the origin competes
        hit = want["model"] >= 0
        for L in (0.005 * 500, 0.005 * 900, np.nextafter(np.float32(0.005 * 650), np.float32(np.inf))):
            got = r.query_occluded(*_dev(rays), float(L)).cpu().numpy()
            assert np.array_equal(got, hit & (want["dist"] < np.float32(L))), f"large scale, L = {L}"
    # origins 0.9e7 ... 3e7 world units away: accepted hits at world distances on both sides of FLOAT_MAX, where the closest hit is a
    # miss, so neither L = inf nor a finite L above FLOAT_MAX may report them
    far = far_rays(centres, 4000, 15)
    wf = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")}).trace(far, 1)
    fhit = wf["model"] >= 0
    assert fhit.sum() > 100 and (~fhit).sum() > 100
    for accel in (ACCEL_BVH, ACCEL_BVH_DEVICE):
        r.set_accel(accel)
        _assert_closest(_records(r.query_closest(*_dev(far))), wf, "far origins", oracle=True)
        for L in (float("inf"), 5e7, 9999999.0, 2e7):
            got = r.query_occluded(*_dev(far), L).cpu().numpy()
            assert np.array_equal(got, fhit & (wf["dist"] < np.float32(L))), f"far origins, accel {accel}, L = {L}: {(got != (fhit & (wf['dist'] < np.float32(L)))).sum()} rays differ"
        _check_occluded(r, far, wf, f"far origins, accel {accel}", 16)
    r.free()


def test_query_occluded_matrices_that_are_not_inverses(libptap, port, golden_scene):
    """model_to_world not the inverse of world_to_model: pruning is off (sc.prune = sc.tie = inf), the early exit never fires, and the
    any-hit traversal is a closest-hit traversal bounded by L."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, Renderer, Scene
    g = golden_scene
    models = g["models"].copy()
    rs = np.random.RandomState(2)
    for k in (0, 4, 7):
        M = models[k]["model_to_world"].reshape(4, 4).T.astype(np.float64)
        M[:3, :3] *= rs.uniform(0.7, 1.4)
        M[:3, 3] += rs.uniform(-30, 30, 3)
        models[k]["model_to_world"] = M.T.astype(np.float32).reshape(16)
    s = Scene.from_arrays(models, g["meshes"], g["vertices"], g["triangles"])
    s.build_bvh()
    r = Renderer(width=32, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    rays = _rays(100_000, 6)
    want = port.OracleScene({"models": models, "meshes": g["meshes"], "vertices": g["vertices"], "triangles": g["triangles"]}).trace(rays, 1)
    for accel in (ACCEL_BVH, ACCEL_BVH_DEVICE):
        r.set_accel(accel)
        _assert_closest(_records(r.query_closest(*_dev(rays))), want, "inconsistent matrices", oracle=True)
        _check_occluded(r, rays, want, f"inconsistent matrices, accel {accel}", 6)
    r.free()


@pytest.mark.parametrize("copies", [3, 12])
def test_query_occluded_coincident_copies(libptap, port, copies):
    """Coincident triangles: exact-t ties inside a model, resolved by the lowest id; every accel against its oracle tier."""
    from pathtracerap_b200 import ACCEL_GRID_EMULATED, Renderer
    s = _stacked_scene(copies)
    a = s.arrays()
    osc = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    rs = np.random.RandomState(5)
    n = 60_000
    o = np.stack([rs.uniform(-150, 100, n), rs.uniform(-80, 80, n), rs.uniform(-100, 100, n)], 1)
    tgt = np.stack([rs.uniform(-120, 60, n), rs.uniform(-50, 50, n), rs.uniform(-40, 40, n)], 1)
    rays = np.concatenate([o, tgt - o], 1).astype(np.float32)
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_GRID_EMULATED)
    r.allocateOnGPU(s)
    for name, accel, tier in ACCELS:
        r.set_accel(accel)
        want = osc.trace(rays, tier)
        assert (want["model"] >= 0).mean() > 0.2
        _assert_closest(_records(r.query_closest(*_dev(rays))), want, f"{copies} copies, {name}", oracle=True)
        _check_occluded(r, rays, want, f"{copies} copies, {name}", 7)
    r.free()


def test_query_occluded_mesh100k_brute_force(libptap, port):
    """The mesh100k scene (a displaced 81,920-triangle icosphere in the bundled box): a seeded subset against brute force (R1)."""
    sys.path.insert(0, ROOT)
    import bench
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, Renderer
    s, arrays = bench.build_scene("mesh100k")
    s.build_bvh()
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    rays = _rays(3000, 8)
    want = port.OracleScene(arrays).trace(rays, 1)
    for accel in (ACCEL_BVH, ACCEL_BVH_DEVICE):
        r.set_accel(accel)
        _assert_closest(_records(r.query_closest(*_dev(rays))), want, "mesh100k", oracle=True)
        _check_occluded(r, rays, want, f"mesh100k, accel {accel}", 9)
    r.free()


def test_shadow_rays_of_a_mesh1m_frame(libptap):
    """Shadow rays as tools/bench_queries.py builds them (round-1 origins of a 1920 x 1080 frame towards points on the lights), more than
    one million, through both occlusion paths of the BVH: equal to the ptap_trace-derived truth."""
    sys.path.insert(0, ROOT)
    import bench
    from tools.bench_queries import shadow_rays
    from pathtracerap_b200 import ACCEL_BVH, Renderer
    s, arrays = bench.build_scene("mesh1m")
    s.build_bvh()
    r = Renderer(width=1920, height=1080, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    o, d, L = shadow_rays(r, arrays, 1920, 1080)
    assert len(o) >= 1_000_000
    ref = r.trace(np.concatenate([o, d], 1))
    truth = (ref["model"] >= 0) & (ref["dist"] < L)
    assert 0.02 < truth.mean() < 0.98
    org, dir_ = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    got = r.query_occluded(org, dir_, torch.from_numpy(L).cuda()).cpu().numpy()
    assert np.array_equal(got, truth), f"mesh1m shadow rays differ on {(got != truth).sum()} rays"
    r.free()


def test_stream_ordering_and_chunks(bundled):
    """Rays made by torch on a side stream, queried and consumed there with no host synchronisation in between; a render enqueued before
    a query keeps its film; a query of more than one chunk (2^22 rays)."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_EMULATED
    r, _ = bundled
    r.set_accel(ACCEL_BVH)
    rays = _rays(300_000, 29)
    want = r.trace(rays)
    base = torch.from_numpy(rays).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(50_000_000)                     # keeps the stream busy: a query not ordered after it would read stale rays
        rays_dev = base * 1.0                             # produced by a torch kernel on `side`
        q = r.query_closest(rays_dev[:, :3].contiguous(), rays_dev[:, 3:].contiguous())
        model_sum = q["model"].to(torch.int64).sum()      # consumed on `side`
        occ = r.query_occluded(rays_dev[:, :3].contiguous(), rays_dev[:, 3:].contiguous(), float("inf"))
        n_occ = occ.sum()
    side.synchronize()
    assert _records(q).tobytes() == want.tobytes()
    assert int(model_sum) == int(want["model"].astype(np.int64).sum())
    assert int(n_occ) == int((want["model"] >= 0).sum())
    # a render enqueued before the query: the film is what it is without the query
    for accel in (ACCEL_BVH, ACCEL_GRID_EMULATED):
        r.set_accel(accel)
        r.set_params(64, 48, 5, first_hit_cache=False)
        r.frame_begin(); r.render(0, 2); film_alone = r.film()
        r.frame_begin(); r.render(0, 2)
        occ = r.query_occluded(*_dev(rays), 100.0)
        film = r.film()
        assert np.array_equal(film, film_alone), f"accel {accel}: the query changed the film"
        assert np.array_equal(occ.cpu().numpy(), (r.trace(rays)["model"] >= 0) & (r.trace(rays)["dist"] < np.float32(100.0)))
    # more than one chunk
    r.set_accel(ACCEL_BVH)
    big = np.concatenate([rays] * 15)                     # 4.5 M rays
    L = np.random.RandomState(1).uniform(0, 1500, len(big)).astype(np.float32)
    got = r.query_occluded(*_dev(big), torch.from_numpy(L).cuda()).cpu().numpy()
    wb = np.concatenate([want] * 15)
    assert np.array_equal(got, (wb["model"] >= 0) & (wb["dist"] < L))
    qb = _records(r.query_closest(*_dev(big)))
    assert qb.tobytes() == wb.tobytes()


def test_rejections(bundled, libptap):
    from pathtracerap_b200 import PtapError
    r, _ = bundled
    rays = _rays(1000, 3)
    org, dir_ = _dev(rays)
    with pytest.raises(TypeError):
        r.query_closest(org.double(), dir_)
    with pytest.raises(TypeError):
        r.query_occluded(org, dir_.half(), 1.0)
    with pytest.raises(TypeError):
        r.query_closest(rays[:, :3], rays[:, 3:])
    with pytest.raises(TypeError):
        r.query_occluded(org, dir_, torch.ones(1000, dtype=torch.float64, device="cuda"))
    with pytest.raises(TypeError):
        r.query_occluded(org, dir_, True)
    # numpy scalars are lengths like Python floats
    assert np.array_equal(r.query_occluded(org, dir_, np.float32(300.0)).cpu().numpy(), r.query_occluded(org, dir_, 300.0).cpu().numpy())
    with pytest.raises(ValueError):
        r.query_closest(org.cpu(), dir_.cpu())
    with pytest.raises(ValueError):
        r.query_closest(org, torch.cat([dir_, dir_], 1)[:, ::2])          # non-contiguous
    with pytest.raises(ValueError):
        r.query_occluded(org, dir_, torch.ones(7, device="cuda"))
    # the C ABI itself: host pointers, misaligned pointers, n < 0
    lib = libptap
    o4 = torch.zeros((1000, 4), device="cuda"); d4 = torch.ones((1000, 4), device="cuda")
    hits = torch.empty((1000, 10), dtype=torch.int32, device="cuda"); occ = torch.empty(1000, dtype=torch.uint8, device="cuda")
    host = np.zeros((1000, 4), np.float32)
    assert lib.ptap_query_closest(r.h, host.ctypes.data, d4.data_ptr(), 1000, hits.data_ptr(), None) == -1
    assert b"org" in lib.ptap_last_error(r.h)
    assert lib.ptap_query_occluded(r.h, o4.data_ptr(), d4.data_ptr() + 4, 999, occ.data_ptr(), None) == -1
    assert b"dir" in lib.ptap_last_error(r.h) and b"aligned" in lib.ptap_last_error(r.h)
    assert lib.ptap_query_occluded(r.h, o4.data_ptr(), d4.data_ptr(), 1000, host.ctypes.data, None) == -1
    assert lib.ptap_query_closest(r.h, o4.data_ptr(), d4.data_ptr(), -1, hits.data_ptr(), None) == -1
    # n = 0: a no-op, null pointers included
    assert lib.ptap_query_closest(r.h, None, None, 0, None, None) == 0
    assert r.query_closest(org[:0], dir_[:0])["model"].shape == (0,)
    assert r.query_occluded(org[:0], dir_[:0], 1.0).shape == (0,)
    with pytest.raises(PtapError):           # a misaligned (n, 4) view through the Python layer reaches the ABI's check
        t = torch.zeros(4001, device="cuda")[1:].view(1000, 4)
        r.query_closest(t, t)
    if torch.cuda.device_count() < 2:
        return
    with pytest.raises(ValueError):
        r.query_closest(org.to("cuda:1"), dir_.to("cuda:1"))
    o1, d1, h1 = o4.to("cuda:1"), d4.to("cuda:1"), hits.to("cuda:1")
    assert lib.ptap_query_closest(r.h, o1.data_ptr(), d1.data_ptr(), 1000, h1.data_ptr(), None) == -1
    assert b"device" in lib.ptap_last_error(r.h)
