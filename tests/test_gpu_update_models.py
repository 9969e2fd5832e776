"""Moving models of an uploaded scene (ptap_update_models, Renderer.update_models; DESIGN.md 4.9).

After an update the renderer must trace, answer queries and render exactly as a fresh renderer over Scene.from_arrays of the same scene
with the moved models and the same accel: hits, films and occlusion bit for bit, and the oracle of the moved scene in every field."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
FIELDS = ("model", "tri", "t_model", "dist", "u", "v", "normal", "mat_type")
ACCELS = [("grid", 0, 0), ("emu", 3, 0), ("bvh", 1, 1), ("bvh_device", 2, 1)]     # name, accel, oracle tier
W, H, DEPTH = 64, 48, 5


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
    from pathtracerap_b200 import HIT
    out = np.zeros(q["model"].shape[0], HIT)
    for f in FIELDS:
        out[f] = q[f].cpu().numpy()
    return out


def _assert_oracle(got, want, what):
    assert np.array_equal(got["model"], want["model"]), f"{what}: model ids differ on {(got['model'] != want['model']).sum()} rays"
    assert np.array_equal(got["tri"], want["tri"]), f"{what}: triangle ids differ"
    hit = want["model"] >= 0
    for f in ("t_model", "dist", "u", "v", "normal"):
        assert np.array_equal(got[f][hit], want[f][hit]), f"{what}: {f} not bit-equal to the oracle"
    assert np.array_equal(got["mat_type"], want["mat_type"]), f"{what}: material types differ"


def _place(models, which, rs, translate=60.0, scale=(0.6, 1.5)):
    """Models `which` rotated about a random axis and scaled non-uniformly in model space, then moved by up to `translate`: model_to_world
    in binary32, world_to_model its inverse (float64, rounded)."""
    out = models.copy()
    for i in which:
        M = out["model_to_world"][i].reshape(4, 4).T.astype(np.float64)       # column-major storage
        q, _ = np.linalg.qr(rs.randn(3, 3))
        if np.linalg.det(q) < 0:
            q[:, 0] *= -1
        R = np.eye(4); R[:3, :3] = q * rs.uniform(*scale, 3)[None, :]
        T = np.eye(4); T[:3, 3] = rs.uniform(-translate, translate, 3)
        Mn = (T @ M @ R).astype(np.float32)
        out["model_to_world"][i] = Mn.T.reshape(16)
        out["world_to_model"][i] = np.linalg.inv(Mn.astype(np.float64)).astype(np.float32).T.reshape(16)
    return out


def _scene(g, models):
    from pathtracerap_b200 import Scene
    s = Scene.from_arrays(models, g["meshes"], g["vertices"], g["triangles"])
    s.build_grids(25, 25, 25)
    return s


def _renderer(scene, accel, **kw):
    from pathtracerap_b200 import Renderer
    r = Renderer(width=W, height=H, depth=DEPTH, accel=accel, **kw)
    r.allocateOnGPU(scene)
    return r


def _film(r, iters=8):
    r.frame_begin()
    r.render(0, iters)
    r.sync()
    return r.film()


@pytest.fixture(scope="module")
def base(libptap, golden_scene):
    """The bundled scene as uploaded (grid indices set by build_grids) and random rays over it."""
    s = _scene(golden_scene, golden_scene["models"])
    return golden_scene, s.models, _rays(300_000, 41)


def _check_occluded(r, rays, want, what):
    """query_occluded at L = dist, one ulp either side and inf, against (model >= 0) & (dist < L)."""
    hit = want["model"] >= 0
    base_len = np.where(hit, want["dist"], np.float32(500.0)).astype(np.float32)
    org, dir_ = _dev(rays)
    for L in (base_len, np.nextafter(base_len, np.float32(0)), np.nextafter(base_len, np.float32(np.inf)), np.full_like(base_len, np.inf)):
        got = r.query_occluded(org, dir_, torch.from_numpy(L).cuda()).cpu().numpy()
        assert np.array_equal(got, hit & (want["dist"] < L)), f"{what}: occlusion differs on {(got != (hit & (want['dist'] < L))).sum()} rays"


@pytest.mark.parametrize("name,accel,tier", ACCELS)
def test_update_hits_equal_fresh_and_oracle(base, port, golden_trace, name, accel, tier):
    g, models, rnd = base
    moved = _place(models, [0, 3, 5, 8, 10], np.random.RandomState(7))
    r = _renderer(_scene(g, models), accel)
    r.update_models(moved)
    fresh = _renderer(_scene(g, moved), accel)
    oracle = port.OracleScene({"models": moved, "meshes": g["meshes"], "vertices": g["vertices"], "triangles": g["triangles"]})
    for rays, what in ((golden_trace["rays"], "golden rays"), (rnd, "300k random rays")):
        got = r.trace(rays)
        assert got.tobytes() == fresh.trace(rays).tobytes(), f"{name}, {what}: trace differs from the fresh renderer"
        assert _records(r.query_closest(*_dev(rays))).tobytes() == got.tobytes(), f"{name}, {what}: query_closest differs from trace"
        sub = slice(None) if len(rays) < 50_000 else slice(None, None, 15)
        _assert_oracle(got[sub], oracle.trace(rays[sub], tier), f"{name}, {what}, oracle R{tier}")
        _check_occluded(r, rays, got, f"{name}, {what}")
    assert (got["model"] >= 0).sum() > 10_000
    r.free(); fresh.free()


@pytest.mark.parametrize("name,accel", [("emu", 3), ("bvh", 1)])
def test_update_films_equal_fresh(base, monkeypatch, name, accel):
    """4 lanes, first-hit cache, 8 iterations; transforms, a material colour and a material type change."""
    from pathtracerap_b200 import METAL
    monkeypatch.setenv("PTAP_LANES", "4")
    g, models, _ = base
    moved = _place(models, [1, 4, 9], np.random.RandomState(11))
    moved["mat"]["color"][2] = (0.2, 0.9, 0.4)
    moved["mat"]["type"][6] = METAL
    r = _renderer(_scene(g, models), accel)
    _film(r)                                           # a first-hit cache of the old placement
    r.update_models(moved)
    fresh = _renderer(_scene(g, moved), accel)
    assert r.stats()["lanes"] == 4
    a, b = _film(r), _film(fresh)
    assert a.tobytes() == b.tobytes(), f"{name}: film differs from the fresh renderer's on {(a != b).sum()} values"
    r.free(); fresh.free()


@pytest.mark.parametrize("name,accel", [("emu", 3), ("bvh_device", 2)])
def test_update_sequences(base, name, accel):
    """Partial ranges, ten successive updates, and back to the original models: exactly the never-moved renderer."""
    g, models, rnd = base
    rays = rnd[:100_000]
    r = _renderer(_scene(g, models), accel)
    ref_trace, ref_film = r.trace(rays), _film(r)
    rs = np.random.RandomState(3)
    cur = models.copy()
    for step in range(10):
        first = int(rs.randint(0, len(models)))
        count = int(rs.randint(1, len(models) - first + 1))
        cur = _place(cur, range(first, first + count), rs, translate=25.0, scale=(0.8, 1.25))
        r.update_models(cur[first:first + count], first)
    fresh = _renderer(_scene(g, cur), accel)
    assert r.trace(rays).tobytes() == fresh.trace(rays).tobytes(), f"{name}: after ten partial updates"
    assert _film(r).tobytes() == _film(fresh).tobytes()
    fresh.free()
    r.update_models(models)
    assert r.trace(rays).tobytes() == ref_trace.tobytes(), f"{name}: back to the original models"
    assert _film(r).tobytes() == ref_film.tobytes()
    r.free()


def _cloud(n, seed):
    """n instances of two small meshes (an 80-triangle icosphere and a 20-triangle one) in a 1000-unit cube."""
    from pathtracerap_b200 import Scene
    rs = np.random.RandomState(seed)
    s = Scene.empty()
    meshes = [s.add_icosphere(1, radius=1.0, displacement=0.05, seed=3), s.add_icosphere(0, radius=1.0, displacement=0.0, seed=4)]
    for k in range(n):
        sc = rs.uniform(2.0, 8.0)
        s.add_model(meshes[k % 2], translate=tuple(rs.uniform(-500, 500, 3)), rotate_y_degrees=float(rs.uniform(0, 360)),
                    scale=(sc, sc * rs.uniform(0.5, 2.0), sc), color=tuple(rs.uniform(0.2, 0.9, 3)))
    return s


@pytest.mark.parametrize("name,accel", [("bvh", 1), ("bvh_device", 2)])
def test_update_many_instances(libptap, port, name, accel):
    """12,000 instances: more clusters than the host SAH top takes, so PLOC builds the lower levels of the device TLAS."""
    from pathtracerap_b200 import Scene
    s = _cloud(12_000, 5)
    a = s.arrays()
    r = _renderer(s, accel)
    moved = _place(a["models"], range(0, 12_000, 2), np.random.RandomState(9), translate=40.0)
    r.update_models(moved)
    fresh = _renderer(Scene.from_arrays(moved, a["meshes"], a["vertices"], a["triangles"]), accel)
    rays = _rays(300_000, 19, -600.0, 600.0)
    got = r.trace(rays)
    assert got.tobytes() == fresh.trace(rays).tobytes(), f"{name}: trace differs from the fresh renderer"
    assert (got["model"] >= 0).sum() > 10_000
    assert _records(r.query_closest(*_dev(rays))).tobytes() == got.tobytes()
    oracle = port.OracleScene({"models": moved, "meshes": a["meshes"], "vertices": a["vertices"], "triangles": a["triangles"]})
    _assert_oracle(got[:2000], oracle.trace(rays[:2000], 1), f"{name}: oracle R1")
    r.free(); fresh.free()


def test_update_matrices_not_inverses(base, port, golden_trace):
    """model_to_world that is not the inverse of world_to_model (the traversal then prunes nothing across instances): still exact."""
    g, models, rnd = base
    moved = _place(models, [2, 7], np.random.RandomState(5))
    moved["world_to_model"][7] *= np.float32(1.02)
    for accel in (1, 2):
        r = _renderer(_scene(g, models), accel)
        r.update_models(moved)
        fresh = _renderer(_scene(g, moved), accel)
        for rays in (golden_trace["rays"], rnd[:100_000]):
            assert r.trace(rays).tobytes() == fresh.trace(rays).tobytes()
        oracle = port.OracleScene({"models": moved, "meshes": g["meshes"], "vertices": g["vertices"], "triangles": g["triangles"]})
        _assert_oracle(r.trace(golden_trace["rays"]), oracle.trace(golden_trace["rays"], 1), f"accel {accel}: oracle R1")
        r.free(); fresh.free()


@pytest.mark.parametrize("name,accel", [("grid", 0), ("bvh", 1)])
def test_update_rejects_bad_input(base, name, accel):
    """A singular world_to_model, a changed mesh or grid index, a bad range: rejected, and the renderer traces exactly as before."""
    from pathtracerap_b200 import PtapError, _native as N
    g, models, rnd = base
    rays = rnd[:50_000]
    r = _renderer(_scene(g, models), accel)
    before = r.trace(rays)
    good = _place(models, range(len(models)), np.random.RandomState(2))
    singular = good.copy(); singular["world_to_model"][4, [0, 4, 8]] = 0.0
    mesh = good.copy(); mesh["mesh_index"][3] = (mesh["mesh_index"][3] + 1) % len(g["meshes"])
    grid = good.copy(); grid["grid_index"][5] += 1
    for bad, first, what in ((singular, 0, "model 4: world_to_model is singular"), (mesh, 0, "model 3: mesh_index"), (grid, 0, "model 5: grid_index"),
                             (good[:3], len(models) - 2, "out of range"), (good[:1], -1, "out of range")):
        with pytest.raises(PtapError, match=what):
            r.update_models(bad, first)
        assert r.trace(rays).tobytes() == before.tobytes(), f"{name}: {what} changed the context"
    with pytest.raises(PtapError, match="dtype"):
        r.update_models(good.view(np.uint8))
    assert N.lib().ptap_update_models(r.h, None, 0, 0) == 0                    # count == 0: a no-op
    assert r.trace(rays).tobytes() == before.tobytes()
    r.free()


def test_update_ordering(base):
    """A render enqueued before the update renders the unmoved scene; an update before any upload is a state error."""
    from pathtracerap_b200 import Renderer, _native as N
    g, models, _ = base
    moved = _place(models, range(len(models)), np.random.RandomState(13))
    ref = _renderer(_scene(g, models), 1)
    want = _film(ref, 6)
    r = _renderer(_scene(g, models), 1)
    r.frame_begin()
    r.render(0, 6)                                     # asynchronous: still running when the update is called
    r.update_models(moved)
    assert r.film().tobytes() == want.tobytes()
    fresh = _renderer(_scene(g, moved), 1)
    assert _film(r, 6).tobytes() == _film(fresh, 6).tobytes()
    for x in (ref, r, fresh):
        x.free()
    empty = Renderer(width=W, height=H, depth=DEPTH)
    assert N.lib().ptap_update_models(empty.h, N.ptr(models), 0, len(models)) == -6
    assert N.lib().ptap_update_models(empty.h, None, 0, 0) == -6
    empty.free()


def test_update_then_rebuild_from_host_copies(base, golden_trace):
    """Builds after an update upload the instance records from the context's host copies: a BVH build of another kind and the device
    grid build must keep the moved models, exactly as a fresh renderer of the moved scene."""
    g, models, rnd = base
    rays = np.concatenate([golden_trace["rays"], rnd[:100_000]])
    moved = _place(models, [0, 2, 6, 9], np.random.RandomState(17))
    s = _scene(g, models)
    r = _renderer(s, 2)
    r.update_models(moved)
    fresh = _renderer(_scene(g, moved), 1)
    r.set_accel(1)                                     # the host BVH: uploadBvh + finishBvh re-upload d_inst
    assert r.trace(rays).tobytes() == fresh.trace(rays).tobytes(), "build_accel(BVH) after the update"
    r.build_grids_device(s)                            # re-uploads d_inst as well; selects the grid walk
    fresh.set_accel(0)
    assert r.trace(rays).tobytes() == fresh.trace(rays).tobytes(), "build_grids_device after the update"
    r.free(); fresh.free()
