"""k_scan + k_shade + film accumulation held to the exact per-slot model (tests/shade_model.py) at production sizes.

ptap_shade at n from 1 to 3 * 2^20 + 7 slots (partial tiles, more than one look-back window of k_scan, CTAs of k_shade that shade more
than one block), and whole frames through ptap_render_probe / ptap_render: survivors, order, origins and throughput exact, directions
within the model's bound, and the film of ptap_render equal to the model's film bit for bit."""
import os

import numpy as np
import pytest

import shade_model as sm
from conftest import have_gpu
from test_gpu_production import _assert_production_hits
from test_shade_model import ITERS, seven_material_models

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_gpu(), reason="no CUDA device")]

SIZES = [1, 31, 32, 33, 255, 256, 257, 2047, 2048, 2049, 65535, 65536, 65537, 3 * (1 << 20) + 7]
REMAINING = [1, 2, 5, 16]


def _albedo(models):
    return np.ascontiguousarray(models["mat"]["color"], np.float32)


def _renderer(scene, W, H, depth, accel, sort=None, lanes=None, first_hit_cache=True):
    from pathtracerap_b200 import Renderer
    old = {k: os.environ.get(k) for k in ("PTAP_SHADE_SORT", "PTAP_LANES")}
    try:
        for k, v in (("PTAP_SHADE_SORT", sort), ("PTAP_LANES", lanes)):
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = str(v)
        r = Renderer(width=W, height=H, depth=depth, accel=accel, first_hit_cache=first_hit_cache)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    r.allocateOnGPU(scene)
    return r


@pytest.fixture(scope="module")
def seven_scene(libptap, golden_scene):
    from pathtracerap_b200 import Scene
    models = seven_material_models(golden_scene["models"])
    s = Scene.from_arrays(models, golden_scene["meshes"], golden_scene["vertices"], golden_scene["triangles"])
    s.build_grids(25, 25, 25)
    s.build_bvh()
    return s, models


# ------------------------------------------------------------------------------------------------------------ a. ptap_shade sweep

def _random_paths(r, models, n, seed):
    """n paths whose hits are real: rays from the camera region and from inside the box, traced by the renderer; about 1 in 8 rays
    points away from the scene and misses.  Throughputs are random."""
    from pathtracerap_b200 import PATH_IN
    rs = np.random.RandomState(seed)
    o = np.zeros((n, 3), np.float32)
    cam = rs.rand(n) < 0.5
    o[cam] = (0.0, 0.0, 920.0)
    o[~cam] = rs.uniform(-300, 300, ((~cam).sum(), 3)) + np.float32([0, 0, 400])
    d = rs.randn(n, 3).astype(np.float32)
    d[cam] = np.stack([rs.uniform(-10, 10, cam.sum()), rs.uniform(-4, 12, cam.sum()), np.full(cam.sum(), -20.0)], 1)
    d[rs.rand(n) < 0.12, 2] = 50.0
    d *= rs.uniform(0.5, 3.0, (n, 1)).astype(np.float32)              # ray directions are not normalised
    hits = r.trace(np.concatenate([o, d], 1))
    p = np.zeros(n, PATH_IN)
    p["orig"], p["dir"] = o, d
    p["color"] = rs.uniform(0.0, 1.0, (n, 3)).astype(np.float32)
    p["ipixel"] = rs.permutation(n)
    p["model"], p["tri"], p["dist"] = hits["model"], hits["tri"], hits["dist"]
    return p, hits


def test_shade_sweep_exact(seven_scene):
    """ptap_shade against the model at every size of SIZES, with remaining bounces, iteration seeds (edge seeds included) and both
    shade schedules (PTAP_SHADE_SORT 0 / 1): alive, order, throughput, origins and film contributions bit-equal, directions in bound."""
    from pathtracerap_b200 import ACCEL_BVH
    scene, models = seven_scene
    alb = _albedo(models)
    rs = [_renderer(scene, 64, 48, 5, ACCEL_BVH, sort=s) for s in (0, 1)]
    pool, hits = _random_paths(rs[0], models, SIZES[-1], 5)
    j = np.nonzero(hits["mat_type"] == sm.DIFFUSE)[0][0]
    for slot in (sm.ZERO_SEED[1], sm.ONE_DRAW[1]):                        # the edge seeds' slots bounce off a DIFFUSE surface
        pool[slot], hits[slot] = pool[j], hits[j]
    hit = pool["model"] >= 0
    typ = np.where(hit, hits["mat_type"], -1)
    assert all(np.mean(typ == t) > 0.005 for t in range(-1, 7)), "every material type and misses must be present"
    cases = [(n, ITERS[k % len(ITERS)], REMAINING[k % len(REMAINING)]) for k, n in enumerate(SIZES)]
    cases += [(SIZES[-1], it, rem) for it, rem in ((ITERS[3], 16), (ITERS[2], 2))]
    cases += [(2049, it, rem) for it in ITERS for rem in REMAINING]
    cases += [(257, *sm.ZERO_SEED[::2]), (257, *sm.ONE_DRAW[::2])]                # the edge seeds' slots are below 256
    worst = 0.0
    for n, it, rem in cases:
        p = pool[:n]
        a = np.ascontiguousarray(alb[np.maximum(p["model"], 0)])
        m = sm.shade(p["orig"], p["dir"], p["color"], hit[:n], p["dist"], hits["normal"][:n], typ[:n], a, it, rem)
        for sort, r in enumerate(rs):
            what = f"n={n} iter={it} remaining={rem} sort={sort}"
            out, order = r.shade(p, it, rem)
            al = m["alive"]
            assert np.array_equal(out["alive"].astype(bool), al), f"{what}: survivors"
            assert np.array_equal(order, m["order"]), f"{what}: compaction order"
            assert np.array_equal(out["color"][al], m["color"][al]), f"{what}: throughput"
            assert np.array_equal(out["color"][~al], m["contrib"][~al]), f"{what}: film contribution sqrt(throughput)"
            assert np.array_equal(out["orig"][order], m["orig"]), f"{what}: origins"
            ratio, same = sm.dir_errors(out["dir"][order], m)
            assert ratio <= 1.0 and same, f"{what}: directions (worst error / bound {ratio:.3f}, exact ones equal: {same})"
            worst = max(worst, ratio)
    print(f"ptap_shade sweep: {len(cases)} cases x 2 schedules, largest n {SIZES[-1]}, worst direction error / bound {worst:.3f}")
    for r in rs:
        r.free()


# ---------------------------------------------------------------------------------------------- b. production frames, round by round

def _probe_iteration(r, it, depth):
    rounds = []
    for rnd in range(depth):
        rays, pix, hits = r.render_probe(it, rnd)
        if len(rays) == 0:
            break
        rounds.append((rays, pix, hits))
    return rounds


def _model_rounds(rounds, alb):
    out = []
    for rays, pix, hits in rounds:
        hit = hits["model"] >= 0
        out.append((pix, hit, np.where(hit, hits["mat_type"], -1), np.ascontiguousarray(alb[np.maximum(hits["model"], 0)])))
    return out


def check_frame(r, alb, W, H, depth, iters, dir_iters=(0,), oracle_scene=None, tier=1):
    """Every round of every iteration of a frame against the model, then ptap_render's film against predict_film bit for bit.
    Directions are compared on the iterations in dir_iters (the others add nothing the first does not); with an oracle scene the first
    iteration's hits are compared with the oracle's tier `tier` (R0: the grid walk, R1: the exact closest hit).  Returns the probes."""
    N = W * H
    probes, lengths, worst = [], [], 0.0
    for it in range(iters):
        rounds = _probe_iteration(r, it, depth)
        assert len(rounds[0][0]) == N and np.array_equal(rounds[0][1], np.arange(N))
        mr = _model_rounds(rounds, alb)
        for k, (rays, pix, hits) in enumerate(rounds):
            what = f"{W}x{H} depth {depth} iter {it} round {k}"
            if oracle_scene is not None and it == 0:
                _assert_production_hits(hits, oracle_scene.trace(rays, tier), what)
            _, hit, typ, a = mr[k]
            m = sm.shade(rays[:, :3], rays[:, 3:], np.ones((len(rays), 3), np.float32), hit, hits["dist"], hits["normal"], typ, a, it,
                         depth - k, directions=it in dir_iters)
            nxt = rounds[k + 1] if k + 1 < len(rounds) else None
            assert (0 if nxt is None else len(nxt[0])) == len(m["order"]), f"{what}: survivor count"
            if nxt is None:
                continue
            assert np.array_equal(nxt[1], pix[m["order"]]), f"{what}: next round's pixels are not the survivors in stable order"
            assert np.array_equal(nxt[0][:, :3], m["orig"]), f"{what}: origins not bit-equal"
            if it in dir_iters:
                ratio, same = sm.dir_errors(nxt[0][:, 3:], m)
                assert ratio <= 1.0 and same, f"{what}: directions (worst error / bound {ratio:.3f}, exact ones equal: {same})"
                worst = max(worst, ratio)
        probes.append(mr)
        lengths.append([len(x[0]) for x in rounds] + [0] * (depth - len(rounds)))
    want = sm.predict_film(probes, H, W, depth)
    r.frame_begin()
    r.render(0, iters)
    film = r.film()
    st = r.stats()
    assert st["active_per_round"][:depth] == lengths[-1]
    assert st["rays_traced"] == int(np.sum(lengths)) - (iters - 1) * N              # the first-hit cache: round 0 is traced once
    diff = int(np.sum(np.any(film != want, axis=-1)))
    assert np.array_equal(film, want), f"{W}x{H} depth {depth}: film differs from the model's on {diff} pixels"
    print(f"{W}x{H} depth {depth} x{iters}: film bit-equal, rounds {lengths[-1]}, worst direction error / bound {worst:.3f}")
    return probes


@pytest.mark.parametrize("config", ["emu", "bvh", "bvh_lanes1", "bvh_sort"])
def test_production_frame_bundled_1000x800(gpu_scene, golden_scene, config):
    """The reference's frame size (800,000 slots, 391 scan blocks) on the bundled scene."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_EMULATED
    accel = ACCEL_GRID_EMULATED if config == "emu" else ACCEL_BVH
    r = _renderer(gpu_scene, 1000, 800, 5, accel, sort=1 if config == "bvh_sort" else None, lanes=1 if config == "bvh_lanes1" else None)
    check_frame(r, _albedo(golden_scene["models"]), 1000, 800, 5, 3)
    r.free()


def test_production_frame_mesh1m_1920x1080(libptap):
    """The benchmark's configuration: the 1.3M-triangle mesh at 1920x1080, depth 5, BVH, 4 lanes (frames above 2^20 pixels)."""
    import bench
    from pathtracerap_b200 import ACCEL_BVH
    scene, arrays = bench.build_scene("mesh1m")
    scene.build_bvh()
    r = _renderer(scene, 1920, 1080, 5, ACCEL_BVH)
    assert r.stats()["lanes"] == 4
    check_frame(r, _albedo(arrays["models"]), 1920, 1080, 5, 4)
    r.free()


def test_production_frame_cornell_and_full_depth(libptap, golden_scene, golden_films):
    """Cornell at 512x512, depth 8 (GRID_EMULATED), and a frame at depth 16 = kMaxDepth."""
    from pathtracerap_b200 import ACCEL_GRID_EMULATED, Scene
    m = golden_films["cornell_models"]
    s = Scene.from_arrays(m, golden_scene["meshes"], golden_scene["vertices"], golden_scene["triangles"])
    s.build_grids()
    r = _renderer(s, 512, 512, 8, ACCEL_GRID_EMULATED)
    check_frame(r, _albedo(m), 512, 512, 8, 2)
    r.set_params(96, 64, sm.K_MAX_DEPTH, first_hit_cache=True)
    probes = check_frame(r, _albedo(m), 96, 64, sm.K_MAX_DEPTH, 2, dir_iters=(0, 1))
    assert len(probes[0]) == sm.K_MAX_DEPTH                           # paths survive into the last round
    r.free()


def test_production_frame_tiny_sizes(gpu_scene, golden_scene):
    """5x7, 31x1 and 1x1 frames, and depth 1, where nothing survives round 0."""
    from pathtracerap_b200 import ACCEL_BVH
    alb = _albedo(golden_scene["models"])
    r = _renderer(gpu_scene, 5, 7, 5, ACCEL_BVH)
    check_frame(r, alb, 5, 7, 5, 3, dir_iters=(0, 1, 2))
    for W, H, depth in ((31, 1, 5), (1, 1, 5), (64, 48, 1)):
        r.set_params(W, H, depth, first_hit_cache=True)
        probes = check_frame(r, alb, W, H, depth, 3, dir_iters=(0, 1, 2))
        if depth == 1:
            assert all(len(p) == 1 for p in probes)
    r.free()


# ------------------------------------------------------------------------------------------------------ c. a seven-material scene

@pytest.mark.parametrize("sort", [0, 1])
def test_seven_material_frame(seven_scene, oracle_scene, port, golden_scene, sort):
    """Every material type 0-6 on a visible surface, at 333x211 = 70,263 slots: more than one look-back window, and not a multiple of
    32, 256 or 2048.  Round by round against the model (and the first iteration's hits against the oracle's R1), the film bit-equal
    to the model's, and the film against the oracle's R1 frame under the statistical bound of the other frame tests (below the tail)."""
    from pathtracerap_b200 import ACCEL_BVH
    scene, models = seven_scene
    W, H, depth, iters = 333, 211, 5, 2
    oscene = port.OracleScene({**{k: golden_scene[k] for k in ("meshes", "vertices", "triangles")}, "models": models})
    r = _renderer(scene, W, H, depth, ACCEL_BVH, sort=sort)
    probes = check_frame(r, _albedo(models), W, H, depth, iters, dir_iters=(0, 1), oracle_scene=oscene)
    types = np.concatenate([p[2] for p in probes[0]])
    assert all((types == t).sum() > 500 for t in range(7))
    film = r.film()
    r.free()
    w = port.OracleWavefront(oscene, W, H, depth, mode=1)
    w.init_image()
    for it in range(iters):
        w.run_iteration(it)
    want = w.image()
    w.close()
    span = (W * H // 32) * 32
    f, g = film.reshape(-1, 3)[:span], want.reshape(-1, 3)[:span]
    rmse = float(np.sqrt(np.mean((f - g) ** 2)))
    exact = float(np.mean(np.all(f == g, axis=-1)))
    print(f"seven-material vs oracle R1: rmse={rmse:.3e} mean={g.mean():.3f} bit-equal pixels={exact:.4f}")
    assert rmse <= 0.005 * g.mean() and exact > 0.97


# ------------------------------------------------------------------------------------------------ d. tail pixels (W * H mod 32 != 0)

def test_tail_pixels_are_rendered(gpu_scene, golden_scene, port):
    """The reference launches N / 32 blocks of 32 (integer division), so its last N mod 32 pixels are never traced and stay black;
    this library renders every pixel (DESIGN 2).  At 100x75 (7,500 = 234 * 32 + 12): the pixels below 7,488 meet the film bound against
    the oracle's R1 frame, the last 12 are zero there and lit here; tail paths sort after every other survivor in every round, so the
    other slots keep the reference's random streams, and the active counts differ exactly by the tail's surviving paths."""
    from pathtracerap_b200 import ACCEL_BVH
    W, H, depth, iters = 100, 75, 5, 4
    N = W * H
    span = (N // 32) * 32
    assert N - span == 12
    r = _renderer(gpu_scene, W, H, depth, ACCEL_BVH)
    probes = check_frame(r, _albedo(golden_scene["models"]), W, H, depth, iters, dir_iters=(0, 1, 2, 3))
    film = r.film().reshape(N, 3)
    r.free()
    w = port.OracleWavefront(port.OracleScene({k: golden_scene[k] for k in ("models", "meshes", "vertices", "triangles")}), W, H, depth, mode=1)
    w.init_image()
    counts = [w.run_iteration(it) for it in range(iters)]
    want = w.image().reshape(N, 3)
    w.close()
    assert (want[span:] == 0).all() and (film[span:] > 0).any(axis=-1).all()
    rmse = float(np.sqrt(np.mean((film[:span] - want[:span]) ** 2)))
    assert rmse <= 0.005 * want[:span].mean() and float(np.mean(np.all(film[:span] == want[:span], axis=-1))) > 0.97
    for it, rounds in enumerate(probes):
        gpu = []
        for k, (pix, _, _, _) in enumerate(rounds):
            tail = pix >= span
            n_tail = int(tail.sum())
            assert not tail[:len(pix) - n_tail].any(), f"iter {it} round {k}: a tail path sorts before another survivor"
            gpu.append(len(pix) - (n_tail if k else 0))
        ref = counts[it] + [0] * (len(gpu) - len(counts[it]))
        assert gpu[:2] == ref[:2], f"iter {it}: active counts {gpu} vs the reference's {ref}"
        assert np.abs(np.array(gpu) - np.array(ref[:len(gpu)])).max() <= 0.01 * N
