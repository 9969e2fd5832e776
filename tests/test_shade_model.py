"""The per-slot shading model (tests/shade_model.py) against the C oracle: draws bit for bit at the RNG's edge seeds, scattered
directions within the model's bound, and whole R1 iterations of the oracle round by round and as a film, bit for bit."""
import numpy as np
import pytest

import shade_model as sm

ITERS = [0, 1, (1 << 22) - 1, 1 << 22, (1 << 22) + 3]               # bits of iter >= 2^22 overlap the remaining-bounce bits
SLOTS = [0, 1, 31, 32, 2047, 2048, 65535, 65536, 1 << 20, 3 * (1 << 20) + 6, 8294399, 8294400]     # up to a 4K wavefront


def test_draws_bit_equal_at_edge_seeds(port):
    for it in ITERS:
        for slot in SLOTS:
            for rem in range(1, sm.K_MAX_DEPTH + 1):
                want = port.rng_u01(it, slot, rem, 6)
                got = sm.rng_draws(sm.rng_seed(it, slot, rem), 6)
                assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (it, slot, rem)


def test_edge_constants(port):
    it, slot, rem = sm.ZERO_SEED
    assert int(sm.seed_hash(it, slot, rem)) % sm.M31 == 0 and int(sm.rng_seed(it, slot, rem)) == 1
    assert np.array_equal(sm.rng_draws(1, 4), port.rng_u01(it, slot, rem, 4))
    it, slot, rem = sm.ONE_DRAW
    u = sm.rng_draws(sm.rng_seed(it, slot, rem), 3)
    assert u[0] == np.float32(1.0) and port.rng_u01(it, slot, rem, 1)[0] == np.float32(1.0)
    assert np.array_equal(u, port.rng_u01(it, slot, rem, 3))
    # u = 1.0f: a DIFFUSE bounce returns the normal itself (up = 1, over = 0), and a COAT bounce takes the diffuse half
    n = np.float32([[0.6, 0.0, 0.8]]); d = np.float32([[0.0, 0.0, -1.0]])
    got, _, _ = sm.scatter(0, n, d, it, slot, rem)
    assert np.array_equal(got.astype(np.float32), n) and np.array_equal(port.scatter(0, n[0], d[0], it, slot, rem), n[0])


def _unit(rs, n):
    v = rs.randn(n, 3)
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_scatter_vs_oracle(port, kind):
    """Several thousand normals, directions and seeds per kind, including axis-aligned normals (the frame switches at 1/sqrt(3)) and
    grazing directions; the oracle runs glibc's sinf / cosf / powf, the model float64: within the model's per-ray bound."""
    rs = np.random.RandomState(100 + kind)
    n_rays = 3000
    nrm = sm.normalize32(_unit(rs, n_rays))
    nrm[:6] = np.float32([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, 0, 0], [0, -1, 0], [0, 0, -1]])
    d = sm.normalize32(_unit(rs, n_rays))
    d[6:50] = sm.normalize32(d[6:50] - nrm[6:50] * (sm.dot32(d[6:50], nrm[6:50]) * np.float32(0.999))[:, None])
    it = rs.choice(ITERS, n_rays); slot = rs.randint(0, 8294400, n_rays); rem = rs.randint(2, 17, n_rays)
    want = np.stack([port.scatter(kind, nrm[i], d[i], int(it[i]), int(slot[i]), int(rem[i])) for i in range(n_rays)])
    got, tol, exact = sm.scatter(kind, nrm, d, it, slot, rem)
    err = np.abs(want.astype(np.float64) - got).max(axis=1)
    print(f"kind {kind}: worst error / bound {(err / tol).max():.3f}, {exact.sum()} exact")
    assert (err <= tol).all()
    assert np.array_equal(want[exact], got[exact].astype(np.float32))
    if kind in (2, 3):
        assert exact.sum() > (n_rays // 3 if kind == 2 else n_rays - 1)


def seven_material_models(models):
    """The bundled scene's 11 models with every material type 0-6 on a visible surface (SPECULAR and REFRACTIVE included)."""
    m = np.array(models, copy=True)
    m["mat"]["type"] = [sm.METAL, sm.COAT, sm.REFLECTIVE, sm.DIFFUSE, sm.SPECULAR, sm.REFRACTIVE, sm.METAL, sm.EMISSIVE, sm.DIFFUSE, sm.COAT, sm.EMISSIVE]
    return m


def run_oracle_checked(port, arrays, W, H, depth, iters, mode=1, rounds_checked=None):
    """R1 iterations of the oracle, each round held to the model; returns (model film, oracle film, per-round counts, worst ratio)."""
    w = port.OracleWavefront(port.OracleScene(arrays), W, H, depth, mode=mode)
    w.init_image()
    probes, counts, worst = [], [], 0.0
    for it in range(iters):
        rounds, state = [], {}

        def on_bounce(b, wf):
            nonlocal worst
            n = wf.nrays
            rays, hits = wf.rays(n), wf.hits(n)
            if "model" in state:                                         # the previous round's prediction of this wavefront
                m = state["model"]
                assert n == len(m["order"]), f"iter {it} round {b}: survivor count"
                assert np.array_equal(rays["ipixel"], state["pix"][m["order"]]), f"iter {it} round {b}: order"
                assert np.array_equal(rays["color"], m["color"][m["order"]]), f"iter {it} round {b}: throughput"
                assert np.array_equal(rays["orig"], m["orig"]), f"iter {it} round {b}: origins"
                ratio, same = sm.dir_errors(rays["dir"], m)
                worst = max(worst, ratio)
                assert ratio <= 1.0 and same, f"iter {it} round {b}: directions (worst error / bound {ratio:.3f}, exact ones equal: {same})"
                assert (rays["remaining_bounces"] == depth - b).all()
            hit = hits["dist"] < sm.FLOAT_MAX
            typ = np.where(hit, hits["mat"]["type"], -1)
            alb = hits["mat"]["color"]
            rounds.append((rays["ipixel"].copy(), hit, typ, alb))
            if rounds_checked is None or b in rounds_checked:
                state["model"] = sm.shade(rays["orig"], rays["dir"], rays["color"], hit, hits["dist"], hits["normal"], typ, alb, it, depth - b)
            else:
                state.pop("model", None)
            state["pix"] = rays["ipixel"].copy()

        counts.append(w.run_iteration(it, on_bounce))
        probes.append(rounds)
    want = w.image()
    w.close()
    return sm.predict_film(probes, H, W, depth), want, counts, worst


@pytest.mark.parametrize("scene", ["bundled", "seven"])
def test_oracle_iterations_round_by_round(port, golden_scene, scene):
    """R1 on the bundled scene and on the seven-material scene: every round's next wavefront (survivors, order, throughput, origins
    exact; directions within the bound, reflections exact) and the film of three iterations bit for bit."""
    arrays = {k: golden_scene[k] for k in ("models", "meshes", "vertices", "triangles")}
    if scene == "seven":
        arrays["models"] = seven_material_models(arrays["models"])
    W, H, depth, iters = 64, 48, 6, 3
    film, want, counts, worst = run_oracle_checked(port, arrays, W, H, depth, iters)
    print(f"{scene}: counts {counts}, worst direction error / bound {worst:.3f}")
    assert np.array_equal(film, want)
    assert all(len(c) == depth for c in counts)                     # paths survive to the last round
    assert want.mean() > 0.05


def test_seven_material_scene_covers_every_type(port, golden_scene):
    """Every material type 0-6 is the first hit of at least 1 % of the frame's pixels (so the GPU tests that use the scene see them)."""
    arrays = {k: golden_scene[k] for k in ("models", "meshes", "vertices", "triangles")}
    arrays["models"] = seven_material_models(arrays["models"])
    W, H = 96, 64
    w = port.OracleWavefront(port.OracleScene(arrays), W, H, 1, mode=1)
    w.generate(); w.trace()
    hits = w.hits(W * H)
    typ = np.where(hits["dist"] < sm.FLOAT_MAX, hits["mat"]["type"], -1)
    w.close()
    share = np.array([np.mean(typ == t) for t in range(7)])
    print("first-hit share per type", np.round(share, 3))
    assert (share >= 0.01).all()
