"""The C restatement (oracle/ptap_oracle.c) against vectors dumped from the reference's own code (tools/make_golden.py).
These run on any machine: they need neither /root/reference nor a GPU."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import live_scenes, ref

FLOAT_MAX = np.float32(9999999.0)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def golden_live():
    z = np.load(os.path.join(GOLDEN, "live_scenes.npz"))
    return {k: z[k] for k in z.files}


def test_hash_and_rng_known_answers(port, golden_kat):
    k = golden_kat
    got = np.array([port.util_hash(int(x)) for x in k["hash_in"]], np.uint32)
    assert np.array_equal(got, k["hash_out"])
    for (it, ix, dp), want in zip(k["rng_args"], k["rng_out"]):
        assert np.array_equal(port.rng_u01(int(it), int(ix), int(dp), 8), want)


def test_rng_can_return_one(port):
    # uniform_real_distribution<float> divides by 2^31 after rounding: the top of the range maps to exactly 1.0f (SURVEY 8a a8)
    import ctypes as C
    st = C.c_uint(0)
    L = port.lib()
    # find the predecessor state of x = 2^31-2 : x = 48271*s mod m  =>  s = x * inv(48271) mod m
    m = 2147483647
    inv = pow(48271, -1, m)
    st.value = ((m - 1) * inv) % m
    assert L.oracle_rng_next(C.byref(st)) == 1.0 and st.value == m - 1


def test_scatter_known_answers(port, golden_kat):
    k = golden_kat
    for i, (kind, it, ix, dp) in enumerate(k["sc_args"]):
        got = port.scatter(int(kind), k["sc_n"][i], k["sc_d"][i], int(it), int(ix), int(dp))
        assert np.array_equal(got, k["sc_out"][i]), (i, kind, got, k["sc_out"][i])


def test_grid_build_matches_reference(port, golden_scene):
    g = golden_scene
    models, grids, voxels, refs = port.build_grids(g["models"], g["meshes"], g["vertices"], g["triangles"])
    assert models.tobytes() == g["models"].tobytes()          # grid_index assignment
    assert grids.tobytes() == g["grids"].tobytes()            # voxel widths, creating model
    assert len(voxels) == int(g["nvoxels"]) == 46875 and len(refs) == int(g["nrefs"]) == 38138
    assert sha(voxels) == str(g["voxels_sha"]) and sha(refs) == str(g["refs_sha"])


def test_trace_r0_r1_golden(oracle_scene, golden_trace):
    t = golden_trace
    for mode, key in ((0, "r0"), (1, "r1")):
        got = oracle_scene.trace(t["rays"], mode)
        want = t[key]
        assert np.array_equal(got["model"], want["model"]) and np.array_equal(got["tri"], want["tri"])
        hit = want["model"] >= 0
        for f in ("t_model", "dist", "u", "v", "normal"):
            assert np.array_equal(got[f][hit], want[f][hit]), (key, f)
        assert np.array_equal(got["mat_type"], want["mat_type"])
        assert (got["dist"][~hit] >= FLOAT_MAX).all()


def test_r0_is_not_exact_closest_hit(golden_trace):
    # SURVEY 0.5: the reference grid walk misses / returns farther hits than brute force, never closer ones
    r0, r1 = golden_trace["r0"], golden_trace["r1"]
    differ = (r0["tri"] != r1["tri"]) | (r0["model"] != r1["model"])
    assert 0 < differ.sum() < 0.01 * len(r0)
    both = (r0["model"] >= 0) & (r1["model"] >= 0)
    assert (r0["dist"][both] >= r1["dist"][both]).all()
    assert not ((r0["model"] >= 0) & (r1["model"] < 0)).any()


def test_wavefront_checkpoints_1000x800(port, oracle_scene, golden_trace):
    w = port.OracleWavefront(oracle_scene, 1000, 800, 5)
    w.init_image()
    hits = []
    counts = w.run_iteration(0, on_bounce=lambda b, ww: hits.append(int((ww.hits(ww.nrays)["dist"] < FLOAT_MAX).sum())))
    assert counts == [800000, 708894, 474310, 348742, 254855] == list(golden_trace["active_per_bounce"])   # SURVEY A.3
    assert hits == [800000, 574891, 409613, 300967, 223986] == list(golden_trace["hits_per_bounce"])
    w.close()


def test_wavefront_states_golden(port, oracle_scene, golden_wavefront):
    g = golden_wavefront
    w = port.OracleWavefront(oracle_scene, 64, 48, 5)
    w.init_image()
    k = 0
    for it in range(2):
        w.generate()
        while w.nrays > 0:
            n = w.nrays
            assert n == int(g["n"][k]) and it == int(g["iter"][k])
            w.trace()
            rays, hits, probe = w.rays(n), w.hits(n), w.probe(n)
            assert np.array_equal(rays["orig"], g[f"pre_orig_{k}"]) and np.array_equal(rays["dir"], g[f"pre_dir_{k}"])
            assert np.array_equal(rays["color"], g[f"pre_color_{k}"]) and np.array_equal(rays["ipixel"], g[f"pre_ipixel_{k}"])
            assert np.array_equal(hits["dist"], g[f"hit_dist_{k}"])
            hit = hits["dist"] < FLOAT_MAX
            assert np.array_equal(probe["model"][hit], g[f"hit_model_{k}"][hit]) and np.array_equal(probe["tri"][hit], g[f"hit_tri_{k}"][hit])
            assert np.array_equal(hits["normal"][hit], g[f"hit_normal_{k}"][hit])
            w.shade(it)
            post = w.rays(n)
            assert np.array_equal(post["orig"], g[f"post_orig_{k}"]) and np.array_equal(post["dir"], g[f"post_dir_{k}"])
            assert np.array_equal(post["color"], g[f"post_color_{k}"]) and np.array_equal(post["remaining_bounces"], g[f"post_bounces_{k}"])
            w.compact()
            k += 1
        w.gather()
    assert k == int(g["nsteps"])
    assert np.array_equal(w.image(), g["film"])
    w.close()


def test_films_golden(port, oracle_scene, golden_scene, golden_films):
    f = golden_films
    W, H, depth, iters = (int(x) for x in f["bundled_params"])
    w = port.OracleWavefront(oracle_scene, W, H, depth)
    w.init_image()
    counts = [w.run_iteration(it) for it in range(iters)]
    assert np.array_equal(np.array(counts), f["bundled_counts"])
    assert np.array_equal(w.image(), f["bundled_film"])
    w.close()
    # the reference's first-hit cache (Renderer.cpp:594-613) must not change the film
    w2 = port.OracleWavefront(oracle_scene, W, H, depth)
    w2.init_image()
    traced = w2.render(0, iters, first_hit_cache=True)
    assert np.array_equal(w2.image(), f["bundled_film"])
    assert traced == int(np.sum(f["bundled_counts"])) - (iters - 1) * W * H
    w2.close()
    # Cornell (config 1): models edited, grids rebuilt by the oracle
    cs = port.OracleScene(dict(models=f["cornell_models"], meshes=golden_scene["meshes"], vertices=golden_scene["vertices"],
                               triangles=golden_scene["triangles"]))
    assert cs.arrays()["grids"].tobytes() == f["cornell_grids"].tobytes()
    Wc, Hc, dc, ic = (int(x) for x in f["cornell_params"])
    wc = port.OracleWavefront(cs, Wc, Hc, dc)
    wc.init_image()
    cc = [wc.run_iteration(it) for it in range(ic)]
    assert np.array_equal(np.array([c + [0] * (dc - len(c)) for c in cc]), f["cornell_counts"])
    assert np.array_equal(wc.image(), f["cornell_film"])
    wc.close()


def test_films_golden_r1(port, oracle_scene, golden_films):
    """Tier R1 of the wavefront (every triangle, the reference's predicate and loop): the fixture was produced by the compiled reference's
    own kernels with only the closest-hit launch swapped (ref_harness.cpp: ref_trace_step_r1).  This is the film an exact BVH must match."""
    f = golden_films
    W, H, depth, iters = (int(x) for x in f["bundled_params"])
    w = port.OracleWavefront(oracle_scene, W, H, depth, mode=1)
    w.init_image()
    counts = [w.run_iteration(it) for it in range(iters)]
    assert np.array_equal(np.array(counts), f["bundled_counts_r1"])
    assert np.array_equal(w.image(), f["bundled_film_r1"])
    assert not np.array_equal(f["bundled_film_r1"], f["bundled_film"])      # the tiers do differ (SURVEY 8c: 0.3-0.6 % of rays)
    w.close()
    w2 = port.OracleWavefront(oracle_scene, W, H, depth, mode=1)
    w2.init_image(); w2.render(0, iters, first_hit_cache=True)
    assert np.array_equal(w2.image(), f["bundled_film_r1"])
    w2.close()


def test_bmp_writer_vs_compiled_reference(port, golden_scene, golden_live, tmp_path):
    """Renderer::renderImage (Renderer.cpp:15-63) of the compiled reference, run on its own film, against the port's writer on the same film:
    the two files must be byte-identical (header, row order, channel order, (char) truncation).  The film and the file are stored in
    tests/golden/live_scenes.npz (its `source` entry names what wrote them); where oracle/_ref is built, the reference renders and
    writes them again live and must match them too."""
    W, H, depth, iters = live_scenes.BMP
    film, want = golden_live["bmp_film"], golden_live["bmp_bytes"].tobytes()
    if ref.available():
        rfilm, rbytes = live_scenes.reference_bmp(golden_scene)
        assert np.array_equal(rfilm, film) and rbytes == want
    _, pfilm = live_scenes.Port().frame(port.OracleScene(golden_scene), W, H, depth, iters, 0)
    assert np.array_equal(pfilm, film)
    port.write_bmp(film, iters, tmp_path / "port.bmp")
    got = (tmp_path / "port.bmp").read_bytes()
    assert len(want) == 54 + 3 * W * H
    assert got == want


def test_bmp_writer(port, tmp_path):
    img = np.zeros((4, 8, 3), np.float32)
    img[1, 2] = (2.0, 1.0, 0.5)
    img[3, 7] = (4.0, 4.0, 4.0)
    p = tmp_path / "o.bmp"
    port.write_bmp(img, 4, p)
    raw = p.read_bytes()
    assert raw[:2] == b"BM" and len(raw) == 54 + 3 * 8 * 4
    assert int.from_bytes(raw[2:6], "little") == len(raw) and int.from_bytes(raw[18:22], "little") == 8 and int.from_bytes(raw[22:26], "little") == 4
    px = np.frombuffer(raw[54:], np.uint8).reshape(4, 8, 3)
    assert tuple(px[1, 2]) == (127, 63, 31)      # (sum/iters*255) truncated, written in x,y,z order (Renderer.cpp:48-51)
    assert tuple(px[3, 7]) == (255, 255, 255)


def test_committed_render_bmp(port, oracle_scene, golden_render_bmp):
    """The reference's only golden artefact: the author's own GPU render of the coded scene, PathTracerAP/Render.bmp (1000x800, iteration
    count unrecorded).  The oracle at 24 iterations must reproduce its per-channel byte means to 0.1/255 and, after an 8x8 box filter
    that averages the Monte-Carlo noise of both images down, agree to PSNR >= 39 dB (measured 41.1 dB at 24 iterations; SURVEY 8c: 48 dB at 100)."""
    from conftest import box8_of_film
    g = golden_render_bmp
    H, W = (int(x) for x in g["shape"])
    iters = 24
    w = port.OracleWavefront(oracle_scene, W, H, 5)
    w.init_image(); w.render(0, iters, True)
    b8, means = box8_of_film(w.image(), iters)
    w.close()
    rmse = float(np.sqrt(np.mean((b8 - g["box8"]) ** 2)))
    psnr = 20 * np.log10(255.0 / rmse)
    print(f"oracle vs Render.bmp: channel means {means} vs {g['channel_means']}, box-filtered rmse {rmse:.2f}/255, psnr {psnr:.1f} dB")
    assert np.abs(means - g["channel_means"]).max() <= 0.1
    assert psnr >= 39.0


def _check_live(scene_list, golden_live, min_hit):
    """The C restatement - and, where oracle/_ref is built, the compiled reference itself - against the stored outputs."""
    impls = [("port", live_scenes.Port())] + ([("reference", live_scenes.Reference())] if ref.available() else [])
    for name, impl in impls:
        got = live_scenes.outputs(impl, scene_list)
        for k, v in got.items():
            want = golden_live[k]
            assert v.dtype == want.dtype and v.shape == want.shape and v.tobytes() == want.tobytes(), f"{name}: {k} differs"
    for key, *_ in scene_list:
        for mode in (0, 1):
            assert (golden_live[f"{key}_r{mode}_model"] >= 0).mean() > min_hit


def test_port_equals_compiled_reference_on_other_scenes(port, golden_scene, golden_live):
    """The golden fixtures pin the C restatement on the bundled scene.  Here it is compared on scenes they do not hold - random rotated /
    non-uniformly scaled instances, all five material branches - for the grid build, both trace tiers on random rays, and two whole
    iterations of the wavefront at both tiers (BVH film parity rests on tier R1 of the port): bit-equal to the outputs stored in
    tests/golden/live_scenes.npz, and, where oracle/_ref is built, the reference's own outputs must equal them as well."""
    _check_live(live_scenes.scenes(golden_scene, ("instances",)), golden_live, 0.05)


def test_port_equals_compiled_reference_on_a_dense_mesh(port, libptap, golden_scene, golden_live):
    """Same comparison on the kind of mesh the throughput workloads use: a displaced icosphere (5120 triangles; the host-side
    generator of libptap needs no GPU), three instances, so that voxels hold many references and the 3D-DDA early exit matters."""
    _check_live(live_scenes.scenes(golden_scene, ("dense",)), golden_live, 0.3)
