#!/usr/bin/env python
"""Generates tests/golden/*.npz from the reference's own sources compiled for the host (oracle/_ref).

Run in the build container, where /root/reference exists:   python tools/make_golden.py
The reference ships no golden vectors of its own (SURVEY.md 4); these files are outputs of ITS code
(Renderer.cpp / Scene.cpp through oracle/ref_harness.cpp) and travel to the GPU box, where /root/reference
does not exist.  Nothing here comes from this repository's own kernels.

    python tools/make_golden.py live_scenes

writes only tests/golden/live_scenes.npz (oracle/live_scenes.py): from the compiled reference where oracle/_ref is built,
otherwise from the C restatement, which tests/test_oracle_golden.py compares with the compiled reference live, bit for bit,
wherever that is built.  The file's `source` entry names which of the two wrote it.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import live_scenes, port, ref  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def cornell_models(models):
    """Config 1 (SURVEY.md 8d): drop the three monkeys, every non-emissive material becomes DIFFUSE."""
    m = models[3:].copy()
    m["mat"]["type"] = np.where(m["mat"]["type"] == 4, 4, 0)
    return m


def write_live_scenes():
    g = np.load(os.path.join(OUT, "bundled_scene.npz"))
    g = {k: g[k] for k in ("models", "meshes", "vertices", "triangles")}
    if ref.available():
        source = "the compiled reference (oracle/_ref)"
        out = live_scenes.outputs(live_scenes.Reference(), live_scenes.scenes(g))
        film, bmp = live_scenes.reference_bmp(g)
    else:
        source = "the C restatement (oracle/ptap_oracle.c), held bit-equal to the compiled reference wherever oracle/_ref is built"
        out = live_scenes.outputs(live_scenes.Port(), live_scenes.scenes(g))
        W, H, depth, iters = live_scenes.BMP
        _, film = live_scenes.Port().frame(port.OracleScene(g), W, H, depth, iters, 0)
        path = os.path.join(OUT, "_bmp.tmp")
        port.write_bmp(film, iters, path)
        bmp = open(path, "rb").read(); os.remove(path)
    np.savez_compressed(os.path.join(OUT, "live_scenes.npz"), source=np.array(source), bmp_film=film,
                        bmp_bytes=np.frombuffer(bmp, np.uint8), **out)
    print("live_scenes.npz from", source, os.path.getsize(os.path.join(OUT, "live_scenes.npz")), "bytes")


def main():
    if sys.argv[1:] == ["live_scenes"]:
        write_live_scenes()
        return
    scene = ref.RefScene.builtin()
    A = scene.arrays()
    np.savez_compressed(os.path.join(OUT, "bundled_scene.npz"), models=A["models"], meshes=A["meshes"], vertices=A["vertices"],
                        triangles=A["triangles"], grids=A["grids"],
                        voxels_sha=sha(A["voxels"]), refs_sha=sha(A["refs"]), nvoxels=len(A["voxels"]), nrefs=len(A["refs"]))

    # ---- known-answer vectors for utility.h:43-170
    rs = np.random.RandomState(7)
    hash_in = np.concatenate([[0, 1, 2, 0x80000000, 0xFFFFFFFF], rs.randint(0, 2**32, 59, dtype=np.uint64)]).astype(np.uint32)
    hash_out = np.array([ref.util_hash(int(x)) for x in hash_in], np.uint32)
    rng_args = np.array([[0, 0, 5], [1, 17, 4], [499, 799999, 1], [3, 262143, 8], [0, 123456, 3]], np.int32)
    rng_out = np.stack([ref.rng_u01(int(a), int(b), int(c), 8) for a, b, c in rng_args])
    sc_n = rs.randn(64, 3).astype(np.float32); sc_n /= np.linalg.norm(sc_n, axis=1, keepdims=True).astype(np.float32)
    sc_d = rs.randn(64, 3).astype(np.float32); sc_d /= np.linalg.norm(sc_d, axis=1, keepdims=True).astype(np.float32)
    sc_args = np.stack([rs.randint(0, 4, 64), rs.randint(0, 500, 64), rs.randint(0, 800000, 64), rs.randint(1, 6, 64)], 1).astype(np.int32)
    sc_out = np.stack([ref.scatter(int(k), sc_n[i], sc_d[i], int(it), int(ix), int(dp)) for i, (k, it, ix, dp) in enumerate(sc_args)])
    np.savez_compressed(os.path.join(OUT, "shade_kat.npz"), hash_in=hash_in, hash_out=hash_out, rng_args=rng_args, rng_out=rng_out,
                        sc_n=sc_n, sc_d=sc_d, sc_args=sc_args, sc_out=sc_out)

    # ---- closest hit on a seeded ray set: rays are the reference's own wavefront (primary + bounces 1..4 of iteration 0)
    W, H, depth = 1000, 800, 5
    r = ref.RefRenderer(scene, W, H, depth)
    r.init_image()
    rs = np.random.RandomState(11)
    ray_sets, counts, hits = [], [], []

    def grab(b, rr):
        n = rr.nrays
        counts.append(n)
        hits.append(int((rr.hits(n)["dist"] < ref.FLOAT_MAX).sum()))
        sel = np.sort(rs.choice(n, size=min(n, 6000), replace=False))
        rays = rr.rays(n)[sel]
        ray_sets.append(np.concatenate([rays["orig"], rays["dir"]], 1))

    r.run_iteration(0, probe=False, on_bounce=grab)
    rays = np.concatenate(ray_sets).astype(np.float32)
    bounce_of = np.concatenate([np.full(len(x), i, np.int32) for i, x in enumerate(ray_sets)])
    r0 = r.trace_rays(rays, 0)
    r1 = r.trace_rays(rays, 1)
    np.savez_compressed(os.path.join(OUT, "trace_bundled.npz"), rays=rays, bounce=bounce_of, r0=r0, r1=r1,
                        active_per_bounce=np.array(counts), hits_per_bounce=np.array(hits))
    print("1000x800 iteration 0: active", counts, "hits", hits)
    print("R0 vs R1 on the fixture rays: differ", int(((r0["tri"] != r1["tri"]) | (r0["model"] != r1["model"])).sum()), "of", len(rays))
    r.close()

    # ---- wavefront states around shadeRayKernel at a small resolution (slot == index matters for the RNG)
    W, H, depth = 64, 48, 5
    r = ref.RefRenderer(scene, W, H, depth)
    r.init_image()
    pre, post, probes, ns, its = [], [], [], [], []
    for it in range(2):
        r.generate()
        while r.nrays > 0:
            n = r.nrays
            r.trace(True)
            pre.append((r.rays(n), r.hits(n))); probes.append(r.probe(n)); ns.append(n); its.append(it)
            r.shade(it)
            post.append(r.rays(n))
            r.compact()
        r.gather()
    film2 = r.image()
    keep = {}
    for k, ((ra, hi), pr, po) in enumerate(zip(pre, probes, post)):
        keep[f"pre_orig_{k}"] = ra["orig"]; keep[f"pre_dir_{k}"] = ra["dir"]; keep[f"pre_color_{k}"] = ra["color"]
        keep[f"pre_ipixel_{k}"] = ra["ipixel"]; keep[f"pre_bounces_{k}"] = ra["remaining_bounces"]
        keep[f"hit_dist_{k}"] = hi["dist"]; keep[f"hit_model_{k}"] = pr["model"]; keep[f"hit_tri_{k}"] = pr["tri"]
        keep[f"hit_normal_{k}"] = hi["normal"]; keep[f"hit_type_{k}"] = hi["mat"]["type"]
        keep[f"post_orig_{k}"] = po["orig"]; keep[f"post_dir_{k}"] = po["dir"]; keep[f"post_color_{k}"] = po["color"]
        keep[f"post_bounces_{k}"] = po["remaining_bounces"]
    np.savez_compressed(os.path.join(OUT, "wavefront_64x48.npz"), nsteps=len(pre), n=np.array(ns), iter=np.array(its), film=film2, **keep)
    r.close()

    # ---- films: bundled scene 128x96 (4 iterations, depth 5) and Cornell 96x96 (4 iterations, depth 8)
    W, H, depth, iters = 128, 96, 5, 4
    r = ref.RefRenderer(scene, W, H, depth)
    r.init_image()
    per_iter = [r.run_iteration(it) for it in range(iters)]
    film = r.image()
    # the reference's own untouched loop (with its first-hit cache) must give the same film
    r2 = ref.RefRenderer(scene, W, H, depth)
    r2.render_loop(iters)
    assert np.array_equal(r2.image(), film), "step-wise harness differs from Renderer::renderLoop"
    # the same frame at tier R1 (brute force with the reference's own predicate and loop): what an exact BVH must reproduce
    r3 = ref.RefRenderer(scene, W, H, depth)
    r3.init_image()
    per_iter_r1 = [r3.run_iteration(it, mode=1) for it in range(iters)]
    film_r1 = r3.image()
    r3.close()
    r.close(); r2.close()

    cm = cornell_models(A["models"])
    cscene = ref.RefScene.from_arrays(cm, A["meshes"], A["vertices"], A["triangles"])
    CA = cscene.arrays()
    Wc, Hc, dc = 96, 96, 8
    rc = ref.RefRenderer(cscene, Wc, Hc, dc)
    rc.init_image()
    c_per_iter = [rc.run_iteration(it) for it in range(iters)]
    cfilm = rc.image()
    rc.close()
    np.savez_compressed(os.path.join(OUT, "films.npz"), bundled_film_r1=film_r1, bundled_counts_r1=np.array(per_iter_r1), bundled_film=film, bundled_counts=np.array(per_iter), bundled_params=np.array([W, H, depth, iters]),
                        cornell_film=cfilm, cornell_counts=np.array([c + [0] * (dc - len(c)) for c in c_per_iter]),
                        cornell_params=np.array([Wc, Hc, dc, iters]), cornell_models=CA["models"], cornell_grids=CA["grids"])
    print("bundled 128x96 per-iteration active counts:", per_iter)
    print("bundled 128x96 per-iteration active counts, tier R1:", per_iter_r1)
    print("cornell 96x96 per-iteration active counts:", c_per_iter)

    # Cornell 512x512 iteration-0 checkpoint (SURVEY.md A.3b)
    rc = ref.RefRenderer(cscene, 512, 512, 8)
    rc.init_image()
    print("cornell 512x512 iteration 0 active:", rc.run_iteration(0))
    rc.close()
    write_live_scenes()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
