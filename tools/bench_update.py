"""Moving models without a re-upload (ptap_update_models, DESIGN.md 4.9) against ptap_upload_scene + ptap_build_accel.

    python tools/bench_update.py [--big mesh1m,mesh5m] [--instances 1000,16000,256000,1000000] [--repeats 3] [--min-seconds 1.0] [--out FILE]

(a) The bench.py workloads (the bundled box plus one displaced icosphere): moving the icosphere model, ptap_update_models against
    ptap_upload_scene + ptap_build_accel for PTAP_ACCEL_BVH with the prebuilt host tree in the view, and for PTAP_ACCEL_BVH_DEVICE (a
    view with packed triangles only).
(b) n instances of a 320-triangle icosphere in a cube whose volume grows with n: every model moved, ptap_update_models against
    ptap_upload_scene + ptap_build_accel(PTAP_ACCEL_BVH); then ptap_query_closest on 8 M random rays through the host median-split TLAS of
    a fresh upload and through the device TLAS of an update to the same transforms (the answers are compared byte for byte).

Times are host clocks around calls that end in a device synchronise; rates come from CUDA events on the query stream.  Each figure is
the median call over at least --min-seconds of work after a warm-up call, and the two arms of every comparison alternate --repeats times
in this one process.  One JSON document goes to stdout and to --out."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def timed(fn, min_seconds):
    """Median wall time (ms) of fn() over at least min_seconds of calls, after one warm-up call."""
    fn()
    ts, t_end = [], time.perf_counter() + min_seconds
    while time.perf_counter() < t_end or len(ts) < 3:
        t0 = time.perf_counter(); fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), len(ts)


def rigid(rs, n, spread, scale):
    """n model records' matrices: rotation about y, uniform scale, translation in [-spread, spread]^3 (model_to_world in binary32,
    world_to_model its inverse rounded from float64), both column-major."""
    a = rs.uniform(0, 2 * np.pi, n); s = rs.uniform(*scale, n)
    M = np.zeros((n, 4, 4)); M[:, 3, 3] = 1
    M[:, 0, 0] = np.cos(a) * s; M[:, 0, 2] = np.sin(a) * s; M[:, 1, 1] = s; M[:, 2, 0] = -np.sin(a) * s; M[:, 2, 2] = np.cos(a) * s
    M[:, :3, 3] = rs.uniform(-spread, spread, (n, 3))
    M = M.astype(np.float32)
    Wm = np.linalg.inv(M.astype(np.float64)).astype(np.float32)
    return M.transpose(0, 2, 1).reshape(n, 16), Wm.transpose(0, 2, 1).reshape(n, 16)


def bench_big(workload, args):
    import bench
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, Renderer
    s_host, a = bench.build_scene(workload)
    s_host.build_bvh()
    s_dev, _ = bench.build_scene(workload)
    s_dev.pack()
    i = len(a["models"]) - 1                                    # the icosphere
    rs = np.random.RandomState(1)
    poses = a["models"][i:i + 1].copy().repeat(2)
    for k in range(2):
        M = poses["model_to_world"][k].reshape(4, 4).T.astype(np.float64)
        M[:3, 3] += rs.uniform(-30, 30, 3)
        poses["model_to_world"][k] = M.astype(np.float32).T.reshape(16)
        poses["world_to_model"][k] = np.linalg.inv(M.astype(np.float32).astype(np.float64)).astype(np.float32).T.reshape(16)
    out = {"workload": workload, "triangles": int(len(a["triangles"])), "models": int(len(a["models"]))}
    for name, accel, scene in (("bvh", ACCEL_BVH, s_host), ("bvh_device", ACCEL_BVH_DEVICE, s_dev)):
        r = Renderer(width=64, height=64, depth=5, accel=accel)
        r.allocateOnGPU(scene)
        flip = [0]

        def update():
            flip[0] ^= 1
            r.update_models(poses[flip[0]:flip[0] + 1], i)

        def upload():
            r.upload(scene)
            r.sync()
        ups, upl = [], []
        for _ in range(args.repeats):
            ups.append(timed(update, args.min_seconds)); upl.append(timed(upload, args.min_seconds))
        out[name] = {"update_ms": [u[0] for u in ups], "update_calls": [u[1] for u in ups],
                     "upload_build_ms": [u[0] for u in upl], "upload_build_calls": [u[1] for u in upl]}
        out[name]["speedup"] = float(np.median(out[name]["upload_build_ms"]) / np.median(out[name]["update_ms"]))
        r.free()
    return out


def bench_instances(n, args):
    import torch
    from pathtracerap_b200 import ACCEL_BVH, DIFFUSE, MODEL, Renderer, Scene
    s0 = Scene.empty()
    mi = s0.add_icosphere(2, radius=1.0, displacement=0.05, seed=7)
    s0.add_model(mi, material=DIFFUSE)
    a = s0.arrays()
    spread = 40.0 * n ** (1 / 3)                                 # about the same density at every n
    rs = np.random.RandomState(n)
    models = np.zeros(n, MODEL)
    models["mesh_index"] = mi; models["grid_index"] = -1
    models["mat"]["type"] = DIFFUSE; models["mat"]["color"] = rs.uniform(0.2, 0.9, (n, 3))
    poses = []
    for _ in range(2):
        m2w, w2m = rigid(rs, n, spread, (2.0, 8.0))
        p = models.copy(); p["model_to_world"] = m2w; p["world_to_model"] = w2m
        poses.append(p)
    scene = Scene.from_arrays(poses[0], a["meshes"], a["vertices"], a["triangles"])
    scene.pack()
    r = Renderer(width=64, height=64, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(scene)
    flip = [0]

    def update():
        flip[0] ^= 1
        r.update_models(poses[flip[0]])

    def upload():
        r.upload(scene)
        r.sync()
    ups, upl = [], []
    for _ in range(args.repeats):
        ups.append(timed(update, args.min_seconds)); upl.append(timed(upload, args.min_seconds))
    out = {"instances": n, "triangles_per_instance": int(len(a["triangles"])),
           "update_all_ms": [u[0] for u in ups], "upload_build_ms": [u[0] for u in upl]}
    out["speedup"] = float(np.median(out["upload_build_ms"]) / np.median(out["update_all_ms"]))
    # query rates: the same transforms through the host TLAS (fresh upload of poses[1]) and the device TLAS (update to poses[1])
    r.update_models(poses[1])
    scene1 = Scene.from_arrays(poses[1], a["meshes"], a["vertices"], a["triangles"])
    scene1.pack()
    fresh = Renderer(width=64, height=64, depth=5, accel=ACCEL_BVH)
    fresh.allocateOnGPU(scene1)
    nr = 8 << 20
    g = torch.Generator(device="cuda").manual_seed(n)
    org = (torch.rand((nr, 3), device="cuda", generator=g) * 2 - 1) * spread
    dir_ = torch.nn.functional.normalize(torch.randn((nr, 3), device="cuda", generator=g), dim=1)
    same = all(torch.equal(r.query_closest(org, dir_)[k], fresh.query_closest(org, dir_)[k]) for k in ("model", "tri", "dist", "t_model", "u", "v"))

    def rate(x):
        x.query_closest(org, dir_); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps, ms = 0, 0.0
        while ms < args.min_seconds * 1e3:
            e0.record(); x.query_closest(org, dir_); e1.record(); e1.synchronize()
            ms += e0.elapsed_time(e1); reps += 1
        return reps * nr / (ms * 1e-3) / 1e6
    host, dev = [], []
    for _ in range(args.repeats):
        host.append(rate(fresh)); dev.append(rate(r))
    out.update(query_rays=nr, query_hit_fraction=float((r.query_closest(org, dir_)["model"] >= 0).float().mean()),
               query_closest_mrays_host_tlas=host, query_closest_mrays_device_tlas=dev, query_answers_identical=bool(same))
    r.free(); fresh.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--big", default="mesh1m,mesh5m")
    ap.add_argument("--instances", default="1000,16000,256000,1000000")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "big": [], "instances": []}
    for w in filter(None, args.big.split(",")):
        res["big"].append(bench_big(w, args)); print(json.dumps(res["big"][-1]), file=sys.stderr)
    for n in filter(None, args.instances.split(",")):
        res["instances"].append(bench_instances(int(n), args)); print(json.dumps(res["instances"][-1]), file=sys.stderr)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
