"""Ray-query rates on the GPU: shadow rays of a real frame through ptap_query_occluded / ptap_query_closest (DESIGN.md 4.8).

    python tools/bench_queries.py [--workloads mesh1m,bundled] [--repeats 3] [--min-seconds 1.0] [--out FILE]

Shadow rays: the origins are the round-1 ray origins of a frame of the workload (ptap_render_probe: surface points offset 0.1 along the
normal, as the reference does), the targets points sampled uniformly by area on the emissive instances' triangles; d = target - o and
L = |target - o| * (1 - 1e-4).  Rates in Mrays/s from CUDA events on the query stream, after warm-up, over at least --min-seconds of work:
  (a) ptap_query_occluded through the any-hit traversal (the default),
  (b) the same call on a context created with PTAP_QUERY_ANYHIT=0: closest hit + compare,
  (c) ptap_query_closest from device tensors,
  (d) ptap_trace on the same rays from host arrays, end to end (host clock around the synchronous call).
(a) and (b) alternate --repeats times to show the spread.  One JSON line goes to stdout (and to --out)."""
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

EMISSIVE = 4


def emissive_points(arrays, n, rs):
    """n points uniform by area on the world-space triangles of the emissive models."""
    models, meshes, verts, tris = arrays["models"], arrays["meshes"], arrays["vertices"], arrays["triangles"]
    P = []
    for m in models[models["mat"]["type"] == EMISSIVE]:
        me = meshes[m["mesh_index"]]
        idx = tris["v"][me["t_start"]:me["t_end"]]
        M = m["model_to_world"].reshape(4, 4).T.astype(np.float64)
        p = verts["position"][idx].astype(np.float64) @ M[:3, :3].T + M[:3, 3]
        P.append(p)
    P = np.concatenate(P)                                             # (ntri, 3 corners, 3)
    area = 0.5 * np.linalg.norm(np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0]), axis=1)
    k = rs.choice(len(P), n, p=area / area.sum())
    u, v = rs.uniform(size=n), rs.uniform(size=n)
    flip = u + v > 1
    u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
    return P[k, 0] + u[:, None] * (P[k, 1] - P[k, 0]) + v[:, None] * (P[k, 2] - P[k, 0])


def shadow_rays(r, arrays, W, H, seed=0):
    """(org (n, 3), dir (n, 3), L (n,)) float32 shadow rays from the round-1 origins of iteration 0 of a W x H frame rendered by `r`."""
    r.set_params(W, H, 5, first_hit_cache=False)
    rays, _, _ = r.render_probe(0, 1)
    r.frame_begin()
    o = rays[:, :3].astype(np.float64)
    tgt = emissive_points(arrays, len(o), np.random.RandomState(seed))
    d = tgt - o
    L = np.linalg.norm(d, axis=1) * (1 - 1e-4)
    return o.astype(np.float32), d.astype(np.float32), L.astype(np.float32)


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def timed(fn, n_rays, min_seconds):
    """Mrays/s of fn() (enqueues one query of n_rays on the current stream) over >= min_seconds, CUDA events on that stream."""
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); e1.synchronize()
    reps = max(3, int(np.ceil(min_seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3))))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    ms = e0.elapsed_time(e1)
    return n_rays * reps / (ms * 1e-3) / 1e6, reps, ms


def run_workload(workload, repeats, min_seconds):
    import torch

    import bench
    from pathtracerap_b200 import ACCEL_BVH, Renderer
    W, H = bench.WORKLOADS[workload][:2]
    s, arrays = bench.build_scene(workload)
    s.build_bvh()
    r = Renderer(width=W, height=H, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    os.environ["PTAP_QUERY_ANYHIT"] = "0"                 # read once, at context creation
    try:
        rc = Renderer(width=W, height=H, depth=5, accel=ACCEL_BVH)
    finally:
        del os.environ["PTAP_QUERY_ANYHIT"]
    rc.allocateOnGPU(s)
    o, d, L = shadow_rays(r, arrays, W, H)
    n = len(o)
    org, dir_, tmax = (torch.from_numpy(x).cuda() for x in (o, d, L))
    # the packed (n, 4) layout the ABI reads, built once, so that the timed window holds the queries alone
    o4 = torch.cat([org, torch.zeros_like(org[:, :1])], 1).contiguous()
    d4 = torch.cat([dir_, tmax[:, None]], 1).contiguous()
    occ_a = r.query_occluded(o4, d4[:, :3].contiguous(), tmax)
    occ_b = rc.query_occluded(o4, d4[:, :3].contiguous(), tmax)
    host = np.concatenate([o, d], 1)
    ref = r.trace(host)
    truth = (ref["model"] >= 0) & (ref["dist"] < L)
    assert np.array_equal(occ_a.cpu().numpy(), truth) and np.array_equal(occ_b.cpu().numpy(), truth), "occlusion differs from ptap_trace"
    occ = torch.empty(n, dtype=torch.bool, device="cuda")
    hits = torch.empty((n, 10), dtype=torch.int32, device="cuda")
    from pathtracerap_b200 import _native as N
    lib = N.lib()

    def q_occ(h):
        stream = torch.cuda.current_stream().cuda_stream or 1
        return lambda: lib.ptap_query_occluded(h, o4.data_ptr(), d4.data_ptr(), n, occ.data_ptr(), stream)

    def q_closest():
        stream = torch.cuda.current_stream().cuda_stream or 1
        lib.ptap_query_closest(r.h, o4.data_ptr(), d4.data_ptr(), n, hits.data_ptr(), stream)

    rates_a, rates_b = [], []
    for _ in range(repeats):
        rates_a.append(timed(q_occ(r.h), n, min_seconds)[0])
        rates_b.append(timed(q_occ(rc.h), n, min_seconds)[0])
    rate_c = timed(q_closest, n, min_seconds)[0]
    r.trace(host)                                          # warm-up of the host path
    t0 = time.perf_counter(); k = 0
    while True:
        r.trace(host); k += 1
        if time.perf_counter() - t0 >= min_seconds:
            break
    rate_d = n * k / (time.perf_counter() - t0) / 1e6
    out = {"workload": workload, "rays": n, "occluded_fraction": round(float(truth.mean()), 4),
           "a_anyhit_mrays": [round(x, 1) for x in rates_a], "b_closest_compare_mrays": [round(x, 1) for x in rates_b],
           "a_over_b_median": round(float(np.median(rates_a) / np.median(rates_b)), 3),
           "c_query_closest_mrays": round(rate_c, 1), "d_trace_host_mrays": round(rate_d, 1)}
    r.free(); rc.free()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="mesh1m,bundled")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_queries: no CUDA device (the rates are GPU measurements; there is nothing to fall back to)")
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit_and_max_sm_clock": power,
           "workloads": [run_workload(w, args.repeats, args.min_seconds) for w in args.workloads.split(",")]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
