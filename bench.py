#!/usr/bin/env python
"""bench.py - headline benchmark of the render hot path (BASELINE.json: Mrays/s, all bounces; ms/frame at 2800x2240, 64 spp).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload mesh100k|mesh1m|mesh5m|bundled|cornell|mesh1m4k]
                    [--accel bvh|lbvh|grid|emu] [--scaling weak|strong] [--impl ptap|reference] [--dump-outputs DIR]

A "step" is one whole frame of the workload: Renderer::renderLoop for `spp` iterations (ray generation, closest hit,
shading + compaction, film accumulation for every bounce).  Rays = rays actually traced, summed over closest-hit launches
(a restored first-hit cache does not count, BASELINE.md).  N > 1: launched under torchrun, one rank per GPU, the scene
replicated, every rank renders its own sample range of the same frame, and the per-rank films are combined with ONE NCCL
reduce issued through the library's C ABI (ptap_reduce) inside the timed region (SURVEY.md 8e).
  --scaling weak (default): every rank renders `spp` iterations (the frame has N * spp samples).
  --scaling strong: the frame's `spp` iterations are split over the ranks (BASELINE configs[4]: --workload mesh1m4k).

Rank 0 prints ONE JSON line (contract in the task statement).  `--impl reference` times the reference's own CPU code
(oracle/_ref, or the C port when that library is absent) on a bounded sample of the same workload; it builds its scene
arrays with the oracle's own generator and never loads the product library.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it

GOLDEN_SCENE = os.path.join(ROOT, "tests", "golden", "bundled_scene.npz")
DIFFUSE, EMISSIVE = 0, 4            # Primitive.h:70-79

# name -> (W, H, spp, depth, description)
WORKLOADS = {
    "mesh100k": (1920, 1080, 64, 5, "configs[1]: displaced icosphere 81,920 tris (DIFFUSE) in the bundled box with its 4 lights, 1920x1080, 64 spp, depth 5, BVH"),
    "mesh1m": (1920, 1080, 64, 5, "configs[3]: displaced icosphere 1,310,720 tris (DIFFUSE) in the bundled box, 1920x1080, 64 spp, depth 5, BVH"),
    "mesh5m": (1920, 1080, 64, 5, "configs[3] upper end: displaced icosphere 5,242,880 tris (DIFFUSE) in the bundled box, 1920x1080, 64 spp, depth 5"),
    "bundled": (2800, 2240, 64, 5, "configs[2]: the reference's coded scene (METAL/COAT/REFLECTIVE/DIFFUSE/EMISSIVE, 11 models), 2800x2240, 64 spp, depth 5, BVH"),
    "mesh1m4k": (3840, 2160, 1024, 5, "configs[4]: the mesh1m scene at 3840x2160, 1024 spp, sample-partitioned, one NCCL reduce of the film (weak scaling: 128 spp per GPU)"),
    "cornell": (512, 512, 16, 8, "configs[0]: Cornell box from Input data, 512x512, 16 spp, depth 8, diffuse only"),
}
ICO = {"mesh100k": (6, 1), "mesh1m": (8, 2), "mesh1m4k": (8, 2), "mesh5m": (9, 2)}       # workload -> (subdivision level, seed)
ICO_MODEL = dict(translate=(25.0, 230.0, -50.0), rotate_y_degrees=30.0, scale=(0.25, 0.25, 0.25), color=(0.75, 0.6, 0.4))
KEEP = [3, 7, 8, 9, 10]             # box + four lights of Scene.cpp:114-124, 175-221


# ------------------------------------------------------------------------------------------------ scenes (host arrays)

def bundled_arrays():
    z = np.load(GOLDEN_SCENE)
    return {k: z[k] for k in ("models", "meshes", "vertices", "triangles")}


def build_scene(workload: str):
    """Product arm: (pathtracerap_b200.Scene, dict of the four reference-layout arrays) for a workload."""
    from pathtracerap_b200 import Scene
    base = bundled_arrays()
    if workload == "bundled":
        s = Scene.from_arrays(base["models"], base["meshes"], base["vertices"], base["triangles"])
    elif workload == "cornell":
        m = base["models"][3:].copy()
        m["mat"]["type"] = np.where(m["mat"]["type"] == EMISSIVE, EMISSIVE, DIFFUSE)
        s = Scene.from_arrays(m, base["meshes"], base["vertices"], base["triangles"])
    else:
        level, seed = ICO[workload]
        s = Scene.from_arrays(base["models"][KEEP], base["meshes"], base["vertices"], base["triangles"])
        mi = s.add_icosphere(level, radius=1000.0, displacement=0.05, seed=seed)
        s.add_model(mi, material=DIFFUSE, **ICO_MODEL)
    a = s.arrays()
    return s, {k: a[k] for k in ("models", "meshes", "vertices", "triangles")}


def reference_arrays(workload: str):
    """CPU arms: the same four arrays built WITHOUT the product library (oracle/synth.c restates the synthetic-mesh generator and the
    glm model-matrix composition; tests/test_host.py asserts byte equality with build_scene)."""
    from oracle import port
    base = bundled_arrays()
    if workload == "bundled":
        return base
    if workload == "cornell":
        m = base["models"][3:].copy()
        m["mat"]["type"] = np.where(m["mat"]["type"] == EMISSIVE, EMISSIVE, DIFFUSE)
        return dict(base, models=m)
    level, seed = ICO[workload]
    v, t, lo, hi = port.icosphere(level, 1000.0, 0.05, seed)
    m2w, w2m = port.compose_trs(ICO_MODEL["translate"], ICO_MODEL["rotate_y_degrees"], ICO_MODEL["scale"])
    return port.scene_with_mesh(base, KEEP, v, t, lo, hi, dict(m2w=m2w, w2m=w2m, type=DIFFUSE, color=ICO_MODEL["color"]))


# ------------------------------------------------------------------------------------------------ clocks

class ClockSampler:
    """Polls nvidia-smi during the timed region (B200_PROFILING.md clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1]); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "power_w_max": max(power) if power else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU arms (oracle/)

def cpu_reference_arm(arrays, depth, sample_w, sample_h, iters, threads=None):
    """The reference's own CPU implementation on a bounded sample: `iters` iterations at sample_w x sample_h of the same
    scene, full bounce loop, 25^3 grid as the reference builds it.  Returns (Mrays/s, rays, seconds, kind, cores, ms_per_iter)."""
    from oracle import ref
    # every host core this process may use: torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently run the
    # reference on one thread and flatter the GPU arm
    threads = threads or len(os.sched_getaffinity(0))
    if ref.available():
        kind = "reference"
        if threads:
            ref.lib().ref_set_threads(threads)
        cores = ref.lib().ref_max_threads()
        scene = ref.RefScene.from_arrays(arrays["models"], arrays["meshes"], arrays["vertices"], arrays["triangles"])
        r = ref.RefRenderer(scene, sample_w, sample_h, depth)
        r.init_image()
        t0 = time.perf_counter()
        rays = sum(sum(r.run_iteration(it)) for it in range(iters))
        dt = time.perf_counter() - t0
        r.close(); scene.close()
    else:
        from oracle import port
        kind = "port"
        if threads:
            port.lib().oracle_set_threads(threads)
        cores = port.lib().oracle_max_threads()
        scene = port.OracleScene(arrays)
        w = port.OracleWavefront(scene, sample_w, sample_h, depth)
        w.init_image()
        t0 = time.perf_counter()
        rays = w.render(0, iters, first_hit_cache=False)
        dt = time.perf_counter() - t0
        w.close()
    return rays / dt / 1e6, rays, dt, kind, cores, dt / iters * 1e3


def sample_size(W, H, target_paths):
    """Largest W/k x H/k (k integer) with at most target_paths paths and a multiple of 32 (Renderer.cpp:573)."""
    k = 1
    while (W // k) * (H // k) > target_paths or ((W // k) * (H // k)) % 32:
        k += 1
    return W // k, H // k


def reference_gpu_arm(device_index: int):
    """The reference's OWN CUDA kernels (Renderer.cpp:363-648, compiled for sm_100a by oracle/build_ref_gpu.sh) on this GPU: its bundled
    scene at its native 1000x800 (Config.h:12-13), 20 iterations, with its cudaDeviceSynchronize after every launch and with those
    synchronisations removed.  The GPU-side "before" number: what the redesign is measured against, where the CPU baseline only
    measures CPU vs GPU."""
    exe = os.path.join(ROOT, "oracle", "_ref", "pt_ref_gpu")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/pt_ref_gpu not built (oracle/build_ref_gpu.sh needs /root/reference)"}
    a = bundled_arrays()
    out = {"scene": "the reference's coded scene (11 models, 1039 triangles, 25^3 grids built by its own Scene::addMeshesToGrid)", "resolution": [1000, 800],
           "kernels": "Renderer.cpp:363-648 as written (patches: duplicate-inline fix, UB return, runtime Config knobs, ray counter)"}
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "scene.bin")
        with open(path, "wb") as f:
            f.write(np.array([len(a["models"]), len(a["meshes"]), len(a["vertices"]), len(a["triangles"])], np.int32).tobytes())
            for k in ("models", "meshes", "vertices", "triangles"):
                f.write(np.ascontiguousarray(a[k]).tobytes())
        vis = [x for x in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if x]
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=vis[device_index] if device_index < len(vis) else str(device_index))
        for name, sync in (("sync_per_launch", 1), ("no_sync", 0)):
            try:
                p = subprocess.run([exe, path, "1000", "800", "20", "2", str(sync), "5"], capture_output=True, text=True, timeout=180, env=env)
                line = [l for l in p.stdout.splitlines() if l.startswith("{")]
                if p.returncode != 0 or not line:
                    out[name] = {"error": (p.stderr or p.stdout)[-300:]}
                    continue
                d = json.loads(line[-1])
                out[name] = {"Mrays_s": d["Mrays_s"], "ms_per_iter": d["ms_per_iter"], "rays": d["rays"], "iters": d["iters"], "film_mean": d["film_mean"]}
            except (subprocess.TimeoutExpired, OSError, ValueError) as e:
                out[name] = {"error": str(e)[:300]}
    return out


# ------------------------------------------------------------------------------------------------ outputs

DUMP_PIXELS = 1 << 22               # 48 MB of float32 RGB: films above this are sampled, so that a dump stays under 64 MB


def dump_outputs(out_dir: str, film: np.ndarray):
    """--dump-outputs: the film of the last timed step (the un-normalised H x W x 3 float32 sum Renderer.film() returns) as
    out_dir/film.npy, so that two builds can be compared output for output.  A film of more than DUMP_PIXELS pixels is written as
    the pixels of one fixed sample (seed 0, ascending pixel index, DUMP_PIXELS x 3): the same pixels for every build at one resolution."""
    os.makedirs(out_dir, exist_ok=True)
    H, W, _ = film.shape
    if H * W > DUMP_PIXELS:
        film = film.reshape(-1, 3)[np.sort(np.random.default_rng(0).choice(H * W, DUMP_PIXELS, replace=False))]
    np.save(os.path.join(out_dir, "film.npy"), film)


# ------------------------------------------------------------------------------------------------ main

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps before the timed ones: at least 3 (1 for --impl reference); the JSON reports the count run")
    ap.add_argument("--impl", default="ptap", choices=["ptap", "reference"])
    ap.add_argument("--workload", default="mesh1m", choices=sorted(WORKLOADS))
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel of the workload")
    ap.add_argument("--accel", default="bvh", choices=["bvh", "lbvh", "grid", "emu"], help="bvh: host-built SAH tree (default); lbvh: tree built on the GPU at upload; grid: the reference's uniform grid, walked; emu: the walk's results (bit-identical) through the BVH")
    ap.add_argument("--grid-dim", type=int, default=25, help="voxels per axis of the uniform grid (--accel grid); the reference fixes 25 (Config.h:8-10)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="N > 1: weak = spp iterations per GPU; strong = the frame's spp split over the GPUs")
    ap.add_argument("--no-cache", action="store_true", help="disable the first-hit cache (Renderer.cpp:594-613)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the second BASELINE metric (bundled 2800x2240), the lbvh end-to-end line and the reference's GPU kernels")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the film of the last timed step to DIR/film.npy (float32; a fixed pixel sample above 4 Mpixels)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ptap":
        ap.error("--dump-outputs writes the film of --impl ptap")
    warmup = max(args.warmup, 3 if args.impl == "ptap" else 1)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    W, H, spp, depth, desc = WORKLOADS[args.workload]
    if args.spp:
        spp = args.spp
    elif args.workload == "mesh1m4k" and args.scaling == "weak":
        spp = 128                          # configs[4] on 8 GPUs: 1024 spp = 128 per GPU
    metric, unit = "Mrays/s (all bounces)", "Mrays/s"

    # -------- reference arm: the reference's CPU implementation on a bounded sample; rank 0 only; never loads the product library
    if args.impl == "reference":
        if rank != 0:
            return
        arrays = reference_arrays(args.workload)
        sw, sh = sample_size(W, H, 140_000)
        ITERS = 8
        for _ in range(warmup):
            cpu_reference_arm(arrays, depth, sw, sh, 1)
        vals, rays_total, t_total = [], 0, 0.0
        for _ in range(args.steps):
            v, rays, dt, kind, cores, _ms = cpu_reference_arm(arrays, depth, sw, sh, ITERS)
            vals.append(v); rays_total += rays; t_total += dt
        value = rays_total / t_total / 1e6
        sample = f"{sw}x{sh} x {ITERS} iterations per step of the {args.workload} scene, full bounce loop, reference 25^3 grid, no first-hit cache"
        print(json.dumps({"impl": "reference", "metric": metric, "value": round(value, 4), "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": warmup, "ms_per_step": round(t_total / args.steps * 1e3, 3), "higher_is_better": True, "scaling": args.scaling,
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": args.workload, "description": desc, "resolution": [W, H], "spp": spp, "depth": depth},
                          "cpu_baseline": {"value": round(value, 4), "unit": unit, "cores": cores, "kind": kind, "sample": sample},
                          "e2e": {"value": round(value, 4), "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # -------- our arm
    # stdout carries exactly ONE line, the JSON: native libraries that print to file descriptor 1 (NCCL announces its version there when
    # a communicator is created) are sent to stderr for the whole run, and the line is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_BVH_DEVICE, ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, Renderer
    from pathtracerap_b200 import _native as N
    from pathtracerap_b200 import multi_gpu

    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = local if world > 1 else 0
    torch.cuda.set_device(dev)
    torch.cuda.init()

    scene, arrays = build_scene(args.workload)
    accel = {"bvh": ACCEL_BVH, "lbvh": ACCEL_BVH_DEVICE, "grid": ACCEL_GRID_COMPAT, "emu": ACCEL_GRID_EMULATED}[args.accel]
    t0 = time.perf_counter()
    if accel == ACCEL_BVH:
        scene.build_bvh()                 # host-side, part of scene construction like the reference's addMeshesToGrid
    elif accel == ACCEL_GRID_COMPAT:
        scene.build_grids(args.grid_dim, args.grid_dim, args.grid_dim)
    elif accel == ACCEL_GRID_EMULATED:
        scene.build_grids(args.grid_dim, args.grid_dim, args.grid_dim); scene.build_bvh()
    else:
        scene.pack()                      # triangle records in page-locked memory; the tree itself is built on the GPU at every upload
    build_s = time.perf_counter() - t0     # lbvh: built on the GPU inside Renderer.allocateOnGPU / upload
    ntris = len(arrays["triangles"])
    cache = not args.no_cache

    r = Renderer(device=dev, width=W, height=H, depth=depth, accel=accel, first_hit_cache=cache, profile=True)
    r.allocateOnGPU(scene)

    # sample partition: weak = every rank renders `spp` iterations of a (world * spp)-sample frame; strong = the frame's spp are split
    total_spp = world * spp if args.scaling == "weak" else spp
    it0, it1 = multi_gpu.iteration_range(rank, world, total_spp)
    reduce_how = None
    if world > 1:
        reduce_how = multi_gpu.nccl_join(r, rank, world)        # the library's own communicator (ptap_nccl_init); None -> torch.distributed
        film_t = None

    def barrier():
        if world > 1:
            dist.barrier()
        r.sync(); torch.cuda.synchronize()

    lib_stream = torch.cuda.ExternalStream(r.stream_ptr(), device=torch.device("cuda", dev))

    def step():
        r.frame_begin()
        if it1 > it0:
            r.render(it0, it1)
        if world > 1:
            if reduce_how is None:
                with torch.cuda.stream(lib_stream):
                    multi_gpu.reduce_film(film_t, 0)
            else:
                r.reduce(0)               # ptap_reduce: ncclReduce on the library's stream, ordered after the render, covered by its timer

    # counting pass (not timed): traversal work per ray of this exact workload, for the algorithmic-bytes figure
    r.set_params(W, H, depth, first_hit_cache=cache, count=True)
    r.render(it0, it0 + 1); r.sync()
    cst = r.stats()
    avg_nodes, avg_tris, avg_cells, avg_refs = cst["avg_nodes"], cst["avg_tris"], cst["avg_cells"], cst["avg_refs"]
    r.set_params(W, H, depth, first_hit_cache=cache, profile=False)
    if world > 1 and reduce_how is None:
        film_t = multi_gpu.film_tensor(r)      # zero-copy torch view of the library's film buffer

    for _ in range(warmup):
        step()
    barrier()
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
    rays = launches = 0
    lanes = r.stats()["lanes"]
    t_wall0 = time.perf_counter()
    ms_dev = 0.0
    for _ in range(args.steps):
        r.timer_start()
        step()
        ms_dev += r.timer_stop()                 # device time on the launching stream (render + reduce; the lanes' streams join it)
        st = r.stats()
        rays += st["rays_traced"]; launches += st["kernel_launches"]
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r.film())      # N > 1: rank 0's film holds the reduced frame

    def over_ranks(t_rank, n_rank):
        if world == 1:
            return t_rank, float(n_rank)
        tt = torch.tensor([t_rank], dtype=torch.float64, device=f"cuda:{dev}"); dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        rr = torch.tensor([float(n_rank)], dtype=torch.float64, device=f"cuda:{dev}"); dist.all_reduce(rr, op=dist.ReduceOp.SUM)
        return float(tt.item()), float(rr.item())

    t_max, rays_all = over_ranks(ms_dev / 1e3, rays)          # CUDA events on the library stream; max over ranks
    value = rays_all / t_max / 1e6

    # -------- end to end through the public API with HOST buffers: upload scene (H2D) + render + film read-back (D2H), every step
    film_host = torch.empty((H, W, 3), dtype=torch.float32, pin_memory=True).numpy()      # page-locked read-back target
    barrier()
    t0 = time.perf_counter()
    e2e_rays = 0
    for _ in range(args.steps):
        r.upload(scene)
        step()
        N.lib().ptap_read_film(r.h, N.ptr(film_host))
        e2e_rays += r.stats()["rays_traced"]
    barrier()
    t_e2e, e2e_rays = over_ranks(time.perf_counter() - t0, e2e_rays)
    h2d = r.stats()["scene_bytes"]
    d2h = film_host.nbytes
    e2e_value = e2e_rays / t_e2e / 1e6

    # -------- stamped pass (not part of `value`): the same K steps in the SAME multi-lane schedule, every closest-hit launch recording
    # its first start / last end on the device's nanosecond clock (two atomics per CTA).  Lanes overlap, so the time a rate may be divided
    # by is the UNION of the launches' residency intervals (<= the step's own duration); the summed residency is reported beside it.
    r.set_params(W, H, depth, first_hit_cache=cache, stamp=True)
    if world > 1 and reduce_how is None:
        film_t = multi_gpu.film_tensor(r)
    step(); r.sync()
    trace_launches = rays_i = 0
    ms_inflight = ms_sum = ms_stamped = 0.0
    for _ in range(args.steps):
        r.timer_start()
        step()
        ms_stamped += r.timer_stop()
        st = r.stats()
        rays_i += st["rays_traced"]; trace_launches += st["trace_launches"]
        ms_inflight += st["ms_trace_inflight"]; ms_sum += st["ms_trace_sum"]
    barrier()

    if rank != 0:
        if world > 1:
            r.nccl_finalize()
            dist.destroy_process_group()
        return

    # -------- roofline of the dominant kernel (closest hit)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # SURVEY 8(d): ray 32 B read + hit 16 B written, 128 B per 4-wide node visited, 48 B per triangle tested (8 B per cell, 4 B per reference
    # for the grid).  For --accel lbvh the per-ray counts are those of the HOST (SAH) tree of the same scene, so that a worse tree, which
    # visits more nodes per ray, cannot raise the fraction: with a fixed numerator per ray the fraction moves only with rays/s.
    ref_nodes, ref_tris, denom = avg_nodes, avg_tris, "this run's tree"
    if accel == ACCEL_BVH_DEVICE:
        scene.build_bvh()
        r2 = Renderer(device=dev, width=W, height=H, depth=depth, accel=ACCEL_BVH, first_hit_cache=cache)
        r2.allocateOnGPU(scene)
        r2.set_params(W, H, depth, first_hit_cache=cache, count=True)
        r2.render(it0, it0 + 1); r2.sync()
        c2 = r2.stats(); ref_nodes, ref_tris, denom = c2["avg_nodes"], c2["avg_tris"], "host SAH tree of the same scene (fixed denominator)"
        r2.free()
    if accel == ACCEL_GRID_EMULATED:
        bytes_per_ray = 48.0 + 128.0 * ref_nodes + 64.0 * ref_tris
        formula = "48 + 128 * nodes_per_ray + 64 * tris_per_ray (leaf-order triangle record; the replayed voxels read nothing)"
    elif accel != ACCEL_GRID_COMPAT:
        bytes_per_ray = 48.0 + 128.0 * ref_nodes + 48.0 * ref_tris
        formula = "48 + 128 * nodes_per_ray + 48 * tris_per_ray"
    else:
        bytes_per_ray = 48.0 + 8.0 * avg_cells + 4.0 * avg_refs + 48.0 * avg_tris
        formula = "48 + 8 * cells_per_ray + 4 * refs_per_ray + 48 * tris_per_ray"
    achieved = bytes_per_ray * rays_i / (ms_inflight / 1e3) / 1e9 if ms_inflight > 0 else None
    # what limits the kernel: measured fractions of the committed `ncu --set full` capture of the same kernel on the same workload
    evidence, traffic = None, None
    ep = os.path.join(ROOT, "profiles", "ncu_evidence.json")
    if os.path.exists(ep):
        evidence = json.load(open(ep)).get(f"{args.workload}:{args.accel}")
        if evidence:
            traffic = evidence.get("dram_bytes_per_launch")
    kernel = "k_trace_emu" if accel == ACCEL_GRID_EMULATED else "k_trace_bvh" if accel != ACCEL_GRID_COMPAT else "k_trace_grid"
    roofline = {"bound": "issue", "bound_note": "instruction issue x SIMT fill; NOT memory-bound: DRAM traffic is a few % of the HBM peak (evidence). `frac` is the "
                "contract's algorithmic-bytes figure against the HBM peak and says how far the kernel is from becoming memory-bound, not what limits it",
                "kernel": kernel, "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                "bytes_per_ray": round(bytes_per_ray, 1), "formula": formula, "denominator_tree": denom,
                "avg_nodes_per_ray": round(avg_nodes, 2), "avg_tris_per_ray": round(avg_tris, 2),
                "avg_cells_per_ray": round(avg_cells, 2), "avg_refs_per_ray": round(avg_refs, 2),
                "trace_launches": trace_launches, "trace_inflight_ms_per_step": round(ms_inflight / args.steps, 3),
                "trace_summed_residency_ms_per_step": round(ms_sum / args.steps, 3), "stamped_ms_per_step": round(ms_stamped / args.steps, 3),
                "avg_launch_ms": round(ms_sum / max(trace_launches, 1), 4),
                "trace_Mrays_per_s": round(rays_i / (ms_inflight / 1e3) / 1e6, 1) if ms_inflight > 0 else None,
                "timing": f"measured inside the timed schedule ({lanes} lanes): %globaltimer stamps by every CTA of every closest-hit launch over {args.steps} steps; "
                          "achieved = algorithmic bytes / union of the launches' residency intervals (<= ms_per_step)",
                "evidence": evidence}

    extras = {}
    if not args.no_extras and world == 1:
        # ---- second half of BASELINE.json's metric: ms/frame at 2800x2240, 64 spp (the reference's coded scene), both acceleration structures
        if args.workload != "bundled":
            bs, _ = build_scene("bundled")
            bs.build_bvh(); bs.build_grids(25, 25, 25)
            rb = Renderer(device=dev, width=2800, height=2240, depth=5, accel=ACCEL_BVH, first_hit_cache=True)
            rb.allocateOnGPU(bs)
            frames = {}
            for name, acc, nfr in (("bvh", ACCEL_BVH, 3), ("grid_compat", ACCEL_GRID_COMPAT, 2), ("grid_emulated", ACCEL_GRID_EMULATED, 3)):
                rb.set_accel(acc)
                rb.set_params(2800, 2240, 5, first_hit_cache=True)
                rb.frame_begin(); rb.render(0, 64); rb.sync()
                ms = rays_b = 0
                for _ in range(nfr):
                    rb.timer_start(); rb.frame_begin(); rb.render(0, 64); ms += rb.timer_stop(); rays_b += rb.stats()["rays_traced"]
                frames[name] = {"ms_per_frame": round(ms / nfr, 2), "Mrays_s": round(rays_b / ms / 1e3, 1), "frames": nfr}
                if acc == ACCEL_GRID_EMULATED:
                    stb = rb.stats()
                    frames[name]["rays_emulated_in_full"] = round(stb["rays_reemulated"] / max(stb["rays_traced"], 1), 5)
                    frames[name]["rays_answered_by_the_walk_itself"] = round(stb["rays_walked"] / max(stb["rays_traced"], 1), 6)
            rb.free()
            extras["ms_per_frame_2800x2240_64spp"] = dict(frames, scene="bundled (configs[2])", note="grid_compat = the reference's own 25^3 grid walk; grid_emulated = the same hits, bit for bit, through the BVH (the drop-in default); bvh = exact closest hit")
        # ---- end to end with the acceleration structure built INSIDE the timed region (tree built on the GPU at upload)
        if accel == ACCEL_BVH and args.workload != "cornell":
            scene_l, _ = build_scene(args.workload)      # the same scene WITHOUT a host tree: triangle records only
            scene_l.pack()
            rl = Renderer(device=dev, width=W, height=H, depth=depth, accel=ACCEL_BVH_DEVICE, first_hit_cache=cache)
            rl.allocateOnGPU(scene_l)
            rl.render(it0, it1); rl.sync()
            t0 = time.perf_counter(); n_l = 0; k = min(args.steps, 3)
            for _ in range(k):
                rl.upload(scene_l); rl.frame_begin(); rl.render(it0, it1)
                N.lib().ptap_read_film(rl.h, N.ptr(film_host)); n_l += rl.stats()["rays_traced"]
            dt = time.perf_counter() - t0
            extras["e2e_build_included"] = {"value": round(n_l / dt / 1e6, 2), "unit": unit, "accel": "lbvh (triangles uploaded, tree built on the GPU by PLOC + a host SAH top inside every step)",
                                            "device_bvh_build_ms": round(rl.stats()["ms_build"], 3), "ms_per_step": round(dt / k * 1e3, 3)}
            rl.free()
    r.free()
    if not args.no_extras and world == 1:
        extras["reference_gpu"] = reference_gpu_arm(dev)

    cpu = None
    if not args.no_cpu_baseline:
        carr = reference_arrays(args.workload)
        sw, sh = sample_size(W, H, 140_000)
        cpu_reference_arm(carr, depth, sw, sh, 1)          # warm the page cache / OpenMP pool
        n_it = 2
        v, rays_c, dt, kind, cores, _ms = cpu_reference_arm(carr, depth, sw, sh, n_it)
        if dt < 5.0:
            n_it = int(min(64, max(2, 12.0 / (dt / n_it))))
            v, rays_c, dt, kind, cores, _ms = cpu_reference_arm(carr, depth, sw, sh, n_it)
        cpu = {"value": round(v, 4), "unit": unit, "cores": cores, "kind": kind,
               "sample": f"{sw}x{sh} x {n_it} iterations of the same scene ({rays_c} rays, {dt:.1f} s), full bounce loop, reference 25^3 grid, no first-hit cache"}

    par = f"sample-partition x{world}"
    if world > 1:
        par += " + 1 NCCL reduce of the film (" + ("ptap_reduce: ncclReduce through the library's C ABI" if reduce_how else "torch.distributed.reduce") + ")"
    out = {"metric": metric, "value": round(value, 2), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": warmup,
           "ms_per_step": round(t_max / args.steps * 1e3, 3), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": args.workload, "description": desc, "resolution": [W, H], "spp_per_gpu": it1 - it0, "spp_total": total_spp, "depth": depth,
                      "triangles": ntris, "models": len(arrays["models"]), "accel": {"grid": f"grid {args.grid_dim}^3 (walked)", "emu": f"grid {args.grid_dim}^3 (emulated through the BVH)"}.get(args.accel, args.accel), "first_hit_cache": cache, "lanes": lanes,
                      "parallelism": par,
                      "l2": "wavefront state (6 float4 queues + hits, >300 MB at 1080p) exceeds L2 every bounce; the scene is small and L2-resident by design",
                      "host_accel_build_s": round(build_s, 3)},
           "rays_per_step": int(rays_all / args.steps), "ms_per_frame_device": round(ms_dev / args.steps, 3), "wall_s_timed_region": round(t_wall, 3),
           "e2e": {"value": round(e2e_value, 2), "unit": unit, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                   "ms_per_step": round(t_e2e / args.steps * 1e3, 3),
                   "what": "per step: Renderer.upload(scene) from host arrays (triangles + the prebuilt acceleration structure; the host-side build itself, "
                           "host_accel_build_s, is done once per scene like the reference's addMeshesToGrid and is NOT in this figure - see extras.e2e_build_included) "
                           "+ renderLoop + film read-back to pinned host memory"},
           "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "extras": extras}
    real_stdout.write(json.dumps(out) + "\n"); real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
