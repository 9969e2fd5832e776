"""Scene::addMeshesToGrid on the GPU (ptap_build_grids_device, csrc/grid_device.cu; SURVEY 8f row 2): cells and reference lists must be
bit-identical to the host builder's - which tests/test_host.py pins to the reference's own output - and the grid walk over them must
reproduce the reference's hits (tier R0)."""
import numpy as np
import pytest

from conftest import have_gpu
from test_host import GRID_SHAPES

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_gpu(), reason="no CUDA device")]


def _host_grids(arrays, shape):
    from pathtracerap_b200 import Scene
    s = Scene.from_arrays(arrays["models"], arrays["meshes"], arrays["vertices"], arrays["triangles"])
    s.build_grids(*shape)
    return s.arrays()


CASES = [("bundled", (25, 25, 25)), ("cornell", (25, 25, 25)), ("mesh100k", (25, 25, 25)), ("mesh100k", (64, 64, 64))]
CASES += [("bundled", shape) for shape in GRID_SHAPES]


def _case_id(workload, shape):
    return f"{workload}-{shape[0]}" if len(set(shape)) == 1 and shape[0] in (25, 64) else f"{workload}-{'x'.join(map(str, shape))}"


@pytest.mark.parametrize("workload,shape", CASES, ids=[_case_id(*c) for c in CASES])
def test_device_grids_equal_host_grids(libptap, port, workload, shape):
    import bench
    from pathtracerap_b200 import ACCEL_BVH, Renderer
    scene, arrays = bench.build_scene(workload)
    want = _host_grids(arrays, shape)
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)         # uploaded WITHOUT grids: nothing host-built can leak in
    r.allocateOnGPU(scene)
    r.build_grids_device(scene, *shape)
    vox, refs = r.read_grids()
    assert len(vox) == len(want["voxels"]) and len(refs) == len(want["refs"])
    assert np.array_equal(vox["start"], want["voxels"]["start"]) and np.array_equal(vox["end"], want["voxels"]["end"])
    assert np.array_equal(refs, want["refs"])                           # ascending triangle order inside every cell, as push_back gives
    assert r.stats()["ms_build"] > 0
    # the grid walk over the device-built grids against the oracle's R0 on its own (restated) grids
    rs = np.random.RandomState(5)
    o = np.stack([rs.uniform(-450, 500, 20000), rs.uniform(-100, 850, 20000), rs.uniform(-450, 900, 20000)], 1)
    d = rs.randn(20000, 3) * rs.uniform(0.1, 30.0, (20000, 1))
    rays = np.concatenate([o, d], 1).astype(np.float32)
    oscene = port.OracleScene(arrays, grid_dim=shape)
    got, ref = r.trace(rays), oscene.trace(rays, 0)
    assert np.array_equal(got["model"], ref["model"]) and np.array_equal(got["tri"], ref["tri"])
    hit = ref["model"] >= 0
    assert hit.mean() > 0.5
    for f in ("t_model", "dist", "u", "v"):
        assert np.array_equal(got[f][hit], ref[f][hit]), f
    # and a frame through it equals the frame through host-built grids bit for bit
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, Scene
    r.set_params(128, 96, 5)
    r.render(0, 2)
    film_dev = r.film()
    s2 = Scene.from_arrays(arrays["models"], arrays["meshes"], arrays["vertices"], arrays["triangles"])
    s2.build_grids(*shape)
    r2 = Renderer(width=128, height=96, depth=5, accel=ACCEL_GRID_COMPAT)
    r2.allocateOnGPU(s2)
    r2.render(0, 2)
    assert np.array_equal(r2.film(), film_dev)
    r.free(); r2.free()
