import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def _build_product():
    lib = os.path.join(ROOT, "pathtracerap_b200", "libptap.so")
    if not os.path.exists(lib):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "pathtracerap_b200", "csrc")])
    return lib


@pytest.fixture(scope="session")
def libptap():
    _build_product()
    from pathtracerap_b200 import _native
    return _native.lib()


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement of the reference (oracle/ptap_oracle.c)."""
    from oracle import port as p
    p.lib()
    return p


@pytest.fixture(scope="session")
def golden_scene():
    z = np.load(os.path.join(GOLDEN, "bundled_scene.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden_trace():
    z = np.load(os.path.join(GOLDEN, "trace_bundled.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden_films():
    z = np.load(os.path.join(GOLDEN, "films.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden_wavefront():
    z = np.load(os.path.join(GOLDEN, "wavefront_64x48.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden_kat():
    z = np.load(os.path.join(GOLDEN, "shade_kat.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden_render_bmp():
    """8x8 box-filtered bytes and channel means of the reference's committed PathTracerAP/Render.bmp (tools/make_render_bmp_fixture.py)."""
    z = np.load(os.path.join(GOLDEN, "render_bmp_8x8.npz"))
    return {k: z[k] for k in z.files}


def box8_of_film(film_sum, iters):
    """The bytes Renderer::renderImage would store (Renderer.cpp:45-52: (char)(sum * (1/ITER) * 255)), 8x8 box-filtered."""
    v = film_sum.astype(np.float32) * np.float32(1.0 / iters) * np.float32(255)
    by = np.minimum(v, 255).astype(np.uint8)
    H, W, _ = by.shape
    return by.astype(np.float64).reshape(H // 8, 8, W // 8, 8, 3).mean(axis=(1, 3)), by.reshape(-1, 3).astype(np.float64).mean(0)


@pytest.fixture(scope="session")
def oracle_scene(port, golden_scene):
    """Bundled scene on the C oracle; its grids come from the oracle's own restatement of addMeshesToGrid."""
    return port.OracleScene(golden_scene)


def have_gpu():
    try:
        import ctypes
        cuda = ctypes.CDLL("libcuda.so.1")
        if cuda.cuInit(0) != 0:
            return False
        n = ctypes.c_int(0)
        return cuda.cuDeviceGetCount(ctypes.byref(n)) == 0 and n.value > 0
    except OSError:
        return False


@pytest.fixture(scope="session")
def gpu_scene(libptap, golden_scene):
    """Bundled scene through the product's own host Scene (grids built by libptap's builder)."""
    from pathtracerap_b200 import Scene
    s = Scene.from_arrays(golden_scene["models"], golden_scene["meshes"], golden_scene["vertices"], golden_scene["triangles"])
    s.build_grids(25, 25, 25)
    return s
