"""The grid paths (PTAP_ACCEL_GRID_COMPAT: k_trace_grid; PTAP_ACCEL_GRID_EMULATED: trace_emu.cu) and both grid builders on grids whose
axes differ, thin grids, 160^3 and both sides of the emulation's 512-per-axis limit (test_host.GRID_SHAPES).  On a cubic grid a stride
or limit swapped between two axes computes the same thing; on these shapes it changes hits.  Every answer is held to the oracle's R0
(the reference's grid walk) at the same shape, the oracle building its own grids.  Also: reference lists between 2^30 and 2^31 entries,
and grids the device builder must refuse because their cells or references overflow 32-bit positions, or because the product of
their dimensions exceeds 2^27 cells."""
import numpy as np
import pytest

from conftest import have_gpu
from test_gpu_queries import _assert_closest, _dev, _records
from test_gpu_trace import _random_rays, assert_hits_equal
from test_gpu_wavefront_exact import _albedo, _renderer, check_frame
from test_host import CONFIG, GRID_SHAPES, WRAPPING_DIMS, box_filling_mesh

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_gpu(), reason="no CUDA device")]

FOUR = ("models", "meshes", "vertices", "triangles")
RAYS = _random_rays(300_000, 29)


def _sid(shape):
    return "x".join(map(str, shape))


def _emulable(shape):
    return max(shape) <= 512


@pytest.fixture(scope="module")
def oracle_at(port, golden_scene):
    """shape -> (OracleScene of the bundled scene gridded at that shape, its R0 hits on RAYS); built once per shape."""
    cache = {}

    def get(shape):
        if shape not in cache:
            osc = port.OracleScene({k: golden_scene[k] for k in FOUR}, grid_dim=shape)
            cache[shape] = (osc, osc.trace(RAYS, 0))
        return cache[shape]
    return get


def _scene(golden_scene, shape=None):
    from pathtracerap_b200 import Scene
    s = Scene.from_arrays(*(golden_scene[k] for k in FOUR))
    if shape is not None:
        s.build_grids(*shape)
    return s


def _check_occluded_at_the_hit(r, want, what):
    """query_occluded at L = the closest hit's distance (not occluded: the hit is not nearer than L) and one ulp either side; misses at
    L = 500 and its neighbours."""
    hit = want["model"] >= 0
    base = np.where(hit, want["dist"], np.float32(500.0)).astype(np.float32)
    org, dir_ = _dev(RAYS)
    import torch
    for L in (base, np.nextafter(base, np.float32(np.inf)), np.nextafter(base, np.float32(-np.inf))):
        got = r.query_occluded(org, dir_, torch.from_numpy(L).cuda()).cpu().numpy()
        truth = hit & (want["dist"] < L)
        assert np.array_equal(got, truth), f"{what}: occlusion differs on {(got != truth).sum()} rays"


@pytest.mark.parametrize("builder", ["host", "device"])
@pytest.mark.parametrize("shape", GRID_SHAPES, ids=_sid)
def test_walk_and_emulation_match_the_oracle(golden_scene, oracle_at, shape, builder):
    """300 k random rays (axis-parallel and zero direction components included) through the walk and the emulation over host- or
    device-built grids: trace and query_closest equal to the oracle's R0 in every field, query_occluded exact at the hit distance.
    Past 512 voxels on an axis the emulation is refused with a message naming the limit, and the walk keeps answering."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, PtapError, Renderer
    _, want = oracle_at(shape)
    assert (want["model"] >= 0).mean() > 0.5
    if builder == "host":
        r = Renderer(width=64, height=32, depth=5, accel=ACCEL_GRID_COMPAT)
        r.allocateOnGPU(_scene(golden_scene, shape))
    else:
        s = _scene(golden_scene)
        r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)         # uploaded without grids
        r.allocateOnGPU(s)
        r.build_grids_device(s, *shape)
    for accel in (ACCEL_GRID_EMULATED, ACCEL_GRID_COMPAT):
        what = f"{_sid(shape)}, {builder} grids, accel {accel}"
        if accel == ACCEL_GRID_EMULATED and not _emulable(shape):
            with pytest.raises(PtapError, match="512"):
                r.set_accel(accel)
            continue
        r.set_accel(accel)
        got = r.trace(RAYS)
        assert_hits_equal(got, want, f"{what}: trace vs oracle R0")
        _assert_closest(_records(r.query_closest(*_dev(RAYS))), got, f"{what}: query_closest vs trace")
        _check_occluded_at_the_hit(r, want, what)
    r.free()


@pytest.mark.parametrize("shape", [(7, 40, 3), (64, 1, 3)], ids=_sid)
def test_production_frames_on_non_cubic_grids(golden_scene, oracle_at, shape):
    """Both grid modes through the production path: every round of two iterations against the shading model, the first iteration's hits
    against the oracle's R0 at the same shape, ptap_render's film equal to the model's bit for bit - and the two modes' films equal."""
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED
    osc, _ = oracle_at(shape)
    s = _scene(golden_scene, shape)
    W, H, depth = 200, 150, 5
    films = []
    for accel in (ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED):
        r = _renderer(s, W, H, depth, accel)
        check_frame(r, _albedo(golden_scene["models"]), W, H, depth, 2, oracle_scene=osc, tier=0)
        films.append(r.film().copy())
        r.free()
    assert np.array_equal(films[0], films[1]), f"{(films[0] != films[1]).any(axis=-1).sum()} pixels differ between the modes"


def test_config_txt_grid_end_to_end(libptap, port, tmp_path):
    """A Config.txt with GRID [7, 40, 3]: Scene(config), allocateOnGPU and round 0 of a frame in both grid modes, against the oracle's R0
    on grids it builds itself at that shape."""
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, Renderer, Scene
    from test_gpu_production import _assert_production_hits
    (tmp_path / "one.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nv 1 1 0\nf 1 2 4 3\n")
    cfg = tmp_path / "Config.txt"
    cfg.write_text(CONFIG + "\nGRID\n[7, 40, 3]\n")
    s = Scene(str(cfg))
    a = s.arrays()
    assert a["grid_dim"] == (7, 40, 3)
    osc = port.OracleScene({k: a[k] for k in FOUR}, grid_dim=(7, 40, 3))
    for accel in (ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED):
        r = Renderer(width=160, height=120, depth=5, accel=accel)
        r.allocateOnGPU(s)
        rays, _, hits = r.render_probe(0, 0)
        want = osc.trace(rays, 0)
        assert (want["model"] >= 0).mean() > 0.5
        _assert_production_hits(hits, want, f"Config.txt GRID [7, 40, 3], accel {accel}")
        r.free()


def _box_rays(n, seed):
    """Rays from outside the box [0, 100]^3 towards points of the box-filling triangle (and 1 in 10 towards random points of the box)."""
    rs = np.random.RandomState(seed)
    a, b, c = np.float64([0, 0, 0]), np.float64([100, 100, 0]), np.float64([0, 100, 100])
    u, v = rs.uniform(0, 1, n), rs.uniform(0, 1, n)
    flip = u + v > 1
    u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
    tgt = a + u[:, None] * (b - a) + v[:, None] * (c - a)
    off = rs.rand(n) < 0.1
    tgt[off] = rs.uniform(0, 100, (off.sum(), 3))
    d = rs.randn(n, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = tgt - d * rs.uniform(180, 400, (n, 1))
    return np.concatenate([o, d * rs.uniform(0.5, 4.0, (n, 1))], 1).astype(np.float32)


def test_reference_list_between_2p30_and_2p31(libptap, port):
    """Nine coincident triangles that fill their mesh's box, gridded at 512^3: 9 * 2^27 = 1.21e9 references, past 2^30, where a binary
    search with midpoint (a + b) / 2 in int overflows.  The device build must equal the closed form (cell c lists [9c, 9c + 9), the ids
    0 ... 8 in every cell), and the walk and the emulation must equal the oracle's R0 at 512^3.
    Footprint, estimated from the sizes, not measured: about 31 GB of device memory (pairs, sort buffers, reference list) and 15 GB of
    host memory (the grids read back, then the oracle's own grids)."""
    from pathtracerap_b200 import ACCEL_BVH, ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, Renderer, Scene
    s = Scene.empty()
    s.add_model(box_filling_mesh(s, 9))
    ncell = 512 ** 3
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_BVH)
    r.allocateOnGPU(s)
    r.build_grids_device(s, 512, 512, 512)
    vox, refs = r.read_grids()
    assert len(vox) == ncell and len(refs) == 9 * ncell
    assert np.array_equal(vox["start"], np.arange(0, 9 * ncell, 9, dtype=np.int32))
    assert np.array_equal(vox["end"] - vox["start"], np.full(ncell, 9, np.int32))
    assert (refs.reshape(ncell, 9) == np.arange(9, dtype=np.int32)).all()
    del vox, refs
    rays = _box_rays(10_000, 3)
    osc = port.OracleScene({k: s.arrays()[k] for k in FOUR}, grid_dim=(512, 512, 512))
    want = osc.trace(rays, 0)
    assert (want["model"] >= 0).mean() > 0.5
    for accel in (ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED):
        r.set_accel(accel)
        assert_hits_equal(r.trace(rays), want, f"9 x 2^27 references, accel {accel}")
    r.free()


DEVICE_REFUSALS = {"17_coincident": (17, 1, (512, 512, 512), str(17 * 2 ** 27) + " references"),
                   "17_meshes": (1, 17, (512, 512, 512), str(17 * 2 ** 27) + " cells"),
                   "2097152_cubed": (1, 1, WRAPPING_DIMS[0], "bad grid dimensions"),
                   "4194304_cubed": (1, 1, WRAPPING_DIMS[1], "bad grid dimensions")}


@pytest.mark.parametrize("case", list(DEVICE_REFUSALS))
def test_device_builder_refuses_32bit_overflow(libptap, case):
    """17 * 2^27 references in one grid (counted in 64 bits: a 32-bit scan wraps), 17 grids of 2^27 cells (refused before anything is
    allocated), or more than 2^27 cells per grid through a product of the dimensions that overflows 64 bits when taken in one step:
    build_grids_device fails with the count or "bad grid dimensions" in the message, and the context keeps its grids and accel and traces
    exactly as before."""
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, ACCEL_GRID_EMULATED, PtapError, Renderer, Scene
    copies, meshes, dims, want = DEVICE_REFUSALS[case]
    s = Scene.empty()
    for _ in range(meshes):
        s.add_model(box_filling_mesh(s, copies))
    s.build_grids(3, 4, 5)
    rays = _box_rays(20_000, 5)
    r = Renderer(width=64, height=32, depth=5, accel=ACCEL_GRID_COMPAT)
    r.allocateOnGPU(s)
    before = {}
    for accel in (ACCEL_GRID_EMULATED, ACCEL_GRID_COMPAT):
        r.set_accel(accel)
        before[accel] = r.trace(rays)
    assert (before[ACCEL_GRID_COMPAT]["model"] >= 0).mean() > 0.5
    with pytest.raises(PtapError, match=want):
        r.build_grids_device(s, *dims)
    assert r.trace(rays).tobytes() == before[ACCEL_GRID_COMPAT].tobytes()
    r.set_accel(ACCEL_GRID_EMULATED)
    assert r.trace(rays).tobytes() == before[ACCEL_GRID_EMULATED].tobytes()
    r.free()
