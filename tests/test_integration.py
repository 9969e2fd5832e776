"""The drop-in boundary in C++ (INTEGRATION.md): the facade headers under include/PathTracerAP/ and the in-tree shim
integration/Renderer_ptap.cpp.  CPU part: everything compiles and links, the reference's own main.cpp included where the
reference tree is mounted, and the binaries fail loudly without a GPU.  GPU part: the C++ flow renders the same BMP as the
Python mirror of the API."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, have_gpu
from oracle.ref import REFERENCE_ROOT

# the original PathTracerAP sources are not part of this repository: tests that build them run where PTAP_REFERENCE points at a checkout
REF_MAIN = os.path.join(REFERENCE_ROOT, "PathTracerAP", "main.cpp")
LIBDIR = os.path.join(ROOT, "pathtracerap_b200")


def _compile_facade(main_cpp, out, defs=()):
    cmd = ["g++", "-std=c++17", "-Wall", "-I" + os.path.join(ROOT, "include", "PathTracerAP"), *defs, main_cpp,
           "-L" + LIBDIR, "-lptap", "-Wl,-rpath," + LIBDIR, "-o", out]
    subprocess.check_call(cmd)
    return out


def write_bundled_objs(dirpath):
    """The three bundled meshes, regenerated from the golden scene arrays as 'Input data/*.obj' (one v/vn pair per face corner)."""
    z = np.load(os.path.join(GOLDEN, "bundled_scene.npz"))
    d = os.path.join(dirpath, "Input data")
    os.makedirs(d, exist_ok=True)
    names = ["enclosing_box.obj", "ceiling_light.obj", "blender_monkey.obj"]          # mesh order of Scene.cpp:6-16
    for mesh, name in zip(z["meshes"], names):
        v = z["vertices"][mesh["v_start"]:mesh["v_end"]]
        t = z["triangles"][mesh["t_start"]:mesh["t_end"]]["v"] - mesh["v_start"]
        with open(os.path.join(d, name), "w") as f:
            for p in v["position"] / 1000.0:
                f.write("v %.9g %.9g %.9g\n" % tuple(p))
            for n in v["normal"] / 1000.0:
                f.write("vn %.9g %.9g %.9g\n" % tuple(n))
            for a, b, c in t + 1:
                f.write(f"f {a}//{a} {b}//{b} {c}//{c}\n")
    return dirpath


def test_facade_compiles_with_the_reference_main(libptap, tmp_path):
    """main.cpp:11-28 against include/PathTracerAP/{Scene,Renderer}.h, unchanged (copied next to nothing so that its quoted
    includes resolve to the facade, not to the reference's own headers)."""
    src = tmp_path / "main.cpp"
    if os.path.exists(REF_MAIN):
        shutil.copy(REF_MAIN, src)
    else:
        shutil.copy(os.path.join(ROOT, "examples", "main.cpp"), src)
    exe = _compile_facade(str(src), str(tmp_path / "pt_main"))
    if not have_gpu():
        write_bundled_objs(str(tmp_path))
        p = subprocess.run([exe], cwd=tmp_path, capture_output=True, text=True)
        assert p.returncode != 0 and "no usable CUDA device" in (p.stderr + p.stdout)      # no CPU fallback: loud failure


@pytest.mark.skipif(not os.path.exists(REF_MAIN), reason="needs the original PathTracerAP sources (PTAP_REFERENCE), which are not part of this repository")
def test_shim_builds_inside_the_reference_tree(libptap):
    """The reference's own main.cpp + Scene.cpp + integration/Renderer_ptap.cpp (instead of Renderer.cpp) link against libptap."""
    subprocess.check_call([os.path.join(ROOT, "integration", "build_in_reference_tree.sh")])
    exe = os.path.join(ROOT, "integration", "_build", "pt_reference_tree")
    assert os.path.exists(exe)
    nm = subprocess.run(["nm", "-C", "--undefined-only", exe], capture_output=True, text=True).stdout
    for sym in ("ptap_create", "ptap_upload_scene", "ptap_build_accel", "ptap_set_render_params", "ptap_render", "ptap_read_film", "ptap_write_bmp"):
        assert sym in nm


def test_objs_round_trip_through_the_loader(libptap, tmp_path):
    """The in-repo OBJ reader (replaces Assimp, Scene.cpp:226-291): regenerated bundled meshes load to the golden topology."""
    from pathtracerap_b200 import Scene
    write_bundled_objs(str(tmp_path))
    s = Scene(None, root=str(tmp_path))
    a = s.arrays()
    z = np.load(os.path.join(GOLDEN, "bundled_scene.npz"))
    assert np.array_equal(a["triangles"]["v"], z["triangles"]["v"])
    assert len(a["models"]) == 11 and np.array_equal(a["models"]["mesh_index"], z["models"]["mesh_index"])
    assert np.allclose(a["vertices"]["position"], z["vertices"]["position"], rtol=1e-6, atol=1e-3)
    assert np.array_equal(a["models"]["model_to_world"], z["models"]["model_to_world"])
    assert np.array_equal(a["models"]["world_to_model"], z["models"]["world_to_model"])


@pytest.mark.gpu
@pytest.mark.skipif(not have_gpu(), reason="no CUDA device")
def test_cpp_flow_matches_python_api(libptap, tmp_path):
    from pathtracerap_b200 import ACCEL_GRID_COMPAT, Renderer, Scene
    write_bundled_objs(str(tmp_path))
    W, H, IT = 200, 160, 3
    exe = _compile_facade(os.path.join(ROOT, "examples", "main.cpp"), str(tmp_path / "pt_main"))
    env = dict(os.environ, PTAP_WIDTH=str(W), PTAP_HEIGHT=str(H), PTAP_ITER=str(IT))
    p = subprocess.run([exe], cwd=tmp_path, env=env, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    assert "Full run:" in p.stdout
    assert "emulated through the BVH" in p.stderr          # the default: the walk's results without the walk (PTAP_ACCEL_GRID_EMULATED)
    # the reference's per-iteration timing lines (Renderer.cpp:641-643), one per iteration, non-negative
    its = [l for l in p.stdout.splitlines() if l.startswith("Iteration ")]
    assert [l.split(":")[0] for l in its] == [f"Iteration {k + 1}" for k in range(IT)]
    assert all(int(l.split(":")[1].split()[0]) >= 0 for l in its)
    one_rank = (tmp_path / "Render.bmp").read_bytes()
    # PTAP_RANKS: several contexts of ONE process share the iterations and the films are summed over peer copies (ptap_reduce_peer).
    # On a one-GPU box both ranks sit on device 0; the image equals the one-rank image up to float reassociation of the film sum.
    p2 = subprocess.run([exe], cwd=tmp_path, env=dict(env, PTAP_RANKS="2", PTAP_RANK_DEVICES="0,0"), capture_output=True, text=True)
    assert p2.returncode == 0, p2.stderr
    assert "on 2 GPU(s)" in p2.stdout
    two_rank = (tmp_path / "Render.bmp").read_bytes()
    a1 = np.frombuffer(one_rank, np.uint8, offset=54).astype(int); a2 = np.frombuffer(two_rank, np.uint8, offset=54).astype(int)
    assert one_rank[:54] == two_rank[:54] and np.abs(a1 - a2).max() <= 1 and np.mean(a1 == a2) > 0.999
    p = subprocess.run([exe], cwd=tmp_path, env=env, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    s = Scene(None, root=str(tmp_path))
    r = Renderer(width=W, height=H, iters=IT, depth=5, accel=ACCEL_GRID_COMPAT)
    r.allocateOnGPU(s)
    r.renderLoop()
    r.renderImage(str(tmp_path / "py.bmp"))
    r.free()
    assert (tmp_path / "Render.bmp").read_bytes() == (tmp_path / "py.bmp").read_bytes()
    # the in-tree build (reference's main.cpp + Scene.cpp + Renderer_ptap.cpp), when it travelled with the snapshot
    exe2 = os.path.join(ROOT, "integration", "_build", "pt_reference_tree")
    if os.path.exists(exe2):
        d2 = tmp_path / "tree"; d2.mkdir()
        write_bundled_objs(str(d2))
        p = subprocess.run([exe2], cwd=d2, env=dict(os.environ, PTAP_ITER="2"), capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        assert "emulated through the BVH" in p.stderr      # the lists the reference's own Scene.cpp builds pass the shape checks
        r = Renderer(width=1000, height=800, iters=2, depth=5, accel=ACCEL_GRID_COMPAT)     # Config.h:12-13
        r.allocateOnGPU(Scene(None, root=str(d2)))
        r.renderLoop()
        r.renderImage(str(d2 / "py.bmp"))
        r.free()
        assert (d2 / "Render.bmp").read_bytes() == (d2 / "py.bmp").read_bytes()
