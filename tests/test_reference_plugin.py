"""The drop-in boundary exercised the way ChameleonRT exercises it: the headless twin of the app
(oracle/ref_build/crt_headless.cpp) loads `libcrt_<backend>.so` through the REFERENCE'S OWN
RenderPlugin class, loads an .obj with the reference's own Scene loader, and drives
initialize / set_scene / render. Binaries live in oracle/_ref/ (built by __graft_entry__.build() where the reference's
sources are; they travel with the tree as built artefacts). Where they are not built, the tests that compare the
reference's loaders with the Python scene model compare with the loaders' recorded frames (tests/golden/ref_loader_frames.json)."""
import os
import subprocess

import numpy as np
import pytest

from chameleonrt_b200.obj_io import write_obj
from chameleonrt_b200.scenes import cornell_box, sponza_like
from helpers import ROOT, assert_parity, digest, reference_result

REF = os.path.join(ROOT, "oracle", "_ref")
HEADLESS = os.path.join(REF, "crt_headless")

needs_ref = pytest.mark.skipif(not os.path.exists(HEADLESS), reason="oracle/_ref not built (needs the reference's sources)")


def run_headless(backend, obj, cam, w, h, spp, frames, tmp_path, depth=5, extra_env=None):
    out = tmp_path / f"accum_{backend}.f32"
    cmd = [HEADLESS, backend, obj, "-img", str(w), str(h), "-spp", str(spp), "-benchmark-frames", str(frames),
           "-accum", str(out), "-eye", *map(str, cam["eye"]), "-center", *map(str, cam["center"]),
           "-up", *map(str, cam["up"]), "-fov", str(cam["fov_y"])]
    env = dict(os.environ, CRT_CUDA_MAX_DEPTH=str(depth), **(extra_env or {}))
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path), env=env, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    cam_line = [l for l in r.stdout.splitlines() if l.startswith("camera:")][0].split()[1:]
    vec = [float.fromhex(x) for x in cam_line]
    accum = np.fromfile(out, np.float32).reshape(h, w, 3)
    assert os.path.exists(tmp_path / "chameleonrt.png")  # main.cpp:306-314 writes the final image
    return accum, vec, r.stdout


def reference_loader_frame(case, path, cam, w, h, tmp_path):
    """`crt_headless oracle <path>` at w x h, 2 spp, 2 frames: the file loaded by the reference's own Scene constructor and
    rendered by the oracle plugin, run where the harness is built, else as recorded: (digest of the float framebuffer's bits,
    camera the harness derived, the loader's scene summary)."""
    def live():
        accum, v, out = run_headless("oracle", path, cam, w, h, 2, 2, tmp_path)
        summary = [l for l in out.splitlines() if l.startswith("Scene '")][0].split("': ", 1)[1]
        return {"accum": digest(accum.view(np.uint32)), "camera": v, "summary": summary}

    rec = reference_result("ref_loader_frames.json", case, live if os.path.exists(HEADLESS) else None)
    return rec["accum"], rec["camera"], rec["summary"]


@pytest.mark.parametrize("name", ["cornell", "sponza"])
def test_reference_loader_matches_python_scene_model(built, tmp_path, name):
    """OBJ written by obj_io -> reference's load_obj (tinyobj, stb_image) -> oracle plugin must be
    bit-identical to the oracle fed the in-memory Python Scene: pins chameleonrt_b200.scene /
    scenes / obj_io against util/scene.cpp:94-228 (materials, generated light, texture flip)."""
    from oracle import OracleBackend

    scene, cam = cornell_box(spp=2) if name == "cornell" else sponza_like(spp=2, detail=0.2, tex_size=64)
    obj = write_obj(scene, str(tmp_path / "scene.obj"))
    accum, v, out = reference_loader_frame(f"obj_{name}", obj, cam, 96, 64, tmp_path)
    assert f"tris {scene.total_tris()} " in out and f"materials {len(scene.materials)} " in out
    o = OracleBackend()
    o.initialize(96, 64)
    o.set_scene(scene)
    for f in range(2):
        o.render(v[0:3], v[3:6], v[6:9], v[9], f == 0)
    assert digest(o.read_accum().view(np.uint32)) == accum


@needs_ref
def test_headless_application_with_the_native_loader(built, tmp_path):
    """The application path with the loader swapped (CRT_NATIVE_LOADER=1: crt_cuda::load_scene_native in place of the Scene
    constructor, backends/cuda/scene_native_load.h): same scene summary line, same camera, same frame for an OBJ with textures
    (tests/test_scene_io.py compares the Scene structs themselves, for every format)."""
    scene, cam = sponza_like(spp=2, detail=0.2, tex_size=32)
    obj = write_obj(scene, str(tmp_path / "scene.obj"))
    runs = [run_headless("oracle", obj, cam, 64, 48, 2, 2, tmp_path, extra_env={"CRT_NATIVE_LOADER": flag}) for flag in ("0", "1")]
    assert "(Scene constructor)" in runs[0][2] and "(native loader)" in runs[1][2]
    summary = [[l for l in r[2].splitlines() if l.startswith("Scene '")][0] for r in runs]
    assert summary[0] == summary[1] and runs[0][1] == runs[1][1]
    assert np.array_equal(runs[0][0].view(np.uint32), runs[1][0].view(np.uint32))


@needs_ref
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell", "sponza"])
def test_cuda_plugin_drop_in(built, tmp_path, name):
    """`crt_headless cuda scene.obj` vs `crt_headless oracle scene.obj`: the whole drop-in path
    (dlopen + POPULATE_PLUGIN_FUNCTIONS + RenderCUDA : RenderBackend + C ABI + kernels)."""
    scene, cam = cornell_box(spp=2) if name == "cornell" else sponza_like(spp=2, detail=0.3, tex_size=64)
    obj = write_obj(scene, str(tmp_path / "scene.obj"))
    a_gpu, v1, out = run_headless("cuda", obj, cam, 160, 96, 2, 2, tmp_path)
    a_cpu, v2, out_cpu = run_headless("oracle", obj, cam, 160, 96, 2, 2, tmp_path)
    assert v1 == v2 and "CUDA wavefront" in out
    assert_parity(a_gpu, a_cpu)
    # both plugins export crt_<backend>_get_stats (SURVEY.md §8b): stage times + counters of the last frame; the ray
    # counts of the two backends agree (closest-hit + occlusion on the GPU side = the CPU side's single count)
    def last_frame(text):
        line = [l for l in text.splitlines() if l.startswith("last frame: stage ms")][0]
        stage, counters = (list(map(float, part.split())) for part in line[len("last frame: stage ms"):].split("| counters"))
        return stage, counters
    (sg, cg), (sc, cc) = last_frame(out), last_frame(out_cpu)
    assert sg[6] > 0 and sc[6] > 0 and cg[0] + cg[1] == cc[0] > 0


def test_gltf_through_reference_loader_matches_python_scene_model(built, tmp_path):
    """The instanced, textured glTF-class scene written by gltf_io -> the reference's load_gltf (tinygltf,
    flatten_gltf, generated light; util/scene.cpp:230-415) -> oracle plugin is bit-identical to the oracle fed the
    in-memory Python Scene: pins scene.py / scenes.san_miguel_like / gltf_io against the reference's glTF import
    (parameterized meshes, instance matrices, sRGB base colour + linear metallic-roughness texture handles)."""
    from chameleonrt_b200.gltf_io import write_gltf
    from chameleonrt_b200.scenes import san_miguel_like
    from oracle import OracleBackend

    scene, cam = san_miguel_like(spp=2, scale=0.02, tex_size=64)
    gltf = write_gltf(scene, str(tmp_path / "scene.gltf"))
    accum, v, out = reference_loader_frame("gltf_san_miguel", gltf, cam, 96, 54, tmp_path)
    assert f"tris {scene.total_tris()} " in out and f"instances {len(scene.instances)} " in out
    assert f"materials {len(scene.materials)} " in out and f"textures {len(scene.textures)} " in out
    o = OracleBackend()
    o.initialize(96, 54)
    o.set_scene(scene)
    for f in range(2):
        o.render(v[0:3], v[3:6], v[6:9], v[9], f == 0)
    assert digest(o.read_accum().view(np.uint32)) == accum


@needs_ref
@pytest.mark.gpu
def test_cuda_plugin_drop_in_gltf_instances(built, tmp_path):
    """`crt_headless cuda scene.gltf`: BASELINE config 3's scene class (glTF, instances with non-identity
    transforms, textures) through the reference's loader into the CUDA plugin. The CUDA path flattens instances
    to world space, the oracle intersects in object space like Embree: parity is statistical, as in
    tests/test_gpu_parity.py::test_instanced_textured_gltf_class_scene."""
    from chameleonrt_b200.gltf_io import write_gltf
    from chameleonrt_b200.scenes import san_miguel_like

    scene, cam = san_miguel_like(spp=2, scale=0.02, tex_size=64)
    gltf = write_gltf(scene, str(tmp_path / "scene.gltf"))
    a_gpu, v1, out = run_headless("cuda", gltf, cam, 192, 108, 2, 2, tmp_path)
    a_cpu, v2, _ = run_headless("oracle", gltf, cam, 192, 108, 2, 2, tmp_path)
    assert v1 == v2 and "CUDA wavefront" in out
    assert_parity(a_gpu, a_cpu, min_frac=0.99, max_rel_l1=1e-2)


def _crts_case(tmp_path):
    """All BSDF lobes + textured scalar parameters + an explicit (axis-aligned) quad light, as a .crts file."""
    from chameleonrt_b200.crts_io import write_crts
    from chameleonrt_b200.scene import QuadLight
    from helpers import synthetic_material_scene

    scene, cam = synthetic_material_scene(spp=2)
    scene.lights = [QuadLight(emission=(12.0, 11.0, 9.0, 1.0), position=(0.5, 4.5, 0.5, 1.0), normal=(0.0, -1.0, 0.0),
                              v_x=(1.0, 0.0, 0.0), width=1.5, v_y=(0.0, 0.0, 1.0), height=1.0)]
    return scene, cam, write_crts(scene, str(tmp_path / "materials.crts"))


def test_crts_through_reference_loader_matches_python_scene_model(built, tmp_path):
    """.crts is the one format whose importer reads every Disney parameter, per-parameter texture handles
    (texture id + channel) and explicit quad lights (util/scene.cpp:417-620). File -> reference loader -> oracle
    plugin is bit-identical to the oracle fed the in-memory Scene, and to crts_io.crts_scene_view()."""
    from chameleonrt_b200.crts_io import crts_scene_view
    from oracle import OracleBackend

    scene, cam, crts = _crts_case(tmp_path)
    accum, v, out = reference_loader_frame("crts_all_lobes", crts, cam, 96, 72, tmp_path)
    assert f"tris {scene.total_tris()} " in out and "lights 1 " in out and f"textures {len(scene.textures)} " in out
    for sc in (scene, crts_scene_view(scene)):
        o = OracleBackend()
        o.initialize(96, 72)
        o.set_scene(sc)
        for f in range(2):
            o.render(v[0:3], v[3:6], v[6:9], v[9], f == 0)
        assert digest(o.read_accum().view(np.uint32)) == accum


@needs_ref
@pytest.mark.gpu
def test_cuda_plugin_drop_in_crts_all_lobes(built, tmp_path):
    """`crt_headless cuda materials.crts`: transmission, anisotropy, clearcoat, sheen and textured metallic /
    roughness through the reference's loader into the CUDA plugin."""
    scene, cam, crts = _crts_case(tmp_path)
    a_gpu, v1, out = run_headless("cuda", crts, cam, 192, 128, 2, 2, tmp_path, depth=6)
    a_cpu, v2, _ = run_headless("oracle", crts, cam, 192, 128, 2, 2, tmp_path, depth=6)
    assert v1 == v2 and "CUDA wavefront" in out
    assert_parity(a_gpu, a_cpu, min_frac=0.99, max_rel_l1=1e-2)


@needs_ref
def test_backends_cuda_cmake_builds_in_a_chameleonrt_like_project(built, tmp_path):
    """backends/cuda/CMakeLists.txt — what ChameleonRT's backends/CMakeLists.txt picks up — configured and built by CMake inside a
    stand-in for the reference's top-level project (oracle/ref_build/cmake_check: the reference's target names and headers; SDL2 /
    OpenGL / GLM headers from third_party/): the CUDA language is enabled, crt_cuda_core.cu compiles for sm_100a, libcrt_cuda.so
    comes out as a MODULE in its interactive (GLDisplay + CUDA-GL interop) form exporting populate_plugin_functions, and the
    optional crt_scene_native library builds."""
    import shutil

    if shutil.which("cmake") is None or not os.path.exists(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")):
        pytest.skip("needs cmake and nvcc")
    build = tmp_path / "cmake_check"
    r = subprocess.run([os.path.join(ROOT, "oracle", "ref_build", "cmake_check", "run.sh"), str(build)], capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    flags = open(build / "backends" / "cuda" / "CMakeFiles" / "crt_cuda.dir" / "flags.make").read()
    assert "arch=compute_100a" in flags and "-fmad=false" in flags
    symbols = subprocess.run(["nm", "-D", str(build / "libcrt_cuda.so")], capture_output=True, text=True).stdout
    assert " T populate_plugin_functions" in symbols
    assert os.path.getsize(build / "backends" / "cuda" / "libcrt_scene_native.a") > 100000
