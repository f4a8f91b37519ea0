"""The oracle against the REFERENCE'S OWN Embree/ISPC backend.

tests/golden/ref_embree_frames.npz was produced by oracle/_ref/libcrt_embree.so, i.e. by
/root/reference/backends/embree/{render_embree.cpp,embree_utils.cpp,render_embree.ispc,*.ih} compiled where
they lie (ISPC kernels as scalar C++; Embree, TBB, GLM replaced by third_party/ stand-ins; see
oracle/ref_build/Makefile and tests/golden/make_ref_embree_golden.py). The oracle has to reproduce those
float framebuffers, per-pixel ray counts, sRGB8 images and pure-function tables BIT FOR BIT: that is what pins
it. Further cases compare with the library live where it is built (oracle/_ref/), including the plugin loaded by the
reference's own RenderPlugin in the headless twin, and elsewhere with what it rendered for them, recorded as digests
in tests/golden/ref_embree_live.json.
"""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import digest, reference_result
from ref_cases import FRAME_CASES, kat_inputs, make_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref_golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "ref_embree_frames.npz"))


def _same(a, b):
    """Bitwise equality of float arrays, NaNs in the same places."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("name", list(FRAME_CASES))
def test_oracle_reproduces_reference_frames_bit_for_bit(built, ref_golden, name):
    from oracle import OracleBackend

    scene, view, w, h, frames, depth = make_case(name)
    cpu = OracleBackend(max_depth=depth)
    cpu.initialize(w, h)
    cpu.set_scene(scene)
    rays = [cpu.render(*view, f == 0, True).num_rays for f in range(frames)]
    assert rays == [int(r) for r in ref_golden[f"{name}.rays"]]
    assert np.array_equal(cpu.read_ray_stats(), ref_golden[f"{name}.ray_stats"])
    assert _same(cpu.read_accum(), ref_golden[f"{name}.accum"])
    assert np.array_equal(cpu.img, ref_golden[f"{name}.img"])


def test_oracle_pure_functions_equal_the_references(built, ref_golden):
    """disney_bsdf.ih, lights.ih, texture2d.ih, lcg_rng.ih, util.ih, miss_shader: the oracle's restatements
    against tables computed by the reference's functions themselves."""
    from oracle import load_oracle_lib

    lib = load_oracle_lib()
    k = kat_inputs()
    ev = np.zeros_like(ref_golden["kat.disney_eval"])
    for mi, m in enumerate(k["mats"]):
        for oi, wo in enumerate(k["dirs"]):
            for ii, wi in enumerate(k["dirs"]):
                lib.oracle_kat_disney_eval(m.ctypes.data, k["n"].ctypes.data, wo.ctypes.data, wi.ctypes.data,
                                           ev[mi, oi, ii].ctypes.data)
    assert _same(ev, ref_golden["kat.disney_eval"])
    sm = np.zeros_like(ref_golden["kat.disney_sample"])
    for mi, m in enumerate(k["mats"]):
        for oi, wo in enumerate(k["dirs"]):
            for si, seed in enumerate(k["seeds"]):
                st = C.c_uint32(int(seed))
                lib.oracle_kat_disney_sample(m.ctypes.data, k["n"].ctypes.data, wo.ctypes.data, C.addressof(st),
                                             sm[mi, oi, si].ctypes.data)
                sm[mi, oi, si, 7] = np.array([st.value], np.uint32).view(np.float32)[0]
    assert _same(sm, ref_golden["kat.disney_sample"])
    lt = np.zeros_like(ref_golden["kat.light"])
    for si, s2 in enumerate(k["light_s"]):
        for di, d in enumerate(k["dirs"]):
            lib.oracle_kat_light(k["light"].ctypes.data, s2.ctypes.data, k["light_orig"].ctypes.data, d.ctypes.data,
                                 lt[si, di].ctypes.data)
    assert _same(lt, ref_golden["kat.light"])
    for ch in (1, 3, 4):
        tex = k[f"tex{ch}"]
        tx = np.zeros((len(k["uv"]), 4), np.float32)
        lib.oracle_kat_texture(tex.ctypes.data, tex.shape[1], tex.shape[0], ch, k["uv"].ctypes.data, len(k["uv"]),
                               tx.ctypes.data)
        assert _same(tx, ref_golden[f"kat.texture{ch}"])
    ms = np.zeros((len(k["miss_dirs"]), 3), np.float32)
    lib.oracle_kat_miss(k["miss_dirs"].ctypes.data, len(k["miss_dirs"]), ms.ctypes.data)
    assert _same(ms, ref_golden["kat.miss"])
    ob = np.zeros((len(k["dirs"]), 6), np.float32)
    for di, d in enumerate(k["dirs"]):
        lib.oracle_kat_ortho_basis(d.ctypes.data, ob[di].ctypes.data)
    assert _same(ob, ref_golden["kat.ortho_basis"])
    for i, (pix, frame) in enumerate(k["rng_keys"]):
        states, floats = np.zeros(16, np.uint32), np.zeros(16, np.float32)
        lib.oracle_kat_rng(int(pix), int(frame), 16, states.ctypes.data, floats.ctypes.data)
        assert np.array_equal(states, ref_golden["kat.rng_states"][i]) and _same(floats, ref_golden["kat.rng_floats"][i])


def _frame_digests(backend, by_value=False):
    """accum (bit for bit; by_value: NaN payloads and signed zeros folded), per-pixel ray counts, sRGB8 image."""
    a = backend.read_accum()
    a = np.where(np.isnan(a), np.float32(np.nan), a + np.float32(0)) if by_value else a.view(np.uint32)
    return {"accum": digest(a), "ray_stats": digest(backend.read_ray_stats()), "img": digest(backend.img)}


def _live(key, compute):
    """The reference build's result for `key`: compute() where the library is built, else the recorded result."""
    from oracle import ref_embree

    return reference_result("ref_embree_live.json", key, compute if ref_embree.available() else None)


# ------------------------------------------------------------------ live, where the library exists
def _ref_mod():
    from oracle import ref_embree

    if not ref_embree.available():
        pytest.skip("oracle/_ref/libcrt_embree.so not built (needs /root/reference at build time)")
    return ref_embree


def test_golden_file_is_what_the_reference_build_produces(built, ref_golden):
    """Guards the fixture itself: regenerating one case from the library gives the committed arrays."""
    ref_embree = _ref_mod()
    scene, view, w, h, frames, depth = make_case("materials")
    ref = ref_embree.RefEmbreeBackend(max_depth=depth)
    assert ref.name() == "Embree (w/ TBB & ISPC)"  # render_embree.cpp:33-36
    ref.initialize(w, h)
    ref.set_scene(scene)
    for f in range(frames):
        ref.render(*view, f == 0, True)
    assert _same(ref.read_accum(), ref_golden["materials.accum"])
    assert np.array_equal(ref.read_ray_stats(), ref_golden["materials.ray_stats"])


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_oracle_equals_reference_build_on_random_views(built, seed):
    """Other cameras, sizes, spp and frame counts than the frozen ones, camera reset included."""
    from chameleonrt_b200 import ArcballCamera
    from chameleonrt_b200.scenes import cornell_box, sponza_like
    from helpers import synthetic_material_scene
    from oracle import OracleBackend

    rng = np.random.default_rng(seed)
    spp = int(rng.integers(1, 4))
    scene, cam = [cornell_box, synthetic_material_scene, lambda spp: sponza_like(spp=spp, detail=0.2, tex_size=32)][seed % 3](spp=spp)
    w, h = int(rng.integers(40, 150)), int(rng.integers(40, 110))
    depth = int(rng.integers(1, 9))
    passes = []
    for k in range(2):  # second pass: camera moved, accumulation restarts
        eye = np.array(cam["eye"], np.float32) + rng.normal(scale=0.15, size=3).astype(np.float32)
        passes.append((ArcballCamera(eye, cam["center"], cam["up"]), int(rng.integers(1, 4))))

    def run(r):
        r.initialize(w, h)
        r.set_scene(scene)
        out = []
        for c, frames in passes:
            rays = [int(r.render(c.eye(), c.dir(), c.up(), cam["fov_y"], f == 0, True).num_rays) for f in range(frames)]
            out.append(dict(_frame_digests(r), rays=rays))
        return out

    from oracle import ref_embree

    ref = _live(f"random_view_{seed}", lambda: run(ref_embree.RefEmbreeBackend(max_depth=depth)))
    assert run(OracleBackend(max_depth=depth)) == ref


def _headless_embree_vs_oracle(case, scene, path, cam, w, h, tmp_path):
    """`crt_headless embree <path>` (2 spp, 2 frames) against `crt_headless oracle <path>`, bit for bit. Where the harness is
    not built, the recorded embree frame against the oracle fed the in-memory scene, which renders what the oracle plugin
    renders from the file (tests/test_reference_plugin.py)."""
    from oracle import OracleBackend
    from test_reference_plugin import HEADLESS, run_headless

    def live():
        a_ref, v, out = run_headless("embree", path, cam, w, h, 2, 2, tmp_path)
        return {"accum": digest(a_ref.view(np.uint32)), "camera": v, "embree": "Embree (w/ TBB & ISPC)" in out}

    ref = _live(f"headless_{case}", live if os.path.exists(HEADLESS) else None)
    assert ref["embree"]
    if os.path.exists(HEADLESS):
        a_cpu, v, _ = run_headless("oracle", path, cam, w, h, 2, 2, tmp_path)
        assert v == ref["camera"]
    else:
        v, o = ref["camera"], OracleBackend()
        o.initialize(w, h)
        o.set_scene(scene)
        for f in range(2):
            o.render(v[0:3], v[3:6], v[6:9], v[9], f == 0)
        a_cpu = o.read_accum()
    assert digest(a_cpu.view(np.uint32)) == ref["accum"]


@pytest.mark.parametrize("name", ["cornell", "sponza"])
def test_headless_embree_plugin_equals_oracle_plugin(built, tmp_path, name):
    """`crt_headless embree scene.obj`: the reference's RenderPlugin loads libcrt_embree.so, the reference's
    Scene::load_obj loads the file, the reference's RenderEmbree renders it (calling thread in FTZ/DAZ mode
    like the real application); the oracle plugin on the same file gives the same float framebuffer bit for
    bit."""
    from chameleonrt_b200.obj_io import write_obj
    from chameleonrt_b200.scenes import cornell_box, sponza_like

    scene, cam = cornell_box(spp=2) if name == "cornell" else sponza_like(spp=2, detail=0.2, tex_size=64)
    obj = write_obj(scene, str(tmp_path / "scene.obj"))
    _headless_embree_vs_oracle(f"obj_{name}", scene, obj, cam, 100, 76, tmp_path)


def test_headless_embree_plugin_on_gltf_instances(built, tmp_path):
    """The reference's glTF loader + the reference's Embree backend (instanced scene: rtcSetGeometryTransform,
    world_to_object normals) against the oracle plugin on the same .gltf: bit for bit."""
    from chameleonrt_b200.gltf_io import write_gltf
    from chameleonrt_b200.scenes import san_miguel_like

    scene, cam = san_miguel_like(spp=2, scale=0.02, tex_size=64)
    gltf = write_gltf(scene, str(tmp_path / "scene.gltf"))
    _headless_embree_vs_oracle("gltf_san_miguel", scene, gltf, cam, 96, 54, tmp_path)


def test_headless_embree_plugin_on_crts_all_lobes(built, tmp_path):
    """Every BSDF lobe, textured scalar parameters and an explicit light, loaded by the reference's .crts
    importer and rendered by the reference's Embree backend, against the oracle plugin: bit for bit."""
    from test_reference_plugin import _crts_case

    scene, cam, crts = _crts_case(tmp_path)
    _headless_embree_vs_oracle("crts_all_lobes", scene, crts, cam, 96, 72, tmp_path)


def test_fuzz_random_scenes_against_reference_build(built):
    """scripts/fuzz_oracle_vs_reference.py on a fixed set of seeds: random triangle soups and primitives, every
    Disney parameter random (textured scalars, transmission -> NaN paths), sheared / mirrored instances, several
    lights, random spp / depth / frames / ragged sizes. 2,100 seeds were clean when this was written; seed 1583 is
    the one that showed the oracle needs ISPC's min / max NaN semantics (minps / maxps return the second operand)."""
    import sys

    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import fuzz_oracle_vs_reference as fuzz
    from oracle import OracleBackend

    for seed in (0, 2, 5, 20, 31, 1583, 5007, 5333):
        c = fuzz.case(seed)
        ref = _live(f"fuzz_{seed}", lambda: _frame_digests(fuzz.render(fuzz.RefEmbreeBackend(max_depth=c[3]), c), by_value=True))
        assert _frame_digests(fuzz.render(OracleBackend(max_depth=c[3]), c), by_value=True) == ref, seed
