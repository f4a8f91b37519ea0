"""The native scene loader (include/crt_scene_io.h, chameleonrt_b200/csrc/scene_io.cpp; SURVEY.md §8(f) rank 4) against its
oracle: the REFERENCE'S OWN Scene::load_obj (util/scene.cpp:94-228 over tinyobjloader + stb_image), compiled from the
reference's sources into oracle/_ref/libcrt_refscene.so by oracle/ref_build/Makefile. Every array of the Scene must be the same,
bit for bit: per geometry the vertices, uvs and indices in the same order (the single-index remap of scene.cpp:116-181 keeps
the order of first use), the material ids, the DisneyMaterials (incl. texture handles), the texture pixels (RGBA, rows
flipped) and the generated light. Where the reference library is not built, the reference's results are read from
tests/golden/ref_scene_loads.json (digests of every array, recorded by that library on the same input files)."""
import ctypes as C
import hashlib
import os
import time

import numpy as np
import pytest

from helpers import ROOT, digest, reference_result, synthetic_material_scene

REFLIB = os.path.join(ROOT, "oracle", "_ref", "libcrt_refscene.so")


NATIVE_SHIM_LIB = os.path.join(ROOT, "oracle", "_ref", "libcrt_refscene_native.so")


def _ref(path=None):
    lib = C.CDLL(path or REFLIB)
    lib.refscene_texture_name.restype = C.c_char_p
    lib.refscene_texture_name.argtypes = [C.c_void_p, C.c_uint32]
    lib.refscene_load.restype = C.c_void_p
    lib.refscene_load.argtypes = [C.c_char_p, C.POINTER(C.c_double)]
    lib.refscene_load_mode.restype = C.c_void_p
    lib.refscene_load_mode.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_double)]
    lib.refscene_error.restype = C.c_char_p
    lib.refscene_free.argtypes = [C.c_void_p]
    lib.refscene_counts.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    lib.refscene_mesh_geometry.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32] + [C.c_void_p] * 7
    lib.refscene_parameterized_mesh.restype = C.POINTER(C.c_uint32)
    lib.refscene_parameterized_mesh.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.refscene_materials.restype = C.POINTER(C.c_uint32)
    lib.refscene_materials.argtypes = [C.c_void_p]
    lib.refscene_light.restype = C.POINTER(C.c_uint32)
    lib.refscene_light.argtypes = [C.c_void_p, C.c_uint32]
    lib.refscene_instance.restype = C.POINTER(C.c_uint32)
    lib.refscene_instance.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.refscene_cameras.restype = C.POINTER(C.c_uint32)
    lib.refscene_cameras.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    lib.refscene_texture.restype = C.POINTER(C.c_uint8)
    lib.refscene_texture.argtypes = [C.c_void_p, C.c_uint32] + [C.POINTER(C.c_int)] * 4
    return lib


def _reference_arrays(path, white_diffuse=False, lib_path=None, refusal_ok=False):
    """What the reference's Scene constructor built, as numpy arrays (bit patterns for everything float). `geometries` lists the
    geometries of all meshes in order; `mesh_sizes` says how many each mesh has. Where the reference refuses the file: None if
    refusal_ok, else an assertion with the reference's error."""
    lib = _ref(lib_path)
    secs = C.c_double(0)
    h = lib.refscene_load_mode(path.encode(), int(white_diffuse), C.byref(secs))
    if not h and refusal_ok:
        return None
    assert h, lib.refscene_error().decode()
    counts = (C.c_uint32 * 7)()
    lib.refscene_counts(h, counts)
    out = dict(counts=list(counts), seconds=secs.value, geometries=[], mesh_sizes=[])
    for m in range(counts[0]):
        g, ng = 0, C.c_uint32(1)
        while g < ng.value:
            v, uv, idx = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint32)()
            nv, nuv, nt = C.c_uint32(), C.c_uint32(), C.c_uint32()
            lib.refscene_mesh_geometry(h, m, g, C.byref(v), C.byref(nv), C.byref(uv), C.byref(nuv), C.byref(idx), C.byref(nt), C.byref(ng))
            out["geometries"].append((np.ctypeslib.as_array(v, (nv.value * 3,)).copy() if nv.value else np.zeros(0, np.uint32),
                                      np.ctypeslib.as_array(uv, (nuv.value * 2,)).copy() if nuv.value else np.zeros(0, np.uint32),
                                      np.ctypeslib.as_array(idx, (nt.value * 3,)).copy() if nt.value else np.zeros(0, np.uint32)))
            g += 1
        out["mesh_sizes"].append(ng.value)
    out["parameterized_meshes"] = []
    for i in range(counts[2]):
        n, mesh_id = C.c_uint32(), C.c_uint32()
        p = lib.refscene_parameterized_mesh(h, i, C.byref(n), C.byref(mesh_id))
        out["parameterized_meshes"].append((mesh_id.value, list(np.ctypeslib.as_array(p, (n.value,)))))
    out["material_ids"] = np.array(out["parameterized_meshes"][0][1], np.uint32) if counts[2] else np.zeros(0, np.uint32)
    out["materials"] = np.ctypeslib.as_array(lib.refscene_materials(h), (counts[4] * 16,)).copy() if counts[4] else np.zeros(0, np.uint32)
    out["lights"] = np.concatenate([np.ctypeslib.as_array(lib.refscene_light(h, i), (20,)).copy() for i in range(counts[6])])
    inst = []
    for i in range(counts[3]):
        pm = C.c_uint32()
        inst.append(np.append(np.ctypeslib.as_array(lib.refscene_instance(h, i, C.byref(pm)), (16,)).copy(), pm.value))
    out["instances"] = np.concatenate(inst) if inst else np.zeros(0, np.uint32)
    n = C.c_uint32()
    cams = lib.refscene_cameras(h, C.byref(n))
    out["cameras"] = np.ctypeslib.as_array(cams, (n.value * 10,)).copy() if n.value else np.zeros(0, np.uint32)
    out["textures"] = []
    for i in range(counts[5]):
        w, hh, ch, cs = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        d = lib.refscene_texture(h, i, C.byref(w), C.byref(hh), C.byref(ch), C.byref(cs))
        out["textures"].append((np.ctypeslib.as_array(d, (hh.value, w.value, ch.value)).copy(), cs.value))
    out["texture_names"] = [lib.refscene_texture_name(h, i).decode() for i in range(counts[5])]
    lib.refscene_free(h)
    return out


def _record(arrays):
    """A loaded scene as counts and digests of its arrays: what the comparison with the reference's loader needs, small enough
    to be stored (tests/golden/ref_scene_loads.json)."""
    return dict(counts=[int(c) for c in arrays["counts"]], mesh_sizes=[int(n) for n in arrays["mesh_sizes"]],
                geometries=[digest(*g) for g in arrays["geometries"]],
                parameterized_meshes=digest(*[np.array([m] + list(ids), np.uint32) for m, ids in arrays["parameterized_meshes"]]),
                **{k: digest(arrays[k]) for k in ("material_ids", "materials", "lights", "instances", "cameras")},
                textures=[[digest(t), int(cs)] for t, cs in arrays["textures"]])


def _load_key(path, white_diffuse):
    """The input a recorded result belongs to: the scene file's name, the material mode and the bytes of every file under the
    scene file's directory (MTL files, textures, buffers — and whatever else the test wrote there, in a fixed order). Many
    textures are written by Pillow, so a Pillow / zlib / libjpeg that encodes them differently makes different input files:
    their lookup then fails with "no recorded result" (the reference's result for the new bytes is not known) rather than
    comparing with a result recorded for other bytes; re-record where the reference library is built."""
    h = hashlib.sha256(f"{os.path.basename(path)}|{int(white_diffuse)}".encode())
    top = os.path.dirname(os.path.abspath(path))
    for d, subdirs, files in os.walk(top):
        subdirs.sort()
        for f in sorted(files):
            h.update(os.path.relpath(os.path.join(d, f), top).encode() + b"\0")
            with open(os.path.join(d, f), "rb") as fh:
                h.update(hashlib.sha256(fh.read()).digest())
    return h.hexdigest()[:32]


def _reference_scene(path, white_diffuse=False, lib_path=None):
    """What the reference's Scene constructor builds from `path`, as a _record(); {"refused": True} where it refuses the file.
    Computed by the reference's own loader where oracle/_ref/libcrt_refscene.so is built (and checked against the recorded
    result), else read from tests/golden/ref_scene_loads.json. "seconds", the reference loader's time, is there only when it
    ran here. (lib_path: another library behind the same API, always run live.)"""
    if lib_path is not None:
        arrays = _reference_arrays(path, white_diffuse, lib_path, refusal_ok=True)
        return {"refused": True} if arrays is None else dict(_record(arrays), texture_names=arrays["texture_names"])
    timing = {}

    def live():
        arrays = _reference_arrays(path, white_diffuse, refusal_ok=True)
        if arrays is None:
            return {"refused": True}
        timing["seconds"] = arrays["seconds"]
        return _record(arrays)

    rec = reference_result("ref_scene_loads.json", _load_key(path, white_diffuse), live if os.path.exists(REFLIB) else None)
    return dict(rec, **timing)


def _native_arrays(path, threads=0, white_diffuse=False):
    from chameleonrt_b200 import scene_io

    loaded = scene_io.load_scene(path, threads, white_diffuse)
    s = loaded.c_scene.contents
    out = dict(counts=[s.num_meshes, s.meshes[0].num_geometries if s.num_meshes else 0, s.num_parameterized_meshes, s.num_instances,
                       s.num_materials, s.num_textures, s.num_lights], seconds=loaded.timings["total_s"], timings=loaded.timings,
               warnings=loaded.warnings, geometries=[], mesh_sizes=[])
    u32 = C.POINTER(C.c_uint32)
    for m in range(s.num_meshes):
        for g in range(s.meshes[m].num_geometries):
            cg = s.meshes[m].geometries[g]
            out["geometries"].append((np.ctypeslib.as_array(C.cast(cg.vertices, u32), (cg.num_vertices * 3,)).copy() if cg.num_vertices else np.zeros(0, np.uint32),
                                      np.ctypeslib.as_array(C.cast(cg.uvs, u32), (cg.num_vertices * 2,)).copy() if cg.uvs else np.zeros(0, np.uint32),
                                      np.ctypeslib.as_array(cg.indices, (cg.num_tris * 3,)).copy() if cg.num_tris else np.zeros(0, np.uint32)))
        out["mesh_sizes"].append(s.meshes[m].num_geometries)
    out["parameterized_meshes"] = []
    for i in range(s.num_parameterized_meshes):
        pm = s.parameterized_meshes[i]
        out["parameterized_meshes"].append((pm.mesh_id, list(np.ctypeslib.as_array(pm.material_ids, (pm.num_material_ids,)))))
    out["material_ids"] = np.array(out["parameterized_meshes"][0][1], np.uint32) if s.num_parameterized_meshes else np.zeros(0, np.uint32)
    out["materials"] = np.ctypeslib.as_array(C.cast(s.materials, u32), (s.num_materials * 16,)).copy() if s.num_materials else np.zeros(0, np.uint32)
    out["lights"] = np.ctypeslib.as_array(C.cast(s.lights, u32), (20 * s.num_lights,)).copy()
    inst = [np.append(np.ctypeslib.as_array(C.cast(C.pointer(s.instances[i]), u32), (16,)).copy(), s.instances[i].parameterized_mesh_id)
            for i in range(s.num_instances)]
    out["instances"] = np.concatenate(inst) if inst else np.zeros(0, np.uint32)
    out["cameras"] = (np.concatenate([np.concatenate([c["position"], c["center"], c["up"], [np.float32(c["fov_y"])]]).astype(np.float32)
                                      for c in loaded.cameras]).view(np.uint32) if loaded.cameras else np.zeros(0, np.uint32))
    out["textures"] = [(np.ctypeslib.as_array(s.textures[i].data, (s.textures[i].height, s.textures[i].width, s.textures[i].channels)).copy(),
                        int(s.textures[i].color_space)) for i in range(s.num_textures)]
    return out, loaded


def _assert_same(a, b):
    """a: the native loader's arrays (or a record), b: the reference's record."""
    assert not b.get("refused"), "the reference's loader refuses the file"
    if not isinstance(a["materials"], str):
        a = _record(a)
    assert a["counts"] == b["counts"] and a["mesh_sizes"] == b["mesh_sizes"]
    assert len(a["geometries"]) == len(b["geometries"])
    for g, (x, y) in enumerate(zip(a["geometries"], b["geometries"])):
        assert x == y, f"geometry {g}: vertices, uvs or indices differ"
    for k in ("parameterized_meshes", "material_ids", "materials", "lights", "instances", "cameras"):
        assert a[k] == b[k], k
    assert len(a["textures"]) == len(b["textures"])
    for t, (x, y) in enumerate(zip(a["textures"], b["textures"])):
        assert x == y, f"texture {t} differs"


def _cases():
    from chameleonrt_b200.scenes import cornell_box, rungholt_like, sponza_like

    return {"cornell": lambda: cornell_box()[0], "sponza_textured": lambda: sponza_like(detail=0.3, tex_size=64)[0],
            "voxels": lambda: rungholt_like(scale=0.02)[0]}


@pytest.mark.parametrize("name", ["cornell", "sponza_textured", "voxels"])
def test_native_obj_loader_builds_the_reference_loaders_scene(built, tmp_path, name):
    from chameleonrt_b200.obj_io import write_obj

    path = write_obj(_cases()[name](), str(tmp_path / f"{name}.obj"))
    ref = _reference_scene(path)
    for threads in (0, 1, 3):
        nat, _ = _native_arrays(path, threads)
        _assert_same(nat, ref)
    print(f"\n{name}: reference loader {ref.get('seconds', float('nan')) * 1e3:.1f} ms, native {nat['timings']}")


def test_native_obj_loader_on_hand_written_obj_quirks(built, tmp_path):
    """What tinyobjloader does with the less regular parts of the format: relative (negative) indices, v//vn and v/vt/vn
    corners (the normal index is part of the remap key), several usemtl inside one group (the first face's material wins,
    with a warning), an `o` statement, faces before any group, a material that no MTL defines (-> the generated default
    material), exponents and signs in numbers, CRLF line ends, comments and blank lines."""
    obj = tmp_path / "quirks.obj"
    (tmp_path / "quirks.mtl").write_text("# materials\nnewmtl red\nKd 0.8 0.1 0.1\nNs 250\n\nnewmtl shiny\nKd 1e-1 2.5E-1 +0.5\nNs 1000\n")
    obj.write_text("mtllib quirks.mtl\r\n# a quad as two triangles, no group yet\r\n"
                   "v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvn 0 0 1\nvn 0 0 -1\nvt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\n"
                   "usemtl red\nf 1/1/1 2/2/1 3/3/1\nf -4/1/1 -2/3/1 -1/4/1\n"
                   "g second\nusemtl shiny\nv 0 0 1.5e0\nv 1 0 1.5\nv 1 1 1.5\n\nf 5//1 6//1 7//1\nf 5//2 6//1 7//1\nusemtl red\nf 7//1 6//1 5//1\n"
                   "o third\nusemtl nowhere\nv -1 -1 -1\nv -2 -1 -1\nv -1 -2 -1\nf 8 9 10\nf 10 9 8\n")
    ref = _reference_scene(str(obj))
    nat, loaded = _native_arrays(str(obj))
    _assert_same(nat, ref)
    assert nat["counts"][1] == 3 and nat["counts"][4] == 3  # three shapes; red, shiny + the generated default material
    assert "per-face material IDs" in loaded.warnings and "generating a default" in loaded.warnings


def _polygon_obj(path, seed, faces=400):
    """An OBJ of faces with 3 to 12 corners: convex and star-shaped (concave) polygons in arbitrary planes, non-planar
    ones, self-intersecting ones (corners in shuffled order), polygons with collinear runs, repeated corners and zero
    area, faces of one and two corners; with and without vt / vn indices; several groups, objects and materials."""
    rng = np.random.default_rng(seed)
    lines, nv, nvt = ["mtllib poly.mtl"], 0, 0
    for i in range(16):
        lines.append(f"vn {rng.normal():.4f} {rng.normal():.4f} {rng.normal():.4f}")
    for f in range(faces):
        if f % 37 in (0, 19):
            lines.append(f"g group{f}" if (f // 37) % 3 else f"o object{f}")
        if f % 23 == 0:
            lines.append(f"usemtl m{(f // 23) % 3}")
        n = int(rng.integers(3, 13))
        kind = int(rng.integers(0, 8))
        origin, ex, ey = rng.normal(size=3) * 3, rng.normal(size=3), rng.normal(size=3)
        ang = np.sort(rng.uniform(0, 2 * np.pi, n))
        rad = np.ones(n)
        if kind == 1:
            rad = np.where(np.arange(n) % 2, 0.35, 1.0)  # a star
        elif kind == 2:
            rad = rng.uniform(0.2, 1.5, n)
        pts = origin + np.outer(np.cos(ang) * rad, ex) + np.outer(np.sin(ang) * rad, ey)
        if kind == 3:
            pts += rng.normal(size=(n, 3)) * 0.2  # not planar
        elif kind == 4:
            pts = pts[rng.permutation(n)]  # self-intersecting
        elif kind == 5:
            pts = origin + np.outer(np.linspace(0, 1, n), ex)  # all on one line
        elif kind == 6 and n > 3:
            pts[1] = pts[0]  # a repeated corner
            pts[n - 1] = 0.5 * (pts[n - 2] + pts[0])  # and a collinear one
        elif kind == 7 and f % 37 not in (0, 19):
            n = int(rng.integers(1, 3))  # a face that is none
            pts = pts[:n]
        if rng.integers(0, 2):
            pts = pts[::-1]
        fmt = "%.6g" if f % 2 else "%.3f"
        for q in pts:
            lines.append("v " + " ".join(fmt % x for x in q))
        style = (1 + 2 * int(rng.integers(0, 2))) if f % 37 > 18 else 2 * int(rng.integers(0, 2))  # (all corners of a shape have uvs or none)
        if style in (1, 3):
            for q in pts:
                lines.append(f"vt {rng.uniform():.4f} {rng.uniform():.4f}")
        corners = []
        for k in range(n):
            v = nv + k + 1 if f % 3 else k - n  # absolute or relative
            vt, vn = nvt + k + 1, int(rng.integers(1, 17))
            corners.append([f"{v}", f"{v}/{vt}", f"{v}//{vn}", f"{v}/{vt}/{vn}"][style])
        lines.append("f " + ("  " if f % 5 == 0 else " ").join(corners) + (" \r" if f % 7 == 0 else ""))
        nv += n
        nvt += n if style in (1, 3) else 0
    with open(path, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    with open(os.path.join(os.path.dirname(path), "poly.mtl"), "w") as fh:
        fh.write("newmtl m0\nKd 0.8 0.2 0.2\nnewmtl m1\nKd 0.2 0.8 0.2\nNs 100\nnewmtl m2\nKd 0.2 0.2 0.8\n")
    return path


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_native_obj_loader_triangulates_polygons_as_tinyobjloader_does(built, tmp_path, seed):
    """Faces of more than three corners: the ear clipping of exportGroupsToShape (tiny_obj_loader.h:1107-1310), restated in
    ear_clip() — same triangles in the same order, also where the clipping gives up on a polygon."""
    path = _polygon_obj(str(tmp_path / "poly.obj"), seed)
    ref = _reference_scene(path)
    for threads in (0, 1):
        nat, _ = _native_arrays(path, threads)
        _assert_same(nat, ref)
    tris = sum(len(g[2]) // 3 for g in nat["geometries"])
    assert tris > 400
    if seed == 1:
        # corners that point at positions the file defines later: the ear clipping sees what was read when the face group
        # was exported (here: at the `g` line), and takes (0, 0) for the rest
        fwd = tmp_path / "forward.obj"
        fwd.write_text("v 0 0 0\nv 2 0 0\nv 2 2 0\nv 1 0.5 0\nf 1 2 3 4 5 6\ng later\nv 0 2 0\nv -1 1 0\nf 1 2 3 4 5 6\nf 1 2 6 3 5 4\n")
        _assert_same(_native_arrays(str(fwd))[0], _reference_scene(str(fwd)))


def test_native_obj_loader_quads_without_the_reference(built, tmp_path):
    """Known answers (hold on the GPU box too): a convex quad is cut into (0, 1, 2) and (0, 2, 3); of a dart the ear that
    would contain the reflex corner is skipped."""
    from chameleonrt_b200 import scene_io

    quad = tmp_path / "quad.obj"
    quad.write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf 1 2 3 4\n")
    loaded = scene_io.load_obj(str(quad))  # (owns the arrays)
    g = loaded.c_scene.contents.meshes[0].geometries[0]
    assert g.num_tris == 2 and g.num_vertices == 4
    assert list(np.ctypeslib.as_array(g.indices, (6,))) == [0, 1, 2, 0, 2, 3]
    dart = tmp_path / "dart.obj"  # corner 2 (0.2, 0.2) is reflex
    dart.write_text("v 0 0 0\nv 1 0 0\nv 0.2 0.2 0\nv 0 1 0\nf 1 2 3 4\n")
    loaded = scene_io.load_obj(str(dart))
    g = loaded.c_scene.contents.meshes[0].geometries[0]
    idx = np.ctypeslib.as_array(g.indices, (g.num_tris * 3,)).reshape(-1, 3)
    v = np.ctypeslib.as_array(g.vertices, (g.num_vertices * 3,)).reshape(-1, 3)
    area = sum(0.5 * np.cross(v[t[1]] - v[t[0]], v[t[2]] - v[t[0]])[2] for t in idx)
    assert g.num_tris == 2 and abs(area - 0.2) < 1e-6  # the dart's area: both triangles inside it


def test_native_obj_loader_errors(built, tmp_path):
    from chameleonrt_b200 import scene_io

    with pytest.raises(RuntimeError, match="cannot open"):
        scene_io.load_obj(str(tmp_path / "missing.obj"))
    flat = tmp_path / "flat.obj"  # (the reference indexes an empty material_ids array here)
    flat.write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nf 1 2\n")
    with pytest.raises(RuntimeError, match="without a triangle"):
        scene_io.load_obj(str(flat))
    glued = tmp_path / "glued.obj"
    glued.write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nf 1/1/1/1 2 3\n")
    with pytest.raises(RuntimeError, match="Failed parse `f' line"):
        scene_io.load_obj(str(glued))
    zero = tmp_path / "zero.obj"
    zero.write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nf 0 1 2\n")
    with pytest.raises(RuntimeError, match="zero value for face index"):
        scene_io.load_obj(str(zero))
    oob = tmp_path / "oob.obj"
    oob.write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nf 1 2 9\n")
    with pytest.raises(RuntimeError, match="out of range"):
        scene_io.load_obj(str(oob))


def test_native_obj_loader_round_trip_and_oracle_frame(built, tmp_path):
    """Without the reference library (the GPU box): the loaded scene equals the scene the OBJ was written from —
    write_obj / Scene::load_obj are inverse to each other for these scenes (tests/test_reference_plugin.py) — and renders
    the same frame through the CPU oracle."""
    from chameleonrt_b200 import ArcballCamera, scene_io
    from chameleonrt_b200.obj_io import write_obj
    from chameleonrt_b200.scenes import cornell_box
    from oracle import OracleBackend

    scene, cam = cornell_box(spp=1)
    path = write_obj(scene, str(tmp_path / "cornell.obj"))
    loaded = scene_io.load_obj(path)
    got = loaded.to_scene(spp=1)
    assert len(got.meshes[0].geometries) == len(scene.meshes[0].geometries)
    c = ArcballCamera(cam["eye"], cam["center"], cam["up"])
    frames = []
    for s in (scene, got):
        o = OracleBackend(max_depth=5)
        o.initialize(48, 32)
        o.set_scene(s)
        o.render(c.eye(), c.dir(), c.up(), cam["fov_y"], True, True)
        frames.append(o.read_accum())
    assert np.array_equal(frames[0].view(np.uint32), frames[1].view(np.uint32))


def test_native_obj_loader_is_faster_on_a_large_file(built, tmp_path):
    """Throughput (the point of the row): a voxel city of a few hundred thousand triangles through both loaders. The bound
    asserted is loose (the suite runs on shared CPUs); the measured times are printed and recorded in DESIGN.md."""
    from chameleonrt_b200.obj_io import write_obj
    from chameleonrt_b200.scenes import rungholt_like

    path = write_obj(rungholt_like(scale=0.12)[0], str(tmp_path / "city.obj"))
    t0 = time.time()
    ref = _reference_scene(path)
    t_ref = time.time() - t0
    best = None
    for _ in range(2):
        nat, loaded = _native_arrays(path)
        best = loaded.timings if best is None or loaded.timings["total_s"] < best["total_s"] else best
    _assert_same(nat, ref)
    tris = sum(len(g[2]) // 3 for g in nat["geometries"])
    print(f"\n{tris} triangles, {os.path.getsize(path) / 1e6:.0f} MB: reference loader {ref.get('seconds', float('nan')):.2f} s (call {t_ref:.2f} s), native {best}")
    if "seconds" in ref:  # (the loaders are timed against each other only on the same host: a recorded time is another machine's)
        assert best["total_s"] < ref["seconds"]


# ---------------------------------------------------------------------------------------------------------------
# .crts (Scene::load_crts, util/scene.cpp:417-625)
def _rotated(seed):
    """A rotation + non-uniform scale + translation as a column-major list of 16 floats (an object's "matrix")."""
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    m = np.eye(4)
    m[:3, :3] = q * rng.uniform(0.5, 2.0, 3)
    m[:3, 3] = rng.normal(size=3) * 4
    return [float(np.float32(x)) for x in m.T.reshape(-1)]


def _crts_file(tmp_path, align=True, name="scene.crts"):
    """Every material parameter and texture handle (helpers.synthetic_material_scene), three instances of the same meshes
    under different matrices (-> shared parameterized meshes), two lights with arbitrary frames, two cameras."""
    from chameleonrt_b200.crts_io import write_crts
    from chameleonrt_b200.scene import Instance

    scene, cam = synthetic_material_scene(spp=1)
    scene.lights = []
    for k in (1, 2):
        scene.instances.append(Instance(np.array(_rotated(k), np.float32).reshape(4, 4).T, 0))
    extra = [dict(type="LIGHT", color=[0.9, 0.8, 0.7], energy=12.5, size=[1.5, 0.75], matrix=_rotated(10)),
             dict(type="CAMERA", fov_y=55.0, matrix=_rotated(11)),
             dict(type="LIGHT", color=[1, 1, 1], energy=3, size=[2, 1], matrix=_rotated(12)),  # (integers in the JSON)
             dict(type="CAMERA", fov_y=40, matrix=_rotated(13))]
    return scene, write_crts(scene, str(tmp_path / name), extra_objects=extra, align=align)


@pytest.mark.parametrize("align", [True, False])
def test_native_crts_loader_builds_the_reference_loaders_scene(built, tmp_path, align):
    """Meshes, (mesh, material) parameterized meshes in order of first use, instances, all 14 material parameters with their
    texture handles, decoded images, lights (frames normalised with glm's vec4 arithmetic), cameras — bit for bit what
    Scene::load_crts builds; also when the data block is not aligned in the file (the arrays are copied then)."""
    pytest.importorskip("PIL")
    scene, path = _crts_file(tmp_path, align)
    ref = _reference_scene(path)
    for threads in (0, 1):
        nat, loaded = _native_arrays(path, threads)
        _assert_same(nat, ref)
    assert nat["counts"] == [5, 1, 5, 15, 5, 2, 2] and len(loaded.cameras) == 2
    assert len(nat["cameras"]) == 20 and nat["lights"].shape == (40,)


def test_native_crts_loader_defaults_and_header_quirks(built, tmp_path):
    """No lights (-> the generated one, emission 10), no materials section and material id -1 (-> the default material), a
    key given twice (the last one counts), escapes in strings, numbers with exponents, an empty images list."""
    import json
    import struct

    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.5]], np.float32).tobytes()
    i = np.array([[0, 1, 2], [2, 1, 3]], np.uint32).tobytes()
    header = {"meshes": [{"positions": 0, "indices": 1}], "images": [],
              "objects": [{"type": "MESH", "mesh": 0, "material": 4294967295, "matrix": _rotated(3)},
                          {"type": "MESH", "mesh": 0.0, "material": 4294967295, "matrix": [1e0, 0, 0, 0, 0, 1.5E+0, 0, 0, 0, 0, 1, 0, -2.5e-1, 0, 0, 1]}],
              "buffer_views": [{"byte_offset": 0, "byte_length": len(v), "type": "VEC3_F32"},
                               {"byte_offset": len(v), "byte_length": len(i), "type": "UINT_32", "näme": "a \"quoted\" \\ name / \t tab"}]}
    js = json.dumps(header)
    js = js[:-1] + ', "objects": ' + json.dumps(header["objects"][::-1]) + "}"  # the second "objects" wins
    path = tmp_path / "quirks.crts"
    path.write_bytes(struct.pack("<Q", len(js)) + js.encode() + v + i)
    ref = _reference_scene(str(path))
    nat, loaded = _native_arrays(str(path))
    _assert_same(nat, ref)
    assert nat["counts"] == [1, 1, 1, 2, 1, 0, 1]
    assert "generating a default" in loaded.warnings and "No lights found" in loaded.warnings


def test_native_crts_loader_errors(built, tmp_path):
    import json
    import struct

    from chameleonrt_b200 import scene_io

    def write(name, header, data=b"", raw=None):
        js = raw if raw is not None else json.dumps(header).encode()
        p = tmp_path / name
        p.write_bytes(struct.pack("<Q", len(js)) + js + data)
        return str(p)

    with pytest.raises(RuntimeError, match="cannot open"):
        scene_io.load_crts(str(tmp_path / "missing.crts"))
    with pytest.raises(RuntimeError, match="Unsupported file"):
        scene_io.load_scene(str(tmp_path / "scene.ply"))
    (tmp_path / "short.crts").write_bytes(b"abc")
    with pytest.raises(RuntimeError, match="too short"):
        scene_io.load_crts(str(tmp_path / "short.crts"))
    (tmp_path / "size.crts").write_bytes(struct.pack("<Q", 1000) + b"{}")
    with pytest.raises(RuntimeError, match="header size past the end"):
        scene_io.load_crts(str(tmp_path / "size.crts"))
    with pytest.raises(RuntimeError, match="malformed JSON"):
        scene_io.load_crts(write("bad.crts", None, raw=b'{"meshes": [1, 2,, ]}'))
    views = [{"byte_offset": 0, "byte_length": 36, "type": "VEC3_F32"}, {"byte_offset": 36, "byte_length": 12, "type": "VEC3_U32"}]
    tri = np.zeros(9, np.float32).tobytes() + np.array([0, 1, 2], np.uint32).tobytes()
    with pytest.raises(RuntimeError, match="past the end"):
        scene_io.load_crts(write("oob.crts", {"meshes": [{"positions": 0, "indices": 1}], "buffer_views": views}, tri[:40]))
    with pytest.raises(RuntimeError, match="has no element 7"):
        scene_io.load_crts(write("view.crts", {"meshes": [{"positions": 7, "indices": 1}], "buffer_views": views}, tri))
    with pytest.raises(RuntimeError, match='has no "indices"'):
        scene_io.load_crts(write("key.crts", {"meshes": [{"positions": 0}], "buffer_views": views}, tri))
    with pytest.raises(RuntimeError, match="Invalid data type string"):
        scene_io.load_crts(write("dtype.crts", {"meshes": [{"positions": 0, "indices": 1}],
                                                "buffer_views": [dict(views[0], type="VEC3_F16"), views[1]]}, tri))
    ok = {"meshes": [{"positions": 0, "indices": 1}], "buffer_views": views}
    with pytest.raises(RuntimeError, match="instances mesh 3 of 1"):
        scene_io.load_crts(write("mesh.crts", dict(ok, objects=[{"type": "MESH", "mesh": 3, "material": 0, "matrix": [0.0] * 16}]), tri))
    with pytest.raises(RuntimeError, match="Unsupported object type"):
        scene_io.load_crts(write("type.crts", dict(ok, objects=[{"type": "EMPTY", "matrix": [0.0] * 16}]), tri))
    with pytest.raises(RuntimeError, match="array of 16 numbers"):
        scene_io.load_crts(write("matrix.crts", dict(ok, objects=[{"type": "MESH", "mesh": 0, "material": 0, "matrix": [1.0] * 12}]), tri))
    img_views = views + [{"byte_offset": 48, "byte_length": 16, "type": "UINT_8"}]
    with pytest.raises(RuntimeError, match="Failed to load wood .*JPEG"):
        scene_io.load_crts(write("image.crts", dict(ok, buffer_views=img_views, images=[{"name": "wood", "view": 2, "color_space": "SRGB"}]),
                                 tri + b"\xff\xd8\xff\xe0JFIF" + bytes(8)))


def test_native_crts_loader_round_trip_and_oracle_frame(built, tmp_path):
    """Without the reference library (the GPU box): the loaded scene renders, through the CPU oracle, the frame of
    crts_io.crts_scene_view(scene) — what Scene::load_crts builds from the file (tests/test_reference_plugin.py pins that)."""
    pytest.importorskip("PIL")
    from chameleonrt_b200 import scene_io
    from chameleonrt_b200.crts_io import crts_scene_view, write_crts
    from chameleonrt_b200.scene import QuadLight
    from helpers import camera_for
    from oracle import OracleBackend

    scene, cam = synthetic_material_scene(spp=1)
    scene.lights = [QuadLight(emission=(12.0, 11.0, 9.0, 1.0), position=(0.5, 4.5, 0.5, 1.0), normal=(0.0, -1.0, 0.0),
                              v_x=(1.0, 0.0, 0.0), width=1.5, v_y=(0.0, 0.0, 1.0), height=1.0)]
    loaded = scene_io.load_scene(write_crts(scene, str(tmp_path / "materials.crts")))
    got = loaded.to_scene(spp=1)
    assert len(got.meshes) == 5 and len(got.instances) == 5 and len(got.textures) == 2
    c = camera_for(cam)
    frames = []
    for s in (crts_scene_view(scene), got):
        o = OracleBackend(max_depth=5)
        o.initialize(48, 32)
        o.set_scene(s)
        o.render(c.eye(), c.dir(), c.up(), cam["fov_y"], True, True)
        frames.append(o.read_accum())
    assert np.array_equal(frames[0].view(np.uint32), frames[1].view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------
# glTF (Scene::load_gltf, util/scene.cpp:230-415 over tinygltf; util/flatten_gltf.cpp)
def _png_bytes(img):
    import io

    from PIL import Image as PILImage

    buf = io.BytesIO()
    mode = {1: "L", 3: "RGB", 4: "RGBA"}[img.shape[2]]
    PILImage.fromarray(img[:, :, 0] if mode == "L" else img, mode).save(buf, format="PNG")
    return buf.getvalue()


def _gltf_hierarchy(tmp_path, container, seed=5):
    """A glTF the way exporters write them: a node hierarchy three levels deep with translation / rotation / scale nodes and
    matrix nodes, meshes instanced from several nodes, an interleaved vertex buffer (byteStride), 16-bit and 32-bit indices,
    accessor byteOffsets, a primitive without material, textures (base colour + metallic-roughness) and a second, unused
    scene. container: "gltf" (external .bin + .png files), "datauri" (everything base64 in the .gltf) or "glb" (one binary
    file, images in buffer views)."""
    import base64
    import json
    import struct

    rng = np.random.default_rng(seed)
    blob = bytearray()
    views, accessors = [], []

    def add_view(raw, stride=None):
        while len(blob) % 4:
            blob.append(0)
        v = {"buffer": 0, "byteOffset": len(blob), "byteLength": len(raw)}
        if stride:
            v["byteStride"] = stride
        views.append(v)
        blob.extend(raw)
        return len(views) - 1

    def add_accessor(view, comp, typ, count, offset=0):
        a = {"bufferView": view, "componentType": comp, "count": count, "type": typ}
        if offset:
            a["byteOffset"] = offset
        accessors.append(a)
        return len(accessors) - 1

    def grid(n):
        xs, ys = np.meshgrid(np.linspace(-1, 1, n), np.linspace(-1, 1, n))
        pos = np.stack([xs.ravel(), ys.ravel(), 0.3 * np.sin(3 * xs.ravel()) * np.cos(2 * ys.ravel())], 1).astype(np.float32)
        uv = np.stack([(xs.ravel() + 1) / 2, (ys.ravel() + 1) / 2], 1).astype(np.float32)
        idx = []
        for j in range(n - 1):
            for i in range(n - 1):
                a = j * n + i
                idx += [a, a + 1, a + n, a + 1, a + n + 1, a + n]
        return pos, uv, np.array(idx, np.uint32)

    prims = []
    # primitive 0: interleaved position / normal / uv (stride 32), 16-bit indices
    pos, uv, idx = grid(7)
    inter = np.zeros((len(pos), 8), np.float32)
    inter[:, 0:3], inter[:, 3:6], inter[:, 6:8] = pos, rng.normal(size=(len(pos), 3)), uv
    v = add_view(inter.tobytes(), stride=32)
    prims.append({"attributes": {"POSITION": add_accessor(v, 5126, "VEC3", len(pos)), "NORMAL": add_accessor(v, 5126, "VEC3", len(pos), 12),
                                 "TEXCOORD_0": add_accessor(v, 5126, "VEC2", len(pos), 24)},
                  "indices": add_accessor(add_view(idx.astype(np.uint16).tobytes() + b"\0\0"), 5123, "SCALAR", len(idx)), "material": 0})
    # primitive 1: packed arrays sharing one view through accessor byteOffsets, 32-bit indices, no uvs, no material
    pos2, _, idx2 = grid(5)
    v = add_view(bytes(8) + pos2.tobytes())
    prims.append({"attributes": {"POSITION": add_accessor(v, 5126, "VEC3", len(pos2), 8)},
                  "indices": add_accessor(add_view(idx2.tobytes()), 5125, "SCALAR", len(idx2)), "mode": 4})
    # primitive 2: packed, uvs, material 1, an index count that is not a multiple of three (the last two are dropped)
    pos3, uv3, idx3 = grid(4)
    prims.append({"attributes": {"POSITION": add_accessor(add_view(pos3.tobytes()), 5126, "VEC3", len(pos3)),
                                 "TEXCOORD_0": add_accessor(add_view(uv3.tobytes()), 5126, "VEC2", len(uv3))},
                  "indices": add_accessor(add_view(np.append(idx3, [0, 1]).astype(np.uint32).tobytes()), 5125, "SCALAR", len(idx3) + 2),
                  "material": 1})
    meshes = [{"primitives": [prims[0], prims[1]], "name": "terrain"}, {"primitives": [prims[2]]}]

    def quat():
        q = rng.normal(size=4)
        return [float(x) for x in q / np.linalg.norm(q)]

    nodes = [
        {"name": "root", "children": [1, 2], "translation": [1.5, -0.25, 3.0]},
        {"name": "arm", "children": [3, 4], "rotation": quat(), "scale": [1.0, 2.0, 0.5], "mesh": 0},
        {"name": "matrix node", "matrix": _rotated(21), "mesh": 1, "children": [5]},
        {"name": "leaf a", "mesh": 1, "translation": [0.1, 0.2, 0.3], "rotation": quat(), "scale": [-1.0, 1.0, 1.0]},
        {"name": "camera holder", "camera": 0, "rotation": quat()},
        {"name": "leaf b", "mesh": 0, "scale": [0.5, 0.5, 0.5]},
        {"name": "second root", "mesh": 0, "rotation": quat()},
        {"name": "not in the scene", "mesh": 1},
    ]
    tex_a = (rng.integers(0, 255, (16, 8, 3))).astype(np.uint8)
    tex_b = (rng.integers(0, 255, (4, 4, 4))).astype(np.uint8)
    pngs = [_png_bytes(tex_a), _png_bytes(tex_b)]
    images = []
    for k, png in enumerate(pngs):
        if container == "gltf":
            (tmp_path / f"tex {k}.png").write_bytes(png)
            images.append({"uri": f"tex%20{k}.png", "name": f"tex{k}"})  # (a percent-encoded file name)
        elif container == "datauri":
            images.append({"uri": "data:image/png;base64," + base64.b64encode(png).decode(), "name": f"tex{k}"})
        else:
            images.append({"bufferView": add_view(png), "mimeType": "image/png", "name": f"tex{k}"})
    doc = {"asset": {"version": "2.0"}, "scene": 1, "scenes": [{"nodes": [7]}, {"nodes": [0, 6], "name": "main"}], "nodes": nodes,
           "cameras": [{"type": "perspective", "perspective": {"yfov": 0.8, "znear": 0.1}}], "meshes": meshes,
           "materials": [{"pbrMetallicRoughness": {"baseColorTexture": {"index": 1}, "baseColorFactor": [1, 0.5, 0.25, 1],
                                                   "metallicRoughnessTexture": {"index": 0}}, "name": "textured"},
                         {"pbrMetallicRoughness": {"metallicFactor": 0.25, "roughnessFactor": 0.6}}, {"name": "all defaults"}],
           "textures": [{"source": 1}, {"source": 0, "sampler": 0}], "samplers": [{}], "images": images,
           "accessors": accessors, "bufferViews": views}
    if container == "gltf":
        (tmp_path / "scene.bin").write_bytes(bytes(blob))
        doc["buffers"] = [{"uri": "scene.bin", "byteLength": len(blob)}]
    elif container == "datauri":
        doc["buffers"] = [{"uri": "data:application/octet-stream;base64," + base64.b64encode(bytes(blob)).decode(), "byteLength": len(blob)}]
    else:
        doc["buffers"] = [{"byteLength": len(blob)}]
    if container != "glb":
        path = tmp_path / "scene.gltf"
        path.write_text(json.dumps(doc))
        return str(path)
    js = json.dumps(doc).encode()
    js += b" " * (-len(js) % 4)
    while len(blob) % 4:
        blob.append(0)
    path = tmp_path / "scene.glb"
    path.write_bytes(struct.pack("<4sII", b"glTF", 2, 12 + 8 + len(js) + 8 + len(blob)) + struct.pack("<II", len(js), 0x4E4F534A) + js +
                     struct.pack("<II", len(blob), 0x004E4942) + bytes(blob))
    return str(path)


@pytest.mark.parametrize("container", ["gltf", "datauri", "glb"])
def test_native_gltf_loader_builds_the_reference_loaders_scene(built, tmp_path, container):
    """Bit for bit what Scene::load_gltf builds through tinygltf + flatten_gltf: geometries (interleaved / offset / 16-bit
    accessors), parameterized meshes with the default material for a primitive without one, the instances of the flattened
    hierarchy (T * R * S and matrix nodes composed in float), materials with texture handles, images (RGBA, not flipped,
    colour spaces set by their use), the generated light."""
    pytest.importorskip("PIL")
    path = _gltf_hierarchy(tmp_path, container)
    ref = _reference_scene(path)
    for threads in (0, 1):
        nat, loaded = _native_arrays(path, threads)
        _assert_same(nat, ref)
    assert nat["counts"] == [2, 2, 2, 5, 4, 2, 1] and nat["mesh_sizes"] == [2, 1]
    assert [cs for _, cs in nat["textures"]] == [1, 0]  # texture 1 -> image 0: base colour (sRGB); texture 0 -> image 1: metallic-roughness
    assert "generating a default" in loaded.warnings


def test_native_gltf_loader_on_the_writers_scene(built, tmp_path):
    """The San-Miguel-like scene of BASELINE configs 3 and 5 as gltf_io writes it (flat node list with matrices, external .bin,
    PNG files)."""
    pytest.importorskip("PIL")
    from chameleonrt_b200.gltf_io import write_gltf
    from chameleonrt_b200.scenes import san_miguel_like

    scene, _ = san_miguel_like(spp=1, scale=0.03, tex_size=32)
    path = write_gltf(scene, str(tmp_path / "scene.gltf"))
    ref = _reference_scene(path)
    nat, loaded = _native_arrays(path)
    _assert_same(nat, ref)
    print(f"\nglTF, {sum(len(g[2]) // 3 for g in nat['geometries'])} unique triangles: reference loader {ref.get('seconds', float('nan')) * 1e3:.1f} ms, "
          f"native {loaded.timings}")


def test_native_gltf_loader_errors(built, tmp_path):
    import json

    from chameleonrt_b200 import scene_io

    def write(name, doc, raw=None):
        p = tmp_path / name
        p.write_bytes(raw if raw is not None else json.dumps(doc).encode())
        return str(p)

    tri = np.zeros(9, np.float32).tobytes() + np.array([0, 1, 2], np.uint32).tobytes()
    (tmp_path / "tri.bin").write_bytes(tri)
    base = {"asset": {"version": "2.0"}, "scenes": [{"nodes": [0]}], "nodes": [{"mesh": 0}], "buffers": [{"uri": "tri.bin", "byteLength": 48}],
            "bufferViews": [{"buffer": 0, "byteLength": 36}, {"buffer": 0, "byteOffset": 36, "byteLength": 12}],
            "accessors": [{"bufferView": 0, "componentType": 5126, "count": 3, "type": "VEC3"},
                          {"bufferView": 1, "componentType": 5125, "count": 3, "type": "SCALAR"}],
            "meshes": [{"primitives": [{"attributes": {"POSITION": 0}, "indices": 1}]}]}
    loaded = scene_io.load_gltf(write("ok.gltf", base))
    assert loaded.c_scene.contents.num_instances == 1 and loaded.c_scene.contents.meshes[0].geometries[0].num_tris == 1

    def broken(**changes):
        doc = json.loads(json.dumps(base))
        for k, v in changes.items():
            doc[k] = v
        return doc

    with pytest.raises(RuntimeError, match="Invalid magic"):
        scene_io.load_scene(write("bad.glb", None, raw=b"not a glb file at all...."))
    with pytest.raises(RuntimeError, match="Too short"):
        scene_io.load_scene(write("short.glb", None, raw=b"glTF"))
    with pytest.raises(RuntimeError, match="malformed JSON"):
        scene_io.load_gltf(write("bad.gltf", None, raw=b"{\"asset\": "))
    with pytest.raises(RuntimeError, match="cannot open"):
        scene_io.load_gltf(write("nobin.gltf", broken(buffers=[{"uri": "missing.bin", "byteLength": 48}])))
    with pytest.raises(RuntimeError, match="byteLength says 480"):
        scene_io.load_gltf(write("shortbin.gltf", broken(buffers=[{"uri": "tri.bin", "byteLength": 480}])))
    with pytest.raises(RuntimeError, match="past the end of its buffer"):
        scene_io.load_gltf(write("view.gltf", broken(bufferViews=[{"buffer": 0, "byteLength": 36}, {"buffer": 0, "byteOffset": 40, "byteLength": 12}])))
    with pytest.raises(RuntimeError, match="past the end of its buffer"):
        scene_io.load_gltf(write("count.gltf", broken(accessors=[{"bufferView": 0, "componentType": 5126, "count": 30, "type": "VEC3"}, base["accessors"][1]])))
    with pytest.raises(RuntimeError, match="POSITION is not FLOAT VEC3"):
        scene_io.load_gltf(write("pos.gltf", broken(accessors=[{"bufferView": 0, "componentType": 5123, "count": 3, "type": "VEC3"}, base["accessors"][1]])))
    with pytest.raises(RuntimeError, match="Unsupported index component type"):
        scene_io.load_gltf(write("idx.gltf", broken(accessors=[base["accessors"][0], {"bufferView": 1, "componentType": 5121, "count": 3, "type": "SCALAR"}])))
    with pytest.raises(RuntimeError, match="Only triangles are supported"):
        scene_io.load_gltf(write("mode.gltf", broken(meshes=[{"primitives": [{"attributes": {"POSITION": 0}, "indices": 1, "mode": 1}]}])))
    with pytest.raises(RuntimeError, match="has no indices"):
        scene_io.load_gltf(write("noidx.gltf", broken(meshes=[{"primitives": [{"attributes": {"POSITION": 0}}]}])))
    with pytest.raises(RuntimeError, match="is sparse"):
        scene_io.load_gltf(write("sparse.gltf", broken(accessors=[dict(base["accessors"][0], sparse={"count": 1}), base["accessors"][1]])))
    with pytest.raises(RuntimeError, match="instances mesh 4 of 1"):
        scene_io.load_gltf(write("mesh.gltf", broken(nodes=[{"mesh": 4}])))
    with pytest.raises(RuntimeError, match="cyclic or too deep"):
        scene_io.load_gltf(write("cycle.gltf", broken(nodes=[{"children": [0], "mesh": 0}])))
    with pytest.raises(RuntimeError, match="JPEG image 0"):  # (a JPEG cut off after its first table)
        scene_io.load_gltf(write("jpeg.gltf", broken(images=[{"uri": "data:image/jpeg;base64,/9j/4AAQSkZJRgABAQAAAQABAAD/2wBDAAgGBgcGBQgHBwcJCQgKDBQNDAsLDBkSEw8UHRofHh0a"}])))
    with pytest.raises(RuntimeError, match="exactly one of"):
        scene_io.load_gltf(write("img.gltf", broken(images=[{"name": "nothing"}])))
    _write_png(str(tmp_path / "deep.png"), np.random.default_rng(0).integers(0, 65536, (4, 4, 3)), 2, 16)
    with pytest.raises(RuntimeError, match="Unsupported image pixel type"):  # (as Scene::load_gltf, scene.cpp:335-338)
        scene_io.load_gltf(write("deep.gltf", broken(images=[{"uri": "deep.png"}])))


def test_native_gltf_loader_round_trip_and_oracle_frame(built, tmp_path):
    """Without the reference library (the GPU box): the scene written by gltf_io comes back as the same scene (write_gltf /
    Scene::load_gltf are inverse to each other for it, tests/test_reference_embree.py) — same frame through the CPU oracle."""
    pytest.importorskip("PIL")
    from chameleonrt_b200 import scene_io
    from chameleonrt_b200.gltf_io import write_gltf
    from chameleonrt_b200.scenes import san_miguel_like
    from helpers import camera_for
    from oracle import OracleBackend

    scene, cam = san_miguel_like(spp=1, scale=0.02, tex_size=32)
    loaded = scene_io.load_scene(write_gltf(scene, str(tmp_path / "scene.gltf")))
    got = loaded.to_scene(spp=1)
    assert len(got.instances) == len(scene.instances) and len(got.materials) == len(scene.materials)
    c = camera_for(cam)
    frames = []
    for s in (scene, got):
        o = OracleBackend(max_depth=5)
        o.initialize(48, 32)
        o.set_scene(s)
        o.render(c.eye(), c.dir(), c.up(), cam["fov_y"], True, True)
        frames.append(o.read_accum())
    assert np.array_equal(frames[0].view(np.uint32), frames[1].view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------
# JPEG textures (chameleonrt_b200/csrc/jpeg_decode.h against stb_image, through the reference's loaders)
def _jpeg_cases(tmp_path):
    """JPEG files as encoders write them: baseline and progressive, 4:4:4 / 4:2:2 / 4:2:0, optimised Huffman tables, restart
    markers, grey images, quality 30 to 100, sizes that are no multiple of the MCU (down to one pixel)."""
    from PIL import Image as PILImage

    rng = np.random.default_rng(0)

    def picture(w, h, kind):
        y, x = np.mgrid[0:h, 0:w]
        if kind == 0:
            img = np.stack([(x * 255 // max(w - 1, 1)), (y * 255 // max(h - 1, 1)), ((x + y) * 7) % 256], 2)
        elif kind == 1:
            img = rng.integers(0, 256, (h, w, 3))
        else:
            img = np.stack([128 + 100 * np.sin(x / 5.0) * np.cos(y / 7.0), 128 + 90 * np.cos(x / 3.0), 128 + 80 * np.sin((x + y) / 9.0)], 2)
        return img.astype(np.uint8)

    options = [dict(quality=75, subsampling=0), dict(quality=90, subsampling=1), dict(quality=50, subsampling=2),
               dict(quality=85, subsampling=2, progressive=True), dict(quality=95, subsampling=0, progressive=True, optimize=True),
               dict(quality=100, subsampling=2, optimize=True), dict(quality=30, subsampling=1, progressive=True),
               dict(quality=80, subsampling=2, restart_marker_blocks=3), dict(quality=80, subsampling=0, progressive=True, restart_marker_rows=1)]
    names = []
    for (w, h) in [(64, 64), (33, 17), (1, 1), (7, 40), (130, 1), (100, 75)]:
        for opts in options:
            names.append(f"t{len(names)}.jpg")
            PILImage.fromarray(picture(w, h, len(names) % 3), "RGB").save(str(tmp_path / names[-1]), format="JPEG", **opts)
        names.append(f"t{len(names)}.jpg")
        PILImage.fromarray(picture(w, h, 2)[:, :, 0], "L").save(str(tmp_path / names[-1]), format="JPEG", quality=80)
        names.append(f"t{len(names)}.jpg")
        PILImage.fromarray(picture(w, h, 1)[:, :, 0], "L").save(str(tmp_path / names[-1]), format="JPEG", quality=60, progressive=True)
    return names


def test_native_jpeg_textures_are_stb_images_bytes(built, tmp_path):
    """OBJ materials with JPEG map_Kd textures (stbi_load, flipped), the same files embedded in a .crts (stbi_load_from_memory,
    flipped) and referenced from a glTF (tinygltf -> stbi_load_from_memory, not flipped): every pixel as stb_image decodes it
    — its integer IDCT, its chroma upsampling filters and its fixed-point YCbCr conversion restated in jpeg_decode.h."""
    pytest.importorskip("PIL")
    import json
    import struct

    names = _jpeg_cases(tmp_path)
    (tmp_path / "tex.mtl").write_text("".join(f"newmtl m{i}\nKd 1 1 1\nmap_Kd {n}\n" for i, n in enumerate(names)))
    (tmp_path / "tex.obj").write_text("mtllib tex.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\n" +
                                      "".join(f"g g{i}\nusemtl m{i}\nf 1/1 2/2 3/3\n" for i in range(len(names))))
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32).tobytes() + np.array([0, 1, 2], np.uint32).tobytes()
    blob = bytearray(tri)
    views = [{"byte_offset": 0, "byte_length": 36, "type": "VEC3_F32"}, {"byte_offset": 36, "byte_length": 12, "type": "VEC3_U32"}]
    images = []
    for n in names[::5]:
        raw = (tmp_path / n).read_bytes()
        views.append({"byte_offset": len(blob), "byte_length": len(raw), "type": "UINT_8"})
        images.append({"name": n, "view": len(views) - 1, "color_space": "SRGB"})
        blob.extend(raw)
    js = json.dumps({"meshes": [{"positions": 0, "indices": 1}], "images": images, "buffer_views": views,
                     "objects": [{"type": "MESH", "mesh": 0, "material": 4294967295, "matrix": _rotated(1)}]}).encode()
    (tmp_path / "tex.crts").write_bytes(struct.pack("<Q", len(js)) + js + bytes(blob))
    (tmp_path / "tri.bin").write_bytes(tri)
    (tmp_path / "tex.gltf").write_text(json.dumps({
        "asset": {"version": "2.0"}, "scenes": [{"nodes": [0]}], "nodes": [{"mesh": 0}], "buffers": [{"uri": "tri.bin", "byteLength": 48}],
        "bufferViews": [{"buffer": 0, "byteLength": 36}, {"buffer": 0, "byteOffset": 36, "byteLength": 12}],
        "accessors": [{"bufferView": 0, "componentType": 5126, "count": 3, "type": "VEC3"}, {"bufferView": 1, "componentType": 5125, "count": 3, "type": "SCALAR"}],
        "meshes": [{"primitives": [{"attributes": {"POSITION": 0}, "indices": 1}]}], "images": [{"uri": n} for n in names[2::5]]}))
    for scene_file, count in (("tex.obj", len(names)), ("tex.crts", len(names[::5])), ("tex.gltf", len(names[2::5]))):
        ref = _reference_scene(str(tmp_path / scene_file))
        nat, _ = _native_arrays(str(tmp_path / scene_file))
        assert len(nat["textures"]) == count
        _assert_same(nat, ref)


def test_native_jpeg_decoder_without_the_reference(built, tmp_path):
    """Properties that hold without stb_image at hand (the GPU box): a flat grey JPEG decodes to its exact level (the DC-only
    path of the IDCT), sizes and the RGBA layout are right, a decoded photo-like image is close to its source, and the bytes
    of one fixed file are pinned by a checksum taken when the decoder agreed with stb_image on it."""
    pytest.importorskip("PIL")
    from PIL import Image as PILImage

    from chameleonrt_b200 import scene_io

    def load(img, mode, **opts):
        PILImage.fromarray(img, mode).save(str(tmp_path / "t.jpg"), format="JPEG", **opts)
        (tmp_path / "t.mtl").write_text("newmtl m\nKd 1 1 1\nmap_Kd t.jpg\n")
        (tmp_path / "t.obj").write_text("mtllib t.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\nusemtl m\nf 1/1 2/2 3/3\n")
        loaded = scene_io.load_obj(str(tmp_path / "t.obj"))
        t = loaded.c_scene.contents.textures[0]
        return np.ctypeslib.as_array(t.data, (t.height, t.width, 4)).copy()

    flat = load(np.full((19, 35), 200, np.uint8), "L", quality=90)
    assert flat.shape == (19, 35, 4) and np.all(flat[..., :3] == 200) and np.all(flat[..., 3] == 255)
    y, x = np.mgrid[0:48, 0:80]
    src = np.stack([128 + 100 * np.sin(x / 9.0), 128 + 90 * np.cos(y / 7.0), 128 + 80 * np.sin((x + y) / 11.0)], 2).astype(np.uint8)
    for opts in (dict(quality=95, subsampling=0), dict(quality=95, subsampling=2, progressive=True)):
        got = load(src, "RGB", **opts)
        assert got.shape == (48, 80, 4)
        assert np.abs(got[::-1, :, :3].astype(int) - src.astype(int)).mean() < 3.0  # (the loader flips rows like stbi)


def test_native_jpeg_decoder_against_committed_stb_output(built):
    """tests/golden/jpeg_*.jpg (baseline 4:2:0, progressive 4:2:2 with optimised tables, 4:4:4 with restart markers, grey)
    against the pixels the reference's stb_image decoded from them (tests/golden/make_jpeg_fixtures.py) — runs anywhere."""
    from chameleonrt_b200 import scene_io

    golden = os.path.join(ROOT, "tests", "golden")
    expected = np.load(os.path.join(golden, "jpeg_expected.npz"))
    loaded = scene_io.load_obj(os.path.join(golden, "jpeg_fixture.obj"))
    s = loaded.c_scene.contents
    assert s.num_textures == len(expected.files) == 4
    for i, name in enumerate(sorted(expected.files)):
        t = s.textures[i]
        got = np.ctypeslib.as_array(t.data, (t.height, t.width, t.channels))
        assert got.shape == expected[name].shape and np.array_equal(got, expected[name]), name


# ---------------------------------------------------------------------------------------------------------------
# PNG in all its variants, TGA
def _write_png(path, samples, color_type, bit_depth, interlace=False, palette=None, trns=None, seed=0):
    """A PNG writer for the variants encoders rarely produce: `samples` (h, w, channels) of integers below 2**bit_depth, any
    colour type / bit depth the format allows, Adam7 interlacing, a random filter type per scanline."""
    import struct
    import zlib

    rng = np.random.default_rng(seed)
    h, w, ch = samples.shape

    def chunk(kind, body):
        return struct.pack(">I", len(body)) + kind + body + struct.pack(">I", zlib.crc32(kind + body) & 0xFFFFFFFF)

    def pack_rows(img):  # (rows, cols, ch) -> (rows, row_bytes) uint8
        rows, cols, _ = img.shape
        if bit_depth == 16:
            return np.stack([(img >> 8) & 255, img & 255], -1).reshape(rows, -1).astype(np.uint8)
        if bit_depth == 8:
            return img.reshape(rows, -1).astype(np.uint8)
        per = 8 // bit_depth
        flat = img.reshape(rows, cols)
        pad = (-cols) % per
        flat = np.concatenate([flat, np.zeros((rows, pad), flat.dtype)], 1).reshape(rows, -1, per)
        shifts = (np.arange(per)[::-1] * bit_depth)
        return (flat << shifts).sum(-1).astype(np.uint8)

    bpp = max(1, ch * bit_depth // 8)

    def filtered(raw):  # raw: (rows, row_bytes)
        out = bytearray()
        prior = np.zeros(raw.shape[1], np.int32)
        for r in raw.astype(np.int32):
            left = np.concatenate([np.zeros(bpp, np.int32), r[:-bpp]]) if len(r) > bpp else np.zeros_like(r)
            upleft = np.concatenate([np.zeros(bpp, np.int32), prior[:-bpp]]) if len(r) > bpp else np.zeros_like(r)
            f = int(rng.integers(0, 5))
            if f == 0:
                enc = r
            elif f == 1:
                enc = r - left
            elif f == 2:
                enc = r - prior
            elif f == 3:
                enc = r - ((left + prior) >> 1)
            else:
                p = left + prior - upleft
                pa, pb, pc = np.abs(p - left), np.abs(p - prior), np.abs(p - upleft)
                enc = r - np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, prior, upleft))
            out.append(f)
            out.extend((enc & 255).astype(np.uint8).tobytes())
            prior = r
        return bytes(out)

    if interlace:
        data = b""
        for x0, y0, dx, dy in zip((0, 4, 0, 2, 0, 1, 0), (0, 0, 4, 0, 2, 0, 1), (8, 8, 4, 4, 2, 2, 1), (8, 8, 8, 4, 4, 2, 2)):
            sub = samples[y0::dy, x0::dx]
            if sub.shape[0] and sub.shape[1]:
                data += filtered(pack_rows(sub))
    else:
        data = filtered(pack_rows(samples))
    png = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, bit_depth, color_type, 0, 0, 1 if interlace else 0))
    if palette is not None:
        png += chunk(b"PLTE", np.asarray(palette).astype(np.uint8).tobytes())
    if trns is not None:
        png += chunk(b"tRNS", np.asarray(trns).astype(np.uint8).tobytes())
    comp = zlib.compress(data, 6)
    half = len(comp) // 2
    png += chunk(b"tEXt", b"Comment\0two IDAT chunks") + chunk(b"IDAT", comp[:half]) + chunk(b"IDAT", comp[half:]) + chunk(b"IEND", b"")
    with open(path, "wb") as f:
        f.write(png)


def _write_tga(path, img, image_type, bpp, top_down=False, rle=False, cmap=None, cmap_bits=24, id_text=b"", seed=0):
    """A TGA writer: `img` (h, w, channels) uint8 in the file's channel order (B, G, R[, A]; grey[, alpha]) — or (h, w) of 16-bit
    pixels / colour-map indices; run-length packets of random lengths when `rle`."""
    import struct

    rng = np.random.default_rng(seed)
    h, w = img.shape[:2]
    px_bytes = (bpp + 7) // 8
    if img.ndim == 2:
        rows = np.stack([(img >> (8 * k)) & 255 for k in range(px_bytes)], -1).astype(np.uint8)
    else:
        rows = img.astype(np.uint8)
    rows = rows if top_down else rows[::-1]
    pixels = rows.reshape(-1, px_bytes)
    body = bytearray()
    if rle:
        i = 0
        while i < len(pixels):
            n = int(min(rng.integers(1, 129), len(pixels) - i))
            if rng.integers(0, 2):
                body.append(0x80 | (n - 1))
                body.extend(pixels[i].tobytes())
                pixels[i:i + n] = pixels[i]  # (what the decoder must produce)
            else:
                body.append(n - 1)
                body.extend(pixels[i:i + n].tobytes())
            i += n
        expected_rows = pixels.reshape(rows.shape)
    header = struct.pack("<BBBHHBHHHHBB", len(id_text), 1 if cmap is not None else 0, image_type + (8 if rle else 0), 0,
                         len(cmap) if cmap is not None else 0, cmap_bits if cmap is not None else 0, 0, 0, w, h, bpp, 0x20 if top_down else 0)
    with open(path, "wb") as f:
        f.write(header + id_text)
        if cmap is not None:
            f.write(np.asarray(cmap).astype(np.uint16 if cmap_bits in (15, 16) else np.uint8).tobytes())
        f.write(bytes(body) if rle else pixels.tobytes())


def _texture_scene(tmp_path, names):
    (tmp_path / "tex.mtl").write_text("".join(f"newmtl m{i}\nKd 1 1 1\nmap_Kd {n}\n" for i, n in enumerate(names)))
    (tmp_path / "tex.obj").write_text("mtllib tex.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\n" +
                                      "".join(f"g g{i}\nusemtl m{i}\nf 1/1 2/2 3/3\n" for i in range(len(names))))
    return str(tmp_path / "tex.obj")


def test_native_png_variants_are_stb_images_bytes(built, tmp_path):
    """Every colour type at every bit depth the format allows (grey 1 / 2 / 4 / 8 / 16, RGB 8 / 16, palette 1 / 2 / 4 / 8,
    grey + alpha and RGBA 8 / 16), with and without Adam7 interlacing, with the tRNS chunk where it applies, all five scanline
    filters, sizes down to 1 x 1 — and what PIL's encoder writes — against stbi_load(..., 4)."""
    rng = np.random.default_rng(3)
    names = []
    for (w, h) in [(1, 1), (5, 3), (9, 17), (33, 8)]:
        for color_type, depths, ch in [(0, (1, 2, 4, 8, 16), 1), (2, (8, 16), 3), (3, (1, 2, 4, 8), 1), (4, (8, 16), 2), (6, (8, 16), 4)]:
            for depth in depths:
                for interlace in (False, True):
                    samples = rng.integers(0, 2 ** depth, (h, w, ch))
                    palette = rng.integers(0, 256, 3 * 2 ** depth) if color_type == 3 else None
                    trns = None
                    if len(names) % 2 == 0:
                        if color_type == 3:
                            trns = rng.integers(0, 256, max(1, 2 ** depth // 2))
                        elif color_type in (0, 2):  # the colour of one of the pixels is the transparent one
                            v = samples[h // 2, w // 2]
                            trns = np.stack([v >> 8, v & 255], -1).reshape(-1)
                    names.append(f"v{len(names)}_{color_type}_{depth}_{int(interlace)}.png")
                    _write_png(str(tmp_path / names[-1]), samples, color_type, depth, interlace, palette, trns, seed=len(names))
    try:
        from PIL import Image as PILImage

        y, x = np.mgrid[0:21, 0:40]
        PILImage.fromarray(((x + y) % 2).astype(bool)).save(str(tmp_path / "pil_1bit.png"))
        PILImage.fromarray((x * 1000 + y * 37).astype(np.uint16)).save(str(tmp_path / "pil_16bit.png"))
        PILImage.fromarray(np.stack([x * 6, y * 12, x + y], 2).astype(np.uint8), "RGB").quantize(16).save(str(tmp_path / "pil_pal.png"), bits=4)
        PILImage.fromarray(np.stack([x * 6, y * 12], 2).astype(np.uint8), "LA").save(str(tmp_path / "pil_la.png"), optimize=True)
        names += ["pil_1bit.png", "pil_16bit.png", "pil_pal.png", "pil_la.png"]
    except ImportError:
        pass
    path = _texture_scene(tmp_path, names)
    ref = _reference_scene(path)
    nat, _ = _native_arrays(path)
    assert len(nat["textures"]) == len(names) >= 112
    for name, a, b in zip(names, _record(nat)["textures"], ref["textures"]):
        assert a == b, name


def test_native_tga_textures_are_stb_images_bytes(built, tmp_path):
    """TGA as stb_image reads it: 24 / 32-bit true colour, 15 / 16-bit (5-5-5), 8-bit grey, 16-bit grey + alpha, colour-mapped
    with 8-bit indices and 24 / 32 / 16-bit map entries, each raw and run-length encoded, bottom-up and top-down, with an
    image id field."""
    rng = np.random.default_rng(4)
    names = []
    for (w, h) in [(1, 1), (13, 7), (40, 9)]:
        for rle in (False, True):
            for top_down in (False, True):
                def add(img, image_type, bpp, **kw):
                    names.append(f"t{len(names)}.tga")
                    _write_tga(str(tmp_path / names[-1]), img, image_type, bpp, top_down=top_down, rle=rle, seed=len(names), **kw)

                add(rng.integers(0, 256, (h, w, 3)), 2, 24)
                add(rng.integers(0, 256, (h, w, 4)), 2, 32, id_text=b"made by a test")
                add(rng.integers(0, 65536, (h, w)), 2, 16)
                add(rng.integers(0, 32768, (h, w)), 2, 15)
                add(rng.integers(0, 256, (h, w, 1)), 3, 8)
                add(rng.integers(0, 256, (h, w, 2)), 3, 16)
                add(rng.integers(0, 20, (h, w, 1)), 1, 8, cmap=rng.integers(0, 256, (16, 3)), cmap_bits=24)  # (indices 16-19: past the map)
                add(rng.integers(0, 8, (h, w, 1)), 1, 8, cmap=rng.integers(0, 256, (8, 4)), cmap_bits=32)
                add(rng.integers(0, 8, (h, w, 1)), 1, 8, cmap=rng.integers(0, 65536, 8), cmap_bits=16)
    path = _texture_scene(tmp_path, names)
    ref = _reference_scene(path)
    nat, _ = _native_arrays(path)
    assert len(nat["textures"]) == len(names) == 108
    for name, a, b in zip(names, _record(nat)["textures"], ref["textures"]):
        assert a == b, name


def test_native_loaders_white_diffuse_material_mode(built, tmp_path):
    """MaterialMode::WHITE_DIFFUSE (main.cpp's -mat-mode white_diffuse) for the three formats: no materials are read (glTF: no
    images either; .crts keeps its images), every geometry ends up with the one default material."""
    pytest.importorskip("PIL")
    from chameleonrt_b200.gltf_io import write_gltf
    from chameleonrt_b200.obj_io import write_obj
    from chameleonrt_b200.scenes import san_miguel_like, sponza_like

    _, crts = _crts_file(tmp_path)
    files = [write_obj(sponza_like(detail=0.25, tex_size=16)[0], str(tmp_path / "sponza.obj")), crts,
             write_gltf(san_miguel_like(spp=1, scale=0.02, tex_size=16)[0], str(tmp_path / "miguel.gltf")), _gltf_hierarchy(tmp_path, "glb")]
    for path in files:
        ref = _reference_scene(path, white_diffuse=True)
        nat, loaded = _native_arrays(path, white_diffuse=True)
        _assert_same(nat, ref)
        assert nat["counts"][4] == 1 and "generating a default" in loaded.warnings
        assert nat["counts"][5] == (2 if path.endswith(".crts") else 0)


@pytest.mark.skipif(not (os.path.exists(REFLIB) and os.path.exists(NATIVE_SHIM_LIB)), reason="oracle/_ref not built (needs /root/reference)")
def test_native_loader_behind_the_references_scene_type(built, tmp_path):
    """backends/cuda/scene_native_load.cpp — `Scene scene = crt_cuda::load_scene_native(file, mode);` in place of main.cpp:186's
    Scene constructor — fills the reference's own Scene struct: compared member by member (texture names included) with the
    constructor's Scene, for the three formats and both material modes."""
    pytest.importorskip("PIL")
    from chameleonrt_b200.obj_io import write_obj
    from chameleonrt_b200.scenes import sponza_like

    _, crts = _crts_file(tmp_path)
    files = [write_obj(sponza_like(detail=0.25, tex_size=16)[0], str(tmp_path / "sponza.obj")), _polygon_obj(str(tmp_path / "poly.obj"), 7, faces=120),
             crts, _gltf_hierarchy(tmp_path, "gltf"), os.path.join(ROOT, "tests", "golden", "jpeg_fixture.obj")]
    for path in files:
        for white in (False, True):
            ref = _reference_scene(path, white, lib_path=REFLIB)
            shim = _reference_scene(path, white, lib_path=NATIVE_SHIM_LIB)
            _assert_same(shim, ref)
            assert shim["texture_names"] == ref["texture_names"], path


def test_native_obj_loader_texture_statements(built, tmp_path):
    """map_Kd as tinyobjloader's ParseTextureNameAndOption reads it: texture options with their arguments in front of the name, a
    file name with blanks in it (the name is the rest of the line), the same file named by two materials (one texture), a
    backslash path (canonicalize_path)."""
    pytest.importorskip("PIL")
    from PIL import Image as PILImage

    rng = np.random.default_rng(2)
    (tmp_path / "sub").mkdir()
    for name in ("plain.png", "with blank.png", "sub/deep.png"):
        PILImage.fromarray(rng.integers(0, 256, (6, 9, 3)).astype(np.uint8)).save(str(tmp_path / name))
    (tmp_path / "m.mtl").write_text("newmtl a\nKd 1 1 1\nmap_Kd -blendu on -s 2 2 1 -o 0.5 0 0 -mm 0 1 -bm 0.3 -clamp off plain.png\n"
                                    "newmtl b\nmap_Kd with blank.png  \nnewmtl c\nmap_Kd   sub\\deep.png\r\nnewmtl d\nmap_Kd -colorspace sRGB plain.png\n"
                                    "newmtl e\nmap_Kd -imfchan r -type sphere -boost 2 -t 1 1 1 with blank.png\n")
    (tmp_path / "m.obj").write_text("mtllib m.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\n" +
                                    "".join(f"g g{k}\nusemtl {k}\nf 1/1 2/2 3/3\n" for k in "abcde"))
    ref = _reference_scene(str(tmp_path / "m.obj"))
    nat, _ = _native_arrays(str(tmp_path / "m.obj"))
    _assert_same(nat, ref)
    assert nat["counts"][4] == 5 and nat["counts"][5] == 3


def _random_obj_text(rng, nfaces=30):
    """A random OBJ file in the spelling real exporters and hand-edited files use: blanks and tabs in any amount, CRLF or LF,
    numbers as fixed / exponent / integer / leading-dot / trailing-dot, positions with 2 to 6 components (w, vertex colours),
    texture coordinates with 1 to 3, absolute and relative indices, v / v/t / v//n / v/t/n corners, faces of 3 to 5 corners,
    g (several names) / o / s / usemtl / mtllib statements anywhere, statements the loaders ignore, comments, empty lines."""
    lines=[]
    nv=nvt=nvn=0
    def ws(): return rng.choice([" ", "  ", "\t", " \t "])
    def num():
        k=rng.integers(0,8)
        x=rng.normal()*10.0**int(rng.integers(-3,4))
        if k==0: return f"{x:.6f}"
        if k==1: return f"{x:.3e}"
        if k==2: return f"{int(x)}"
        if k==3: return f"{x:+.4f}"
        if k==4: return f"{x:.10g}"
        if k==5: return f"{x:.2E}"
        if k==6: return f".{rng.integers(0,1000)}"
        return f"{int(x)}."
    if rng.integers(0,2): lines.append("mtllib"+ws()+"fz.mtl")
    mats=["red","green","blue shade","nomat"]
    file_vt=rng.integers(0,2)
    for f in range(nfaces):
        r=rng.integers(0,20)
        if r==0: lines.append("# comment "+num())
        if r==1: lines.append("")
        if r==2: lines.append("g"+ws()+" ".join(rng.choice(["a","b","c_d","e1"], rng.integers(1,3))))
        if r==3: lines.append("o"+ws()+"obj"+str(f))
        if r==4: lines.append("usemtl"+ws()+str(rng.choice(mats)))
        if r==5: lines.append("s"+ws()+str(rng.choice(["off","1","0","3"])))
        if r==6: lines.append(rng.choice(["vp 0.1 0.2","l 1 2","p 1","mg 1 0.5","cstype bezier","g"]))
        if r==7: lines.append("usemtl"+ws()+str(rng.choice(mats))+("  " if rng.integers(0,2) else ""))
        n=int(rng.integers(3,6)) if rng.integers(0,4)==0 else 3
        for k in range(n):
            comps=[num() for _ in range(int(rng.choice([3,3,3,4,6,2])))]
            lines.append((ws() if rng.integers(0,6)==0 else "")+"v"+ws()+ws().join(comps)); nv+=1
        has_vt=file_vt; has_vn=rng.integers(0,2)
        if has_vt:
            for k in range(n):
                lines.append("vt"+ws()+ws().join(num() for _ in range(int(rng.choice([2,2,3,1]))))); nvt+=1
        if has_vn:
            for k in range(n):
                lines.append("vn"+ws()+ws().join(num() for _ in range(3))); nvn+=1
        corners=[]
        rel=rng.integers(0,2)
        for k in range(n):
            v = (k-n) if rel else nv-n+k+1
            vt= (k-n) if rel else nvt-n+k+1
            vn= (k-n) if rel else nvn-n+k+1
            if has_vt and has_vn: c=f"{v}/{vt}/{vn}"
            elif has_vt: c=f"{v}/{vt}"
            elif has_vn: c=f"{v}//{vn}"
            else: c=f"{v}"
            corners.append(c)
        lines.append("f"+ws()+ws().join(corners)+(ws() if rng.integers(0,4)==0 else ""))
    eol = "\r\n" if rng.integers(0,3)==0 else "\n"
    text=eol.join(lines)+(eol if rng.integers(0,4) else "")
    return text


def test_native_obj_loader_differential_fuzz(built, tmp_path):
    """Random OBJ files through both loaders: the same Scene, array for array, or an error from both. (One spelling is left
    out: a `g` statement followed only by blanks — the reference's loader crashes on it, this one reads an unnamed group.)"""
    (tmp_path / "fz.mtl").write_text("newmtl red\nKd 0.8 0.1 0.1\nNs 200\nnewmtl green\n  Kd 0.1 .8 1e-1\nNs 5e2\n\nnewmtl blue shade\nKd 0 0 1\nd 0.5\n"
                                     "illum 2\nKa 1 1 1\n")
    path = str(tmp_path / "f.obj")
    loaded_ok = 0
    for seed in range(int(os.environ.get("CRT_OBJ_FUZZ_FILES", "60"))):
        rng = np.random.default_rng(seed)
        with open(path, "w", newline="") as f:
            f.write(_random_obj_text(rng, int(rng.integers(1, 40))))
        ref = _reference_scene(path)
        try:
            nat, _ = _native_arrays(path, threads=1 + seed % 3)
        except RuntimeError:
            nat = None
        assert (nat is None) == bool(ref.get("refused")), f"seed {seed}: one loader accepts the file, the other does not"
        if nat is not None:
            _assert_same(nat, ref)
            loaded_ok += 1
    assert loaded_ok >= 40


def test_native_mtl_reader_differential_fuzz(built, tmp_path):
    """Random material files through both loaders: statements in any spelling (Kd with 1 to 4 numbers, Ns, map_Kd with and
    without options and with blanks in the name, indented statements, comments, statements that do not matter, look-alikes such
    as Kdx / map_Kdx), material names with blanks and trailing blanks, names defined twice (the first definition is the one a
    usemtl finds), a usemtl of a name no file defines. (`Tr` next to `d` is left out: the reference's reader crashes on it.)"""
    pytest.importorskip("PIL")
    from PIL import Image as PILImage

    for n in ("a.png", "b c.png"):
        PILImage.fromarray(np.random.default_rng(1).integers(0, 256, (4, 4, 3)).astype(np.uint8)).save(str(tmp_path / n))

    def ws(rng):
        return str(rng.choice([" ", "  ", "\t", " \t "]))

    def num(rng):
        x = rng.normal() * 10.0 ** int(rng.integers(-2, 4))
        return [f"{x:.4f}", f"{x:.2e}", f"{int(x)}", f"{abs(x):.3f}", f".{rng.integers(0, 99)}"][rng.integers(0, 5)]

    ignored = ["Ka 1 1 1", "Ks 0.5 0.5 0.5", "d 0.5", "illum 2", "Ni 1.5", "map_Bump a.png", "Ke 1 1 1", "Pr 0.5", "Kdx 1 1 1", "map_Kdx a.png", "Nsx 1"]
    path = str(tmp_path / "f.obj")
    for seed in range(int(os.environ.get("CRT_MTL_FUZZ_FILES", "80"))):
        rng = np.random.default_rng(seed)
        lines, names = [], []
        for _ in range(int(rng.integers(1, 6))):
            names.append(str(rng.choice(["red", "green", "blue shade", "x", "red"])))
            lines.append((ws(rng) if rng.integers(0, 4) == 0 else "") + "newmtl" + ws(rng) + names[-1] + ("  " if rng.integers(0, 3) == 0 else ""))
            for _ in range(int(rng.integers(0, 7))):
                r = rng.integers(0, 12)
                if r == 0:
                    lines.append("Kd" + ws(rng) + ws(rng).join(num(rng) for _ in range(int(rng.choice([3, 3, 1, 2, 4])))))
                elif r == 1:
                    lines.append("Ns" + ws(rng) + num(rng))
                elif r == 2:
                    lines.append("map_Kd" + ws(rng) + str(rng.choice(["a.png", "b c.png", "-s 1 1 1 a.png", "-clamp on b c.png"])))
                elif r == 3:
                    lines.append(str(rng.choice(["# c", "", "\tKd 0.5 0.25 0.125"])))
                elif r == 4:
                    lines.append(str(rng.choice(ignored)))
        (tmp_path / "f.mtl").write_text("\n".join(lines) + ("\n" if rng.integers(0, 3) else ""))
        (tmp_path / "f.obj").write_text("mtllib f.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\n" +
                                        "".join(f"g g{i}\nusemtl {n}\nf 1/1 2/2 3/3\n" for i, n in enumerate(names + ["zzz"])))
        nat, _ = _native_arrays(path)
        _assert_same(nat, _reference_scene(path))


def _random_gltf(rng, d):
    """A random glTF 2.0 scene: 1-3 meshes of 1-3 primitives (interleaved / packed / offset accessors, 16- or 32-bit indices whose
    count need not be a multiple of three, with and without uvs and materials), up to 8 nodes in a random forest with matrix,
    T / R / S (any subset; quaternions not always normalised, negative scales) or both, camera nodes, one or two scenes, written
    as .gltf + .bin, as .gltf with a data: URI, or as .glb."""
    import base64
    import json
    import struct

    blob=bytearray(); views=[]; accessors=[]
    def add_view(raw, stride=None, align=4):
        while len(blob)%align: blob.append(0)
        v={"buffer":0,"byteOffset":len(blob),"byteLength":len(raw)}
        if stride: v["byteStride"]=stride
        if rng.integers(0,3)==0: v["target"]=34962
        views.append(v); blob.extend(raw); return len(views)-1
    def acc(view,comp,typ,count,offset=0):
        a={"bufferView":view,"componentType":comp,"count":count,"type":typ}
        if offset or rng.integers(0,4)==0: a["byteOffset"]=offset
        accessors.append(a); return len(accessors)-1
    meshes=[]
    for m in range(int(rng.integers(1,4))):
        prims=[]
        for p in range(int(rng.integers(1,4))):
            n=int(rng.integers(3,12)); ntri=int(rng.integers(1,8))
            pos=rng.normal(size=(n,3)).astype(np.float32); uv=rng.uniform(size=(n,2)).astype(np.float32)
            idx=rng.integers(0,n,ntri*3+int(rng.integers(0,3)))
            layout=int(rng.integers(0,3)); attrs={}
            has_uv=bool(rng.integers(0,2))
            if layout==0:  # interleaved
                stride=int(rng.choice([20,24,32]))
                inter=np.zeros((n,stride//4),np.float32); inter[:,0:3]=pos; inter[:,3:5]=uv
                v=add_view(inter.tobytes(),stride)
                attrs["POSITION"]=acc(v,5126,"VEC3",n)
                if has_uv: attrs["TEXCOORD_0"]=acc(v,5126,"VEC2",n,12)
            elif layout==1:  # packed separate
                attrs["POSITION"]=acc(add_view(pos.tobytes()),5126,"VEC3",n)
                if has_uv: attrs["TEXCOORD_0"]=acc(add_view(uv.tobytes()),5126,"VEC2",n)
            else:  # one view, accessor offsets, possibly misaligned start (2 mod 4 is not allowed by gltf but tinygltf reads it)
                pad=int(rng.choice([0,4,8]))
                v=add_view(bytes(pad)+pos.tobytes()+uv.tobytes())
                attrs["POSITION"]=acc(v,5126,"VEC3",n,pad)
                if has_uv: attrs["TEXCOORD_0"]=acc(v,5126,"VEC2",n,pad+12*n)
            if rng.integers(0,2):
                ia=acc(add_view(idx.astype(np.uint16).tobytes(),align=2),5123,"SCALAR",len(idx))
            else:
                ia=acc(add_view(idx.astype(np.uint32).tobytes()),5125,"SCALAR",len(idx))
            prim={"attributes":attrs,"indices":ia}
            if rng.integers(0,3): prim["material"]=int(rng.integers(0,3))
            if rng.integers(0,3)==0: prim["mode"]=4
            prims.append(prim)
        meshes.append({"primitives":prims})
    def quat():
        q=rng.normal(size=4)
        if rng.integers(0,3): q=q/np.linalg.norm(q)
        return [float(x) for x in q]
    nn=int(rng.integers(1,9)); nodes=[]
    for i in range(nn):
        node={}
        if rng.integers(0,4): node["mesh"]=int(rng.integers(0,len(meshes)))
        k=rng.integers(0,5)
        if k==0: node["matrix"]=_rotated(int(rng.integers(0,1000)))
        if k in (1,2):
            if rng.integers(0,2): node["translation"]=[float(x) for x in rng.normal(size=3)]
            if rng.integers(0,2): node["rotation"]=quat()
            if rng.integers(0,2): node["scale"]=[float(x) for x in rng.uniform(-2,2,3)]
        if k==3: node["matrix"]=_rotated(int(rng.integers(0,1000))); node["translation"]=[1.0,2.0,3.0]
        if rng.integers(0,5)==0: node["camera"]=0
        nodes.append(node)
    # children: node i may have children among later nodes (tree)
    parent={}
    roots=[]
    for i in range(nn):
        if i>0 and rng.integers(0,2):
            par=int(rng.integers(0,i)); nodes[par].setdefault("children",[]).append(i); parent[i]=par
        else: roots.append(i)
    scenes=[{"nodes":roots}]
    doc={"asset":{"version":"2.0"},"scenes":scenes,"nodes":nodes,"meshes":meshes,"accessors":accessors,"bufferViews":views,
         "cameras":[{"type":"perspective","perspective":{"yfov":0.8,"znear":0.1}}],
         "materials":[{"pbrMetallicRoughness":{"baseColorFactor":[float(x) for x in rng.uniform(size=4)],"metallicFactor":float(rng.uniform())}},
                      {"pbrMetallicRoughness":{"roughnessFactor":float(rng.uniform())}}, {}]}
    if rng.integers(0,2): doc["scene"]=0
    if rng.integers(0,3)==0:
        doc["scenes"].insert(0,{"nodes":[roots[0]]}); doc["scene"]=1
    kind=int(rng.integers(0,3))
    if kind==0:
        open(f'{d}/s.bin','wb').write(bytes(blob)); doc["buffers"]=[{"uri":"s.bin","byteLength":len(blob)}]
        p=f'{d}/s.gltf'; open(p,'w').write(json.dumps(doc)); return p
    if kind==1:
        doc["buffers"]=[{"uri":"data:application/octet-stream;base64,"+base64.b64encode(bytes(blob)).decode(),"byteLength":len(blob)}]
        p=f'{d}/s.gltf'; open(p,'w').write(json.dumps(doc, indent=int(rng.integers(0,3)) or None)); return p
    doc["buffers"]=[{"byteLength":len(blob)}]
    js=json.dumps(doc).encode(); js+=b" "*(-len(js)%4)
    while len(blob)%4: blob.append(0)
    p=f'{d}/s.glb'
    open(p,'wb').write(struct.pack("<4sII",b"glTF",2,12+8+len(js)+8+len(blob))+struct.pack("<II",len(js),0x4E4F534A)+js+struct.pack("<II",len(blob),0x004E4942)+bytes(blob))
    return p


def test_native_gltf_loader_differential_fuzz(built, tmp_path):
    """Random glTF scenes through both loaders: the same Scene — geometry arrays, parameterized meshes, materials and, above
    all, the instance transforms the flattening of the node hierarchy computes in float."""
    for seed in range(int(os.environ.get("CRT_GLTF_FUZZ_FILES", "60"))):
        path = _random_gltf(np.random.default_rng(seed), str(tmp_path))
        nat, _ = _native_arrays(path, threads=1 + seed % 2)
        _assert_same(nat, _reference_scene(path))


_CRTS_PARAMS = ["metallic","specular","roughness","specular_tint","anisotropic","sheen","sheen_tint","clearcoat","clearcoat_roughness","ior","transmission"]
def _crts_number_text(rng):
    k=rng.integers(0,9); x=rng.normal()*10.0**int(rng.integers(-3,4))
    return [f"{x:.6f}",f"{x:.3e}",f"{int(x)}",f"{x:.17g}",f"{abs(int(x))}",f"{x:.2E}","0","-0.0","1e-40"][k]
def _random_crts(rng, d):
    """A random .crts file: 1-3 meshes (indices typed VEC3_U32 or UINT_32, with and without texcoords), 0-2 embedded PNG images,
    0-3 materials with numbers in every JSON spelling (fixed, exponent, integer, 17 digits, -0.0, a float32 denormal) and random
    texture handles, 1-7 MESH / LIGHT / CAMERA objects with arbitrary matrices, a padded or unpadded header."""
    import json
    import re
    import struct

    blob=bytearray(); views=[]
    def view(raw,typ,align=8):
        while len(blob)%align: blob.append(0)
        views.append({"byte_offset":len(blob),"byte_length":len(raw),"type":typ}); blob.extend(raw); return len(views)-1
    meshes=[]
    for m in range(int(rng.integers(1,4))):
        n=int(rng.integers(3,10)); nt=int(rng.integers(1,6))
        e={"positions":view(rng.normal(size=(n,3)).astype(np.float32).tobytes(),"VEC3_F32"),
           "indices":view(rng.integers(0,n,(nt,3)).astype(np.uint32).tobytes(), str(rng.choice(["VEC3_U32","UINT_32"])))}
        if rng.integers(0,2): e["texcoords"]=view(rng.uniform(size=(n,2)).astype(np.float32).tobytes(),"VEC2_F32")
        meshes.append(e)
    images=[]
    for i in range(int(rng.integers(0,3))):
        png=_png_bytes(rng.integers(0,256,(int(rng.integers(1,6)),int(rng.integers(1,6)),int(rng.choice([1,3,4])))).astype(np.uint8))
        images.append({"name":f"img {i}","view":view(png,"UINT_8",align=1),"color_space":str(rng.choice(["SRGB","LINEAR","srgb"]))})
    nmat=int(rng.integers(0,4)); mats=[]
    for i in range(nmat):
        jm={"base_color":"@[%s, %s, %s]"%(_crts_number_text(rng),_crts_number_text(rng),_crts_number_text(rng))}
        if images and rng.integers(0,2): jm["base_color_texture"]=int(rng.integers(0,len(images)))
        for pn in _CRTS_PARAMS:
            jm[pn]="@"+_crts_number_text(rng)
            if images and rng.integers(0,5)==0: jm[pn+"_texture"]={"texture":int(rng.integers(0,len(images))),"channel":int(rng.integers(0,4))}
        mats.append(jm)
    objs=[]
    for i in range(int(rng.integers(1,8))):
        k=rng.integers(0,6)
        mat="@["+", ".join(_crts_number_text(rng) for _ in range(16))+"]"
        if k<4: objs.append({"type":"MESH","mesh":int(rng.integers(0,len(meshes))),"material":int(rng.integers(0,nmat)) if nmat and rng.integers(0,4) else 4294967295,"matrix":mat})
        elif k==4: objs.append({"type":"LIGHT","color":"@[%s, %s, %s]"%(_crts_number_text(rng),_crts_number_text(rng),_crts_number_text(rng)),"energy":"@"+_crts_number_text(rng),"size":"@[%s, %s]"%(_crts_number_text(rng),_crts_number_text(rng)),"matrix":mat})
        else: objs.append({"type":"CAMERA","fov_y":"@"+_crts_number_text(rng),"matrix":mat})
    hdr={"meshes":meshes,"images":images,"materials":mats,"objects":objs,"buffer_views":views}
    js=json.dumps(hdr, indent=int(rng.integers(0,3)) or None)
    # "@..." strings become raw number text
    js = re.sub(r'"@([^"]*)"', lambda m: m.group(1), js)
    js=js.encode()
    if rng.integers(0,2): js+=b" "*((-(len(js)+8))%8)
    p=f'{d}/s.crts'
    open(p,'wb').write(struct.pack("<Q",len(js))+js+bytes(blob))
    return p


def test_native_crts_loader_differential_fuzz(built, tmp_path):
    """Random .crts files through both loaders: the same Scene (numbers through the JSON reader and the float casts, material
    handles, (mesh, material) pairs, light and camera frames)."""
    pytest.importorskip("PIL")
    for seed in range(int(os.environ.get("CRT_CRTS_FUZZ_FILES", "60"))):
        path = _random_crts(np.random.default_rng(seed), str(tmp_path))
        nat, _ = _native_arrays(path)
        _assert_same(nat, _reference_scene(path))


def test_native_png_decoder_refuses_what_stb_image_refuses(built, tmp_path):
    """Structurally wrong PNG files (stbi__parse_png_file's checks): a tRNS chunk in an image with alpha, of the wrong length,
    longer than the palette, before the palette or after the data; a palette image without palette; a palette of a length that
    is no multiple of three; an unknown critical chunk; a second header; no data — each refused by both loaders, while the
    untouched file and harmless variations (an unknown ancillary chunk, a wrong CRC) load to the same pixels."""
    import struct
    import zlib

    rng = np.random.default_rng(5)

    def chunk(kind, body, crc_ok=True):
        return struct.pack(">I", len(body)) + kind + body + struct.pack(">I", (zlib.crc32(kind + body) & 0xFFFFFFFF) ^ (0 if crc_ok else 0x5a5a))

    def png(color_type, depth, chunks_before_idat=(), chunks_after_idat=(), palette=None, idat=True, header_twice=False, ihdr_tail=(0, 0, 0)):
        ch = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[color_type]
        w, h = 5, 4
        raw = b"".join(b"\0" + bytes(rng.integers(0, 2 ** min(depth, 8) if color_type != 3 else 4, (w * ch * depth + 7) // 8, dtype=np.uint8)) for _ in range(h))
        out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, color_type, *ihdr_tail))
        if header_twice:
            out += chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, color_type, 0, 0, 0))
        if palette is not None:
            out += chunk(b"PLTE", bytes(palette))
        for c in chunks_before_idat:
            out += c
        if idat:
            out += chunk(b"IDAT", zlib.compress(raw))
        for c in chunks_after_idat:
            out += c
        return out + chunk(b"IEND", b"")

    pal = list(rng.integers(0, 256, 12))
    cases = {
        "ok_rgb": (png(2, 8), True), "ok_pal": (png(3, 8, palette=pal), True), "ok_pal_trns": (png(3, 8, [chunk(b"tRNS", bytes([1, 2, 3]))], palette=pal), True),
        "ok_ancillary": (png(2, 8, [chunk(b"teSt", b"hello")]), True), "ok_bad_crc": (png(2, 8, [chunk(b"teXt", b"hello", crc_ok=False)]), True),
        "trns_with_alpha": (png(6, 8, [chunk(b"tRNS", bytes(6))]), False), "trns_short": (png(2, 8, [chunk(b"tRNS", bytes(2))]), False),
        "trns_long_grey": (png(0, 8, [chunk(b"tRNS", bytes(6))]), False), "trns_longer_than_palette": (png(3, 8, [chunk(b"tRNS", bytes(5))], palette=pal), False),
        "trns_after_idat": (png(2, 8, (), [chunk(b"tRNS", bytes(6))]), False), "no_palette": (png(3, 8), False),
        "palette_length": (png(3, 8, palette=pal[:11]), False), "critical_chunk": (png(2, 8, [chunk(b"TEST", b"x")]), False),
        "two_headers": (png(2, 8, header_twice=True), False), "no_idat": (png(2, 8, idat=False), False),
        "compression_method": (png(2, 8, ihdr_tail=(1, 0, 0)), False), "filter_method": (png(2, 8, ihdr_tail=(0, 1, 0)), False),
        "interlace_method": (png(2, 8, ihdr_tail=(0, 0, 2)), False), "palette_16_bit": (png(3, 16, palette=pal), False), "colour_type_5": (png(5, 8) if False else None, False),
    }
    from chameleonrt_b200 import scene_io

    for name, (data, should_load) in cases.items():
        if data is None:
            continue
        (tmp_path / f"{name}.png").write_bytes(data)
        path = _texture_scene(tmp_path, [f"{name}.png"])
        ref = _reference_scene(path)
        assert (not ref.get("refused")) == should_load, f"{name}: the reference {'refuses' if ref.get('refused') else 'loads'} it"
        if should_load:
            nat, _ = _native_arrays(path)
            assert _record(nat)["textures"][0] == ref["textures"][0], name
        else:
            with pytest.raises(RuntimeError):
                scene_io.load_scene(path)


def _write_bmp(path, rows, bpp, header=40, top_down=False, masks=None, palette=None, compression=None, gap=0):
    """A BMP writer for the variants of the format: `rows` (h, w) of pixel values (palette indices, or packed 16 / 32-bit pixels)
    or (h, w, 3 / 4) of B, G, R[, A] bytes; header = 12 (OS/2 core), 40 (info), 56, 108 (V4) or 124 (V5); bit-field masks;
    `gap` unused bytes between the headers and the pixel data."""
    import struct

    rows = np.asarray(rows)
    h, w = rows.shape[:2]
    if rows.ndim == 3:
        raw_rows = [bytes(rows[y].astype(np.uint8).tobytes()) for y in range(h)]
    elif bpp in (16, 32):
        raw_rows = [rows[y].astype("<u2" if bpp == 16 else "<u4").tobytes() for y in range(h)]
    elif bpp == 8:
        raw_rows = [rows[y].astype(np.uint8).tobytes() for y in range(h)]
    else:
        per = 8 // bpp
        raw_rows = []
        for y in range(h):
            r = np.concatenate([rows[y], np.zeros((-w) % per, rows.dtype)]).reshape(-1, per)
            raw_rows.append(bytes((r << (np.arange(per)[::-1] * bpp)).sum(1).astype(np.uint8)))
    raw_rows = [r + bytes((-len(r)) % 4) for r in raw_rows]
    if not top_down:
        raw_rows = raw_rows[::-1]
    pal = b""
    if palette is not None:
        pal = b"".join(bytes([c[2], c[1], c[0]] + ([] if header == 12 else [0])) for c in palette)
    compression = (3 if masks and header == 40 else 0) if compression is None else compression
    if header == 12:
        info = struct.pack("<IHHHH", 12, w, h, 1, bpp)
    else:
        info = struct.pack("<IiiHHIIiiII", header, w, -h if top_down else h, 1, bpp, compression, 0, 2835, 2835, 0, 0)
        if header == 40 and masks:
            info += struct.pack("<III", *masks[:3])
        elif header >= 56:
            m = list(masks) + [0] * (4 - len(masks)) if masks else [0, 0, 0, 0]
            info += struct.pack("<IIII", *m)
            info += bytes(header - 56)
            if header == 56 and compression == 3:
                info += struct.pack("<III", *m[:3])  # (stb_image skips the mask fields of a 56-byte header and reads three masks behind it)
    offset = 14 + len(info) + len(pal) + gap
    data = b"".join(raw_rows)
    with open(path, "wb") as f:
        f.write(b"BM" + struct.pack("<IHHI", offset + len(data), 0, 0, offset) + info + pal + bytes(gap) + data)


def test_native_bmp_textures_are_stb_images_bytes(built, tmp_path):
    """BMP as stb_image reads it: 24-bit, 32-bit BGRA (with alpha, and with an all-zero alpha channel, which counts as opaque),
    32- and 16-bit with bit-field masks of 1 to 8 bits per channel in info / V4 / V5 headers, 16-bit 5-5-5, 8 / 4 / 1-bit palettes,
    the OS/2 core header, bottom-up and top-down rows, widths that need row padding, a gap before the pixel data — plus PIL's files."""
    rng = np.random.default_rng(6)
    names = []

    def add(*args, **kw):
        names.append(f"b{len(names)}.bmp")
        _write_bmp(str(tmp_path / names[-1]), *args, **kw)

    for (w, h) in [(1, 1), (5, 3), (14, 9), (33, 4)]:
        for top_down in (False, True):
            add(rng.integers(0, 256, (h, w, 3)), 24, top_down=top_down)
            add(rng.integers(0, 256, (h, w, 4)), 32, top_down=top_down)
            add(np.concatenate([rng.integers(0, 256, (h, w, 3)), np.zeros((h, w, 1), int)], 2), 32, top_down=top_down)  # alpha all 0
            add(rng.integers(0, 2 ** 32, (h, w), dtype=np.uint64), 32, masks=(0x00FF0000, 0x0000FF00, 0x000000FF), top_down=top_down)
            add(rng.integers(0, 2 ** 32, (h, w), dtype=np.uint64), 32, header=108, masks=(0x000000FF, 0x0000FF00, 0x00FF0000, 0xFF000000), top_down=top_down)
            add(rng.integers(0, 2 ** 32, (h, w), dtype=np.uint64), 32, header=124, masks=(0xF8000000, 0x07E00000, 0x001F0000, 0x0000000F), top_down=top_down)
            add(rng.integers(0, 2 ** 16, (h, w)), 16, top_down=top_down)
            add(rng.integers(0, 2 ** 16, (h, w)), 16, masks=(0xF800, 0x07E0, 0x001F), top_down=top_down)
            add(rng.integers(0, 2 ** 16, (h, w)), 16, header=56, masks=(0x0F00, 0x00F0, 0x000F, 0xF000), compression=3, top_down=top_down)
            add(rng.integers(0, 2 ** 16, (h, w)), 16, header=108, masks=(0x7000, 0x0380, 0x0003, 0x8000), compression=3, top_down=top_down)
            add(rng.integers(0, 256, (h, w)), 8, palette=rng.integers(0, 256, (256, 3)), top_down=top_down)
            add(rng.integers(0, 16, (h, w)), 4, palette=rng.integers(0, 256, (16, 3)), top_down=top_down, gap=0)
            add(rng.integers(0, 2, (h, w)), 1, palette=rng.integers(0, 256, (2, 3)), top_down=top_down)
            add(rng.integers(0, 7, (h, w)), 8, palette=rng.integers(0, 256, (7, 3)), header=108, top_down=top_down, gap=8)
        add(rng.integers(0, 256, (h, w, 3)), 24, header=12)
        # (stb_image counts the palette of a core-header file from offset - 38: of 256 entries it reads 252; the rest is uninitialised there)
        add(rng.integers(0, 252, (h, w)), 8, header=12, palette=rng.integers(0, 256, (256, 3)))
    names = [n for n in names if os.path.exists(tmp_path / n)]
    try:
        from PIL import Image as PILImage

        y, x = np.mgrid[0:13, 0:22]
        rgb = np.stack([x * 11, y * 19, x + y], 2).astype(np.uint8)
        PILImage.fromarray(rgb, "RGB").save(str(tmp_path / "pil_rgb.bmp"))
        PILImage.fromarray(rgb[:, :, 0], "L").save(str(tmp_path / "pil_l.bmp"))
        PILImage.fromarray(rgb, "RGB").quantize(16).save(str(tmp_path / "pil_p.bmp"))
        PILImage.fromarray(((x + y) % 2).astype(bool)).save(str(tmp_path / "pil_1.bmp"))
        PILImage.fromarray(np.dstack([rgb, (x * 9).astype(np.uint8)]), "RGBA").save(str(tmp_path / "pil_rgba.bmp"))
        names += ["pil_rgb.bmp", "pil_l.bmp", "pil_p.bmp", "pil_1.bmp", "pil_rgba.bmp"]
    except ImportError:
        pass
    path = _texture_scene(tmp_path, names)
    ref = _reference_scene(path)
    nat, _ = _native_arrays(path)
    assert len(nat["textures"]) == len(names) >= 120
    for name, a, b in zip(names, _record(nat)["textures"], ref["textures"]):
        assert a == b, name
