"""Shared test helpers: scenes, the host-check binding, the parity metric and the recorded results of the reference."""
import ctypes as C
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Parity tolerance for the accumulated float framebuffer (stated per BASELINE.json north_star):
# a pixel matches when every channel satisfies |gpu - oracle| <= ABS_TOL + REL_TOL * |oracle|.
# Differences come only from libm-vs-CUDA transcendental rounding (sin/cos/pow/log/atan2/acos,
# <= 2 ulp) and, for spp > 1, the per-sample summation order; a handful of pixels differ more
# because a last-bit change in a sampled direction flips a discrete event (a ray grazing an
# edge). Hence a fraction threshold, plus a bound on the whole-image relative L1 error.
ABS_TOL = 1e-4
REL_TOL = 1e-3
MIN_MATCH_FRACTION = 0.999
MAX_REL_L1 = 2e-3


def digest(*arrays):
    """Short fingerprint of arrays (dtype, shape and bytes): bit-exact comparison with a result stored as text."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()[:16]


def reference_result(table, key, compute=None):
    """What the reference computed for `key`. compute() runs the reference's own code, where its binaries are built
    (oracle/_ref/); pass None where they are not, and the result recorded in tests/golden/<table> is returned. A live result
    must equal the recorded one, so that the table keeps what the reference computes. With CRT_RECORD_REFERENCE=1, every live
    result is written into the table instead (how the table is regenerated)."""
    path = os.path.join(ROOT, "tests", "golden", table)
    recs = {}
    if os.path.exists(path):
        with open(path) as f:
            recs = json.load(f)
    if compute is None:
        assert key in recs, f"{key}: no recorded result of the reference in tests/golden/{table} (the input has changed?)"
        return recs[key]
    rec = json.loads(json.dumps(compute()))  # (as stored: lists for tuples)
    if os.environ.get("CRT_RECORD_REFERENCE") != "1":
        assert key in recs, f"{key}: no recorded result of the reference in tests/golden/{table}; record it with CRT_RECORD_REFERENCE=1"
        assert rec == recs[key], f"{key}: the reference's result differs from the one recorded in tests/golden/{table}"
    else:
        recs[key] = rec
        with open(path, "w") as f:  # one record per line
            f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(recs[k], separators=(',', ':'))}" for k in sorted(recs)) + "\n}\n")
    return rec


def parity(gpu_accum, ref_accum):
    """(fraction of matching pixels, relative L1 over the pixels finite in both). The reference's
    transmission lobe can produce NaN ("need to debug the transmissive materials",
    util/scene.cpp:196); a pixel that is non-finite in the oracle must be non-finite on the GPU."""
    g, r = gpu_accum.astype(np.float64), ref_accum.astype(np.float64)
    fin_g, fin_r = np.isfinite(g).all(axis=-1), np.isfinite(r).all(axis=-1)
    both = fin_g & fin_r
    d = np.abs(np.where(both[..., None], g - r, 0.0))
    ok = (d <= ABS_TOL + REL_TOL * np.abs(np.where(both[..., None], r, 0.0))).all(axis=-1)
    ok = np.where(both, ok, fin_g == fin_r)
    rel_l1 = d.sum() / max(1e-12, np.abs(r[both]).sum())
    return float(ok.mean()), float(rel_l1)


def assert_parity(gpu_accum, ref_accum, min_frac=MIN_MATCH_FRACTION, max_rel_l1=MAX_REL_L1):
    assert np.isfinite(gpu_accum).all() or not np.isfinite(ref_accum).all(), "GPU produced non-finite pixels the oracle does not"
    frac, rel_l1 = parity(gpu_accum, ref_accum)
    assert frac >= min_frac, f"only {frac:.5f} of pixels within tolerance (rel_l1={rel_l1:.3e})"
    assert rel_l1 <= max_rel_l1, f"relative L1 {rel_l1:.3e} too large (frac={frac:.5f})"
    return frac, rel_l1


class HostCheck:
    """ctypes binding of the TEST-ONLY libcrt_bvh8_hostcheck.so (host instantiation of the
    product's BVH8 builder + traversal)."""

    def __init__(self, scene, threads=0):
        from chameleonrt_b200.scene import CScene

        lib = C.CDLL(os.path.join(ROOT, "chameleonrt_b200", "csrc", "libcrt_bvh8_hostcheck.so"))
        lib.crt_hostcheck_create.restype = C.c_void_p
        lib.crt_hostcheck_create.argtypes = [C.POINTER(CScene), C.c_int]
        lib.crt_hostcheck_destroy.argtypes = [C.c_void_p]
        lib.crt_hostcheck_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crt_hostcheck_stats.argtypes = [C.c_void_p, C.c_void_p]
        lib.crt_hostcheck_last_error.restype = C.c_char_p
        lib.crt_hostcheck_digest.restype = C.c_uint64
        lib.crt_hostcheck_digest.argtypes = [C.c_void_p]
        self.lib = lib
        ms = scene.to_c()
        self.h = lib.crt_hostcheck_create(C.byref(ms.c), threads)
        if not self.h:
            raise RuntimeError(lib.crt_hostcheck_last_error().decode())

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.crt_hostcheck_destroy(self.h)
            self.h = None

    def stats(self):
        a = (C.c_double * 5)()
        self.lib.crt_hostcheck_stats(self.h, a)
        return dict(nodes=int(a[0]), tris=int(a[1]), depth=int(a[2]), sah=a[3], build_ms=a[4])

    def digest(self) -> int:
        return int(self.lib.crt_hostcheck_digest(self.h))

    def trace(self, rays, any_hit=False, normals=False, counters=False, far_first=False):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        n = len(rays)
        hits = np.zeros((n, 4), np.float32)
        nrm = np.zeros((n, 3), np.float32) if normals else None
        cnt = np.zeros((n, 2), np.uint32) if counters else None
        self.lib.crt_hostcheck_trace(self.h, rays.ctypes.data, n, (2 if far_first else 1) if any_hit else 0, hits.ctypes.data,
                                     nrm.ctypes.data if normals else None, cnt.ctypes.data if counters else None)
        return hits, nrm, cnt


def bounce_rays(rays, hits, seed=1):
    """Incoherent secondary rays leaving the hit points of ``rays`` (tnear = 1e-4)."""
    rng = np.random.default_rng(seed)
    hit = hits[:, 3].view(np.uint32) != 0xFFFFFFFF
    p = rays[:, :3] + hits[:, :1] * rays[:, 4:7]
    d = rng.normal(size=(len(rays), 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    out = np.concatenate([p, np.full((len(rays), 1), 1e-4, np.float32), d, np.full((len(rays), 1), 1e20, np.float32)], 1)
    return np.ascontiguousarray(out[hit], np.float32)


def camera_for(cam):
    from chameleonrt_b200 import ArcballCamera

    return ArcballCamera(cam["eye"], cam["center"], cam["up"])


def synthetic_material_scene(spp=1):
    """Small scene exercising every BSDF lobe incl. transmission, anisotropy, clearcoat, sheen and
    textured scalar parameters (the .crts-only features of SURVEY App. A #9)."""
    from chameleonrt_b200.scene import (LINEAR, SRGB, DisneyMaterial, Geometry, Image, Instance, Mesh,
                                        ParameterizedMesh, Scene, default_obj_light, textured_param)
    from chameleonrt_b200.scenes import MeshBuilder, box, grid, make_texture, sphere

    textures = [Image("albedo", make_texture("tiles", 3, 64), SRGB), Image("mr", make_texture("stone", 5, 32), LINEAR)]
    mats = [
        DisneyMaterial(base_color=(textured_param(0), 0.5, 0.5), roughness=0.6, specular=0.4),
        DisneyMaterial(base_color=(0.9, 0.9, 0.95), roughness=0.15, specular_transmission=0.9, ior=1.45, specular=0.5),
        DisneyMaterial(base_color=(0.9, 0.6, 0.2), metallic=0.9, roughness=0.3, anisotropy=0.7, specular=0.6),
        DisneyMaterial(base_color=(0.2, 0.3, 0.8), roughness=0.5, clearcoat=1.0, clearcoat_gloss=0.8, sheen=0.8,
                       sheen_tint=0.5, specular_tint=0.6, specular=0.5),
        DisneyMaterial(base_color=(0.7, 0.7, 0.7), metallic=textured_param(1, 2), roughness=textured_param(1, 1)),
    ]
    geoms = []
    b = MeshBuilder(); b.add(*grid((-3, 0, -3), (0, 0, 6), (6, 0, 0), 4, 4, (3, 3))); geoms.append(b.geometry())
    b = MeshBuilder(); b.add(*sphere((-1.2, 0.8, 0.0), 0.8, 24, 16)); geoms.append(b.geometry())
    b = MeshBuilder(); b.add(*sphere((0.9, 0.7, 0.6), 0.7, 24, 16)); geoms.append(b.geometry())
    b = MeshBuilder()
    for part in box((-0.4, 0.0, -2.0), (0.6, 1.4, -1.2), (2, 2, 2)):
        b.add(*part)
    geoms.append(b.geometry())
    b = MeshBuilder(); b.add(*grid((-3, 0, -3), (6, 0, 0), (0, 3, 0), 4, 2, (2, 1))); geoms.append(b.geometry())
    scene = Scene(meshes=[Mesh(geoms)], parameterized_meshes=[ParameterizedMesh(0, [0, 1, 2, 3, 4])],
                  instances=[Instance(np.eye(4, dtype=np.float32), 0)], materials=mats, textures=textures,
                  lights=[default_obj_light()], samples_per_pixel=spp)
    cam = dict(eye=(0.3, 1.6, 4.2), center=(0.0, 0.6, 0.0), up=(0.0, 1.0, 0.0), fov_y=50.0)
    return scene, cam
