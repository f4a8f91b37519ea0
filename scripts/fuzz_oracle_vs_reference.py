"""Randomised comparison of the CPU oracle with the reference's own Embree backend build
(oracle/_ref/libcrt_embree.so): random triangle soups + structured pieces, every Disney parameter random
(including textured scalar parameters and transmission), random textures, several instances with random
affine transforms (also mirrored / sheared), random lights, cameras, spp, depth, frame counts and ragged
framebuffer sizes. Any difference in the float framebuffer, the per-pixel ray counts or the sRGB8 image is
printed with the seed that reproduces it. CPU only.   python scripts/fuzz_oracle_vs_reference.py [n] [first_seed]
"""
import os
import sys
import warnings

import numpy as np

warnings.filterwarnings("ignore")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from chameleonrt_b200 import ArcballCamera  # noqa: E402
from chameleonrt_b200.scene import (LINEAR, SRGB, DisneyMaterial, Geometry, Image, Instance, Mesh, ParameterizedMesh,  # noqa: E402
                                    QuadLight, Scene, textured_param)
from chameleonrt_b200.scenes import MeshBuilder, box, grid, sphere  # noqa: E402
from oracle import OracleBackend  # noqa: E402
from oracle.ref_embree import RefEmbreeBackend  # noqa: E402


def random_scene(rng):
    ntex = int(rng.integers(0, 4))
    textures = [Image(f"t{i}", rng.integers(0, 256, size=(int(rng.integers(1, 9)), int(rng.integers(1, 9)), int(rng.choice([3, 4]))),
                                             dtype=np.uint8), int(rng.choice([LINEAR, SRGB]))) for i in range(ntex)]

    def param(lo=0.0, hi=1.0):
        if ntex and rng.random() < 0.2:
            t = int(rng.integers(0, ntex))
            # a channel the texture has (the reference's loaders always deliver RGBA; reading channel 3 of an
            # RGB image would read the next texel's red, texture2d.ih:32-34)
            return textured_param(t, int(rng.integers(0, textures[t].channels)))
        return float(np.float32(rng.uniform(lo, hi)))

    mats = []
    for _ in range(int(rng.integers(1, 6))):
        bc0 = textured_param(int(rng.integers(0, ntex))) if ntex and rng.random() < 0.3 else float(np.float32(rng.random()))
        mats.append(DisneyMaterial(base_color=(bc0, float(np.float32(rng.random())), float(np.float32(rng.random()))),
                                   metallic=param(), specular=param(), roughness=param(), specular_tint=param(),
                                   anisotropy=param() if rng.random() < 0.5 else 0.0, sheen=param(), sheen_tint=param(),
                                   clearcoat=param(), clearcoat_gloss=param(), ior=param(1.0, 2.0),
                                   specular_transmission=param() if rng.random() < 0.3 else 0.0))
    meshes, pms, instances = [], [], []
    for _ in range(int(rng.integers(1, 4))):
        geoms = []
        for _ in range(int(rng.integers(1, 4))):
            b = MeshBuilder()
            kind = rng.integers(0, 4)
            if kind == 0:
                n = int(rng.integers(1, 200))
                v = (rng.normal(size=(n, 3, 3)) * rng.uniform(0.05, 1.5) + rng.normal(size=(n, 1, 3)) * 2.0).astype(np.float32)
                b.add(v.reshape(-1, 3), rng.random((3 * n, 2)).astype(np.float32), np.arange(3 * n, dtype=np.uint32).reshape(-1, 3))
            elif kind == 1:
                b.add(*grid(tuple(rng.uniform(-3, 3, 3)), tuple(rng.uniform(-4, 4, 3)), tuple(rng.uniform(-4, 4, 3)),
                            int(rng.integers(1, 9)), int(rng.integers(1, 9)), (2, 2)))
            elif kind == 2:
                b.add(*sphere(tuple(rng.uniform(-2, 2, 3)), float(rng.uniform(0.3, 1.5)), int(rng.integers(3, 12)), int(rng.integers(2, 8))))
            else:
                lo = rng.uniform(-3, 2, 3)
                for part in box(tuple(lo), tuple(lo + rng.uniform(0.2, 2.5, 3)), (1, 1, 1)):
                    b.add(*part)
            g = b.geometry()
            if rng.random() < 0.25:
                g.uvs = None  # geometries without texture coordinates sample textures at uv = (0, 0)
            geoms.append(g)
        meshes.append(Mesh(geoms))
    for _ in range(int(rng.integers(1, 5))):
        mid = int(rng.integers(0, len(meshes)))
        pms.append(ParameterizedMesh(mid, [int(rng.integers(0, len(mats))) for _ in meshes[mid].geometries]))
        t = np.eye(4, dtype=np.float32)
        if rng.random() < 0.7:
            t[:3, :3] = (np.eye(3) + rng.normal(scale=0.5, size=(3, 3))).astype(np.float32)  # shear / mirror / scale
            t[:3, 3] = rng.uniform(-3, 3, 3).astype(np.float32)
        instances.append(Instance(t, len(pms) - 1))
    lights = []
    for _ in range(int(rng.integers(1, 3))):
        n = rng.normal(size=3)
        n /= np.linalg.norm(n)
        a = np.cross(n, rng.normal(size=3))
        a /= np.linalg.norm(a)
        bb = np.cross(n, a)
        e = rng.uniform(2, 30, 3)
        lights.append(QuadLight(emission=(float(e[0]), float(e[1]), float(e[2]), 1.0), position=tuple(float(x) for x in rng.uniform(-6, 6, 3)) + (1.0,),
                                normal=tuple(float(np.float32(x)) for x in n), v_x=tuple(float(np.float32(x)) for x in a),
                                width=float(rng.uniform(0.2, 4)), v_y=tuple(float(np.float32(x)) for x in bb), height=float(rng.uniform(0.2, 4))))
    return Scene(meshes=meshes, parameterized_meshes=pms, instances=instances, materials=mats, textures=textures, lights=lights,
                 samples_per_pixel=int(rng.integers(1, 4)))


def case(seed):
    """The random scene, framebuffer size, depth, frame count, camera and field of view of one seed."""
    rng = np.random.default_rng(seed)
    scene = random_scene(rng)
    w, h, depth, frames = int(rng.integers(8, 90)), int(rng.integers(8, 80)), int(rng.integers(1, 9)), int(rng.integers(1, 4))
    eye = rng.uniform(-9, 9, 3)
    cam = ArcballCamera(tuple(eye), tuple(rng.uniform(-1, 1, 3)), (0.0, 1.0, 0.0))
    fov = float(rng.uniform(20, 90))
    return scene, w, h, depth, frames, cam, fov


def render(backend, c):
    """Renders case c on a fresh backend; returns it."""
    scene, w, h, depth, frames, cam, fov = c
    backend.initialize(w, h)
    backend.set_scene(scene)
    for f in range(frames):
        backend.render(cam.eye(), cam.dir(), cam.up(), fov, f == 0, True)
    return backend


def one(seed):
    c = case(seed)
    scene, w, h, depth, frames = c[:5]
    ref, cpu = render(RefEmbreeBackend(max_depth=depth), c), render(OracleBackend(max_depth=depth), c)
    a, b = ref.read_accum(), cpu.read_accum()
    same = np.array_equal(a.view(np.uint32), b.view(np.uint32)) or bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())
    same_rays = np.array_equal(ref.read_ray_stats(), cpu.read_ray_stats())
    same_img = np.array_equal(ref.img, cpu.img)
    return same and same_rays and same_img, (same, same_rays, same_img, scene.total_tris(), w, h, depth, frames, int(np.isnan(a).any()))


if __name__ == "__main__":
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 100
    first = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    bad = 0
    nan_scenes = 0
    for seed in range(first, first + n):
        ok, info = one(seed)
        nan_scenes += info[-1]
        if not ok:
            bad += 1
            print("MISMATCH seed", seed, info)
    print(f"{n} random scenes, {bad} mismatches, {nan_scenes} scenes with NaN pixels (in both)")
