#!/usr/bin/env python
"""bench.py — MRays/s and ms/frame of the per-frame render path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          # the CUDA wavefront backend
  python bench.py --impl reference --gpus N ...           # the CPU path (oracle), rank 0 only
  python bench.py ... --dump-outputs DIR                  # also write the last timed step's outputs to DIR/*.npy

A "step" is one frame: one pass of the hot path (raygen -> [closest-hit traversal -> shade ->
any-hit traversal -> NEE resolve] x depth -> resolve/tonemap) over the whole image at the
configured samples per pixel. Workload = BASELINE.json configs[1]: Sponza-class OBJ scene
(seeded procedural stand-in, the asset is not on the box), 1280x720, 4 spp, max depth 8.

N > 1 (torchrun, one process per GPU): the image's 64x64 tiles are sharded round-robin across
ranks (scene + BVH replicated), every rank renders its tiles with no communication, and the
accumulated tiles are gathered to rank 0 over NCCL/NVLink at frame end, inside the timed
region. Total work is fixed, so scaling is "strong".

One JSON line on stdout (rank 0). Keys follow the driver contract; `roofline` describes
k_traverse, `cpu_baseline` the CPU oracle timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# BASELINE.json configs. The default (what the driver runs) is configs[1] = "c2"; c3 / c4 are the
# HBM-resident stress cases and are run by hand (results under profiles/).
WORKLOADS = {
    # configs[0] is the reference's own CPU-runnable plumbing case; here for completeness (a 34-triangle scene says
    # nothing about a GPU)
    "c1": dict(name="C1 cornell_box OBJ-class scene (34 tris), 512x512, 1 spp, max depth 5", gen="cornell_box", kw={}, w=512, h=512,
               spp=1, depth=5),
    "c2": dict(name="C2 sponza_like OBJ-class scene (263,792 tris, 25 materials, 8 sRGB 1024^2 textures), "
                    "1280x720, 4 spp, max depth 8", gen="sponza_like", kw={}, w=1280, h=720, spp=4, depth=8),
    "c3": dict(name="C3 san_miguel_like glTF-class scene (10.5 M instanced tris, 961 instances, 100 materials, "
                    "11 textures), 1920x1080, 8 spp, max depth 8", gen="san_miguel_like", kw={}, w=1920, h=1080, spp=8, depth=8),
    "c4": dict(name="C4 rungholt_like OBJ-class voxel city (6.7 M tris, 80 untextured materials), "
                    "1920x1080, 4 spp, max depth 8", gen="rungholt_like", kw={"scale": 1.24}, w=1920, h=1080, spp=4, depth=8),
    "c5": dict(name="C5 san_miguel_like glTF-class scene (10.5 M instanced tris), 3840x2160, 8 spp per step (64 spp accumulated "
                    "after 8 steps), max depth 8; meant for --gpus 8", gen="san_miguel_like", kw={}, w=3840, h=2160, spp=8, depth=8),
    # not a benchmark: a frame small enough for the CPU emulation of the renderer, used by tests/test_bench_contract.py
    # to dry-run this file's GPU arm where no GPU exists
    "dev": dict(name="DEV cornell_box, 128x48, 1 spp, max depth 5 (dry run, not a benchmark)", gen="cornell_box", kw={}, w=128, h=48,
                spp=1, depth=5),
}
WORKLOAD = WORKLOADS["c2"]["name"]
WIDTH, HEIGHT, SPP, MAX_DEPTH = 1280, 720, 4, 8
S_NODE, S_TRI, S_RAY, S_HIT = 80, 48, 32, 16  # algorithmic bytes, SURVEY.md §8d / DESIGN.md §5


def select_workload(key: str) -> None:
    global WORKLOAD, WIDTH, HEIGHT, SPP, MAX_DEPTH, _GEN
    w = WORKLOADS[key]
    WORKLOAD, WIDTH, HEIGHT, SPP, MAX_DEPTH = w["name"], w["w"], w["h"], w["spp"], w["depth"]
    _GEN = (w["gen"], w["kw"])


_GEN = ("sponza_like", {})


def make_workload():
    from chameleonrt_b200 import ArcballCamera
    from chameleonrt_b200 import scenes

    scene, cam = getattr(scenes, _GEN[0])(spp=SPP, **_GEN[1])
    camera = ArcballCamera(cam["eye"], cam["center"], cam["up"])
    return scene, (camera.eye(), camera.dir(), camera.up(), cam["fov_y"])


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons while the timed region runs."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thread.join(timeout=10)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_budget():
    """What this process may actually use: the affinity mask says how many cores it may be scheduled ON, a cgroup CPU
    quota (cpu.max, or cfs_quota_us / cfs_period_us under cgroup v1) says how much CPU TIME it gets — round 1's
    reference arm reported "128 cores" on two boxes whose frames took 1964 ms and 369 ms (VERDICT r1, weak #1)."""
    out = {"affinity_cores": cpu_cores(), "os_cpu_count": os.cpu_count(), "cgroup_quota_cores": None}
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        out["cgroup_quota_cores"] = None if quota == "max" else float(quota) / float(period)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            pr = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            out["cgroup_quota_cores"] = None if q <= 0 else q / pr
        except Exception:
            pass
    try:
        import re

        m = re.search(r"model name\s*:\s*(.+)", open("/proc/cpuinfo").read())
        out["cpu_model"] = m.group(1).strip() if m else None
    except Exception:
        out["cpu_model"] = None
    return out


class CpuMeter:
    """CPU time this process (all threads) spent inside the block / wall time = the cores it really had."""

    def __enter__(self):
        import resource

        ru = resource.getrusage(resource.RUSAGE_SELF)
        self._cpu0, self._t0 = ru.ru_utime + ru.ru_stime, time.perf_counter()
        return self

    def __exit__(self, *a):
        import resource

        ru = resource.getrusage(resource.RUSAGE_SELF)
        self.cpu_s = ru.ru_utime + ru.ru_stime - self._cpu0
        self.wall_s = time.perf_counter() - self._t0
        self.effective_cores = self.cpu_s / max(1e-9, self.wall_s)


CPU_ARM_LABEL = ("scalar C++ build of the reference's ISPC kernel over a stand-in 4-wide BVH (NOT Embree + ISPC SIMD: a real "
                 "Embree/ISPC build would be several times faster)")


def describe_cpu_arm(value, meter, threads):
    b = cpu_budget()
    eff = meter.effective_cores
    return {"cores": b["affinity_cores"], "threads_spawned": threads, "effective_cores": round(eff, 1),
            "cgroup_quota_cores": b["cgroup_quota_cores"], "cpu_model": b["cpu_model"],
            "mrays_per_effective_core": value / max(1e-9, eff), "label": CPU_ARM_LABEL}


def cpu_reference_backend():
    """The CPU implementation of the path that is timed beside the GPU. Where the reference's own Embree
    backend was compiled (oracle/_ref/libcrt_embree_fast.so: /root/reference/backends/embree sources, ISPC
    kernels as scalar C++, Embree/TBB replaced by stand-ins; oracle/ref_build/Makefile) that is used and the
    kind is "reference"; otherwise the oracle port. Both render bit-identical frames in their strict builds
    (tests/test_reference_embree.py); these are the -O3 builds of each."""
    from oracle import ref_embree

    if ref_embree.available(fast=True) and os.environ.get("CRT_BENCH_CPU", "reference") != "port":
        return (ref_embree.RefEmbreeBackend(max_depth=MAX_DEPTH, fast=True), "reference",
                "the reference's backends/embree sources (render_embree.cpp + render_embree.ispc/.ih compiled as "
                "scalar C++, -O3 x86-64-v3; Embree replaced by an own 4-wide BVH, TBB by std::thread), all host threads")
    from oracle import OracleBackend

    return (OracleBackend(max_depth=MAX_DEPTH, fast=True), "port",
            "CPU oracle = Embree/ISPC backend restated with an own BVH2, -O3 x86-64-v3, all host threads")


def time_oracle(scene, view, budget_s: float, frames_cap: int):
    """Times the CPU implementation (all host threads) on the workload; returns per-frame list."""
    cpu, kind, desc = cpu_reference_backend()
    cpu.initialize(WIDTH, HEIGHT)
    cpu.set_scene(scene)
    results = []
    t0 = time.time()
    f = 0
    with CpuMeter() as meter:
        while True:
            st = cpu.render(*view, f == 0, True)
            results.append((st.render_time, st.num_rays))
            f += 1
            if f >= frames_cap or (time.time() - t0) > budget_s:
                break
    return results, kind, desc, meter


def run_reference_arm(args):
    """--impl reference: the CPU implementation of the path on this box's host cores, with every host
    thread: the reference's own Embree backend sources where they were compiled (oracle/_ref, prebuilt for
    the GPU box), else the oracle port (cpu_reference_backend)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    scene, view = make_workload()
    budget_s = float(os.environ.get("CRT_BENCH_REF_BUDGET", "240"))
    cpu, kind, desc = cpu_reference_backend()
    cpu.initialize(WIDTH, HEIGHT)
    cpu.set_scene(scene)
    # probe: one full frame. Each step is a full frame of the workload when K + W of them fit the
    # budget on this box's cores; otherwise a step keeps every pixel and takes fewer samples per pixel
    # (same rays, same scene, same depth: MRays/s is unchanged in meaning, the sample is smaller).
    t0 = time.time()
    cpu.render(*view, True, True)
    probe_s = time.time() - t0
    spp_step = SPP
    est = probe_s * (args.steps + args.warmup)
    if est > budget_s and SPP > 1:
        spp_step = max(1, int(SPP * budget_s / est))
        scene.samples_per_pixel = spp_step
        # a fresh backend: the reference's set_scene appends to its material/texture tables
        # (render_embree.cpp:106-131), it is meant to be called once per renderer
        cpu, kind, desc = cpu_reference_backend()
        cpu.initialize(WIDTH, HEIGHT)
        cpu.set_scene(scene)
    f = 0
    for _ in range(args.warmup):
        cpu.render(*view, f == 0, True)
        f += 1
    rays, ms = 0, 0.0
    with CpuMeter() as meter:
        for _ in range(args.steps):
            st = cpu.render(*view, f == 0, True)
            f += 1
            rays += st.num_rays
            ms += st.render_time
    if args.dump_outputs:
        # (a step keeps the workload's spp only where the frames fit CRT_BENCH_REF_BUDGET on this host, see above: with
        # fewer, the outputs differ accordingly)
        dump_outputs(args.dump_outputs, cpu.read_accum(), cpu.img, int(st.num_rays))
    value = rays / (ms * 1e3)
    cores = cpu_cores()
    line = {
        "impl": "reference", "metric": "MRays/s", "value": value, "unit": "MRays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "width": WIDTH, "height": HEIGHT, "spp": SPP, "max_depth": MAX_DEPTH},
        "cpu_baseline": {"value": value, "unit": "MRays/s", "kind": kind,
                         **describe_cpu_arm(value, meter, os.cpu_count()),
                         "sample": f"{args.steps} frames of the workload at {spp_step} of {SPP} spp per step after 1 "
                                   f"probe + {args.warmup} warm-up frames; {desc}"},
        "e2e": {"value": value, "unit": "MRays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_set_scene_probe() -> None:
    """Sub-process of the N=1 run (`--probe-set-scene`): crtc_set_scene of the bench scene with the BVH8 built on the
    host (binned SAH, the default and what the timed region renders over) and on the device (bvh8_device.cuh, SURVEY.md
    §8(f) rank 1), wall-clock around the call, then two frames over each tree: they must be bit-identical, and the
    instrumented counters tell what the faster build costs in traversal work. Its own process, so that a fault in
    the newer device builder cannot take the bench line with it."""
    import time

    import numpy as np

    from chameleonrt_b200 import RenderCUDA

    scene, view = make_workload()
    out, frames = {}, {}
    for builder in ("host", "device"):
        r = RenderCUDA(0, max_depth=MAX_DEPTH, bvh_builder=builder, count_traversal=True, any_far_first=0)
        r.initialize(WIDTH, HEIGHT)
        t0 = time.perf_counter()
        r.set_scene(scene)
        wall = (time.perf_counter() - t0) * 1e3
        for f in range(2):
            r.render(*view, f == 0, False)
        info, c, st = r.scene_info(), r.counters(), r.stage_times()
        out[builder] = {"set_scene_ms": wall, "bvh_build_ms": info["bvh_build_ms"],
                        "phases_ms": {k: round(info[k + "_ms"], 3) for k in ("flatten", "sort", "tree", "emit", "pack")},
                        "ploc_rounds": int(info["ploc_rounds"]), "bvh8_nodes": int(info["bvh8_nodes"]),
                        "bvh8_depth": int(info["bvh8_depth"]),
                        "closest_nodes_per_ray": c["closest_nodes_visited"] / max(1, c["closest_rays"]),
                        "any_hit_nodes_per_ray": c["any_nodes_visited"] / max(1, c["occlusion_rays"]),
                        "traverse_ms_instrumented": st["traverse"] + st["traverse_primary"]}
        frames[builder] = r.read_accum()
        del r
    out["triangles"] = int(info["triangles"])
    out["frames_bit_identical"] = bool(np.array_equal(frames["host"].view(np.uint32), frames["device"].view(np.uint32)))
    emit(out)


def set_scene_probe(workload_key: str):
    """Runs run_set_scene_probe() in a child process; returns its dict, or {"error": ...}."""
    import subprocess

    try:
        # (CRT_BENCH_PROBE_SCRIPT: tests/test_bench_contract.py dry-runs this through its own launcher)
        script = os.environ.get("CRT_BENCH_PROBE_SCRIPT", os.path.abspath(__file__))
        p = subprocess.run([sys.executable, script, "--probe-set-scene", "--workload", workload_key],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=int(os.environ.get("CRT_BENCH_PROBE_TIMEOUT", "240")))
        if p.returncode != 0:
            return {"error": f"exit code {p.returncode}: " + p.stderr.decode(errors="replace").strip().splitlines()[-1][:300]}
        return json.loads(p.stdout.decode().strip().splitlines()[-1])
    except Exception as e:  # timeout, unparsable output
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def kernel_source_sha():
    """Fingerprint of the traversal kernel's source: a measured DRAM-traffic figure is only quoted next to the kernel it
    was captured from."""
    import hashlib

    h = hashlib.sha256()
    for name in ("kernels.cuh", "bvh8_traverse.h"):
        with open(os.path.join(ROOT, "chameleonrt_b200", "csrc", name), "rb") as fsrc:
            h.update(fsrc.read())
    return h.hexdigest()[:16]


def measured_traffic(workload_key):
    """dram__bytes_read + dram__bytes_write per k_traverse launch from the committed ncu capture of THIS
    workload (profiles/traffic_k_traverse.json, written by scripts/update_traffic.py from the .ncu-rep): returned only
    if the capture was taken from the kernel source that is in the tree now; otherwise null and the reason."""
    path = os.path.join(ROOT, "profiles", "traffic_k_traverse.json")
    try:
        entry = json.load(open(path))["workloads"][workload_key]
    except Exception:
        return None, "no committed ncu capture of this workload"
    if entry.get("kernel_src_sha") != kernel_source_sha():
        return None, f"stale: the committed capture ({entry.get('capture')}) is of an older k_traverse"
    return entry["dram_bytes_per_launch"], (f"mean over the {entry['launches']} k_traverse launches of one frame, ncu dram__bytes_read + "
                                            f"dram__bytes_write, {entry.get('capture')}")


def run_workload_probe(args) -> None:
    """Sub-process of the N=1 run (`--probe-workload --workload cX`): a short measurement of another BASELINE
    configuration — the HBM-resident scenes, where the traversal's DRAM traffic is real — with the same method as the
    main line (W warm-up frames, instrumented counting pass, K frames enqueued back to back, CUDA events)."""
    import torch

    from chameleonrt_b200 import RenderCUDA

    steps, warm = args.steps, max(3, args.warmup)
    scene, view = make_workload()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    t0 = time.perf_counter()
    gpu = RenderCUDA(0, max_depth=MAX_DEPTH, stream=stream.cuda_stream)
    gpu.initialize(WIDTH, HEIGHT)
    gpu.set_scene(scene)
    set_scene_s = time.perf_counter() - t0
    for fi in range(warm):
        gpu.render(*view, fi == 0, False)
    far = gpu.get_option("any_far_first_decision")
    inst = RenderCUDA(0, max_depth=MAX_DEPTH, count_traversal=True, stream=stream.cuda_stream, any_far_first=1 if far == 1 else 0)
    inst.initialize(WIDTH, HEIGHT)
    inst.set_scene(scene)
    acc = np.zeros(6, np.float64)
    for fi in range(warm + steps):
        inst.render(*view, fi == 0, False)
        if fi >= warm:
            c = inst.counters()
            acc += [c["closest_rays"], c["closest_nodes_visited"], c["closest_tris_tested"], c["occlusion_rays"],
                    c["any_nodes_visited"], c["any_tris_tested"]]
    del inst
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(steps):
        gpu.render_async(*view, False, 1)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    totals, stage_acc, csum, nframes = gpu.sync()
    ms = e0.elapsed_time(e1)
    t_trav = stage_acc["traverse_primary"] + stage_acc["traverse"]
    trav_bytes = acc[1] * S_NODE + acc[2] * S_TRI + acc[0] * (S_RAY + S_HIT) + acc[4] * S_NODE + acc[5] * S_TRI + acc[3] * (S_RAY + 1)
    achieved = trav_bytes / (t_trav * 1e-3) / 1e9
    peak, _ = hbm_peak()
    traffic, note = measured_traffic(args.workload)
    n_launch = steps * (MAX_DEPTH + 1)
    info = gpu.scene_info()
    emit({"workload": WORKLOAD, "value": totals.num_rays / (ms * 1e3), "unit": "MRays/s", "ms_per_step": ms / steps, "steps": steps,
          "stage_ms_per_step": {k: v / steps for k, v in stage_acc.items()},
          "scene_mb": {"nodes": info["node_bytes"] / 1e6, "triangles_and_shading": 2 * info["triangle_bytes"] / 1e6},
          "set_scene_s": set_scene_s, "tri_pass_defer": gpu.get_option("tri_pass_defer"),
          "roofline": {"kernel": "k_traverse", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                       "algorithmic_bytes_per_launch": trav_bytes / n_launch, "traffic": traffic, "traffic_note": note,
                       "dram_over_algorithmic": (traffic / (trav_bytes / n_launch)) if traffic else None,
                       "closest_nodes_per_ray": acc[1] / max(1.0, acc[0]), "any_hit_nodes_per_ray": acc[4] / max(1.0, acc[3])}})


def extra_workload_probe(workload_key: str):
    """Runs run_workload_probe() for another workload in a child process; returns its dict, or {"error": ...}."""
    try:
        script = os.environ.get("CRT_BENCH_PROBE_SCRIPT", os.path.abspath(__file__))
        p = subprocess.run([sys.executable, script, "--probe-workload", "--workload", workload_key, "--steps", "5", "--warmup", "3"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=int(os.environ.get("CRT_BENCH_PROBE_TIMEOUT", "240")))
        if p.returncode != 0:
            return {"error": f"exit code {p.returncode}: " + p.stderr.decode(errors="replace").strip().splitlines()[-1][:300]}
        return json.loads(p.stdout.decode().strip().splitlines()[-1])
    except Exception as e:  # timeout, unparsable output
        return {"error": f"{type(e).__name__}: {e}"[:300]}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, accum, img, num_rays: int, limit: int = DUMP_BYTES) -> None:
    """--dump-outputs: what a caller of the render path holds after the last timed step, as .npy files, so that two builds
    can be compared output for output. accum.npy: the accumulated radiance (float32, height x width x 3); img.npy: the
    sRGB8 frame (`img`, one packed RGBA8 uint32 per pixel) as float32 R, G, B, A values 0..255 (height x width x 4);
    num_rays.npy: the rays of that frame (float64). A frame whose two arrays exceed `limit` bytes is sampled at the same
    seeded pixels every run: the arrays are then (n, 3) and (n, 4), and pixel_index.npy holds the row-major pixel indices
    (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    rgba = img.view(np.uint8).reshape(img.shape + (4,)).astype(np.float32)
    pixels = accum.shape[0] * accum.shape[1]
    per_pixel = accum.itemsize * 3 + rgba.itemsize * 4
    if pixels * per_pixel > limit:
        n = (limit - 4096) // (per_pixel + 8)  # (4 KB for the .npy headers and num_rays.npy)
        idx = np.sort(np.random.default_rng(0).choice(pixels, n, replace=False))
        accum, rgba = accum.reshape(-1, 3)[idx], rgba.reshape(-1, 4)[idx]
        np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "accum.npy"), accum)
    np.save(os.path.join(out_dir, "img.npy"), rgba)
    np.save(os.path.join(out_dir, "num_rays.npy"), np.array([num_rays], np.float64))


def emit(line: dict) -> None:
    """The contract is ONE JSON line on stdout. Libraries (NCCL prints its version banner) write
    to fd 1 too, so main() points fd 1 at stderr for the whole run and the result goes to the
    saved real stdout."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


_REAL_STDOUT = None


def main():
    global _REAL_STDOUT
    # watchdog: a run that does not finish is killed with a traceback instead of hanging its caller
    import faulthandler

    faulthandler.dump_traceback_later(int(os.environ.get("CRT_BENCH_WATCHDOG", "600")), repeat=False, file=sys.stderr,
                                      exit=True)
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-mode", action="store_true",
                    help="for runs under ncu: skip the instrumented counting pass and the CPU baseline")
    ap.add_argument("--repeats", type=int, default=5, help="repetitions of the K-step device-timed region (dispersion)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's framebuffers and ray count to DIR/<name>.npy")
    ap.add_argument("--probe-set-scene", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--probe-workload", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "cuda" else max(args.warmup, 1)
    select_workload(args.workload)
    if args.probe_set_scene:
        run_set_scene_probe()
        return
    if args.probe_workload:
        run_workload_probe(args)
        return

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    from chameleonrt_b200 import RenderCUDA
    from chameleonrt_b200.distributed import FrameGatherer, PeerFrame

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; the backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"

    scene, view = make_workload()
    # a dedicated (non-default) torch stream: the renderer launches on it, so torch.cuda.Event
    # brackets exactly the kernels of the timed region
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    gpu = RenderCUDA(local_rank, max_depth=MAX_DEPTH, rank=rank, world_size=world, stream=stream.cuda_stream)
    gpu.set_option("pin_read_img", 1)  # the e2e loop reads every frame into the same host buffer
    gpu.initialize(WIDTH, HEIGHT)
    gpu.set_scene(scene)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # Frame assembly at N > 1. "peer" (default since round 2: measured faster, profiles/r2_experiments.md): no gather,
    # every rank's resolve kernel writes its tiles into rank 0's frame over NVLink (PeerFrame). "gather": NCCL gather of
    # the tile-local buffers + k_assemble on rank 0 (FrameGatherer).
    peer_frame = os.environ.get("CRT_BENCH_FRAME", "peer") == "peer"
    gatherer = (PeerFrame(gpu) if peer_frame else FrameGatherer(gpu)) if world > 1 else None

    def frame(f, readback):
        """One step through the public call. N = 1: the blocking RenderBackend::render with `img` read back. N > 1:
        without readback (warm-up) the blocking call, the frame-end exchange left pending; with readback the frame is
        enqueued, rank 0's stream waits for every rank's tiles (completion flags over peer memory, or the gather), rank 0
        reads `img` into its page-locked host buffer, and every rank waits for its own frame (one host wait per frame)."""
        if world == 1:
            return gpu.render(*view, f == 0, readback)
        if not readback:
            st = gpu.render(*view, f == 0, False)
            gatherer.submit()
            return st
        gpu.render_async(*view, f == 0, 1)
        gatherer.submit()
        gatherer.finish()
        if rank == 0:
            gpu.read_img(gpu.img)
        totals, _, _, _ = gpu.sync()
        return totals

    def flush():
        if world > 1:
            gatherer.finish()

    # Frames in flight: with N GPUs each rank owns 1/N of the image, so N consecutive frames are
    # rendered as one wavefront (crtc_render_async num_frames) — every GPU keeps one full frame's worth
    # of samples in flight, whatever N. The result is bit-identical to frame-by-frame rendering; the
    # accumulated tiles are exchanged once per batch. (The e2e region below stays frame by frame.)
    frames_in_flight = max(1, min(world, args.steps))
    n_warm = args.warmup + frames_in_flight
    repeats = max(1, args.repeats)

    f = 0
    for _ in range(args.warmup):
        frame(f, False)
        f += 1
    flush()  # no collective in flight while the batch-sized path state is (re)allocated
    # The renderer has by now settled the descent order of its shadow rays for this scene (option any_far_first =
    # 2: frames 1 and 2 try one order each; the image does not depend on it). The counting pass must use the same.
    shadow_far_first = gpu.get_option("any_far_first_decision")

    # ---- instrumented pass (not timed): exact node/triangle visit counts of the first repetition's frames ----
    counts = np.zeros(6, np.float64)
    if not args.profile_mode:
        inst = RenderCUDA(local_rank, max_depth=MAX_DEPTH, rank=rank, world_size=world, count_traversal=True,
                          stream=stream.cuda_stream, any_far_first=1 if shadow_far_first == 1 else 0)
        inst.initialize(WIDTH, HEIGHT)
        inst.set_scene(scene)
        acc = np.zeros(6, np.float64)
        for fi in range(n_warm + args.steps):
            inst.render(*view, fi == 0, False)
            if fi >= n_warm:
                c = inst.counters()
                acc += [c["closest_rays"], c["closest_nodes_visited"], c["closest_tris_tested"], c["occlusion_rays"],
                        c["any_nodes_visited"], c["any_tris_tested"]]
        counts = acc
        del inst

    barrier()
    gpu.render_async(*view, False, frames_in_flight)  # warm-up batch (allocates the batch-sized path state)
    f += frames_in_flight
    if world > 1:
        gatherer.submit()
        gatherer.finish()
    flush()
    barrier()
    gpu.sync()  # drop the warm-up batch's record

    def timed_region(batch):
        """Exactly args.steps frames, `batch` frames per wavefront, enqueued back to back (crtc_render_async): the host
        never waits inside the region (it stays at most two batches ahead). Returns (ms, rays, stage sums, launches)."""
        nonlocal f
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        done = 0
        batch_done = []
        while done < args.steps:
            if len(batch_done) >= 2:
                batch_done[-2].synchronize()
            nb = min(batch, args.steps - done)
            gpu.render_async(*view, f == 0, nb)
            f += nb
            done += nb
            if world > 1:
                # one exchange per batch, completed right away (stream-ordered, no host wait)
                gatherer.submit()
                gatherer.finish()
            ev = torch.cuda.Event()
            ev.record(stream)
            batch_done.append(ev)
        flush()
        e1.record(stream)
        barrier()
        totals, stage_acc, csum, nframes = gpu.sync()
        assert nframes == args.steps
        n_batches = -(-args.steps // batch)
        launches = csum["kernel_launches"] + (n_batches * world if (world > 1 and rank == 0 and not peer_frame) else 0)  # + k_assemble
        return e0.elapsed_time(e1), totals.num_rays, stage_acc, launches

    # ---- device-timed region: inputs resident in HBM, no readback; `repeats` repetitions of K steps ----
    # The first repetition records a CUDA event after every launch (the per-stage times the roofline needs); the others —
    # and the frame-by-frame and end-to-end regions — only at the start and the end of a frame: the 28 event records of a
    # frame cost ~0.07 ms (0.8 % of a full C2 frame, 5.5 % of a 1/8 shard's; profiles/r2_experiments.md).
    reps = []
    with ClockSampler(local_rank) as clocks:
        for rep in range(repeats):
            gpu.set_option("stage_events", 1 if rep == 0 else 0)
            reps.append(timed_region(frames_in_flight))
    clock_summary = clocks.summary()
    # frame by frame (one frame per wavefront) on the device clock as well, for N > 1: what a camera that moves every
    # frame gets
    fbf = timed_region(1) if world > 1 else None

    # ---- end-to-end region: the public blocking call with host buffers (img readback every frame) ----
    e2e_reps = []
    for _ in range(min(repeats, 3)):
        barrier()
        t0 = time.perf_counter()
        e2e_rays = 0
        for _ in range(args.steps):
            st = frame(f, True)
            f += 1
            e2e_rays += st.num_rays
        barrier()
        e2e_reps.append(((time.perf_counter() - t0) * 1e3, e2e_rays))
    last_frame_rays = st.num_rays

    def over_ranks(values, op):
        if world == 1:
            return [float(v) for v in values]
        t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return [float(v) for v in t]

    MAX, SUM = (dist.ReduceOp.MAX, dist.ReduceOp.SUM) if world > 1 else (None, None)
    rep_ms = over_ranks([r[0] for r in reps], MAX)
    rep_rays = over_ranks([r[1] for r in reps], SUM)
    launches = over_ranks([reps[0][3]], SUM)[0]
    e2e_ms = over_ranks([r[0] for r in e2e_reps], MAX)
    e2e_rays_all = over_ranks([r[1] for r in e2e_reps], SUM)
    counts = np.array(over_ranks(counts, SUM))
    stage_keys = sorted(reps[0][2])
    stage_acc = dict(zip(stage_keys, over_ranks([reps[0][2][k] for k in stage_keys], MAX)))
    if fbf is not None:
        fbf_ms, fbf_rays = over_ranks([fbf[0]], MAX)[0], over_ranks([fbf[1]], SUM)[0]
    last_rays_all = over_ranks([last_frame_rays], SUM)[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gpu.read_accum(), gpu.read_img(), int(last_rays_all))

    # ---- N > 1: is the assembled multi-GPU frame the single-GPU frame, bit for bit? (rank 0 re-renders the same
    # frame ids on its own GPU alone: accum + img + ray count of the last frame) ----
    mgpu_check = None
    if world > 1:
        barrier()
        if rank == 0:
            try:
                solo = RenderCUDA(local_rank, max_depth=MAX_DEPTH, stream=stream.cuda_stream)
                solo.initialize(WIDTH, HEIGHT)
                solo.set_scene(scene)
                # the same frame ids 0 .. f-1 (accumulation never restarted), in wavefronts of at most ~32 M paths
                per_wave = max(1, min(16, (32 << 20) // max(1, WIDTH * HEIGHT * SPP)))
                done = 0
                while done < f - 1:
                    nb = min(per_wave, f - 1 - done)
                    solo.render_async(*view, done == 0, nb)
                    solo.sync()
                    done += nb
                st_solo = solo.render(*view, f == 1, False)
                same_accum = bool(np.array_equal(solo.read_accum().view(np.uint32), gpu.read_accum().view(np.uint32)))
                same_img = bool(np.array_equal(solo.read_img(), gpu.read_img()))
                mgpu_check = {"mgpu_bit_identical": bool(same_accum and same_img and int(st_solo.num_rays) == int(last_rays_all)),
                              "accum": same_accum, "img": same_img, "frames_accumulated": f,
                              "rays_last_frame": [int(last_rays_all), int(st_solo.num_rays)]}
            except Exception as e:  # (e.g. out of memory: the check must not cost the line its measurements)
                mgpu_check = {"mgpu_bit_identical": None, "mgpu_check_error": f"{type(e).__name__}: {e}"[:300]}
                solo = None
            del solo
        barrier()

    if rank == 0:
        order = np.argsort(rep_ms)
        med = int(order[len(order) // 2])
        elapsed_ms, rays = rep_ms[med], rep_rays[med]
        value = rays / (elapsed_ms * 1e3)  # MRays/s
        rep_value = [r / (m * 1e3) for r, m in zip(rep_rays, rep_ms)]
        e2e_order = np.argsort(e2e_ms)
        e2e_med = int(e2e_order[len(e2e_order) // 2])
        e2e_value = [r / (m * 1e3) for r, m in zip(e2e_rays_all, e2e_ms)]
        peak, peak_src = hbm_peak()
        # dominant kernel: k_traverse (persistent BVH8 traversal; every launch but the first carries
        # the shadow rays of bounce b and the continuation rays of bounce b+1)
        closest_bytes = counts[1] * S_NODE + counts[2] * S_TRI + counts[0] * (S_RAY + S_HIT)
        any_bytes = counts[4] * S_NODE + counts[5] * S_TRI + counts[3] * (S_RAY + 1)
        trav_bytes = closest_bytes + any_bytes
        t_trav_ms = stage_acc["traverse_primary"] + stage_acc["traverse"]  # max over ranks of per-rank sums (first repetition)
        n_batches = -(-args.steps // frames_in_flight)
        n_launch = n_batches * (MAX_DEPTH + 1)  # k_traverse launches per rank in one repetition
        achieved = trav_bytes / world / (t_trav_ms * 1e-3) / 1e9  # per GPU GB/s
        traffic, traffic_note = measured_traffic(args.workload)
        line = {
            "metric": "MRays/s", "value": value, "unit": "MRays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "width": WIDTH, "height": HEIGHT, "spp": SPP, "max_depth": MAX_DEPTH,
                       "parallelism": (f"image tiles 64x64 round-robin over {world} GPUs, scene replicated; {frames_in_flight} "
                                       "consecutive frames per wavefront (bit-identical to frame-by-frame), " +
                                       ("tiles written into rank 0's frame by every rank's resolve kernel through peer-mapped "
                                        "memory (no gather; a one-element all-reduce per batch as the barrier)" if peer_frame else
                                        "NCCL gather of the accumulated tiles to rank 0 once per batch (stream-ordered, not overlapped)") +
                                       "; e2e: frame by frame, assembly + readback every frame") if world > 1 else "single GPU",
                       "frames_in_flight": frames_in_flight,
                       "bvh_builder": ("host (binned SAH)", "device (PLOC)", "device (LBVH)")[gpu.get_option("bvh_builder")],
                       "traversal_variant": {"tri_pass_defer": gpu.get_option("tri_pass_defer"), "refill_idle": gpu.get_option("refill_idle"),
                                             "shade_sort": gpu.get_option("shade_sort")},
                       "shadow_ray_order": {1: "far-first", 0: "near-first"}.get(shadow_far_first, "undecided (near-first)") +
                                           " (chosen per scene from the traversal times of warm-up frames 1 and 2; same image either way)",
                       "l2": f"inputs larger than L2: ~{WIDTH * HEIGHT * SPP * 250 / 1e9:.1f} GB of per-frame path state "
                             f"streams through every bounce (L2 126 MB); scene = {gpu.scene_info()['node_bytes'] / 1e6:.0f} MB "
                             f"nodes + {2 * gpu.scene_info()['triangle_bytes'] / 1e6:.0f} MB triangle/shading records"},
            # value / ms_per_step are the MEDIAN repetition of `repeats` repetitions of `steps` frames each
            "dispersion": {"repeats": len(rep_ms), "of": "the device-timed region, repeated (repetition 1 with a CUDA event after every launch, "
                                                          "for the stage times; the others with frame start / end events only)",
                           "ms_per_step": {"min": min(rep_ms) / args.steps, "median": elapsed_ms / args.steps, "max": max(rep_ms) / args.steps},
                           "value": {"min": min(rep_value), "median": value, "max": max(rep_value)},
                           "e2e_value": {"min": min(e2e_value), "median": e2e_value[e2e_med], "max": max(e2e_value), "repeats": len(e2e_ms)}},
            "roofline": {"kernel": "k_traverse", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": trav_bytes / n_launch / world,
                         "avg_launch_ms": t_trav_ms / n_launch,
                         "note": "achieved = ALGORITHMIC bytes (80 B x nodes visited + 48 B x triangles tested + ray/hit records, counted by the "
                                 "instrumented kernel on the same frames) / CUDA-event time of the k_traverse launches; on C2 the 27 MB scene is "
                                 "L2-resident, so this is L2/issue throughput expressed in the contract's unit, not DRAM traffic (see traffic)",
                         "closest": {"rays": counts[0], "nodes_per_ray": counts[1] / max(1.0, counts[0]),
                                     "tris_per_ray": counts[2] / max(1.0, counts[0])},
                         "any_hit": {"rays": counts[3], "nodes_per_ray": counts[4] / max(1.0, counts[3]),
                                     "tris_per_ray": counts[5] / max(1.0, counts[3])}},
            "stage_ms_per_step": {k: v / args.steps for k, v in stage_acc.items()},
            "e2e": {"value": e2e_value[e2e_med], "unit": "MRays/s", "ms_per_step": e2e_ms[e2e_med] / args.steps,
                    "h2d_bytes_per_step": 52,  # ViewParams (camera basis + frame id) as kernel parameters
                    "d2h_bytes_per_step": WIDTH * HEIGHT * 4 + 36 * 4,
                    "host_buffer": "RenderBackend::img, page-locked by the backend on first use (cudaHostRegister)"},
            "gpu_launches": int(launches),
            "clocks": clock_summary,
        }
        if fbf is not None:
            line["frame_by_frame"] = {"value": fbf_rays / (fbf_ms * 1e3), "unit": "MRays/s", "ms_per_step": fbf_ms / args.steps,
                                      "what": "device-timed like `value`, but ONE frame per wavefront (frames_in_flight = 1) and "
                                              "the frame assembled on rank 0 after every frame"}
        if mgpu_check is not None:
            line.update(mgpu_check)
        if not args.no_cpu_baseline and not args.profile_mode and world == 1:
            res, cpu_kind, cpu_desc, meter = time_oracle(scene, view, budget_s=20.0, frames_cap=6)
            warm = res[1:] if len(res) > 1 else res
            cms = sum(r[0] for r in warm)
            crays = sum(r[1] for r in warm)
            cval = crays / (cms * 1e3)
            line["cpu_baseline"] = {
                "value": cval, "unit": "MRays/s", "kind": cpu_kind, **describe_cpu_arm(cval, meter, os.cpu_count()),
                "ms_per_frame": cms / len(warm),
                "sample": f"{len(warm)} full frame(s) of the same workload (1 warm-up frame discarded); {cpu_desc}"}
        if world == 1 and not args.profile_mode and os.environ.get("CRT_BENCH_SET_SCENE_PROBE", "1") != "0":
            # outside the timed region, in a child process: set_scene with the host and with the device BVH builder
            line["set_scene"] = set_scene_probe(args.workload)
        if world == 1 and not args.profile_mode and args.workload == "c2" and os.environ.get("CRT_BENCH_EXTRA", "1") != "0":
            # the HBM-resident configurations (BASELINE configs[3], [2]) in short form, each in its own child process
            line["extra"] = {"workloads": {k: extra_workload_probe(k) for k in os.environ.get("CRT_BENCH_EXTRA_WORKLOADS", "c4,c3").split(",") if k}}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
