"""bench.py's output contract, as far as it can be exercised without a GPU: the reference arm (`--impl
reference`: the CPU implementation of the path on this box's cores) prints exactly ONE JSON line on stdout with
the keys the driver reads, whatever libraries write to fd 1; non-zero ranks of a multi-rank launch print nothing;
and the GPU arm refuses to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ, CRT_BENCH_REF_BUDGET="2")  # tiny budget: one sample per pixel per step
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=ROOT,
                          env=e, timeout=timeout)


def test_reference_arm_prints_one_json_line(built, tmp_path):
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "outputs")])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "MRays/s" and d["unit"] == "MRays/s" and d["higher_is_better"] is True
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["vs_baseline"] is None  # warm-up is at least 1
    assert d["config"]["workload"].startswith("C2") and d["config"]["width"] == 1280 and d["config"]["max_depth"] == 8
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    import numpy as np

    out = {p.stem: np.load(p) for p in (tmp_path / "outputs").glob("*.npy")}
    assert sorted(out) == ["accum", "img", "num_rays"]
    assert out["accum"].shape == (720, 1280, 3) and out["img"].shape == (720, 1280, 4) and out["num_rays"][0] > 0


def test_dump_outputs_samples_a_large_frame_at_fixed_pixels(tmp_path):
    """A frame over the size limit is written as the same seeded sample of pixels every time, with their indices."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    rng = np.random.default_rng(7)
    accum = rng.normal(size=(30, 40, 3)).astype(np.float32)
    img = rng.integers(0, 2 ** 32, size=(30, 40), dtype=np.uint64).astype(np.uint32)
    limit = 4096 + 36 * 200  # 200 pixels of 12 + 16 bytes, plus an 8-byte index each
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), accum, img, 1234, limit=limit)
    a, b = ({n: np.load(tmp_path / d / f"{n}.npy") for n in ("accum", "img", "num_rays", "pixel_index")} for d in ("a", "b"))
    assert all(np.array_equal(a[n], b[n]) for n in a)
    idx = a["pixel_index"].astype(np.int64)
    assert a["pixel_index"].dtype == np.float64 and len(idx) == 200 and (np.diff(idx) > 0).all() and 0 <= idx[0] and idx[-1] < 30 * 40
    assert a["accum"].dtype == np.float32 and np.array_equal(a["accum"], accum.reshape(-1, 3)[idx])
    assert a["img"].dtype == np.float32 and np.array_equal(a["img"], img.view(np.uint8).reshape(-1, 4)[idx].astype(np.float32))
    assert a["num_rays"].dtype == np.float64 and a["num_rays"].tolist() == [1234.0]
    bench.dump_outputs(str(tmp_path / "whole"), accum, img, 1234)  # under the limit: the whole frame
    assert np.array_equal(np.load(tmp_path / "whole" / "accum.npy"), accum) and not (tmp_path / "whole" / "pixel_index.npy").exists()


def test_reference_arm_is_silent_on_other_ranks(built):
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_gpu(built):
    import torch

    if torch.cuda.is_available():
        import pytest

        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "0"])
    assert r.returncode != 0 and r.stdout.strip() == ""
    assert "CUDA device" in r.stderr


# Frames bench.py renders on its timed renderer with --steps 2 --warmup 3 and the default 5 repeats: 3 warm-up, 1 untimed
# batch, 5 x 2 device-timed, 3 x 2 end-to-end.
REPLAY_FRAMES = 3 + 1 + 5 * 2 + 3 * 2


def test_gpu_arm_dry_run_on_the_emulated_renderer(built, tmp_path):
    """bench.py's GPU arm, every line of it — warm-up, the renderer's shadow-order decision, the counting pass, the
    untimed batch, the device-timed loop with frames in flight, the end-to-end loop, the CPU baseline, the JSON — run
    in a subprocess where `torch.cuda` is a thin fake over wall-clock time and RenderCUDA loads the CPU emulation of
    the renderer (tests/simt_emu), on the tiny `dev` workload. Numbers are meaningless; the point is that the code
    path the driver runs on the B200 executes and prints one well-formed line."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "simt_emu"))
    import build as simt_build

    lib = simt_build.build()
    driver = tmp_path / "dry_run.py"
    driver.write_text(f'''
import os, sys, time, types
sys.path.insert(0, {ROOT!r})
import torch
class _Stream:
    cuda_stream = 0
    def __init__(self, *a, **k): pass
    def synchronize(self): pass
class _Event:
    def __init__(self, enable_timing=False): self.t = None
    def record(self, stream=None): self.t = time.perf_counter()
    def synchronize(self): pass
    def elapsed_time(self, other): return (other.t - self.t) * 1e3
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda d: None
torch.cuda.Stream = _Stream
torch.cuda.set_stream = lambda s: None
torch.cuda.current_stream = lambda d=None: _Stream()
torch.cuda.Event = _Event
torch.cuda.synchronize = lambda d=None: None
import chameleonrt_b200.backend as backend
backend._LIB_PATH, backend._lib = {lib!r}, None
import bench
sys.argv = ["bench.py"] + (sys.argv[1:] or ["--workload", "dev", "--steps", "2", "--warmup", "3"])
bench.main()
replay = os.environ.get("CRT_DRY_RUN_REPLAY")
if replay and "--probe-set-scene" not in sys.argv and "--probe-workload" not in sys.argv:
    # the same frames on a fresh renderer, one blocking call each: what the dumped outputs must be
    import numpy as np
    from chameleonrt_b200 import RenderCUDA
    scene, view = bench.make_workload()
    r = RenderCUDA(0, max_depth=bench.MAX_DEPTH)
    r.initialize(bench.WIDTH, bench.HEIGHT)
    r.set_scene(scene)
    for f in range(int(replay.split(":")[0])):
        st = r.render(*view, f == 0, True)
    out = replay.split(":")[1]
    os.makedirs(out)
    np.save(out + "/accum.npy", r.read_accum())
    np.save(out + "/img.npy", r.read_img())
    np.save(out + "/num_rays.npy", np.array([st.num_rays], np.float64))
''')
    dump = tmp_path / "outputs"
    r = subprocess.run([sys.executable, str(driver), "--workload", "dev", "--steps", "2", "--warmup", "3", "--dump-outputs", str(dump)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900,
                       env=dict(os.environ, CRT_BENCH_REF_BUDGET="2", CRT_BENCH_PROBE_SCRIPT=str(driver),
                                CRT_DRY_RUN_REPLAY=f"{REPLAY_FRAMES}:{tmp_path / 'replay'}"))
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "stage_ms_per_step"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["value"] > 0 and d["gpu_launches"] == 2 * (2 + 3 * 5 + 1)
    # the timed region is repeated: value / ms_per_step are the median repetition, the spread is in the line
    disp = d["dispersion"]
    assert disp["repeats"] == 5 and disp["ms_per_step"]["min"] <= d["ms_per_step"] <= disp["ms_per_step"]["max"]
    assert disp["value"]["min"] <= d["value"] <= disp["value"]["max"] and disp["e2e_value"]["min"] <= d["e2e"]["value"] <= disp["e2e_value"]["max"]
    # the CPU arm says what it is and what CPU budget it really had
    cb = d["cpu_baseline"]
    assert cb["effective_cores"] > 0 and cb["mrays_per_effective_core"] > 0 and "NOT Embree" in cb["label"] and "cgroup_quota_cores" in cb
    assert "traffic_note" in d["roofline"]
    assert d["config"]["workload"].startswith("DEV") and d["config"]["frames_in_flight"] == 1
    assert d["config"]["shadow_ray_order"].split()[0] in ("far-first", "near-first")
    rf = d["roofline"]
    assert rf["kernel"] == "k_traverse" and rf["bound"] == "hbm" and rf["achieved"] > 0 and 0 < rf["frac"] and rf["closest"]["nodes_per_ray"] > 0
    assert d["e2e"]["value"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 128 * 48 * 4 + 36 * 4
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] > 0
    # the set_scene probe (child process): host-built and device-built BVH8, same frames
    ss = d["set_scene"]
    assert "error" not in ss, ss
    assert ss["frames_bit_identical"] is True and ss["triangles"] == 34
    assert ss["host"]["set_scene_ms"] > 0 and ss["device"]["bvh8_nodes"] >= 1 and ss["device"]["closest_nodes_per_ray"] > 0
    # --dump-outputs: the last timed step's framebuffers and ray count
    import numpy as np

    out = {p.stem: np.load(p) for p in dump.glob("*.npy")}
    assert sorted(out) == ["accum", "img", "num_rays"]
    assert out["accum"].dtype == np.float32 and out["accum"].shape == (48, 128, 3) and np.isfinite(out["accum"]).all()
    assert out["img"].dtype == np.float32 and out["img"].shape == (48, 128, 4) and out["img"].max() <= 255 and out["img"].max() > 0
    assert out["num_rays"].dtype == np.float64 and out["num_rays"].shape == (1,) and out["num_rays"][0] > 0
    # ... and they are the last timed frame's: the same frames rendered again one by one give the same bits
    replay = {n: np.load(tmp_path / "replay" / f"{n}.npy") for n in ("accum", "img", "num_rays")}
    assert np.array_equal(out["accum"].view(np.uint32), replay["accum"].view(np.uint32))
    assert np.array_equal(out["img"], replay["img"].view(np.uint8).reshape(48, 128, 4).astype(np.float32))
    assert out["num_rays"].tolist() == replay["num_rays"].tolist()


def test_gpu_arm_dry_run_two_ranks(built, tmp_path):
    """The N = 2 path of bench.py — tile sharding, two frames in flight per wavefront, the per-batch gather and
    assembly on rank 0, the reductions over ranks — dry-run as two processes: gloo instead of NCCL, host tensors
    aliasing the emulated renderer's "device" buffers instead of CUDA tensors. Rank 0 prints the one line."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "simt_emu"))
    import build as simt_build
    import socket

    lib = simt_build.build()
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    driver = tmp_path / "dry_run2.py"
    driver.write_text(f'''
import ctypes, sys, time
sys.path.insert(0, {ROOT!r})
import numpy as np
import torch
import torch.distributed as dist
class _Stream:
    cuda_stream = 0
    def __init__(self, *a, **k): pass
    def synchronize(self): pass
class _Event:
    def __init__(self, enable_timing=False): self.t = None
    def record(self, stream=None): self.t = time.perf_counter()
    def synchronize(self): pass
    def elapsed_time(self, other): return (other.t - self.t) * 1e3
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda d: None
torch.cuda.Stream = _Stream
torch.cuda.set_stream = lambda s: None
torch.cuda.current_stream = lambda d=None: _Stream()
torch.cuda.Event = _Event
torch.cuda.synchronize = lambda d=None: None
_real_device = torch.device
torch.device = lambda *a, **k: _real_device("cpu")
_real_init = dist.init_process_group
dist.init_process_group = lambda backend=None, **k: _real_init("gloo")
import chameleonrt_b200.backend as backend
backend._LIB_PATH, backend._lib = {lib!r}, None
import chameleonrt_b200.distributed as cd
cd.device_tensor = lambda ptr, nbytes, device: torch.from_numpy(np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(ptr)))
import bench
sys.argv = ["bench.py", "--gpus", "2", "--workload", "dev", "--steps", "4", "--warmup", "3"]
bench.main()
''')
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   CRT_BENCH_REF_BUDGET="2", CRT_BENCH_FRAME="gather")  # (peer-written frames need real CUDA IPC between processes)
        procs.append(subprocess.Popen([sys.executable, str(driver)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, env=env))
    outs = [p.communicate(timeout=900) for p in procs]
    for p, (so, se) in zip(procs, outs):
        assert p.returncode == 0, se[-3000:]
    assert outs[1][0].strip() == ""
    lines = [l for l in outs[0][0].splitlines() if l.strip()]
    assert len(lines) == 1, outs[0][0]
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and d["steps"] == 4 and d["config"]["frames_in_flight"] == 2 and d["value"] > 0 and d["e2e"]["value"] > 0
    assert d["gpu_launches"] == 2 * 2 * (2 + 3 * 5 + 1) + 2 * 2  # 2 ranks x 2 batches x launches per wavefront + k_assemble on rank 0
    assert "cpu_baseline" not in d and d["roofline"]["closest"]["rays"] > 0 and "image tiles 64x64" in d["config"]["parallelism"]
    # correctness travels with the scaling line: the assembled 2-rank frame equals the frame one renderer alone renders
    assert d["mgpu_bit_identical"] is True and d["accum"] is True and d["img"] is True and d["rays_last_frame"][0] == d["rays_last_frame"][1]
    assert d["frame_by_frame"]["value"] > 0 and d["dispersion"]["repeats"] == 5
