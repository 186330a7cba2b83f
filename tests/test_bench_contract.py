"""bench.py's reference arm (`--impl reference`): the CPU restatement of the reference algorithm on the
host's cores, printed as one JSON line with the keys the driver reads.  Needs no GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                       env=e, timeout=300)
    return r


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("Mrays/s") and d["unit"] == "Mrays/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "1024x768" in d["config"]["workload"]


def _dumped_rgb_sha256(path):
    import hashlib
    import numpy as np
    px = np.load(path)
    assert px.dtype == np.float32 and px.shape == (1024 * 768, 4)
    assert (px == np.round(px)).all() and px.min() >= 0 and px.max() <= 255
    return hashlib.sha256(np.ascontiguousarray(px[:, :3].astype(np.uint8)).tobytes()).hexdigest()


def test_reference_arm_dumps_the_frame_it_rendered(tmp_path):
    """--dump-outputs: c1 (`make image`) is small enough to be written whole; its pixels are the reference's image."""
    r = run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0",
                  "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "rtrace_output_1024x768.json")))
    assert os.listdir(tmp_path / "out") == ["c1.npy"]
    assert _dumped_rgb_sha256(tmp_path / "out" / "c1.npy") == gold["rgb_sha256"]


def test_dump_of_a_large_frame_is_a_fixed_sample():
    """A frame larger than the run's share of the dump budget is sampled: the same pixels in every run, row-major."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    h, w = 2160, 3840
    frame = np.full((h, w, 4), 7, np.uint8)
    idx = np.arange(h * w, dtype=np.int64)   # every pixel's index, spelled in base 251 over R, G, B
    frame[:, :, 0] = (idx % 251).reshape(h, w)
    frame[:, :, 1] = (idx // 251 % 251).reshape(h, w)
    frame[:, :, 2] = (idx // 251 ** 2 % 251).reshape(h, w)
    n = bench.dump_pixels(3)
    a, b = bench.sample_pixels(frame, n), bench.sample_pixels(frame.copy(), n)
    assert a.dtype == np.float32 and a.shape == (n, 4) and n < h * w and np.array_equal(a, b)
    where = a[:, 0].astype(np.int64) + 251 * a[:, 1].astype(np.int64) + 251 ** 2 * a[:, 2].astype(np.int64)
    assert (np.diff(where) > 0).all() and where[-1] < h * w
    assert np.array_equal(a, frame.reshape(-1, 4)[where].astype(np.float32))


@pytest.mark.parametrize("argv", [[], ["--no-also"], ["--workload", "c4"], ["--workload", "c4", "--mode", "bands"],
                                  ["--impl", "reference"]], ids=lambda a: " ".join(a) or "default")
def test_dumps_of_a_run_stay_within_64_mb_at_any_gpu_count(tmp_path, argv):
    """--dump-outputs writes one file per measurement, from rank 0 only, and sizes the samples so that all files of a
    run together stay within 64 MB whatever the number of ranks; a file outside that plan is refused."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    frames = {}
    for world in (1, 2, 8):
        out = tmp_path / str(world)
        args = bench.parse_args(argv + ["--gpus", str(world), "--dump-outputs", str(out)])
        names = bench.dump_names(args, world)
        for name in names:
            w, h = bench.WORKLOADS[name.replace("_bands", "")][:2]
            if (w, h) not in frames:
                frames[w, h] = np.zeros((h, w, 4), np.uint8)
            bench.dump_frame(args, world, name, frames[w, h])
        assert sorted(os.listdir(out)) == sorted(n + ".npy" for n in names)
        assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 * 10 ** 6, (argv, world)
        with pytest.raises(RuntimeError):
            bench.dump_frame(args, world, "c3", frames[next(iter(frames))])
    if not argv:   # the default run: c5 + c2 + c4 on one rank, + the 8K band split on more
        assert bench.dump_names(bench.parse_args([]), 1) == ["c5", "c2", "c4"]
        assert bench.dump_names(bench.parse_args([]), 8) == ["c5", "c2", "c4", "c4_bands"]


@pytest.mark.gpu
def test_native_arm_dumps_its_last_frames_and_times_every_step(tmp_path, oracle):
    """A default run at --steps 2: every measurement (c5 and the c2 / c4 sub-records, kernel-only and end to end) times
    exactly 2 steps, and the dumped c2 sample is the oracle's frame at the same pixels."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    r = run_bench("--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout)
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2
    for sub in ("c2", "c4"):
        assert d["also"][sub]["steps"] == 2 and d["also"][sub]["e2e"]["steps"] == 2, sub
    files = sorted(os.listdir(tmp_path / "out"))
    assert files == ["c2.npy", "c4.npy", "c5.npy"]
    assert sum(os.path.getsize(tmp_path / "out" / f) for f in files) <= 64 * 10 ** 6
    got = np.load(tmp_path / "out" / "c2.npy")
    w, h, spp, level = bench.WORKLOADS["c2"]
    ref, _ = oracle.Scene(level=level).render(w, h, spp)
    assert np.array_equal(got, bench.sample_pixels(ref, len(got)))


def test_reference_arm_runs_on_rank_zero_only():
    r = run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--gpus", "2",
                  env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_library_banners_cannot_reach_stdout():
    """bench.py keeps stdout to one JSON line: what a library writes to fd 1 while the process group is
    created (NCCL's version banner) lands on stderr, and stdout works again afterwards."""
    code = ("import os, sys; sys.path.insert(0, %r); import bench\n"
            "print('before')\n"
            "with bench.stdout_to_stderr():\n"
            "    os.write(1, b'banner\\n')\n"
            "print('after')\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["before", "after"] and "banner" in r.stderr


def test_native_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = run_bench("--steps", "1", "--warmup", "3", "--no-cpu-baseline")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_c5_orbit_cameras_are_the_bindings_orbit_cameras():
    """bench.py --workload c5 and --impl reference use bench.orbit_basis; the binding (and the CLI's --frames)
    use rtrace_b200.orbit_camera.  Same f32 camera for every frame, frame 0 = the reference camera exactly."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
    import bench
    import rtrace_b200 as rt
    for f in range(bench.ORBIT_FRAMES):
        a = rt.make_camera(*bench.orbit_basis(f))
        b = rt.orbit_camera(f, bench.ORBIT_FRAMES)
        for name in ("eye", "right", "up", "forward"):
            assert list(getattr(a, name)) == list(getattr(b, name)), (f, name)
    ref = rt.make_camera(*bench.orbit_basis(0))
    assert list(ref.eye) == [0.0, 0.0, -4.0] and list(ref.right) == [1.0, 0.0, 0.0] and list(ref.forward) == [0.0, 0.0, 1.0]


def test_job_frames_are_spread_evenly_over_the_orbit():
    """bench.orbit_frame: a job's frames cover the 120-frame orbit evenly whatever its size, so that runs at
    different GPU counts render the same mix of cheap and expensive frames; 120 frames are the orbit itself."""
    sys.path.insert(0, ROOT)
    import bench
    assert [bench.orbit_frame(k, 120) for k in range(120)] == list(range(120))
    for total in (20, 40, 80, 160):
        frames = [bench.orbit_frame(k, total) for k in range(total)]
        assert frames[0] == 0 and all(0 <= f < 120 for f in frames) and frames == sorted(frames)
        # every sixth of the orbit gets its share of the job
        for part in range(6):
            n = sum(1 for f in frames if 20 * part <= f < 20 * (part + 1))
            assert abs(n - total / 6) <= 1, (total, part, n)
    assert bench.orbit_frame(0, 0) == 0


def test_committed_profile_summary_belongs_to_the_committed_kernels():
    """bench.py's executed-work roofline uses profiles/latest_summary.json only if it was captured from the same
    kernel sources: the committed capture must match the committed sources, or the bench line's roofline.frac
    would silently be null at the end of a round."""
    sys.path.insert(0, ROOT)
    import bench
    summ = json.load(open(os.path.join(ROOT, "profiles", "latest_summary.json")))
    assert summ["kernel_source_hash"] == bench.kernel_source_hash(), "re-run tools/round_close.sh after kernel changes"
    for w in ("c2", "c3", "c4", "c5"):
        assert w in summ["workloads"], w
    c3 = summ["workloads"]["c3"]
    # the packed f32x2 instructions carry most of the flops: the scalar op counters alone see a fraction of them
    assert c3["fp32_flop_per_frame"] > 3 * c3["fp32_flop_per_frame_scalar_op_counters"]
    assert len(summ["workloads"]["c5"]["fp32_flop_per_orbit_frame"]) == bench.ORBIT_FRAMES
    for mode in ("mode2", "mode3"):   # calibration: the op counters are blind to FFMA2 / FMUL2 chains
        assert summ["calibration"][mode]["counted_flop"] < 1e-3 * summ["calibration"][mode]["true_flop"]


def test_strided_orbit_captures_interpolate_over_a_closed_orbit():
    """tools/round_profiles.sh may capture every k-th orbit frame (C5_STRIDE); tools/orbit_interp.py fills the
    frames in between linearly, and the frame after the last one is frame 0 again."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from orbit_interp import interpolate_orbit, stride_of
    assert stride_of(120, 120) == 1 and stride_of(120, 40) == 3 and stride_of(120, 30) == 4 and stride_of(120, 17) is None
    cap = [100.0 + 3 * i for i in range(40)]           # frames 0, 3, ..., 117
    full = interpolate_orbit(cap, 120, 3)
    assert len(full) == 120 and full[0::3] == cap
    assert full[1] == pytest.approx(101.0) and full[2] == pytest.approx(102.0)
    # between frame 117 and frame 120 == frame 0 the values return to frame 0's
    assert full[118] == pytest.approx(cap[-1] + (cap[0] - cap[-1]) / 3) and full[119] == pytest.approx(cap[-1] + 2 * (cap[0] - cap[-1]) / 3)
    assert interpolate_orbit([1.0, 2.0, 3.0], 3, 1) == [1.0, 2.0, 3.0]
    # a stride that does not divide the orbit: the last span is shorter (frames 119 -> 120 == 0)
    cap7 = [float(f) for f in range(0, 120, 7)]
    full7 = interpolate_orbit(cap7, 120, 7)
    assert full7[119] == 119.0 and len(full7) == 120
    summ = json.load(open(os.path.join(ROOT, "profiles", "latest_summary.json")))
    c5 = summ["workloads"]["c5"]
    cf = c5.get("captured_orbit_frames")
    if cf:   # the committed capture: captured frames keep their own counts
        w = c5["warp_instructions_per_orbit_frame"]
        assert len(w) == 120 and cf[0] == 0 and all(w[f] > 0 for f in cf)
