"""Float output against RGBA8 on the GPU, measured with CUDA events and host clocks only; writes one JSON file.

  python tools/f32_bench.py --out profiles/r06_f32_bench.json

* frames: C2, C3 and C4 rendered into device memory, RGBA8 (rt_render_frame) and float (rt_render_frame_multi_f32
  on one GPU) alternating frame by frame after a warm-up of both; the kernel time of each frame is rt_stats.kernel_ms
  (CUDA events around the frame's launches); the median, minimum and maximum of each are reported, and the f32
  excess over RGBA8 next to the extra bytes the float store writes (12 per pixel).
* cli: `rtrace --format pfm` against the default P6 output at C1 and at 4K (C3 geometry), alternating, wall time of
  the whole process and bytes written.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
import rtrace_b200 as rt  # noqa: E402

FRAME_CASES = [("C2", 3840, 2160, 1, 8), ("C3", 3840, 2160, 4, 9), ("C4", 7680, 4320, 4, 9)]
CLI_CASES = [("C1", 1024, 768, 4, 8), ("C3", 3840, 2160, 4, 9)]
BIN = os.path.join(ROOT, "target", "release", "rtrace")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.strip().splitlines()]


def summary(xs):
    return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4), "n": len(xs)}


def frame_case(name, w, h, spp, level, rounds, warmup):
    scene = rt.Scene(level=level)
    o = rt.RenderOptions(w, h, spp)
    d8, d32 = rt.device_alloc(w * h * 4), rt.device_alloc(w * h * 16)
    try:
        def rgba8():
            _, st = rt.Renderer.render(o, scene, out_ptr=d8, want_stats=True)
            return st

        def f32():
            _, st = rt.Renderer.render_f32(o, scene, out_ptr=d32, want_stats=True)
            return st
        for _ in range(warmup):
            rgba8(), f32()
        k8, k32, used = [], [], set()
        for _ in range(rounds):
            st8, st32 = rgba8(), f32()
            k8.append(st8.kernel_ms)
            k32.append(st32.kernel_ms)
            used.add((int(st8.variant_used), int(st32.variant_used)))
        m8, m32 = statistics.median(k8), statistics.median(k32)
        return {"case": name, "width": w, "height": h, "spp": spp, "level": level, "rounds": rounds, "warmup": warmup,
                "variants_used_rgba8_f32": sorted(used), "rgba8_kernel_ms": summary(k8), "f32_kernel_ms": summary(k32),
                "f32_excess_pct": round((m32 / m8 - 1.0) * 100.0, 2), "extra_store_mb": round(w * h * 12 / 1e6, 1)}
    finally:
        rt.device_free(d8)
        rt.device_free(d32)
        scene.close()


def cli_case(name, w, h, spp, level, rounds):
    out = {"case": name, "width": w, "height": h, "spp": spp, "level": level, "rounds": rounds}
    with tempfile.TemporaryDirectory() as tmp:
        times = {"ppm": [], "pfm": []}
        sizes = {}
        for _ in range(rounds):
            for fmt, path in (("ppm", "o.tga"), ("pfm", "o.pfm")):
                args = [BIN, "--width=%d" % w, "--height=%d" % h, "--samples-per-pixel=%d" % spp, "--level=%d" % level]
                if fmt == "pfm":
                    args.append("--format=pfm")
                t0 = time.perf_counter()
                subprocess.run(args + [path], cwd=tmp, check=True, capture_output=True)
                times[fmt].append((time.perf_counter() - t0) * 1e3)
                sizes[fmt] = os.path.getsize(os.path.join(tmp, path))
        for fmt in times:
            out[fmt + "_wall_ms"] = summary(times[fmt])
            out[fmt + "_bytes"] = sizes[fmt]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--cli-rounds", type=int, default=3)
    a = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("f32_bench: no CUDA device")
    rt.set_device(0)
    res = {"gpu": gpu_info(), "frames": [], "cli": []}
    for c in FRAME_CASES:
        res["frames"].append(frame_case(*c, rounds=a.rounds, warmup=a.warmup))
        print(json.dumps(res["frames"][-1]), flush=True)
    for c in CLI_CASES:
        res["cli"].append(cli_case(*c, rounds=a.cli_rounds))
        print(json.dumps(res["cli"][-1]), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
