"""AOV output against RGBA8 on the GPU, measured with CUDA events; writes one JSON file.

  python tools/aov_bench.py --out profiles/r07_aov_bench.json

C2, C3 and C4 rendered into device memory, RGBA8 (rt_render_frame) and AOV (rt_render_frame_multi_aov on one GPU)
alternating frame by frame after a warm-up of both.  The kernel time of each frame is rt_stats.kernel_ms (CUDA events
around the frame's launches: K1-K4 for RGBA8, K1, K2 and the AOV store for AOVs); the median, minimum and maximum of
each are reported, with the AOV frame's time relative to the RGBA8 frame and the bytes each stores (4 and 32 per
pixel).  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
import rtrace_b200 as rt  # noqa: E402

FRAME_CASES = [("C2", 3840, 2160, 1, 8), ("C3", 3840, 2160, 4, 9), ("C4", 7680, 4320, 4, 9)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.strip().splitlines()]


def summary(xs):
    return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4), "n": len(xs)}


def frame_case(name, w, h, spp, level, rounds, warmup):
    scene = rt.Scene(level=level)
    o = rt.RenderOptions(w, h, spp)
    d8, daov = rt.device_alloc(w * h * 4), rt.device_alloc(w * h * 32)
    try:
        def rgba8():
            _, st = rt.Renderer.render(o, scene, out_ptr=d8, want_stats=True)
            return st

        def aov():
            _, st = rt.Renderer.render_aov(o, scene, out_ptr=daov, want_stats=True)
            return st
        for _ in range(warmup):
            rgba8(), aov()
        k8, ka, used = [], [], set()
        for _ in range(rounds):
            st8, sta = rgba8(), aov()
            k8.append(st8.kernel_ms)
            ka.append(sta.kernel_ms)
            used.add((int(st8.variant_used), int(sta.variant_used), int(st8.kernel_launches), int(sta.kernel_launches)))
        m8, ma = statistics.median(k8), statistics.median(ka)
        return {"case": name, "width": w, "height": h, "spp": spp, "level": level, "rounds": rounds, "warmup": warmup,
                "variant_rgba8_aov_launches_rgba8_aov": sorted(used), "rgba8_kernel_ms": summary(k8),
                "aov_kernel_ms": summary(ka), "aov_over_rgba8": round(ma / m8, 4),
                "rgba8_store_mb": round(w * h * 4 / 1e6, 1), "aov_store_mb": round(w * h * 32 / 1e6, 1),
                "aov_store_gb_per_s_over_aov_frame": round(w * h * 32 / (ma * 1e-3) / 1e9, 1)}
    finally:
        rt.device_free(d8)
        rt.device_free(daov)
        scene.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("aov_bench: no CUDA device")
    rt.set_device(0)
    res = {"gpu": gpu_info(), "frames": []}
    for c in FRAME_CASES:
        res["frames"].append(frame_case(*c, rounds=a.rounds, warmup=a.warmup))
        print(json.dumps(res["frames"][-1]), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
