"""JPEG output on the GPU, measured with CUDA events, torch.profiler and host clocks; writes one JSON file.

  python tools/jpeg_bench.py --out profiles/r10_jpeg_bench.json

* encode: C1..C4 frames resident on the device, at q 75, 90 and 100: `iters` back-to-back rt_encode_jpeg calls into
  a device buffer after warm-up (host clock around the calls, each of which waits for its stream), then the three
  encoder kernels' device time from torch.profiler in a separate pass, each kernel's share, and the file size.
* sweep: the C5 orbit (120 frames, 3840x2160, 4x4 samples, level 9) delivered end to end through
  rt_render_sweep_jpeg (q90), rt_render_sweep_png and rt_render_sweep_multi(rgb=1), alternating the three kinds,
  `rounds` rounds each, at N = 1 and at N = 2 and 8 GPUs when the box has them; the median and the spread.
The card's name, power limit and max SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
import rtrace_b200 as rt  # noqa: E402

ENCODE_CASES = [("C1", 1024, 768, 4, 8), ("C2", 3840, 2160, 1, 8), ("C3", 3840, 2160, 4, 9), ("C4", 7680, 4320, 4, 9)]
QUALITIES = (75, 90, 100)
KERNELS = ("jpeg_transform", "jpeg_encode_rows", "jpeg_assemble")
C5 = (3840, 2160, 4, 9, 120)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.strip().splitlines()]


def profile_kernels(fn, iters):
    """Mean device time per call of each encoder kernel (torch.profiler, CUDA activity)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        for k in KERNELS:
            if k in e.name and e.device_type.name == "CUDA":
                tot[k] = tot.get(k, 0.0) + e.device_time
                break
    return {k: v / iters for k, v in tot.items()}


def encode_case(name, w, h, spp, level, iters):
    L = rt.lib()
    scene = rt.Scene(level=level)
    frame = rt.device_alloc(w * h * 4)
    cap = rt.jpeg_bound(w, h)
    out = rt.device_alloc(cap)
    n = C.c_size_t()
    rows = []
    try:
        rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, out_ptr=frame)
        for q in QUALITIES:
            def one():
                rc = L.rt_encode_jpeg(C.c_void_p(frame), w, h, 0, q, C.c_void_p(out), cap, C.byref(n), None)
                if rc != rt.RT_OK:
                    raise rt.RtError(rc, L.rt_last_error().decode())
            for _ in range(5):
                one()
            t0 = time.perf_counter()
            for _ in range(iters):
                one()
            call_ms = (time.perf_counter() - t0) * 1e3 / iters
            kernel_us = profile_kernels(one, iters)
            total = sum(kernel_us.values())
            rows.append({"case": name, "width": w, "height": h, "spp": spp, "level": level, "quality": q,
                         "iters": iters, "bytes_out": n.value, "rgb_bytes": w * h * 3,
                         "ratio_to_rgb": round(w * h * 3 / n.value, 1), "call_ms": round(call_ms, 4),
                         "kernel_us": {k: round(v, 2) for k, v in kernel_us.items()},
                         "kernel_share": {k: round(v / total, 3) for k, v in kernel_us.items()},
                         "kernel_total_us": round(total, 2)})
            print(json.dumps(rows[-1]), flush=True)
    finally:
        rt.device_free(frame)
        rt.device_free(out)
        scene.close()
    return rows


def sweep(kind, scenes, cams):
    w, h, spp, level, _ = C5
    n = len(cams)
    lens = []
    opts = rt.RenderOptions(w, h, spp)
    t0 = time.perf_counter()
    if kind == "jpeg":
        st = rt.Renderer.render_sweep_jpeg(opts, scenes, n, cameras=cams, quality=90,
                                           on_frame=lambda f, d: lens.append(len(d)))
    elif kind == "png":
        st = rt.Renderer.render_sweep_png(opts, scenes, n, cameras=cams, on_frame=lambda f, d: lens.append(len(d)))
    else:
        st = rt.Renderer.render_sweep_multi(opts, scenes, n, cameras=cams, rgb=True,
                                            on_frame=lambda f, a: lens.append(a.size))
    el = time.perf_counter() - t0
    return {"ms_per_frame": round(el * 1e3 / n, 4), "bytes_per_frame": round(sum(lens) / len(lens)),
            "frames": len(lens), "launches": st.kernel_launches}


def sweep_section(rounds):
    w, h, spp, level, n = C5
    cams = [rt.orbit_camera(f, n) for f in range(n)]
    out = []
    avail = rt.device_count()
    kinds = ("jpeg", "png", "rgb")
    for ngpu in [g for g in (1, 2, 8) if g <= avail]:
        scenes = []
        for g in range(ngpu):
            rt.set_device(g)
            scenes.append(rt.Scene(level=level))
        rt.set_device(0)
        for kind in kinds:  # warm-up: scratch, ring buffers, modules on every GPU
            sweep(kind, scenes, cams[:8])
        res = {k: [] for k in kinds}
        for _ in range(rounds):
            for kind in kinds:
                res[kind].append(sweep(kind, scenes, cams))
        row = {"gpus": ngpu}
        for kind in kinds:
            ms = sorted(r["ms_per_frame"] for r in res[kind])
            row[kind] = {"ms_per_frame_rounds": [r["ms_per_frame"] for r in res[kind]],
                         "ms_per_frame_median": ms[len(ms) // 2], "spread_ms": round(ms[-1] - ms[0], 4),
                         "bytes_per_frame": res[kind][0]["bytes_per_frame"], "frames": res[kind][0]["frames"],
                         "launches": res[kind][0]["launches"]}
        row["jpeg_over_rgb_ms"] = round(row["jpeg"]["ms_per_frame_median"] / row["rgb"]["ms_per_frame_median"], 3)
        row["jpeg_over_png_ms"] = round(row["jpeg"]["ms_per_frame_median"] / row["png"]["ms_per_frame_median"], 3)
        print(json.dumps(row), flush=True)
        out.append(row)
        for s in scenes:
            s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("jpeg_bench: no CUDA device")
    rt.set_device(0)
    import torch
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "devices": rt.device_count(), "library": rt.version()}
    res["encode"] = [r for c in ENCODE_CASES for r in encode_case(*c, a.iters)]
    res["sweep_c5"] = sweep_section(a.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
