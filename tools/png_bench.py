"""PNG output on the GPU, measured with CUDA events and host clocks only; writes one JSON file.

  python tools/png_bench.py --out profiles/r03_png_bench.json

* encode: C1..C4 frames resident on the device, 50 back-to-back rt_encode_png calls into a device buffer after
  warm-up (host clock around the calls, each of which waits for its stream), then the two encoder kernels' own
  device time from torch.profiler in a separate pass; bytes out and GB/s of RGBA read over the kernel time.  The same
  profile of rt_encode_apng_frame (frame 1 of 120) gives apng_assemble's time against png_assemble's.
* sweep: the C5 orbit (120 frames, 3840x2160, 4x4 samples, level 9) delivered end to end through
  rt_render_sweep_png and rt_render_sweep_multi(rgb=1), alternating, three rounds each, at N = 1 and at N = 2 and 8
  GPUs when the box has them.  The callback keeps each frame's length and a CRC of its first KB, never a full hash.
* cli: `rtrace --frames 48` with and without `--format png` (C5 geometry), wall time and bytes written.
The card's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
import rtrace_b200 as rt  # noqa: E402

ENCODE_CASES = [("C1", 1024, 768, 4, 8), ("C2", 3840, 2160, 1, 8), ("C3", 3840, 2160, 4, 9), ("C4", 7680, 4320, 4, 9)]
C5 = (3840, 2160, 4, 9, 120)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.strip().splitlines()]


def encode_case(name, w, h, spp, level, iters):
    L = rt.lib()
    scene = rt.Scene(level=level)
    frame = rt.device_alloc(w * h * 4)
    cap, apng_cap = rt.png_bound(w, h), rt.apng_bound(w, h, 120)
    out = rt.device_alloc(apng_cap)
    n = C.c_size_t()
    try:
        rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, out_ptr=frame, want_stats=True)

        def one():
            rc = L.rt_encode_png(C.c_void_p(frame), w, h, 0, C.c_void_p(out), cap, C.byref(n), None)
            if rc != rt.RT_OK:
                raise rt.RtError(rc, L.rt_last_error().decode())
        for _ in range(5):
            one()
        t0 = time.perf_counter()
        for _ in range(iters):
            one()
        call_ms = (time.perf_counter() - t0) * 1e3 / iters
        kernel_us = profile_kernels(one, iters)
        bytes_out = n.value

        def one_apng():
            rc = L.rt_encode_apng_frame(C.c_void_p(frame), w, h, 0, 1, 120, 1, 24, C.c_void_p(out), apng_cap, C.byref(n),
                                        None)
            if rc != rt.RT_OK:
                raise rt.RtError(rc, L.rt_last_error().decode())
        for _ in range(5):
            one_apng()
        apng_kernel_us = profile_kernels(one_apng, iters)
        rgba = w * h * 4
        return {"case": name, "width": w, "height": h, "spp": spp, "level": level, "iters": iters,
                "bytes_out": bytes_out, "rgb_bytes": w * h * 3, "ratio": round(w * h * 3 / bytes_out, 2),
                "call_ms": round(call_ms, 4), "kernel_us": {k: round(v, 2) for k, v in kernel_us.items()},
                "kernel_total_us": round(sum(kernel_us.values()), 2),
                "apng_frame_kernel_us": {k: round(v, 2) for k, v in apng_kernel_us.items()},
                "rgba_read_gb_per_s": round(rgba / (sum(kernel_us.values()) * 1e-6) / 1e9, 1)}
    finally:
        rt.device_free(frame)
        rt.device_free(out)
        scene.close()


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
        for k in ("png_encode_rows", "apng_assemble", "png_assemble"):
            if k in e.name and e.device_type.name == "CUDA":
                tot[k] = tot.get(k, 0.0) + e.device_time
                break
    return {k: v / iters for k, v in tot.items()}


def sweep(kind, scenes, cams):
    w, h, spp, level, _ = C5
    n = len(cams)
    lens, crcs = [], []

    def cb(f, data):
        lens.append(len(data))
        crcs.append(zlib.crc32(data[:1024]))
    opts = rt.RenderOptions(w, h, spp)
    t0 = time.perf_counter()
    if kind == "png":
        st = rt.Renderer.render_sweep_png(opts, scenes, n, cameras=cams, on_frame=cb)
    else:
        def cb_rgb(f, a):
            buf = a.reshape(-1)
            lens.append(buf.size)
            crcs.append(zlib.crc32(buf[:1024].tobytes()))
        st = rt.Renderer.render_sweep_multi(opts, scenes, n, cameras=cams, rgb=True, on_frame=cb_rgb)
    el = time.perf_counter() - t0
    return {"ms_per_frame": round(el * 1e3 / n, 4), "primary_grays_per_s": round(st.primary_rays / el / 1e9, 2),
            "bytes_per_frame": round(sum(lens) / len(lens)), "frames": len(lens), "first_kb_crc": crcs[:3]}


def sweep_section(rounds):
    w, h, spp, level, n = C5
    cams = [rt.orbit_camera(f, n) for f in range(n)]
    out = []
    avail = rt.device_count()
    for ngpu in [g for g in (1, 2, 8) if g <= avail]:
        scenes = []
        for g in range(ngpu):
            rt.set_device(g)
            scenes.append(rt.Scene(level=level))
        rt.set_device(0)
        sweep("png", scenes, cams[:8])   # warm-up: scratch, ring buffers, modules on every GPU
        sweep("rgb", scenes, cams[:8])
        res = {"png": [], "rgb": []}
        for _ in range(rounds):
            for kind in ("png", "rgb"):
                res[kind].append(sweep(kind, scenes, cams))
        row = {"gpus": ngpu}
        for kind in ("png", "rgb"):
            ms = sorted(r["ms_per_frame"] for r in res[kind])
            row[kind] = {"ms_per_frame_rounds": [r["ms_per_frame"] for r in res[kind]], "ms_per_frame_median": ms[len(ms) // 2],
                         "primary_grays_per_s_best": max(r["primary_grays_per_s"] for r in res[kind]),
                         "bytes_per_frame": res[kind][0]["bytes_per_frame"], "frames": res[kind][0]["frames"]}
        row["png_over_rgb_ms"] = round(row["png"]["ms_per_frame_median"] / row["rgb"]["ms_per_frame_median"], 3)
        out.append(row)
        for s in scenes:
            s.close()
    return out


def cli_section(frames, gpus):
    w, h, spp, level, _ = C5
    binary = os.path.join(ROOT, "target", "release", "rtrace")
    out = []
    for g in gpus:
        for fmt in ("ppm", "png", "ppm", "png"):
            with tempfile.TemporaryDirectory() as d:
                name = "s.png" if fmt == "png" else "s.tga"
                args = [binary, "--width=%d" % w, "--height=%d" % h, "--samples-per-pixel=%d" % spp, "--level=%d" % level,
                        "--frames=%d" % frames, "--gpus=%d" % g, "--stats"] + (["--format=png"] if fmt == "png" else []) + [name]
                t0 = time.perf_counter()
                r = subprocess.run(args, cwd=d, capture_output=True, text=True)
                el = time.perf_counter() - t0
                if r.returncode != 0:
                    raise RuntimeError(r.stderr)
                written = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))
                out.append({"gpus": g, "format": fmt, "frames": frames, "wall_s": round(el, 3), "bytes_written": written,
                            "stats": r.stderr.strip().splitlines()[-1]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cli-frames", type=int, default=48)
    a = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("png_bench: no CUDA device")
    rt.set_device(0)
    import torch
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "devices": rt.device_count(), "library": rt.version()}
    res["encode"] = [encode_case(*c, a.iters) for c in ENCODE_CASES]
    print(json.dumps(res["encode"]), flush=True)
    res["sweep_c5"] = sweep_section(a.rounds)
    print(json.dumps(res["sweep_c5"]), flush=True)
    gpus = sorted({1, min(8, rt.device_count())})
    res["cli_frames"] = cli_section(a.cli_frames, gpus)
    print(json.dumps(res["cli_frames"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
