"""Animated PNG output on the GPU, measured with host clocks around whole sweeps; writes one JSON file.

  python tools/apng_bench.py --out profiles/r04_apng_bench.json

* sweep: the C5 orbit (120 frames, 3840x2160, 4x4 samples, level 9) delivered end to end through
  rt_render_sweep_apng and rt_render_sweep_png, alternating, three rounds each, at N = 1 and at N = 2 and 8 GPUs when
  the box has them.  The callbacks keep each frame's length, never the 170 MB animation.  Every APNG round is checked
  against the size identity of DESIGN.md "Animated PNG" with the PNG round's frame lengths, and every payload against
  rt_apng_bound.
* cli: `rtrace --frames 48` with `--format apng` and with `--format png` (C5 geometry), wall time and bytes written;
  the animation's size is checked against the identity with the PNG files' sizes.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
import rtrace_b200 as rt  # noqa: E402

C5 = (3840, 2160, 4, 9, 120)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.strip().splitlines()]


def size_identity(png_sizes, h):
    """Length of the animation of frames whose stand-alone PNGs have `png_sizes` bytes (DESIGN.md "Animated PNG")."""
    n, c = len(png_sizes), (h + 15) // 16 + 2
    return sum(png_sizes) - 45 * (n - 1) + 20 + 38 * n + 4 * c * (n - 1)


def sweep(kind, scenes, cams):
    w, h, spp, _, _ = C5
    n = len(cams)
    lens = []
    opts = rt.RenderOptions(w, h, spp)
    t0 = time.perf_counter()
    if kind == "apng":
        st = rt.Renderer.render_sweep_apng(opts, scenes, n, cameras=cams, fps=24, on_frame=lambda f, b: lens.append(len(b)))
    else:
        st = rt.Renderer.render_sweep_png(opts, scenes, n, cameras=cams, on_frame=lambda f, b: lens.append(len(b)))
    el = time.perf_counter() - t0
    if len(lens) != n:
        raise RuntimeError("%s sweep delivered %d of %d frames" % (kind, len(lens), n))
    return {"ms_per_frame": round(el * 1e3 / n, 4), "primary_grays_per_s": round(st.primary_rays / el / 1e9, 2),
            "lens": lens}


def sweep_section(rounds):
    w, h, spp, level, n = C5
    cams = [rt.orbit_camera(f, n) for f in range(n)]
    bound = rt.apng_bound(w, h, n)
    out = []
    avail = rt.device_count()
    for ngpu in [g for g in (1, 2, 8) if g <= avail]:
        scenes = []
        for g in range(ngpu):
            rt.set_device(g)
            scenes.append(rt.Scene(level=level))
        rt.set_device(0)
        sweep("apng", scenes, cams[:8])   # warm-up: scratch, ring buffers, modules on every GPU
        sweep("png", scenes, cams[:8])
        res = {"apng": [], "png": []}
        checks = []
        for _ in range(rounds):
            for kind in ("apng", "png"):
                res[kind].append(sweep(kind, scenes, cams))
            a, p = res["apng"][-1]["lens"], res["png"][-1]["lens"]
            if sum(a) != size_identity(p, h) or max(a) > bound:
                raise RuntimeError("APNG size identity or bound violated: %d vs %d, max %d, bound %d"
                                   % (sum(a), size_identity(p, h), max(a), bound))
            checks.append({"apng_bytes": sum(a), "identity_bytes": size_identity(p, h), "max_payload": max(a),
                           "bound": bound})
        row = {"gpus": ngpu, "size_identity_checks": checks}
        for kind in ("apng", "png"):
            ms = sorted(r["ms_per_frame"] for r in res[kind])
            lens = res[kind][0]["lens"]
            row[kind] = {"ms_per_frame_rounds": [r["ms_per_frame"] for r in res[kind]], "ms_per_frame_median": ms[len(ms) // 2],
                         "primary_grays_per_s_best": max(r["primary_grays_per_s"] for r in res[kind]),
                         "bytes_per_frame": round(sum(lens) / len(lens)), "bytes_total": sum(lens), "frames": len(lens)}
        row["apng_over_png_ms"] = round(row["apng"]["ms_per_frame_median"] / row["png"]["ms_per_frame_median"], 3)
        out.append(row)
        for s in scenes:
            s.close()
    return out


def cli_section(frames, gpus):
    w, h, spp, level, _ = C5
    binary = os.path.join(ROOT, "target", "release", "rtrace")
    out = []
    for g in gpus:
        sizes = {}
        for fmt in ("apng", "png", "apng", "png"):
            with tempfile.TemporaryDirectory() as d:
                args = [binary, "--width=%d" % w, "--height=%d" % h, "--samples-per-pixel=%d" % spp, "--level=%d" % level,
                        "--frames=%d" % frames, "--gpus=%d" % g, "--stats", "--format=%s" % fmt, "s.png"]
                t0 = time.perf_counter()
                r = subprocess.run(args, cwd=d, capture_output=True, text=True)
                el = time.perf_counter() - t0
                if r.returncode != 0:
                    raise RuntimeError(r.stderr)
                files = sorted(os.listdir(d))
                sizes[fmt] = [os.path.getsize(os.path.join(d, f)) for f in files]
                out.append({"gpus": g, "format": fmt, "frames": frames, "files": len(files), "wall_s": round(el, 3),
                            "bytes_written": sum(sizes[fmt]), "stats": r.stderr.strip().splitlines()[-1]})
        if sizes["apng"] != [size_identity(sizes["png"], h)]:
            raise RuntimeError("rtrace --format apng wrote %s bytes, the identity gives %d"
                               % (sizes["apng"], size_identity(sizes["png"], h)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cli-frames", type=int, default=48)
    a = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("apng_bench: no CUDA device")
    rt.set_device(0)
    res = {"gpu": gpu_info(), "devices": rt.device_count(), "library": rt.version()}
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
