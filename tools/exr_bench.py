"""OpenEXR encoding on the GPU, measured; writes one JSON file.

  python tools/exr_bench.py --out profiles/r08_exr_bench.json

For C1-C4 the float colour frame and the AOV frame are rendered into device memory (rt_render_frame_multi_f32 / _aov,
one GPU; their kernel times from rt_stats), then encoded as the colour-only (4 channels) and the 12-channel file.
Per file: the encode kernels' mean time from torch.profiler (exr_encode_pieces + exr_assemble per encode, over
`--rounds` encodes after a warm-up), the time of a whole rt_encode_exr call into device memory from CUDA events, and
the file size against the raw float bytes and against the PFM files `--format pfm [--aov]` writes.  Then the wall
time of `rtrace --format exr --aov` against `rtrace --format pfm --aov` at C3 geometry, alternating.  The card's name
and power limit are read in the same run."""
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

CASES = [("C1", 1024, 768, 4, 8), ("C2", 3840, 2160, 1, 8), ("C3", 3840, 2160, 4, 9), ("C4", 7680, 4320, 4, 9)]
KERNELS = ("exr_encode_pieces", "exr_assemble")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.strip().splitlines()]


def summary(xs):
    return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4), "n": len(xs)}


def pfm_bytes(w, h, channels):
    return len(b"PF\n%d %d\n-1.0\n" % (w, h)) + w * h * 4 * channels


def encode_case(name, w, h, spp, level, rounds, warmup):
    import torch
    scene = rt.Scene(level=level)
    o = rt.RenderOptions(w, h, spp)
    rgba = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    aov = torch.empty((h, w, 8), dtype=torch.float32, device="cuda")
    render = {}
    for what, fn, t in (("f32", rt.Renderer.render_f32, rgba), ("aov", rt.Renderer.render_aov, aov)):
        ks = []
        for _ in range(warmup + 5):
            _, st = fn(o, scene, out_ptr=t.data_ptr(), want_stats=True)
            ks.append(st.kernel_ms)
        render[what + "_kernel_ms"] = summary(ks[warmup:])
    scene.close()
    L, n = rt.lib(), rt.C.c_size_t()
    stream = torch.cuda.current_stream()
    res = {"case": name, "width": w, "height": h, "spp": spp, "level": level, **render, "files": []}
    for channels, aov_ptr in ((4, None), (12, aov.data_ptr())):
        cap = rt.exr_bound(w, h, aov_ptr is not None)
        out = torch.empty(cap, dtype=torch.uint8, device="cuda")

        def enc():
            rc = L.rt_encode_exr(rgba.data_ptr(), 0, aov_ptr, 0, w, h, out.data_ptr(), cap, rt.C.byref(n),
                                 stream.cuda_stream)
            assert rc == rt.RT_OK, rt.lib().rt_last_error()
        for _ in range(warmup):
            enc()
        calls = []
        for _ in range(rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            enc()
            e1.record(stream)
            e1.synchronize()
            calls.append(e0.elapsed_time(e1))
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(rounds):
                enc()
            torch.cuda.synchronize()
        per = {}   # mean device time per launch of each kernel, ms
        for ev in prof.key_averages():
            for k in KERNELS:
                if k in ev.key and ev.count:
                    total = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                    per[k] = total / ev.count / 1e3
        kern = sum(per.values()) if len(per) == len(KERNELS) else None
        raw = w * h * 4 * channels
        pfm = pfm_bytes(w, h, 3) + (pfm_bytes(w, h, 3) * 2 + pfm_bytes(w, h, 1) * 2 if channels == 12 else 0)
        f = {"channels": channels, "bytes": n.value, "raw_float_bytes": raw, "over_raw": round(n.value / raw, 4),
             "pfm_bytes": pfm, "over_pfm": round(n.value / pfm, 4),
             "encode_kernels_mean_ms": round(kern, 4) if kern else None,
             "per_kernel_mean_ms": {k: round(v, 4) for k, v in per.items()},
             "rt_encode_exr_call_ms": summary(calls),
             "read_gb_per_s_over_kernels": round(raw / (kern * 1e-3) / 1e9, 1) if kern else None}
        res["files"].append(f)
        del out
    return res


def cli_case(rounds):
    bin_ = os.path.join(ROOT, "target", "release", "rtrace")
    w, h, spp, level = 3840, 2160, 4, 9
    times = {"exr": [], "pfm": []}
    with tempfile.TemporaryDirectory() as d:
        for r in range(rounds + 1):
            for fmt in ("exr", "pfm"):
                t0 = time.perf_counter()
                p = subprocess.run([bin_, "--format=" + fmt, "--aov", "--level=%d" % level, "--width=%d" % w,
                                    "--height=%d" % h, "--samples-per-pixel=%d" % spp, "--stats",
                                    os.path.join(d, "o." + fmt)], capture_output=True, text=True)
                dt = time.perf_counter() - t0
                assert p.returncode == 0, p.stderr
                if r:   # the first round warms the file system and the driver
                    times[fmt].append({"wall_s": round(dt, 3), "stats": p.stderr.strip()})
        sizes = {f: os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)}
    return {"geometry": [w, h, spp, level], "runs": times, "files": sizes,
            "exr_wall_s": summary([t["wall_s"] for t in times["exr"]]),
            "pfm_wall_s": summary([t["wall_s"] for t in times["pfm"]])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cli-rounds", type=int, default=3)
    a = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("exr_bench: no CUDA device")
    rt.set_device(0)
    res = {"gpu": gpu_info(), "cases": []}
    for c in CASES:
        res["cases"].append(encode_case(*c, rounds=a.rounds, warmup=a.warmup))
        print(json.dumps(res["cases"][-1]), flush=True)
    res["cli_c3_aov"] = cli_case(a.cli_rounds)
    print(json.dumps(res["cli_c3_aov"]), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
