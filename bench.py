#!/usr/bin/env python
"""bench.py -- throughput of the rust-tracer hot path on B200 (one JSON line).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

A *step* is one pass of the hot path over one frame: ray generation, primary and shadow traversal, shading,
supersample averaging and RGBA8 quantisation of every pixel.

Default line = BASELINE.json configs[4] ("c5"), the largest single-GPU configuration: the 120-frame orbit of
the camera about the level-9 flake (87,381 spheres) at 3840x2160 with 4x4 samples; the job's K x N frames are
spread evenly over the orbit and step i of rank r renders the (i*N + r)-th of them, so N ranks shard the sweep by
frame (no data-path collective, weak scaling) and every N renders the same mix of cheap and expensive frames.
Frame 0 is BASELINE configs[2] ("c3").  The same invocation also measures, as sub-records under `also`:
  c2        configs[1]: the reference's 20k-sphere scene at 3840x2160, 1 spp (the headline 4K render)
  c4        configs[3], 8K multi-frame: 7680x4320, 4x4, level-9 frames, whole frames per rank (weak scaling)
  c4_bands  configs[3] at N>1: ONE such frame split into interleaved 16-row blocks over the N ranks (strong
            scaling); kernel-only the blocks land in rank 0's device frame through CUDA-IPC peer stores over
            NVLink, end to end every rank copies its blocks into one shared pinned host frame over its own
            PCIe link; a cross-rank barrier closes every frame (frame latency, not throughput)
`--workload X` measures one workload alone (c1/c2/c3/c3l10/c4/c5), `--mode bands` its row-band split.
`--steps K` is the number of timed steps of every measurement (kernel-only and end to end, sub-records included).
`--dump-outputs DIR` writes, after the timed steps, the frame the kernel-only path computed in its last step as
DIR/<workload>.npy (float32 RGBA values; rank 0's frame; a fixed seeded sample of a frame too large for the run's
DUMP_BYTES), so that two builds can be compared output for output: the scenes and cameras of a run depend on its
arguments only.

metric  = Mrays/s (primary + shadow rays, counted as the reference's work is counted)
value   = whole-job rays / device time of the K steps (CUDA events on the launch stream, max over ranks),
          frames written to HBM, nothing leaves the GPU
e2e     = the same metric through the C ABI with HOST output buffers: rt_render_sweep_rgb, every frame delivered
          to pinned host memory (device-to-host copy inside the timed region)
roofline.frac = EXECUTED FP32 work / measured FFMA peak (hardware view, <= 1); roofline.reference_work is
          SURVEY 8(d)'s figure (rays x the reference algorithm's flop/ray / time), which exceeds the peak
          because the candidate lists skip most of the reference's sphere tests.
"""
import argparse
import hashlib
import json
import mmap
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))

WORKLOADS = {
    # name: (width, height, spp, level)
    "c1": (1024, 768, 4, 8),     # `make image`
    "c2": (3840, 2160, 1, 8),    # BASELINE configs[1]: the headline single-GPU 4K render
    "c3": (3840, 2160, 4, 9),    # deeper flake (87,381 spheres), 4x4 supersampling
    "c3l10": (3840, 2160, 4, 10),
    "c4": (7680, 4320, 4, 9),
    "c5": (3840, 2160, 4, 9),    # BASELINE configs[4]: 120-frame orbit sweep of C3-sized frames, frame f -> rank f mod N
}
DEFAULT_WORKLOAD = "c5"
ORBIT_FRAMES = 120               # c5: eye and camera basis rotated about the flake's axis by 2 pi f / 120 (SURVEY F6)
# SURVEY 8(d): algorithmic flop per ray of REFERENCE work (17 T + 3 P + 19 U + 20 f_p + 30 f_s),
# from the oracle's counters (tests/golden/oracle_derived.json); used when the fixture lacks the config.
FLOP_PER_RAY_FALLBACK = 645.0
METRIC = "Mrays/s (primary+shadow)"
DUMP_BYTES = 64 * 10 ** 6        # --dump-outputs: all files of one run together, .npy headers included
DUMP_SEED = 20261020
KERNEL_SOURCES = ("rt_phased.cu", "rt_cull.cuh", "rt_pack.cuh", "rt_device.cuh", "rt_kernels.cu", "rt_tile.cu")


def orbit_basis(frame, n_frames=ORBIT_FRAMES, eye=(0.0, 0.0, -4.0)):
    """(eye, right, up, forward) of orbit frame `frame`: the reference camera (render.rs:145-166, 238-243)
    rotated about the vertical axis; frame 0 is the reference camera exactly.  Same arithmetic as
    rtrace_b200.orbit_camera and the CLI's --frames (host/main.cpp)."""
    import math
    th = 2.0 * math.pi * frame / n_frames
    c, s = (1.0, 0.0) if frame % n_frames == 0 else (math.cos(th), math.sin(th))

    def rot(v):
        return (c * v[0] + s * v[2], v[1], -s * v[0] + c * v[2])
    return rot(eye), rot((1, 0, 0)), (0, 1, 0), rot((0, 0, 1))


def orbit_frame(k, total):
    """Orbit frame of the k-th of a job's `total` frames: the job's frames are spread evenly over the 120-frame orbit
    (frame cost varies 1.6x around it), so that runs with different step counts or GPU counts render the same mix and
    their throughputs compare; with total = 120 it is frame k."""
    return (k * ORBIT_FRAMES // max(total, 1)) % ORBIT_FRAMES


def workload_name(name, level, width, height, spp):
    s = "%s: pyramid level %d (%d spheres) at %dx%d, %d spp" % (name, level, (4 ** level - 1) // 3, width, height,
                                                               spp * spp)
    if name == "c5":
        s += ", %d-frame orbit sweep (the job's steps x N frames spread evenly over the orbit; frame i*N + r on rank r)" % ORBIT_FRAMES
    return s


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_names(args, world):
    """The files a run with these arguments writes under --dump-outputs, one per measurement; rank 0 writes them all."""
    workload = args.workload or DEFAULT_WORKLOAD
    if args.impl == "reference":
        return [workload]
    names = [workload + "_bands" if args.mode == "bands" and world > 1 else workload]
    if args.workload is None and not args.no_also:
        names += ["c2", "c4"] + (["c4_bands"] if world > 1 else [])
    return names


def dump_pixels(n_files):
    """Pixels kept per frame when a run writes n_files frames: DUMP_BYTES split evenly, 16 bytes a pixel (float32
    RGBA), 4 KiB per file left for the .npy header."""
    return (DUMP_BYTES // n_files - 4096) // 16


def sample_pixels(frame, pixels):
    """An (h, w, 4) RGBA8 frame as float32 (n, 4), pixels in row-major order: the whole frame if it has at most
    `pixels` pixels, else the same seeded sample of `pixels` of them in every run."""
    import numpy as np
    px = np.asarray(frame).reshape(-1, 4)
    if len(px) > pixels:
        px = px[np.sort(np.random.default_rng(DUMP_SEED).choice(len(px), pixels, replace=False))]
    return px.astype(np.float32)


def dump_frame(args, world, name, frame):
    """--dump-outputs: the frame as <DIR>/<name>.npy, sampled so that the run's files stay within DUMP_BYTES."""
    import numpy as np
    names = dump_names(args, world)
    if name not in names:
        raise RuntimeError("bench.py: %s is not among the files this run writes (%s)" % (name, names))
    os.makedirs(args.dump_outputs, exist_ok=True)
    path = os.path.join(args.dump_outputs, name + ".npy")
    np.save(path, sample_pixels(frame, dump_pixels(len(names))))
    log("bench.py: wrote", path)


def oracle_case(width, height, spp, level):
    try:
        for c in json.load(open(os.path.join(ROOT, "tests", "golden", "oracle_derived.json")))["cases"]:
            if (c["width"], c["height"], c["spp"], c["level"]) == (width, height, spp, level):
                return c
    except Exception:
        pass
    return None


def flop_per_ray(width, height, spp, level):
    c = oracle_case(width, height, spp, level)
    if c:
        return c["flop_per_ray"], "oracle counters for this exact config (tests/golden/oracle_derived.json)"
    try:
        for c in json.load(open(os.path.join(ROOT, "tests", "golden", "oracle_derived.json")))["cases"]:
            if (c["width"], c["height"]) == (width, height):   # same resolution, other level: flat in depth (BASELINE.md 2)
                return c["flop_per_ray"], "oracle counters at %dx%d level %d" % (width, height, c["level"])
    except Exception:
        pass
    return FLOP_PER_RAY_FALLBACK, "SURVEY 8(d) figure for C2"


def kernel_source_hash():
    """sha256 over the kernel sources: a committed ncu capture describes the running kernels only if it was
    taken from the same sources (profiles/latest_summary.json records the hash it was captured at)."""
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        try:
            h.update(open(os.path.join(ROOT, "rust-tracer_b200", "csrc", name), "rb").read())
        except OSError:
            h.update(b"?")
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the benchmark runs (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, windows):
        """windows: [(t_begin, t_end)] of the timed regions; samples inside them are 'under load'."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        ok = [(t, r) for (t, r) in self.rows if len(r) >= 7]
        rows = [r for (t, r) in ok if any(a - 0.02 <= t <= b + 0.05 for a, b in windows)]
        under_load = len(rows)
        if not rows:
            rows = [r for (_, r) in ok]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]

        def num(s):
            try:
                return float(s)
            except ValueError:
                return None
        sm = [num(r[0]) for r in rows if num(r[0]) is not None]
        pw = [num(r[2]) for r in rows if num(r[2]) is not None]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": num(rows[0][1]),
                "power_w_max": max(pw) if pw else None, "samples": len(ok), "samples_under_load": under_load,
                "reasons": reasons}


class stdout_to_stderr:
    """File descriptor 1 points at stderr inside the block.  NCCL prints "NCCL version ..." on stdout when the
    first communicator is created; bench.py's stdout carries exactly one JSON line, so that goes to stderr."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def pin_to_gpu_cpus(local_rank):
    """Keep this rank's host threads (and so its pinned frame buffers, first touch) on the CPUs NVML reports as
    local to its GPU, so that frames copied out do not cross sockets (at N=1 too: the end-to-end number is a
    host-link number)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d cpus local to GPU %d" % (len(cpus), idx)
    except Exception as e:   # best effort
        return "not pinned (%s)" % type(e).__name__
    return "not pinned"


# ---------------------------------------------------------------------------------------------------
# CPU legs (the oracle: test infrastructure, allowed here as the reported baseline only)
# ---------------------------------------------------------------------------------------------------
def cpu_frames(workload, width, height, spp, level, frames, threads):
    """Whole frames of the workload on `threads` host threads -> (rays, seconds, flop/ray of the last frame, last frame)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle as o   # bench.py's cpu_baseline / reference legs are allowed to run the oracle
    s = o.Scene(level=level)
    rays = secs = 0.0
    ctr = img = None
    for f in frames:
        cam = o.make_camera(*orbit_basis(f % ORBIT_FRAMES)) if workload == "c5" else None   # f: an orbit frame index
        t0 = time.perf_counter()
        img, ctr = s.render_rows(width, height, spp, 0, 1, height, threads=threads, camera=cam)
        secs += time.perf_counter() - t0
        rays += ctr.primary_rays + ctr.shadow_rays
    return rays, secs, (ctr.flop_per_ray() if ctr else None), img


def cpu_leg(workload, width, height, spp, level, budget_s=12.0):
    """cpu_baseline of the native line: whole frames of the same workload on every host core, bounded to about
    `budget_s` seconds (at least one frame)."""
    cores = os.cpu_count() or 1
    rays = secs = 0.0
    n, fpr = 0, None
    while n == 0 or (secs < budget_s and secs / n * (n + 1) < 2.5 * budget_s):
        r, s, fpr, _ = cpu_frames(workload, width, height, spp, level, [(n * 47) % ORBIT_FRAMES], cores)   # 0, 47, 94, 21, ..: spread
        rays, secs, n = rays + r, secs + s, n + 1
    what = "orbit frame(s) %s" % [(k * 47) % ORBIT_FRAMES for k in range(n)] if workload == "c5" else "%d repeat(s) of the frame" % n
    return {"value": rays / secs / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": "%s, whole %dx%d spp %d level %d frames, %.1f s" % (what, width, height, spp, level, secs),
            "flop_per_ray": fpr}


def run_reference(args, workload):
    """--impl reference: the reference's CPU algorithm (oracle port; the Rust crate cannot be built here: no
    cargo/rustc) on all host threads -- same metric, same config, whole frames, the same warm-up and step counts
    as the native arm.  Rank 0 only.  A run that would pass ~200 s stops early and says so in `steps`."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    width, height, spp, level = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    t_all = time.perf_counter()
    wdone = 0
    for i in range(args.warmup):
        cpu_frames(workload, width, height, spp, level, [orbit_frame(i, args.steps)], cores)
        wdone += 1
        if time.perf_counter() - t_all > 60.0:
            break
    rays = secs = 0.0
    done = 0
    for i in range(args.steps):
        r, s, _, img = cpu_frames(workload, width, height, spp, level, [orbit_frame(i, args.steps)], cores)   # the native arm's mix
        rays, secs, done = rays + r, secs + s, done + 1
        if time.perf_counter() - t_all > 200.0:   # keep the whole run within a few minutes on any host
            break
    if args.dump_outputs:   # the last frame rendered; only c5's frame changes from step to step
        if done < args.steps and workload == "c5":
            log("bench.py: the reference arm stopped after %d of %d steps; %s.npy holds orbit frame %d, the native arm's "
                "holds orbit frame %d" % (done, args.steps, workload, orbit_frame(done - 1, args.steps),
                                          orbit_frame(args.steps - 1, args.steps)))
        dump_frame(args, 1, workload, img)
    v = rays / secs / 1e6
    sample = "each step = one whole %dx%d spp %d level %d frame%s on %d host threads; %d of %d steps timed" % (
        width, height, spp, level, " (orbit frame i)" if workload == "c5" else "", cores, done, args.steps)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": done,
        "warmup": wdone, "ms_per_step": secs / done * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(workload, level, width, height, spp)},
        "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------------------
# native arm
# ---------------------------------------------------------------------------------------------------
class Job:
    """Process-wide state of the native arm: rank / world, device, library, clocks."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import rtrace_b200 as rt   # raises ImportError if the CUDA library is not built: no fallback
        self.torch, self.dist, self.rt, self.args = torch, dist, rt, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.cpu_note = None if os.environ.get("RTRACE_NO_PIN") else pin_to_gpu_cpus(self.local_rank)
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU fallback (use --impl reference)")
        torch.cuda.set_device(self.local_rank)
        rt.set_device(self.local_rank)
        if self.world > 1:
            with stdout_to_stderr():   # communicator creation and the first collective: NCCL's banner
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
                dist.barrier()
        rt.set_variant(args.variant)
        self.stream = torch.cuda.current_stream()
        self.flush = None if args.no_l2_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        self.windows = []
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        self.sampler = ClockSampler(vis.split(",")[self.local_rank] if vis else torch.cuda.current_device()) \
            if self.rank == 0 else None
        self.peaks = {}
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        self._fp32 = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values):
        """(max over ranks, sum over ranks) of a list of floats."""
        t = self.torch.tensor(values, dtype=self.torch.float64, device="cuda")
        if self.world == 1:
            return t.tolist(), t.tolist()
        tmax, tsum = t.clone(), t.clone()
        self.dist.all_reduce(tmax, op=self.dist.ReduceOp.MAX)
        self.dist.all_reduce(tsum, op=self.dist.ReduceOp.SUM)
        return tmax.tolist(), tsum.tolist()

    def fp32_peak(self):
        if self._fp32 is None:
            try:
                tf, mhz = self.rt.measure_fp32_peak(self.local_rank)
                self._fp32 = (tf, "measured live: FFMA chains on all SMs (rt_measure_fp32_peak), effective %.0f MHz; "
                                  "MEASURED_PEAKS.json has no FP32 entry" % mhz)
            except Exception as e:   # pragma: no cover
                self._fp32 = (148 * 128 * 2 * 1.965e9 / 1e12, "nominal 148 SM x 128 lanes x 2 x 1965 MHz (%s)" % e)
        return self._fp32

    def timed(self, steps, step_fn, pre_fn=None):
        """K steps between CUDA events on the launch stream, L2 flushed before each (outside the events).
        Returns (device ms summed over the steps, wall ms)."""
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t_begin = time.time()
        w0 = time.perf_counter()
        for i, (a, b) in enumerate(ev):
            if self.flush is not None:
                self.flush.zero_()          # evict L2 (126 MB) between timed steps; outside the event pair
            if pre_fn:
                pre_fn(i)
            a.record(self.stream)
            step_fn(i)
            b.record(self.stream)
        self.barrier()
        wall_ms = (time.perf_counter() - w0) * 1e3
        self.windows.append((t_begin, time.time()))
        return sum(a.elapsed_time(b) for a, b in ev), wall_ms

    def pcie(self, nbytes):
        """Copy-only ceiling of the end-to-end numbers: after a barrier every rank copies `nbytes` frames device ->
        pinned host (a ring of three buffers, as the sweep's) at the same time.  Returns (job ceiling, rank 0's own
        rate, fastest rank's rate) in GB/s; the ceiling is world x the SLOWEST rank's rate: every rank delivers the
        same number of frames, so the slowest host link bounds the job (the sum of the ranks' rates would count the
        speed-up the fast ranks see once the slow ones are the only ones left copying)."""
        self.barrier()
        g = self.rt.microbench_d2h(nbytes, 24, 3)
        t = self.torch.tensor([g, -g], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        gmax, gmin = t[0].item(), -t[1].item()
        return gmin * self.world, g, gmax


def roofline_block(job, workload, width, height, spp, level, rays_per_launch, ms_per_step, fb_bytes, frames=None):
    """Hardware view first: executed FP32 flops per frame (from the committed ncu capture of THIS workload, used
    only if it was taken from the same kernel sources) / live time / live FFMA peak.  SURVEY 8(d)'s reference-work
    figure travels beside it under its own name.  frames: the orbit frames the timed steps rendered (c5)."""
    peak_tf, peak_src = job.fp32_peak()
    fpr, fpr_src = flop_per_ray(width, height, spp, level)
    ref_tf = rays_per_launch * fpr / (ms_per_step * 1e-3) / 1e12
    cap, note = None, "no ncu capture of this workload in profiles/latest_summary.json"
    try:
        summ = json.load(open(os.path.join(ROOT, "profiles", "latest_summary.json")))
        c = summ.get("workloads", {}).get(workload)
        if c and summ.get("kernel_source_hash") == kernel_source_hash():
            cap, note = dict(c), None
            if "fp32_flop_per_orbit_frame" in c:   # c5: mean over the orbit frames this run timed
                tab, fr = c["fp32_flop_per_orbit_frame"], (frames or [0])
                cap["fp32_flop_per_frame"] = sum(tab[f % len(tab)] for f in fr) / len(fr)
                wtab = c.get("warp_instructions_per_orbit_frame")
                if wtab:
                    cap["warp_instructions_per_frame"] = sum(wtab[f % len(wtab)] for f in fr) / len(fr)
        elif c:
            note = "the committed capture (%s) was taken from other kernel sources: not used" % summ.get("kernel_source_hash")
    except Exception:
        pass
    hbm_peak = job.peaks.get("hbm_gbs", 6650.0)
    out = {"bound": "fp32", "unit": "TFLOP/s", "peak": peak_tf, "peak_source": peak_src}
    if cap:
        ex_tf = cap["fp32_flop_per_frame"] / (ms_per_step * 1e-3) / 1e12
        out.update({
            "achieved": ex_tf, "frac": ex_tf / peak_tf, "traffic": cap.get("dram_bytes_per_frame"),
            "executed": {k: cap[k] for k in ("fp32_flop_per_frame", "warp_instructions_per_frame", "fma_pipe_active_pct",
                                             "issue_active_pct", "dominant_kernel", "dominant_kernel_share", "source")
                         if k in cap},
            "note": "achieved = FP32 flops the kernels EXECUTE per frame (ncu thread-level FADD + FMUL + 2 FFMA counts of this "
                    "workload, committed capture of the same kernel sources; the work is deterministic) / live event time; "
                    "traffic = DRAM bytes per frame of the same capture (cold L2: ncu flushes it between replays); "
                    "fma_pipe_active_pct = ncu's own FMA-pipe utilisation over the frame's elapsed cycles"})
    else:
        out.update({"achieved": None, "frac": None, "traffic": None, "executed": None, "note": note})
    out["reference_work"] = {
        "achieved": ref_tf, "frac_of_peak": ref_tf / peak_tf, "flop_per_ray": fpr,
        "note": "SURVEY 8(d): rays/launch x algorithmic flop/ray of the REFERENCE walk (%s) / event time. Not a hardware "
                "roofline: the candidate lists replace ~34 sphere tests per ray by 1-2 exact tests, so this exceeds the "
                "FP32 peak on supersampled frames" % fpr_src}
    hb = fb_bytes / (ms_per_step * 1e-3) / 1e9
    out["hbm"] = {"achieved": hb, "peak": hbm_peak, "unit": "GB/s", "frac": hb / hbm_peak,
                  "note": "algorithmic HBM bytes = framebuffer written once (4 B/pixel); peak = MEASURED_PEAKS.json hbm_gbs"
                          if job.peaks else "peak = fallback 6.65 TB/s"}
    return out


def measure_frames(job, workload, steps, warmup, cpu_baseline=False):
    """Whole frames per rank (frame-sharded; for c5 the orbit): kernel-only `value` and the end-to-end sweep."""
    rt, torch = job.rt, job.torch
    rank, world = job.rank, job.world
    width, height, spp, level = WORKLOADS[workload]
    sweep = workload == "c5"
    scene = rt.Scene(level=level)
    opts = rt.RenderOptions(width, height, spp)
    cams = [rt.make_camera(*orbit_basis(f)) for f in range(ORBIT_FRAMES)] if sweep else None

    def frame_of(i):   # c5: step i of this rank is frame i * world + rank of the job's steps * world frames
        return orbit_frame(i * world + rank, steps * world)
    fb = torch.zeros((height, width, 4), dtype=torch.uint8, device="cuda")
    _, st0 = rt.Renderer.render_rows(opts, scene, out_ptr=fb.data_ptr(), stream=job.stream.cuda_stream, want_stats=True)
    launches_per_step, variant_used = int(st0.kernel_launches), int(st0.variant_used)
    e2e_steps = steps
    # rays of this rank's steps, counted on the device the way the reference's work is counted
    if sweep:
        table = {f: scene.count_rays(width, height, spp, camera=cams[f]) for f in sorted({frame_of(i) for i in range(steps)})}
        primary = sum(table[frame_of(i)][0] for i in range(steps)) / steps
        shadow = sum(table[frame_of(i)][1] for i in range(steps)) / steps
    else:
        primary, shadow = scene.count_rays(width, height, spp)
    rays_rank = primary + shadow

    def step(i):
        rt.Renderer.render_rows(opts, scene, camera=cams[frame_of(i)] if sweep else None, out_ptr=fb.data_ptr(),
                                stream=job.stream.cuda_stream)
    for i in range(warmup):
        step(i)
    job.barrier()
    dev_ms, wall_ms = job.timed(steps, step)
    if job.args.dump_outputs and rank == 0:   # fb holds the frame of the last timed step (job.timed synchronises)
        dump_frame(job.args, world, workload, fb.cpu().numpy())

    # ---- e2e: the C-ABI call a user makes, every frame delivered to HOST memory ----
    # All ranks PULL frames from one queue (a counter in shared memory, rt_render_sweep_pull): the job is
    # e2e_steps x world frames, and a rank whose host link is slower under load takes fewer of them.
    seen = []

    def on_frame(f, arr):
        seen.append(int(arr[0, 0, 0]))   # touch the host copy of every frame

    queue = SharedCounter(job, workload)

    def e2e_run(total):
        queue.reset()
        job.barrier()
        taken = [0]

        def next_frame():
            i = rt.atomic_fetch_add_u64(queue.ptr, 1)
            if i >= total:
                return None
            taken[0] += 1
            return i, (cams[orbit_frame(i, total)] if sweep else None)
        rt.Renderer.render_sweep_pull(opts, scene, next_frame, on_frame=on_frame, rgb=True)
        return taken[0]
    e2e_run(3 * world)
    job.barrier()
    t_begin = time.time()
    e0 = time.perf_counter()
    my_frames = e2e_run(e2e_steps * world)
    job.barrier()
    e2e_ms = (time.perf_counter() - e0) * 1e3
    job.windows.append((t_begin, time.time()))
    queue.close()
    if sweep:   # rays of the job's e2e_steps * world frames, counted on the device
        total = e2e_steps * world
        if rank == 0:
            for f in sorted({orbit_frame(i, total) for i in range(total)}):
                if f not in table:
                    table[f] = scene.count_rays(width, height, spp, camera=cams[f])
        e2e_rays_job_total = sum(sum(table[orbit_frame(i, total)]) for i in range(total)) if rank == 0 else 0.0
    else:
        e2e_rays_job_total = float(primary + shadow) * e2e_steps * world
    d2h = width * height * 3
    pcie_sum, pcie_own, pcie_fast = job.pcie(d2h)

    (dev_ms, e2e_ms, _, fr_max), (_, _, rays_job, _) = job.reduce([dev_ms, e2e_ms, float(rays_rank), float(my_frames)])
    (_, fr_min), _ = job.reduce([0.0, -float(my_frames)])
    if rank != 0:
        return None
    ms_per_step = dev_ms / steps
    e2e_step = e2e_ms / e2e_steps          # time per `world` frames = per frame per GPU on average
    e2e_rays_job = e2e_rays_job_total / e2e_steps
    rec = {
        "metric": METRIC, "value": rays_job / (ms_per_step * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": workload_name(workload, level, width, height, spp),
            "partition": "one whole frame per rank per step (frame-sharded sweep), no collective",
            "l2": "not flushed" if job.flush is None else "flushed between steps (256 MiB memset, outside the timed events)",
            "rays_per_frame": {"primary": primary, "shadow": shadow},
            "mpixels_per_s": width * height * world / (ms_per_step * 1e-3) / 1e6,
            "variant": job.args.variant, "variant_used": variant_used,
            "wall_ms_per_step_incl_flush": wall_ms / steps, "host_cpus": job.cpu_note,
        },
        "roofline": roofline_block(job, workload, width, height, spp, level, rays_job / world, ms_per_step, width * height * 4,
                                   frames=[frame_of(i) for i in range(steps)] if sweep else None),
        "e2e": {"value": e2e_rays_job / (e2e_step * 1e-3) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": 512,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_step,
                "pcie": {"achieved_gbs": d2h * world / (e2e_step * 1e-3) / 1e9, "ceiling_gbs": pcie_sum,
                         "frac": d2h * world / (e2e_step * 1e-3) / 1e9 / pcie_sum, "rank0_gbs": pcie_own,
                         "fastest_rank_gbs": pcie_fast,
                         "note": "achieved = frame bytes leaving all GPUs / e2e time; ceiling = world x the slowest rank's copy-only "
                                 "rate with every rank copying at once into a ring of three pinned host buffers, as the "
                                 "sweep does (rt_microbench_d2h, no kernels)"},
                "frames_per_rank": {"min": -fr_min, "max": fr_max, "job": e2e_steps * world},
                "note": "rt_render_sweep_pull (the engine under `rtrace --frames K --gpus N`): the job's steps x N frames sit in one "
                        "queue (a counter in shared memory) and every rank pulls the next one when its pipeline has room; per "
                        "frame the kernel-parameter blocks (camera, options) go in and the RGB8 frame -- the body of the "
                        "reference's P6 file, its sink drops alpha (render.rs:389-397) -- comes out to pinned host memory; two "
                        "frames render at a time while an earlier one is copied out.  ms_per_step = job time / steps"},
        "gpu_launches": steps * world * launches_per_step,
    }
    if cpu_baseline:
        rec["cpu_baseline"] = cpu_leg(workload, width, height, spp, level)
    return rec


class SharedCounter:
    """A 64-bit counter in a POSIX shared-memory segment every rank maps: the frame queue of the end-to-end sweep."""

    def __init__(self, job, tag):
        import ctypes
        self.job = job
        self.path = "/dev/shm/rtrace_bench_%s_%s_queue" % (os.environ.get("MASTER_PORT", "0"), tag)
        if job.rank == 0:
            with open(self.path, "wb") as f:
                f.write(b"\0" * 64)
        job.barrier()
        self.f = open(self.path, "r+b")
        self.mm = mmap.mmap(self.f.fileno(), 64)
        self.ptr = ctypes.addressof(ctypes.c_char.from_buffer(self.mm))

    def reset(self):
        self.job.barrier()
        if self.job.rank == 0:
            self.mm[:8] = b"\0" * 8
        self.job.barrier()

    def close(self):
        self.job.barrier()
        if self.job.rank == 0:
            try:
                os.unlink(self.path)
            except OSError:
                pass


class SharedHostFrame:
    """One frame in a POSIX shared-memory segment, page-locked in every rank: each GPU copies its row blocks into
    it over its own PCIe link, rank 0 (the sink) reads the whole frame."""

    def __init__(self, job, nbytes, tag):
        self.job, self.nbytes = job, nbytes
        self.path = "/dev/shm/rtrace_bench_%s_%s" % (os.environ.get("MASTER_PORT", "0"), tag)
        if job.rank == 0:
            with open(self.path, "wb") as f:
                f.truncate(nbytes)
        job.barrier()
        self.f = open(self.path, "r+b")
        self.mm = mmap.mmap(self.f.fileno(), nbytes)
        import ctypes
        import numpy as np
        self.array = np.frombuffer(self.mm, dtype=np.uint8)
        self.ptr = ctypes.addressof(ctypes.c_char.from_buffer(self.mm))
        job.rt.host_register(self.ptr, nbytes)

    def close(self):
        try:
            self.job.rt.host_unregister(self.ptr)
        except Exception:
            pass
        self.job.barrier()
        self.array = None
        if self.job.rank == 0:
            try:
                os.unlink(self.path)
            except OSError:
                pass


def measure_bands(job, workload, steps, warmup, gather="peer"):
    """ONE frame per step split over the ranks in interleaved 16-row blocks (strong scaling).  Kernel-only: the
    kernels store straight into rank 0's device frame through CUDA-IPC peer memory (NVLink), a cross-rank barrier
    closes every frame.  End to end: every rank renders its blocks and copies them into one shared pinned HOST
    frame over its own PCIe link; barrier; the frame is complete in rank 0's address space."""
    rt, torch, dist = job.rt, job.torch, job.dist
    rank, world = job.rank, job.world
    from rtrace_b200 import partition
    width, height, spp, level = WORKLOADS[workload]
    scene = rt.Scene(level=level)
    opts = rt.RenderOptions(width, height, spp)
    block = 16
    row_start, row_stride, row_block, my_rows = partition.block_band_spec(height, rank, world, block)
    row_bytes = width * 4
    # rank 0 owns the device frame; the others map it through a CUDA IPC handle
    handle = torch.zeros(64, dtype=torch.uint8, device="cuda")
    if rank == 0:
        frame_base = rt.device_alloc(height * row_bytes)
        handle.copy_(torch.frombuffer(bytearray(rt.ipc_export(frame_base)), dtype=torch.uint8))
    if world > 1:
        dist.broadcast(handle, src=0)
    if rank != 0:
        frame_base = rt.ipc_open(bytes(handle.cpu().numpy().tobytes()))
    own = torch.zeros((height, width, 4), dtype=torch.uint8, device="cuda")   # e2e: this rank's blocks at their image rows
    nccl_band = torch.zeros((partition.band_capacity(height, world), width, 4), dtype=torch.uint8, device="cuda")
    gathered = [torch.zeros_like(nccl_band) for _ in range(world)] if (gather == "nccl" and rank == 0) else None

    st0 = rt.Renderer.render_row_blocks(opts, scene, row_start, row_stride, row_block, my_rows, own.data_ptr(),
                                        pitch=row_bytes, absolute_rows=True, stream=job.stream.cuda_stream, want_stats=True)
    launches_per_step = int(st0.kernel_launches)
    primary_all, shadow_all = scene.count_rays(width, height, spp)
    rays_frame = primary_all + shadow_all
    sync_flag = torch.zeros(1, device="cuda")

    def frame_sync():   # cross-rank: every rank's kernels of this frame have finished (NCCL all-reduce on the stream)
        if world > 1:
            dist.all_reduce(sync_flag)

    def step(i, synced=True):
        if gather == "nccl":
            s0, s1, n = partition.band_spec(height, rank, world)
            rt.Renderer.render_rows(opts, scene, row_start=s0, row_stride=s1, row_count=n, out_ptr=nccl_band.data_ptr(),
                                    stream=job.stream.cuda_stream)
            dist.gather(nccl_band, gathered, dst=0)
            return
        rt.Renderer.render_row_blocks(opts, scene, row_start, row_stride, row_block, my_rows, frame_base, pitch=row_bytes,
                                      absolute_rows=True, stream=job.stream.cuda_stream)
        if synced:
            frame_sync()
    for i in range(warmup):
        step(i)
    job.barrier()
    dev_ms, wall_ms = job.timed(steps, step)
    thr_ms, _ = job.timed(steps, lambda i: step(i, synced=False)) if gather == "peer" else (dev_ms, 0)

    # the gathered device frame against the ORACLE's hash of this configuration
    verified = None
    job.barrier()
    case = oracle_case(width, height, spp, level)
    if rank == 0 and gather == "peer":
        got = rt.PinnedBuffer(height * row_bytes)
        rt.memcpy(got.ptr, frame_base, got.nbytes)
        verified = (hashlib.sha256(got.array.tobytes()).hexdigest() == case["rgba_sha256"]) if case else None
        if job.args.dump_outputs:
            dump_frame(job.args, world, workload + "_bands", got.array)
        got.close()
    elif rank == 0 and job.args.dump_outputs:
        dump_frame(job.args, world, workload + "_bands", partition.deinterleave(gathered, height).cpu().numpy())
    job.barrier()

    # ---- e2e: one shared pinned host frame (RGB8, the body of the P6 file), every rank copies its own blocks into it ----
    # The rank's blocks go in `chunks` groups: group c is rendered on the launch stream while group c-1 is packed to
    # RGB8 on the device (the sink drops alpha, render.rs:389-397) and copied out on a second stream.
    rgb_row = width * 3
    host = SharedHostFrame(job, height * rgb_row, workload)
    own_rgb = torch.zeros((height, width, 3), dtype=torch.uint8, device="cuda")
    copy_stream = torch.cuda.Stream()
    n_blocks = (my_rows + block - 1) // block
    chunks = max(1, min(job.args.band_chunks, n_blocks))
    groups = []   # (first image row, blocks, rows) of each group of this rank's blocks
    for c in range(chunks):
        b0, b1 = c * n_blocks // chunks, (c + 1) * n_blocks // chunks
        if b1 > b0:
            first = row_start + b0 * row_stride
            rows = sum(min(block, height - (row_start + b * row_stride)) for b in range(b0, b1))
            groups.append((first, b1 - b0, rows))
    done_events = [torch.cuda.Event() for _ in groups]

    def e2e_step(i):
        for (first, nb, rows), ev in zip(groups, done_events):
            rt.Renderer.render_row_blocks(opts, scene, first, row_stride, row_block, rows, own.data_ptr(),
                                          pitch=row_bytes, absolute_rows=True, stream=job.stream.cuda_stream)
            ev.record(job.stream)
            copy_stream.wait_event(ev)
            cs = copy_stream.cuda_stream
            last = first + (nb - 1) * row_stride
            rt.pack_rgb_rows(own.data_ptr(), own_rgb.data_ptr(), width, min(height, last + block), first, row_stride, block, cs)
            whole = nb if last + block <= height else nb - 1
            off, pitch = first * rgb_row, row_stride * rgb_row
            if whole:
                rt.memcpy2d_async(host.ptr + off, pitch, own_rgb.data_ptr() + off, pitch, block * rgb_row, whole, cs)
            if whole < nb:   # the image's partial last block
                rt.memcpy2d_async(host.ptr + last * rgb_row, pitch, own_rgb.data_ptr() + last * rgb_row, pitch,
                                  (height - last) * rgb_row, 1, cs)
        job.barrier()          # every rank's copies have landed: the frame is complete in host memory
        if rank == 0:
            _ = int(host.array[0]) + int(host.array[-1])   # the sink touches the frame
        if world > 1:
            dist.barrier()     # nobody overwrites the frame before the sink is done with it
    for i in range(3):
        e2e_step(i)
    e2e_steps = steps
    job.barrier()
    t_begin = time.time()
    e0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    e2e_ms = (time.perf_counter() - e0) * 1e3
    job.windows.append((t_begin, time.time()))
    e2e_verified = None
    if rank == 0 and case:   # the oracle's committed hash of the P6 file of this configuration
        e2e_verified = hashlib.sha256(b"P6\n%d %d\n255\n" % (width, height) + host.array.tobytes()).hexdigest() == case["ppm_sha256"]
    my_bytes = my_rows * rgb_row
    pcie_sum, pcie_own, pcie_fast = job.pcie(max(my_bytes, 1 << 20))
    host.close()
    if rank == 0:
        rt.device_free(frame_base)
    else:
        rt.ipc_close(frame_base)

    (dev_ms, thr_ms, e2e_ms), _ = job.reduce([dev_ms, thr_ms, e2e_ms])
    if rank != 0:
        return None
    ms_per_step, e2e_step_ms = dev_ms / steps, e2e_ms / e2e_steps
    return {
        "metric": METRIC, "value": rays_frame / (ms_per_step * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": workload_name(workload, level, width, height, spp),
            "partition": ("ONE frame per step in interleaved blocks of 16 rows; kernels store into rank 0's frame through IPC "
                          "peer memory (NVLink); an all-reduce on the stream closes every frame (ms_per_step is a frame latency)"
                          if gather == "peer" else "interleaved row bands + NCCL gather to rank 0"),
            "l2": "not flushed" if job.flush is None else "flushed between steps (256 MiB memset, outside the timed events)",
            "rays_per_frame": {"primary": primary_all, "shadow": shadow_all},
            "mpixels_per_s": width * height / (ms_per_step * 1e-3) / 1e6,
            "unsynchronised_throughput_mrays_s": rays_frame / (thr_ms / steps * 1e-3) / 1e6,
            "wall_ms_per_step_incl_flush": wall_ms / steps,
        },
        "e2e": {"value": rays_frame / (e2e_step_ms * 1e-3) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": 512,
                "d2h_bytes_per_step": height * rgb_row, "steps": e2e_steps, "ms_per_step": e2e_step_ms,
                "gathered_frame_verified": e2e_verified, "chunks": len(groups),
                "pcie": {"achieved_gbs": height * rgb_row / (e2e_step_ms * 1e-3) / 1e9, "ceiling_gbs": pcie_sum,
                         "frac": height * rgb_row / (e2e_step_ms * 1e-3) / 1e9 / pcie_sum, "rank0_gbs": pcie_own,
                         "fastest_rank_gbs": pcie_fast},
                "note": "per frame: every rank renders its row blocks in `chunks` groups, packs each group to RGB8 on the device and "
                        "copies it into ONE shared pinned host frame (POSIX shm, cudaHostRegister in every rank; the body of the "
                        "P6 file) over its own PCIe link while the next group renders; barrier; rank 0 reads the frame; barrier.  "
                        "ms_per_step is the latency of one gathered frame in host memory; verified = sha256 of the P6 file == "
                        "the oracle's"},
        "gpu_launches": steps * world * launches_per_step,
        "gathered_frame_verified": verified,
        "gathered_frame_check": "sha256 of rank 0's device frame == the oracle's committed hash for this configuration",
    }


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="measure this workload alone (default: c5 plus the `also` sub-records)")
    ap.add_argument("--mode", default="frames", choices=["frames", "bands"],
                    help="with --workload and N>1: 'frames' = each rank renders whole frames (weak); 'bands' = one frame "
                         "split into interleaved row blocks (strong)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="bands: 'peer' = kernels store into rank 0's frame through CUDA-IPC peer memory over NVLink; "
                         "'nccl' = dist.gather of the bands")
    ap.add_argument("--band-chunks", type=int, default=4,
                    help="bands e2e: groups a rank's row blocks are rendered / copied out in (copy of one overlaps the next's render)")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-l2-flush", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="default run without the sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of each measurement's last timed step to DIR/<workload>.npy (float32)")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def main():
    args = parse_args()
    workload = args.workload or DEFAULT_WORKLOAD

    if args.impl == "reference":
        run_reference(args, workload)
        return
    if args.warmup < 3:
        args.warmup = 3   # timing rule: at least 3 warm-up steps

    job = Job(args)
    rank, world = job.rank, job.world
    if args.mode == "bands" and workload == "c5":
        raise SystemExit("bench.py: c5 is the frame-sharded orbit sweep; use --mode frames")
    if args.mode == "bands" and world > 1:
        out = measure_bands(job, workload, args.steps, args.warmup, args.gather)
    else:
        out = measure_frames(job, workload, args.steps, args.warmup, cpu_baseline=(world == 1 and not args.no_cpu_baseline))
    also = {}
    if args.workload is None and not args.no_also:
        def sub(name, rec):
            if rec is not None:
                for k in ("metric", "unit", "higher_is_better", "vs_baseline", "dtype", "data"):
                    rec.pop(k, None)
                also[name] = rec
        sub("c2", measure_frames(job, "c2", args.steps, args.warmup))
        # 8K frames: whole frames per rank from one queue at every N ("8K multi-frame"), and at N > 1 ONE frame split
        sub("c4", measure_frames(job, "c4", args.steps, args.warmup))
        if world > 1:
            sub("c4_bands", measure_bands(job, "c4", args.steps, args.warmup))
    clocks = job.sampler.stop(job.windows) if job.sampler else None
    if rank == 0:
        out["also"] = also or None
        out["clocks"] = clocks
        print(json.dumps(out))
    if world > 1:
        job.dist.destroy_process_group()


if __name__ == "__main__":
    main()
