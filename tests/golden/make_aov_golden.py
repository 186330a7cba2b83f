"""Regenerates tests/golden/oracle_aov.json on the CPU:

    python tests/golden/make_aov_golden.py

The sha256 of the oracle's AOV frames -- (h, w, 8) float32 {nx, ny, nz, coverage, distance, px, py, pz}
(include/rtrace.h "geometry output"), little-endian -- for the full-size cases of oracle_derived.json: every BASELINE
configuration (C1, C2 at levels 8/9/10, C3, C4) and the C5 orbit frames 7, 41 and 88.  Each frame is checked on the
way against the pinned oracle (tests/_aov_ref.py): over the whole frame, the covered samples add up to the
primary_hits oracle_derived.json records where it records them; on every 37th row and the last one, coverage equals
orc_render_region's count of non-background samples, and distance, normal and position equal what orc_trace_rays'
per-sample hits give."""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def frame_entry(aov_scene, pinned, case, camera=None, extra=None):
    import _aov_ref
    import _oracle as o
    w, h, spp = case["width"], case["height"], case["spp"]
    cam = o.make_camera(*camera) if camera else None
    a = aov_scene.render_aov(w, h, spp, camera=cam)
    if "counters" in case:
        covered = np.rint(a[..., 3].astype(np.float64) * spp * spp).sum()
        assert covered == case["counters"]["primary_hits"], (case, covered)
    rows = sorted(set(range(0, h, 37)) | {h - 1})
    eye = camera[0] if camera else pinned.eye()
    basis = np.array(camera[1:], np.float32) if camera else None
    _aov_ref.check_rows_coverage(a[rows], pinned, w, h, spp, rows, cam)
    _aov_ref.check_rows_against_traced_rays(a[rows], pinned, w, h, spp, rows, eye, basis)
    entry = {"width": w, "height": h, "spp": spp, "level": case["level"],
             "aov_sha256": hashlib.sha256(a.astype("<f4").tobytes()).hexdigest()}
    entry.update(extra or {})
    print(entry, flush=True)
    return entry


def main():
    import _oracle
    import _oracle_aov
    import bench
    derived = json.load(open(os.path.join(HERE, "oracle_derived.json")))
    scenes = {}

    def scene(level):
        if level not in scenes:
            scenes[level] = (_oracle_aov.Scene(level=level), _oracle.Scene(level=level))
        return scenes[level]

    cases = [frame_entry(*scene(c["level"]), c) for c in derived["cases"] if c["width"] * c["height"] >= 1024 * 768]
    c5 = [frame_entry(*scene(c["level"]), c, bench.orbit_basis(c["frame"]), {"frame": c["frame"], "n_frames": c["n_frames"]})
          for c in derived["c5_cases"]]
    json.dump({"source": "tests/_oracle_aov.cpp orc_render_rows_aov on the pinned oracle/oracle_rt.cpp (checked against its "
                         "orc_render_region kinds and orc_trace_rays hits, tests/_aov_ref.py)",
               "cases": cases, "c5_cases": c5}, open(os.path.join(HERE, "oracle_aov.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
