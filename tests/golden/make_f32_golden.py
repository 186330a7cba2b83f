"""Regenerates tests/golden/oracle_f32.json on the CPU:

    python tests/golden/make_f32_golden.py

The sha256 of the oracle's float frames -- (h, w, 4) float32 {r, g, b, alpha} before quantisation, little-endian --
for the full-size cases of oracle_derived.json: every BASELINE configuration (C1, C2 at levels 8/9/10, C3, C4) and
the C5 orbit frames 7, 41 and 88.  Each frame is checked on the way: quantised with the reference's rule it must
give the RGBA8 hash oracle_derived.json pins, so this file rests on the same pinned oracle."""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def quantise(v):
    """render.rs:96-103: trunc(0.5 + 255 v) in f32, > 255 -> 255, NaN or <= 0 -> 0."""
    r = np.float32(0.5) + np.float32(255.0) * np.asarray(v, np.float32)
    with np.errstate(invalid="ignore"):
        r = np.where(r > np.float32(255.0), np.float32(255.0), np.where(r > np.float32(0.0), r, np.float32(0.0)))
    return np.trunc(r).astype(np.uint8)


def frame_entry(scene, case, camera=None, extra=None):
    import _oracle as o
    w, h, spp = case["width"], case["height"], case["spp"]
    f, _ = scene.render_f32(w, h, spp, camera=o.make_camera(*camera) if camera else None)
    assert hashlib.sha256(quantise(f).tobytes()).hexdigest() == case["rgba_sha256"], case
    entry = {"width": w, "height": h, "spp": spp, "level": case["level"],
             "f32_sha256": hashlib.sha256(f.astype("<f4").tobytes()).hexdigest(), "rgba_sha256": case["rgba_sha256"]}
    entry.update(extra or {})
    print(entry)
    return entry


def main():
    import _oracle_f32
    import bench
    derived = json.load(open(os.path.join(HERE, "oracle_derived.json")))
    scenes = {}

    def scene(level):
        if level not in scenes:
            scenes[level] = _oracle_f32.Scene(level=level)
        return scenes[level]

    cases = [frame_entry(scene(c["level"]), c) for c in derived["cases"] if c["width"] * c["height"] >= 1024 * 768]
    c5 = [frame_entry(scene(c["level"]), c, bench.orbit_basis(c["frame"]), {"frame": c["frame"], "n_frames": c["n_frames"]})
          for c in derived["c5_cases"]]
    json.dump({"source": "tests/_oracle_f32.cpp orc_render_rows_f32 on the pinned oracle/oracle_rt.cpp (quantised: the hashes of oracle_derived.json)",
               "cases": cases, "c5_cases": c5}, open(os.path.join(HERE, "oracle_f32.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
