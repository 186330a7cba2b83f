"""Regenerates the golden fixtures under tests/golden/.

Needs a checkout of the reference (Byron/rust-tracer) and PIL:
    python tests/golden/make_golden.py <reference checkout>

1. rtrace_output_1024x768.json -- derived from the REFERENCE's own artefact
   src/img/rtrace-output.png (the README hero image = exact output of `make image`,
   SURVEY F2): payload sha256, per-row CRC32s, spot pixels, background count.
   This is what pins the oracle.  rtrace_output_1024x768_rows.npz holds the same
   image's pixels, every 4th row, so that a mismatch can be located without the reference.
2. oracle_derived.json -- outputs of the (pinned) oracle for configurations the
   reference ships no image for: frame hashes and ray counts.  These pin the
   oracle against accidental edits; they are NOT independent evidence.
"""
import hashlib
import json
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
STORED_ROW_STEP = 4


def from_reference_png(ref_png):
    from PIL import Image
    rgb = np.array(Image.open(ref_png).convert("RGB"))
    h, w, _ = rgb.shape
    spots = [(0, 0), (384, 512), (600, 400), (700, 512), (200, 300), (300, 512), (767, 1023), (100, 512), (500, 100)]
    out = {
        "source": "reference src/img/rtrace-output.png (make image: 1024x768, spp 4, level 8)",
        "png_sha256": hashlib.sha256(open(ref_png, "rb").read()).hexdigest(),
        "width": w, "height": h, "spp": 4, "level": 8,
        "rgb_sha256": hashlib.sha256(rgb.tobytes()).hexdigest(),
        "ppm_sha256": hashlib.sha256(b"P6\n%d %d\n255\n" % (w, h) + rgb.tobytes()).hexdigest(),
        "row_crc32": [zlib.crc32(rgb[y].tobytes()) for y in range(h)],
        "spot_pixels": [{"row": r, "col": c, "rgb": [int(v) for v in rgb[r, c]]} for r, c in spots],
        "background_rgb": [34, 10, 10],
        "background_pixels": int((rgb.reshape(-1, 3) == np.array([34, 10, 10])).all(axis=1).sum()),
        "unique_colours": int(len(np.unique(rgb.reshape(-1, 3), axis=0))),
    }
    json.dump(out, open(os.path.join(HERE, "rtrace_output_1024x768.json"), "w"), indent=1)
    rows = np.arange(0, h, STORED_ROW_STEP, dtype=np.uint16)
    np.savez_compressed(os.path.join(HERE, "rtrace_output_1024x768_rows.npz"), rows=rows, rgb=rgb[rows])
    print("reference golden:", out["rgb_sha256"])


def from_oracle():
    import _oracle as o
    cases = []
    # (width, height, spp, level): small parity cases + BASELINE C2 at levels 8/9/10
    for (w, h, spp, level) in [(64, 128, 2, 8), (160, 120, 1, 8), (160, 120, 3, 8), (200, 150, 4, 5), (97, 61, 2, 9),
                               (256, 144, 1, 10), (1024, 768, 1, 8), (3840, 2160, 1, 8), (3840, 2160, 1, 9),
                               (3840, 2160, 1, 10), (3840, 2160, 4, 9), (1024, 768, 4, 8),
                               (7680, 4320, 4, 9)]:   # last three: BASELINE C3 (= C5 frame 0), C1, C4
        s = o.Scene(level=level)
        img, ctr = s.render(w, h, spp)
        cases.append({"width": w, "height": h, "spp": spp, "level": level,
                      "rgba_sha256": hashlib.sha256(img.tobytes()).hexdigest(),
                      "ppm_sha256": hashlib.sha256(b"P6\n%d %d\n255\n" % (w, h) + img[:, :, :3].tobytes()).hexdigest(),
                      "counters": ctr.as_dict(), "flop_per_ray": ctr.flop_per_ray()})
        print(w, h, spp, level, cases[-1]["rgba_sha256"][:16], ctr.shadow_rays)
    # camera extension (SURVEY F6): frames of the 120-frame orbit, small enough for the CPU suite
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    import bench
    orbit = []
    s = o.Scene(level=8)
    for f in (0, 7, 41, 60, 88):
        w, h, spp = 320, 240, 2
        img, ctr = s.render(w, h, spp, camera=o.make_camera(*bench.orbit_basis(f)))
        orbit.append({"frame": f, "n_frames": bench.ORBIT_FRAMES, "width": w, "height": h, "spp": spp, "level": 8,
                      "rgba_sha256": hashlib.sha256(img.tobytes()).hexdigest(), "counters": ctr.as_dict()})
        print("orbit", f, orbit[-1]["rgba_sha256"][:16], ctr.shadow_rays)
    json.dump({"source": "oracle/liboracle_rt.so (pinned by rtrace_output_1024x768.json)", "cases": cases,
               "orbit_cases": orbit, "c5_cases": c5_frames()},
              open(os.path.join(HERE, "oracle_derived.json"), "w"), indent=1)


def c5_frames(frames=(7, 41, 88)):
    """BASELINE configs[4] at REAL size: orbit frames of the 120-frame sweep at 3840x2160, 4x4 samples,
    level 9 (87,381 spheres).  Frame 0 is the C3 case above (the reference camera)."""
    import _oracle as o
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    import bench
    s = o.Scene(level=9)
    out = []
    for f in frames:
        w, h, spp = 3840, 2160, 4
        img, ctr = s.render(w, h, spp, camera=o.make_camera(*bench.orbit_basis(f)))
        out.append({"frame": f, "n_frames": bench.ORBIT_FRAMES, "width": w, "height": h, "spp": spp, "level": 9,
                    "rgba_sha256": hashlib.sha256(img.tobytes()).hexdigest(),
                    "rgb_sha256": hashlib.sha256(np.ascontiguousarray(img[:, :, :3]).tobytes()).hexdigest(),
                    "counters": ctr.as_dict(), "flop_per_ray": ctr.flop_per_ray()})
        print("c5 frame", f, out[-1]["rgba_sha256"][:16], ctr.shadow_rays)
    return out


if __name__ == "__main__":
    if "--only-c5" in sys.argv:   # add / refresh the real-size C5 frames without re-rendering the rest
        path = os.path.join(HERE, "oracle_derived.json")
        d = json.load(open(path))
        d["c5_cases"] = c5_frames()
        json.dump(d, open(path, "w"), indent=1)
    else:
        if len(sys.argv) < 2:
            raise SystemExit("usage: make_golden.py <reference checkout> | --only-c5")
        from_reference_png(os.path.join(sys.argv[1], "src", "img", "rtrace-output.png"))
        from_oracle()
