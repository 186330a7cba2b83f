"""Renders a list of cases in a process of its own.  TEST INFRASTRUCTURE (not collected by pytest).

RTRACE_TILE_SHAPE is read once per process (forced_tile_shape in rt_api.cpp), so tests/test_phased_paths.py runs
one of these per shape with the variable set in its environment:

    python _shape_worker.py cases.json out_dir

cases.json is a list of {"id", "variant", "width", "height", "spp", "camera": null or [eye, right, up, forward],
"kinds": bool, "tiles": bool}.  For each case out_dir receives <id>_img.npy, <id>_kinds.npy (kinds cases) and
<id>_tiles.npy (rt_debug_phased_tiles right after the frame, tiles cases); variants.json maps each id to
rt_stats.variant_used."""
import json
import os
import sys

import numpy as np

import rtrace_b200 as rt


def main(cases_path, out_dir):
    cases = json.load(open(cases_path))
    used = {}
    scene = rt.Scene()
    try:
        for c in cases:
            o = rt.RenderOptions(c["width"], c["height"], c["spp"])
            cam = rt.make_camera(*c["camera"]) if c["camera"] else None
            rt.set_variant(c["variant"])
            try:
                res = rt.Renderer.render_rows(o, scene, camera=cam, kinds=c["kinds"], want_stats=True)
                tiles = rt.debug_phased_tiles(scene) if c["tiles"] else None
            finally:
                rt.set_variant(rt.VARIANT_AUTO)
            np.save(os.path.join(out_dir, c["id"] + "_img.npy"), res[0])
            if c["kinds"]:
                np.save(os.path.join(out_dir, c["id"] + "_kinds.npy"), res[1])
            if tiles is not None:
                np.save(os.path.join(out_dir, c["id"] + "_tiles.npy"), tiles)
            used[c["id"]] = int(res[-1].variant_used)
    finally:
        scene.close()
    json.dump(used, open(os.path.join(out_dir, "variants.json"), "w"))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
