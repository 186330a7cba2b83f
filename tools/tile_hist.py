"""Distribution of candidate counts per cull tile (PHASED) for one configuration."""
import sys, os, json
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust-tracer_b200"))
import rtrace_b200 as rt
w, h, spp, level = [int(v) for v in (sys.argv[1:5] if len(sys.argv) > 4 else (3840, 2160, 1, 8))]
cw = int(sys.argv[5]) if len(sys.argv) > 5 else 32   # cull tile width in pixels
s = rt.Scene(level=level)
rt.set_variant(rt.VARIANT_PHASED)
rt.Renderer.render(rt.RenderOptions(w, h, spp), s)
t = rt.debug_phased_tiles(s)
ctx = (w + cw - 1) // cw
WALK, COVERED = 0xffffffff, 0xfffffffd   # per-lane walk / one leaf occludes every shadow ray of the tile
for k, name in ((0, "primary"), (1, "shadow")):
    c = t[:, k].astype(np.int64)
    listed = (c != WALK) & (c != COVERED)
    print(name, "per-lane walk", int((c == WALK).sum()), "covered", int((c == COVERED).sum()))
    c = np.where(listed, c, 0)
    nz = c[c > 0]
    print(name, "tiles", int(listed.sum()), "nonempty", len(nz), "sum", int(c.sum()), "mean(nonempty) %.1f" % (nz.mean() if len(nz) else 0),
          "pcts 50/90/99/99.9/max:", [int(np.percentile(nz, q)) for q in (50, 90, 99, 99.9, 100)] if len(nz) else [])
    top = np.argsort(-c)[:12]
    print("   top tiles (count @ tile x,y):", [(int(c[i]), int(i % ctx), int(i // ctx)) for i in top])
    hist = np.bincount(np.minimum(c[listed], 1023) // 32)
    print("   hist by 32s:", hist.tolist())
