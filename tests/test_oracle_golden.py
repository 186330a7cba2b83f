"""Pins the oracle: it must reproduce the reference's shipped `make image` output
(src/img/rtrace-output.png) bit for bit.  The fixtures hold hashes of that PNG's
pixels and every 4th row of the pixels themselves (tests/golden/make_golden.py)."""
import hashlib
import json
import os
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "rtrace_output_1024x768.json")))
DERIVED = json.load(open(os.path.join(HERE, "golden", "oracle_derived.json")))
REF_ROWS = os.path.join(HERE, "golden", "rtrace_output_1024x768_rows.npz")


@pytest.fixture(scope="module")
def make_image(oracle_scene8):
    return oracle_scene8.render(GOLD["width"], GOLD["height"], GOLD["spp"])


def test_make_image_matches_reference_png_hash(make_image):
    img, _ = make_image
    rgb = np.ascontiguousarray(img[:, :, :3])
    bad = [y for y in range(GOLD["height"]) if zlib.crc32(rgb[y].tobytes()) != GOLD["row_crc32"][y]]
    assert not bad, "rows differing from the reference image: %s" % bad[:10]
    assert hashlib.sha256(rgb.tobytes()).hexdigest() == GOLD["rgb_sha256"]
    ppm = b"P6\n%d %d\n255\n" % (GOLD["width"], GOLD["height"]) + rgb.tobytes()
    assert hashlib.sha256(ppm).hexdigest() == GOLD["ppm_sha256"]


def test_make_image_spot_pixels_and_background(make_image):
    img, _ = make_image
    for sp in GOLD["spot_pixels"]:
        assert [int(v) for v in img[sp["row"], sp["col"], :3]] == sp["rgb"]
    bg = (img[:, :, :3].reshape(-1, 3) == np.array(GOLD["background_rgb"])).all(axis=1).sum()
    assert int(bg) == GOLD["background_pixels"]


def test_make_image_ray_counts(make_image):
    # SURVEY 8(d): C1 = 12,582,912 primary + 7,211,901 shadow rays, ~615 flop/ray of reference work
    _, ctr = make_image
    assert ctr.primary_rays == 1024 * 768 * 16
    assert ctr.shadow_rays == 7211901
    assert ctr.primary_hits == 9430527
    assert 600.0 < ctr.flop_per_ray() < 630.0


def test_make_image_matches_reference_png_pixels(make_image):
    """Pixel for pixel against the stored rows of the reference PNG; their CRC32s are the PNG's own rows."""
    img, _ = make_image
    ref = np.load(REF_ROWS)
    rows, png = ref["rows"].astype(np.int64), ref["rgb"]
    assert rows.tolist() == list(range(0, GOLD["height"], 4)) and png.shape == (len(rows), GOLD["width"], 3)
    assert [zlib.crc32(png[i].tobytes()) for i in range(len(rows))] == [GOLD["row_crc32"][y] for y in rows]
    got = img[rows, :, :3]
    if not np.array_equal(got, png):
        bad = np.argwhere((got != png).any(axis=-1))
        raise AssertionError("%d pixels differ from the reference image, first at row %d col %d: %s != %s" % (
            len(bad), rows[bad[0][0]], bad[0][1], got[tuple(bad[0])], png[tuple(bad[0])]))
    assert hashlib.sha256(np.ascontiguousarray(img[:, :, :3]).tobytes()).hexdigest() == GOLD["rgb_sha256"]


@pytest.mark.parametrize("case", DERIVED.get("orbit_cases", []), ids=lambda c: "orbit_frame_%d" % c["frame"])
def test_oracle_orbit_fixtures(oracle, case):
    """The camera extension (orbit about the flake's axis, SURVEY F6) as the oracle renders it: committed hashes
    keep the oracle, bench.orbit_basis and the fixture generator in step.  Frame 0 is the reference camera."""
    sys.path.insert(0, os.path.dirname(HERE))
    import bench
    s = oracle.Scene(level=case["level"])
    cam = oracle.make_camera(*bench.orbit_basis(case["frame"], case["n_frames"]))
    img, ctr = s.render(case["width"], case["height"], case["spp"], camera=cam)
    assert hashlib.sha256(img.tobytes()).hexdigest() == case["rgba_sha256"]
    assert ctr.as_dict() == case["counters"]
    if case["frame"] == 0:
        plain, _ = s.render(case["width"], case["height"], case["spp"])
        assert np.array_equal(plain, img)


@pytest.mark.parametrize("case", [c for c in DERIVED["cases"] if c["width"] * c["height"] * c["spp"] ** 2 <= 1 << 20],
                         ids=lambda c: "%dx%d_spp%d_L%d" % (c["width"], c["height"], c["spp"], c["level"]))
def test_oracle_derived_fixtures(oracle, case):
    s = oracle.Scene(level=case["level"])
    img, ctr = s.render(case["width"], case["height"], case["spp"])
    assert hashlib.sha256(img.tobytes()).hexdigest() == case["rgba_sha256"]
    assert ctr.as_dict() == case["counters"]
