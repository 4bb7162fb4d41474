"""The LSD oracle (oracle/lsd_oracle.cpp) against the REFERENCE'S OWN lsd.cpp, compiled from the reference's sources into
oracle/_ref/liblsd_ref.so (oracle/Makefile target `ref`, oracle/ref/lsd_ref.cpp + minicv.hpp: the reference file is included from
where it lies, nothing of it is copied).  Raw segments -- createLineSegmentDetector(LSD_REFINE_ADV)->detect(gray), what
LSDDetector::detectImpl (line_lbd/libs/LSDDetector.cpp:120-170) gets for octave 0 -- must be equal bit for bit, count and order.

What the reference returned is recorded in tests/golden/reference/ (tests/reference_outputs.py), so these tests run without it."""
import numpy as np
import pytest

from reference_outputs import Reference, assert_same


@pytest.fixture(scope="module")
def ref(oracle):
    r = Reference(oracle, __name__)
    yield r
    r.save()


def _same(ref, img):
    got = ref.lsd_detect(img, 15.0)["raw_lines"]
    want = ref.ref_lsd_detect(img)
    assert got.shape == want.shape
    assert_same(got, want)
    return len(want)


def test_demo_frame(ref, fixture_a):
    assert _same(ref, fixture_a["img"]) == 450


def test_sequence_frames(ref, fixture_b):
    for i in range(0, len(fixture_b["frames"]), 7):
        assert _same(ref, fixture_b["frames"][i][0]) > 0


@pytest.mark.parametrize("seed,w,h,kind", [(7, 640, 480, "indoor"), (8, 1242, 375, "kitti")])
def test_synthetic_frames(ref, seed, w, h, kind):
    from cube_slam_b200 import synthetic as S
    imgs = S.make_batch(seed, 2, w, h, 3, kind=kind, poisson=(kind == "indoor"))[0]
    for f in range(2):
        assert _same(ref, imgs[f]) > 50


def test_odd_sizes_and_degenerate_images(ref):
    rng = np.random.default_rng(5)
    # ragged sizes (the 0.8 resize rounds differently), noise (thousands of seeds, few accepted), constant (no defined pixel)
    for shape in [(97, 211), (61, 64), (200, 333)]:
        _same(ref, rng.integers(0, 256, shape, dtype=np.uint8))
    assert _same(ref, np.full((120, 160), 77, np.uint8)) == 0
    # a few sharp rectangles: long regions, the reduce-radius / refine branches
    img = np.full((240, 320), 30, np.uint8)
    img[40:200, 60:260] = 200
    img[90:150, 120:180] = 90
    img += rng.integers(0, 6, img.shape, dtype=np.uint8)
    assert _same(ref, img) >= 6
    # a blurred disc: curved regions that fail the density test and get cut
    yy, xx = np.mgrid[:300, :300]
    disc = (np.hypot(yy - 150, xx - 150) < 100).astype(np.float64) * 180 + 40
    _same(ref, np.clip(disc + rng.normal(0, 2, disc.shape), 0, 255).astype(np.uint8))
