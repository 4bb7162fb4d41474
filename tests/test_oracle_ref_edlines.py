"""The EDLines oracle (oracle/edl_oracle.cpp) against the REFERENCE'S OWN detector: line_lbd/libs/binary_descriptor.cpp (BinaryDescriptor
with its nested EDLineDetector) and the reference's headers, compiled from the reference's sources into oracle/_ref/libedl_ref.so
(oracle/Makefile target `ref`, oracle/ref/edl_ref.cpp + minicv.hpp + fakecv/: the reference files are included from where they lie,
nothing of them is copied) and driven as line_lbd_detect::detect_raw_lines drives it for use_LSD = false
(line_lbd/class/line_lbd_allclass.cpp:110-124,165-169).  The key lines of octave 0 must be equal bit for bit, count and order.

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
    got = ref.edl_detect(img, 15.0)["raw_lines"]
    want = ref.ref_edl_detect(img)
    assert got.shape == want.shape
    assert_same(got, want)
    return len(want)


def test_demo_frame(ref, fixture_a):
    assert _same(ref, fixture_a["img"]) == 88


def test_sequence_frames(ref, fixture_b):
    for i in range(0, len(fixture_b["frames"]), 5):
        assert _same(ref, fixture_b["frames"][i][0]) > 0


@pytest.mark.parametrize("seed,w,h,kind", [(7, 640, 480, "indoor"), (8, 1242, 375, "kitti"), (9, 1280, 960, "indoor")])
def test_synthetic_frames(ref, seed, w, h, kind):
    from cube_slam_b200 import synthetic as S
    imgs = S.make_batch(seed, 2, w, h, 3, kind=kind, poisson=(kind == "indoor"))[0]
    for f in range(2):
        assert _same(ref, imgs[f]) > 20


def test_odd_sizes_and_degenerate_images(ref):
    rng = np.random.default_rng(5)
    for shape in [(97, 211), (61, 64), (200, 333)]:       # noise: thousands of anchors, short chains, few lines
        _same(ref, rng.integers(0, 256, shape, dtype=np.uint8))
    assert _same(ref, np.full((120, 160), 77, np.uint8)) == 0   # no gradient, no anchor
    img = np.full((240, 320), 30, np.uint8)                 # sharp rectangles: long chains, corners, the incremental fit
    img[40:200, 60:260] = 200
    img[90:150, 120:180] = 90
    img += rng.integers(0, 6, img.shape, dtype=np.uint8)
    assert _same(ref, img) >= 6
    # NOT compared: one long curved chain (a disc outline).  EDLineDetector::EDline sizes lines.sId as 5 x (number of chains)
    # (binary_descriptor.cpp:2394) and writes one entry per fitted segment (:2438): a chain that splits into more than five segments per chain on
    # average overruns the heap in the reference itself (AddressSanitizer: heap-buffer-overflow at :2438).  The oracle and the CUDA path
    # keep every segment; on such inputs the reference has no defined output to compare with.
    tri = np.full((200, 260), 40, np.uint8)                 # a triangle and a square: chains with two to four segments each
    for y in range(30, 170):
        tri[y, 30 + (y - 30) // 2: 130 - (y - 30) // 3] = 190
    tri[60:150, 160:240] = 120
    tri += rng.integers(0, 5, tri.shape, dtype=np.uint8)
    assert _same(ref, tri) >= 4
