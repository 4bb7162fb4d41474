"""Stage (i) of the north star, `line_lbd_detect::detect_filter_lines(image, lines_mat)`, executed by the REFERENCE'S OWN code from the
first line to the last: line_lbd/class/line_lbd_allclass.cpp + libs/LSDDetector.cpp + libs/lsd.cpp + libs/binary_descriptor.cpp compiled
from the reference's sources into oracle/_ref/liblinelbd_ref.so (oracle/ref/linelbd_ref.cpp; OpenCV replaced by oracle/ref/minicv.hpp) and
called as object_slam/src/main_obj.cpp:363-366,428 calls it.  The oracle's detect_filter_lines (what every CUDA parity test compares with)
must return the same n x 4 float matrix bit for bit: colour conversion, detector, KeyLine fill, border rejection, octave and length filter,
keylines_to_mat -- both detectors, two thresholds.

What the reference returned is recorded in tests/golden/reference/ (tests/reference_outputs.py), so these tests run without it."""
import numpy as np
import pytest

from reference_outputs import Reference, assert_same


@pytest.fixture(scope="module")
def ref(oracle):
    r = Reference(oracle, __name__)
    yield r
    r.save()


def _same(ref, img, use_lsd, thres):
    got = (ref.lsd_detect(img, thres) if use_lsd else ref.edl_detect(img, thres))["lines"]
    want = ref.ref_detect_filter_lines(img, use_lsd, thres)
    assert got.shape == want.shape
    assert_same(got, want)
    return len(want)


@pytest.mark.parametrize("use_lsd", [True, False])
def test_demo_frame_and_sequence(ref, fixture_a, fixture_b, use_lsd):
    assert _same(ref, fixture_a["img"], use_lsd, 15.0) == (271 if use_lsd else 88)
    _same(ref, fixture_a["img"], use_lsd, 50.0)            # the class default threshold (line_lbd_allclass.cpp:122)
    for i in range(0, len(fixture_b["frames"]), 8):
        _same(ref, fixture_b["frames"][i][0], use_lsd, 15.0)


@pytest.mark.parametrize("use_lsd", [True, False])
def test_synthetic_frames_colour_and_gray(ref, use_lsd):
    from cube_slam_b200 import synthetic as S
    for seed, w, h, kind in ((7, 640, 480, "indoor"), (8, 1242, 375, "kitti")):
        imgs = S.make_batch(seed, 2, w, h, 3, kind=kind, poisson=(kind == "indoor"))[0]
        assert _same(ref, imgs[0], use_lsd, 15.0) > 10
        _same(ref, np.ascontiguousarray(ref.bgr2gray(imgs[1])), use_lsd, 15.0)   # a single-channel input skips cvtColor
