"""More than one octave.  The product detects octave 0 and accepts numoctaves >= 1 wherever the reference's result is octave 0 only:
filter_lines (line_lbd_allclass.cpp:200-207) and both detect_descrip_lines overloads (:239,266) drop every other octave, and octave 0 is
detected first and independently of the higher ones in both detectors (LSDDetector.cpp:176-199; binary_descriptor.cpp:805-843,862-886).
Here the REFERENCE'S OWN class (oracle/_ref/liblinelbd_ref.so), built with 2 and 3 octaves as line_lbd/src/detect_lines.cpp:57-60
parameterises it, returns the one-octave matrix bit for bit while its raw key-line list does grow.

The higher octaves run on images made by the stand-in's pyrDown / resize: pyrDown is pinned to cv2 here; the EDLines flavour is tried with
two octaves (a third needs an 8-bit Gaussian of sigma sqrt(2), which the stand-in does not provide).

What the reference returned is recorded in tests/golden/reference/ (tests/reference_outputs.py), so these tests run without it."""
import numpy as np
import pytest

from reference_outputs import Reference, assert_same


@pytest.fixture(scope="module")
def ref(oracle):
    r = Reference(oracle, __name__)
    yield r
    r.save()


@pytest.mark.parametrize("use_lsd,octaves", [(True, (2, 3)), (False, (2,))])
def test_filtered_lines_do_not_depend_on_the_octave_count(ref, fixture_a, fixture_b, use_lsd, octaves):
    for img in (fixture_a["img"], fixture_b["frames"][5][0], fixture_b["frames"][30][0]):
        one = (ref.lsd_detect(img, 15.0) if use_lsd else ref.edl_detect(img, 15.0))["lines"]
        base, raw1 = ref.ref_detect_filter_lines_octaves(img, use_lsd, 15.0, 1)
        assert_same(one, base)
        for n in octaves:
            got, raw_n = ref.ref_detect_filter_lines_octaves(img, use_lsd, 15.0, n)
            assert_same(one, got)
            assert raw_n > raw1                      # the higher octaves did run and did find lines


def test_pyrdown_and_halving_stand_ins_equal_cv2(ref):
    import cv2
    rng = np.random.default_rng(0)
    for shape in [(480, 640), (375, 1242), (97, 211), (120, 161)]:
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        h, w = shape
        assert_same(cv2.pyrDown(a, dstsize=(w // 2, h // 2)), ref.ref_minicv_pyrdown(a, w // 2, h // 2))
        if w % 2 == 0 and h % 2 == 0:
            assert_same(cv2.resize(a, None, fx=0.5, fy=0.5), ref.ref_minicv_resize_half(a))
