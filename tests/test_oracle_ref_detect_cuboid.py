"""Stage (ii) of the north star, `detect_3d_cuboid::detect_cuboid`, executed by the REFERENCE'S OWN code: detect_3d_cuboid/src/matrix_utils.cpp,
object_3d_util.cpp and box_proposal_detail.cpp compiled from the reference's sources into oracle/_ref/libcuboid_ref.so (oracle/ref/cuboid_ref.cpp;
Eigen replaced by oracle/ref/minieigen.hpp, OpenCV by oracle/ref/minicv.hpp with Canny / distanceTransform / cvtColor forwarded to the
cv2-pinned restatements) and driven as object_slam/src/main_obj.cpp:354-361,449 drives it.  Every cuboid the reference returns -- which
proposal wins, its rank among the top k, position, yaw, scale, the 2-D and 3-D corners, both errors, the normalised score, the roll /
pitch deltas -- must equal the oracle's record, here asserted with ==, not a tolerance (the oracle runs with libm's atan2 for this
comparison, as the reference does; tests/test_pmath.py ties the arithmetic atan2 the parity tests use to libm's).

What the reference returned is recorded in tests/golden/reference/ (tests/reference_outputs.py), so these tests run without it."""
import numpy as np
import pytest

from reference_outputs import Reference, assert_same

FIELDS = ("pos", "rotY", "scale", "box_config_type", "box_corners_2d", "box_corners_3d_world", "rect_detect_2d", "edge_distance_error",
          "edge_angle_error", "normalized_error", "skew_ratio", "down_expand_height", "camera_roll_delta", "camera_pitch_delta")
MODES = [("default", {}), ("top5", dict(max_cuboid_num=5)), ("roll_pitch", dict(whether_sample_cam_roll_pitch=1)),
         ("no_height_samples", dict(whether_sample_bbox_height=0)), ("one_config", dict(consider_config_2=0))]


@pytest.fixture(scope="module")
def ref(oracle):
    r = Reference(oracle, __name__)
    oracle.lib().orc_set_portable_atan2(0)
    yield r
    oracle.lib().orc_set_portable_atan2(1)
    r.save()


def _same(ref, img, K, T, boxes, lines, p):
    k = max(int(p.max_cuboid_num), 1)
    got = ref.detect_cuboid(img, K, T, boxes, lines, p, topk_cap=k)["cuboids"]
    want = ref.ref_detect_cuboid(img, K, T, boxes, lines, p, cap_per_box=k)
    n = 0
    for b in range(len(want)):
        assert len(got[b]) == len(want[b]), b
        for f in FIELDS:   # every rank of the box at once
            assert_same(np.asarray(got[b][f], np.float64), want[b][f], err_msg="%s box %d" % (f, b))
        n += len(want[b])
    return n


@pytest.mark.parametrize("mode,kw", MODES)
def test_demo_frame(ref, fixture_a, mode, kw):
    assert _same(ref, fixture_a["img"], fixture_a["K"], fixture_a["T"], fixture_a["boxes"], fixture_a["lines"], ref.default_params(**kw)) >= 1


@pytest.mark.parametrize("mode,kw", MODES[:3])
def test_sequence_frames_with_detected_lines(ref, fixture_b, mode, kw):
    n = 0
    for i in range(0, len(fixture_b["frames"]), 6):
        img, boxes = fixture_b["frames"][i]
        lines = ref.lsd_detect(img, 15.0)["lines"].astype(np.float64)          # main_obj.cpp:428-433
        n += _same(ref, img, fixture_b["K"], fixture_b["T"], boxes, lines, ref.default_params(nominal_skew_ratio=2.0, **kw))
    assert n >= 6


@pytest.mark.parametrize("seed,w,h,kind,nb", [(101, 640, 480, "indoor", 3), (102, 1242, 375, "kitti", 8)])
def test_synthetic_frames_with_several_boxes(ref, seed, w, h, kind, nb):
    from cube_slam_b200 import synthetic as S
    imgs, Ts, boxes, lines, K = S.make_batch(seed, 2, w, h, nb, kind=kind, poisson=(kind == "indoor"))
    for f in range(2):
        ln = ref.lsd_detect(imgs[f], 15.0)["lines"].astype(np.float64)
        for _, kw in MODES[:3]:   # roll / pitch sampling with several boxes: the reference's carried-over cam_pose included
            _same(ref, imgs[f], K, Ts[f], boxes[f], ln, ref.default_params(**kw))
        _same(ref, imgs[f], K, Ts[f], boxes[f], lines[f], ref.default_params())   # the generator's own segments as input
