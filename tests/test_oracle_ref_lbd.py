"""The LBD descriptor / matcher oracle (oracle/lbd_oracle.cpp, SURVEY.md section 8 row f4) against the REFERENCE'S OWN code:
line_lbd/class/line_lbd_allclass.cpp, libs/binary_descriptor.cpp (computeImpl, computeLBD) and libs/binary_descriptor_matcher.cpp compiled
from the reference's sources into oracle/_ref/liblinelbd_ref.so (oracle/ref/linelbd_ref.cpp: the reference files are included from where
they lie).

 * detect_descrip_lines(gray, keylines_out, line_descrips) (line_lbd_allclass.cpp:253-272), both detector flavours: the kept key lines --
   end points, angle, lineLength, response, size, numOfPixels -- and their 32-byte descriptors are equal bit for bit, count and order;
 * BinaryDescriptor::compute on given key lines (what get_line_descriptors calls, :191-198): the 72-float descriptors are == too;
 * match_line_descrip (:341-356): the same (query, train, distance) triples, including which of several equally near codes the multi-index
   hash meets first.

What the reference returned is recorded in tests/golden/reference/ (tests/reference_outputs.py), so these tests run without it."""
import numpy as np
import pytest

from reference_outputs import Reference, assert_same


@pytest.fixture(scope="module")
def ref(oracle):
    r = Reference(oracle, __name__)
    yield r
    r.save()


FIELDS = ("sx", "sy", "ex", "ey", "angle", "line_length", "response", "size", "num_pixels")


def _same_frame(ref, img, use_lsd, thres=15.0):
    kr, dr = ref.ref_detect_descrip_lines(img, use_lsd, thres)
    ko = ref.lbd_detect_keylines(img, use_lsd, thres)
    assert len(kr) == len(ko)
    for f in FIELDS:
        assert_same(ko[f], kr[f], err_msg=f)
    do, fo = ref.lbd_compute(img, ko, want_float=True)
    assert_same(do, dr)
    if len(ko):
        d2, f2 = ref.ref_lbd_compute(img, ko, want_float=True)   # class_id 0 .. n-1, as computeImpl requires
        assert_same(do, d2)
        assert_same(fo, f2)
        assert np.isfinite(fo).all()
    return ko, do


@pytest.mark.parametrize("use_lsd,n", [(True, 271), (False, 88)])
def test_demo_frame(ref, fixture_a, use_lsd, n):
    ko, do = _same_frame(ref, fixture_a["img"], use_lsd)
    assert len(ko) == n
    assert len(np.unique(do, axis=0)) > 0.9 * n          # descriptors are distinctive, not constant


def test_sequence_frames_and_matches_between_neighbours(ref, fixture_b):
    prev = None
    for i in range(0, len(fixture_b["frames"]), 6):
        img = fixture_b["frames"][i][0]
        for use_lsd in (True, False):
            _same_frame(ref, img, use_lsd)
        ko, do = _same_frame(ref, img, True, 30.0)
        if prev is not None and len(do) and len(prev):
            for thres in (25.0, 60.0):
                a, b = ref.lbd_match(do, prev, thres), ref.ref_match_line_descrip(do, prev, thres)
                for x, y in zip(a, b):
                    assert_same(x, y)
        prev = do
    # neighbouring frames of a real sequence (the camera moves a fair way between them): some lines do match
    f0, f1 = fixture_b["frames"][0][0], fixture_b["frames"][1][0]
    d0 = ref.lbd_compute(f0, ref.lbd_detect_keylines(f0, True, 30.0))
    d1 = ref.lbd_compute(f1, ref.lbd_detect_keylines(f1, True, 30.0))
    assert len(ref.lbd_match(d0, d1, 40.0)[0]) >= 3


@pytest.mark.parametrize("use_lsd", [True, False])
def test_octaves_variant_orders_the_ends(ref, fixture_a, use_lsd):
    """detect_descrip_lines_octaves (line_lbd_allclass.cpp:285-339): start x <= end x, the angle folded by normalize_to_PI in double."""
    img = fixture_a["img"]
    kr, dr = ref.ref_detect_descrip_lines_octaves(img, use_lsd, 15.0)
    ko = ref.lbd_detect_keylines(img, use_lsd, 15.0)
    do = ref.lbd_compute(img, ko)
    kz = ref.lbd_order_keylines(ko)
    assert len(kr) == len(kz) and (kz["sx"] != ko["sx"]).any()
    for f in FIELDS:
        assert_same(kz[f], kr[f], err_msg=f)
    assert_same(np.arange(len(kr)), kr["class_id"])
    assert_same(do, dr)                                         # descriptors are computed before the swap


@pytest.mark.parametrize("seed,w,h,kind", [(7, 640, 480, "indoor"), (8, 1242, 375, "kitti")])
def test_synthetic_frames(ref, seed, w, h, kind):
    from cube_slam_b200 import synthetic as S
    imgs = S.make_batch(seed, 2, w, h, 3, kind=kind, poisson=(kind == "indoor"))[0]
    for f in range(2):
        for use_lsd in (True, False):
            ko, _ = _same_frame(ref, imgs[f], use_lsd)
            assert len(ko) > 10


def test_given_keylines_gray_input_and_border_lines(ref):
    """compute() on caller-made key lines: support regions that leave the image on every side (coordinates clamp), a one-pixel line,
    gray input."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (120, 160), dtype=np.uint8)
    img[30:90, 40:120] = 220
    rows = np.array([[2, 2, 150, 3], [5, 110, 5, 4], [158, 1, 158, 118], [0, 0, 159, 119], [80, 60, 80.4, 60.2], [10, 117, 150, 118.5],
                     [40, 30, 120, 30], [40.5, 90.2, 120.3, 89.7]], np.float32)
    kl = ref.lbd_keylines_from_lsd(rows, 160, 120)
    d, f = ref.lbd_compute(img, kl, want_float=True)
    d2, f2 = ref.ref_lbd_compute(img, kl, want_float=True)
    assert_same(d, d2)
    assert_same(f, f2)


def test_matcher_ties_and_far_codes(ref):
    rng = np.random.default_rng(11)

    def flip(c, bits):
        c = c.copy()
        for b in bits:
            c[b // 8] ^= np.uint8(1 << (b % 8))
        return c

    for trial in range(30):
        nq, nt = int(rng.integers(1, 40)), int(rng.integers(6, 70))
        t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
        q = np.stack([flip(t[int(rng.integers(0, nt))], rng.integers(0, 256, int(rng.integers(0, 40)))) for _ in range(nq)])
        # planted ties: for query 0, several train codes at the same distance that differ in WHICH byte is close and by which bit pattern
        base = q[0]
        k = int(rng.integers(2, 7))
        for j in range(min(6, nt)):
            bits = [int(x) for x in rng.choice(256, k, replace=False)]
            t[(j * 7) % nt] = flip(base, bits)
        t[nt - 1] = t[0]                                   # an exact duplicate: bucket order decides
        for thres in (25.0, 300.0):
            a, b = ref.lbd_match(q, t, thres), ref.ref_match_line_descrip(q, t, thres)
            assert_same(a[0], b[0])
            assert_same(a[2], b[2])
            near = a[2] <= 128        # beyond D = 128 the reference never writes results[]: its trainIdx is uninitialised memory, the oracle says -1
            assert_same(a[1][near], b[1][near])
            assert (a[1][~near] == -1).all()
    # unrelated codes: distances around 128; every query still gets its nearest code while that is within D = 128
    q = rng.integers(0, 256, (300, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (40, 32), dtype=np.uint8)
    a, b = ref.lbd_match(q, t, 300.0), ref.ref_match_line_descrip(q, t, 300.0)
    assert_same(a[0], b[0])
    assert_same(a[2], b[2])
    near = a[2] <= 128
    assert_same(a[1][near], b[1][near])
    assert (a[1][~near] == -1).all()
    # the distances themselves are the true minima
    dmin = np.array([[int(np.unpackbits(x ^ y).sum()) for y in t] for x in q]).min(1)
    np.testing.assert_array_equal(a[2], dmin[a[0]].astype(np.float32))
    # empty sides
    assert len(ref.lbd_match(q[:0], t)[0]) == 0 and len(ref.lbd_match(q, t[:0])[0]) == 0


def test_tables(ref):
    G, L, rank = ref.lbd_tables()
    assert G[31] == 1.0 and L[10] == 1.0 and np.all(np.diff(G[:32]) > 0) and np.allclose(G, G[::-1]) and np.allclose(L, L[::-1])
    for s, n in enumerate((1, 8, 28, 56, 70)):                # every s-bit pattern of a byte is looked up once, s = 0 .. 4
        r = sorted(int(rank[i]) for i in range(256) if bin(i).count("1") == s)
        assert r == list(range(n))
    assert all(rank[i] == -1 for i in range(256) if bin(i).count("1") > 4)
