"""CPU: tests/prenet_port.py -- the checker of the device pre-network stage -- against cv2 itself.

The uint8 bicubic resize is bit-exact against cv2 with IPP off and within 1 of cv2's default (IPP on); the whole item
(resize, pad, / 255, rotation, mirror) equals the lines of evaluate.py:98-116 run with IPP off."""
import numpy as np
import pytest

import prenet_port as P

cv2 = pytest.importorskip("cv2")


@pytest.fixture
def ipp():
    """Yields a setter for cv2's IPP switch and restores the switch afterwards."""
    saved = cv2.ipp.useIPP()
    yield cv2.ipp.setUseIPP
    cv2.ipp.setUseIPP(saved)


def _image(seed, h, w):
    """Random BGR with saturated patches, so the resize's overshoot is clamped at both ends."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    img[: h // 3, : w // 3] = 255
    img[h // 2:, w // 2:] = 0
    return img


COCO = [(480, 640), (427, 640), (333, 500), (640, 480), (375, 500)]
GEOMETRIES = (
    [(h, w, x * 640 / h) for h, w in COCO for x in (0.5, 1.0, 2.0)]                  # scale_search x boxsize / h
    + [(h, w, s) for h, w in ((480, 640), (100, 77)) for s in (0.37, 0.5, 0.9, 1.33, 2.0, 3.7)]
    + [(100, 77, 10.24), (480, 640, 1.0), (100, 77, 1.0), (100, 77, 1.001)]          # scale 1; dsize == ssize, scale != 1
    + [(60, 300, min(2600 / 60, 3800 / 300))]                                          # evaluate.py:94-96's clamp
    + [(50, 4, 1.2), (30, 3, 0.5), (9, 2, 0.6), (23, 5, 0.9), (17, 1, 2.3), (40, 6, 0.77)]  # rows of < 16 values
    + [(1, 40, 0.8), (1, 40, 3.0), (40, 1, 2.5), (1, 1, 3.0), (1, 9, 1.6), (2, 1, 7.0)]     # one pixel high / wide
)


def _cv2_resize(img, s):
    out = cv2.resize(img, (0, 0), fx=s, fy=s, interpolation=cv2.INTER_CUBIC)
    return out.reshape(out.shape[0], out.shape[1], -1)


def test_geometry_list_covers_the_cases():
    assert len(GEOMETRIES) >= 40
    widths = [P.resized_size(h, w, s)[1] for h, w, s in GEOMETRIES]
    assert sum(3 * W < 16 for W in widths) >= 6
    assert any(P.resized_size(h, w, s) == (h, w) and s != 1 for h, w, s in GEOMETRIES)


@pytest.mark.parametrize("h,w,scale", GEOMETRIES)
def test_resize_equals_cv2_without_ipp(ipp, h, w, scale):
    ipp(False)
    img = _image(h * 7 + w, h, w)
    want = _cv2_resize(img, scale)
    got = P.resize_cubic_u8(img, scale)
    assert got.shape == want.shape and got.dtype == np.uint8
    assert np.array_equal(got, want), f"{int((got != want).sum())} values differ"


def test_narrow_rows_take_the_integer_tail(ipp):
    """Rows shorter than OpenCV's vector loop are computed with the scalar integer form: on outputs where the float and
    the integer form differ, the port equals cv2 only because it uses the integer form there."""
    ipp(False)
    rng = np.random.default_rng(5)
    found = 0
    for _ in range(20000):
        h, w, s = int(rng.integers(2, 60)), int(rng.integers(1, 6)), float(rng.uniform(0.2, 2.5))
        H, W = P.resized_size(h, w, s)
        if min(H, W) < 1 or (H, W) == (h, w) or 3 * W >= P.VEC_LANES:
            continue
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        saved = P.VEC_LANES
        try:
            P.VEC_LANES = 1  # float form everywhere
            all_float = P.resize_cubic_u8(img, s)
        finally:
            P.VEC_LANES = saved
        got = P.resize_cubic_u8(img, s)
        if np.array_equal(all_float, got):
            continue
        want = _cv2_resize(img, s)
        assert np.array_equal(got, want) and not np.array_equal(all_float, want)
        found += 1
        if found == 5:
            break
    assert found == 5


@pytest.mark.parametrize("h,w,scale", [(480, 640, 640 / 480), (427, 640, 0.75), (333, 500, 3.84), (100, 77, 0.37),
                                       (9, 2, 0.6)])
def test_resize_within_one_of_default_cv2(ipp, h, w, scale):
    ipp(True)
    img = _image(h + w, h, w)
    want = _cv2_resize(img, scale).astype(np.int16)
    got = P.resize_cubic_u8(img, scale).astype(np.int16)
    assert got.shape == want.shape and int(np.abs(got - want).max()) <= 1


def _reference_item(image, scale, angle, max_downsample, pad_value):
    """evaluate.py:98-116's operations on the host with cv2."""
    from improved_body_parts_b200.dropin import pad_right_down_corner
    resized = cv2.resize(image, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)
    padded, pad = pad_right_down_corner(resized, max_downsample, pad_value)
    x = np.float32(padded / 255)
    if angle != 0:
        x = cv2.warpAffine(x, cv2.getRotationMatrix2D((x.shape[0] / 2, x.shape[1] / 2), angle, 1), (0, 0))
    return np.concatenate((x[None, ...], x[:, ::-1, :].copy()[None, ...]), axis=0), resized.shape[:2], pad


@pytest.mark.parametrize("angle", [0.0, 5.0, -5.0, 22.5, 90.0, 180.0, -37.3])
@pytest.mark.parametrize("h,w,scale,md,pv", [(150, 210, 160 / 150, 64, 128), (333, 500, 0.5 * 640 / 333, 8, 0)])
def test_item_equals_the_reference_lines(ipp, angle, h, w, scale, md, pv):
    ipp(False)
    img = _image(int(abs(angle) * 10) + h, h, w)
    want, crop, pad = _reference_item(img, scale, angle, md, pv)
    got, got_crop, got_pad = P.network_input(img, scale, angle, md, pv)
    assert got.dtype == np.float32 and got.shape == want.shape
    assert np.array_equal(got, want) and got_crop == crop and got_pad == pad


def test_network_inputs_stacks_the_angles_of_one_scale(ipp):
    ipp(False)
    img = _image(3, 90, 120)
    pairs, crop = P.network_inputs(img, 1.3, [-5.0, 0.0, 5.0], 64, 128)
    assert pairs.shape == (3, 2, 128, 192, 3) and crop == (117, 156)
    for k, a in enumerate((-5.0, 0.0, 5.0)):
        assert np.array_equal(pairs[k], _reference_item(img, 1.3, a, 64, 128)[0])


def test_prenet_size_agrees_with_the_port():
    """spg_prenet_size is host code: the library answers without a GPU."""
    import __graft_entry__ as ge
    from improved_body_parts_b200.grouping import GroupingError, prenet_size

    ge.build()
    for h, w, s in GEOMETRIES + [(480, 640, 2.5 / 480), (7, 9, 0.5 / 7 + 1e-12)]:
        for md in (64, 8, 1):
            H, W = P.resized_size(h, w, s)
            if min(H, W) < 1:
                with pytest.raises(GroupingError):
                    prenet_size(h, w, s, md)
                continue
            assert prenet_size(h, w, s, md) == ((H, W), P.padded_size(H, W, md))
    for args in ((480, 640, 0.0), (480, 640, -1.0), (480, 640, float("inf")), (480, 640, float("nan")),
                 (480, 640, 1.0, 0), (480, 640, 100.0), (0, 640, 1.0), (1, 1, 0.4)):
        with pytest.raises(GroupingError):
            prenet_size(*args)
