"""CPU: tests/rotation_port.py -- the rotation search of the reference's post-network stage -- against OpenCV.

``cv2.warpAffine`` with its defaults is a fixed-point routine OpenCV defines step by step, so unlike the bicubic resize
(Intel IPP in the reference's wheels) the port can be pinned to it bit for bit.  The whole item -- flip ensemble,
resize, warp, crop, resize -- is pinned to the reference's lines run with cv2 within the resize's existing tolerance.
"""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

import rotation_port as rp
from improved_body_parts_b200 import skeleton
from oracle import postnet_port as pp

ANGLES = [5.0, -5.0, 22.5, 90.0, 180.0, -37.3]
SHAPES = [(128, 128), (96, 160), (75, 131)]  # square, non-square, odd


@pytest.mark.parametrize("shape", SHAPES + [(512, 384)])
@pytest.mark.parametrize("angle", ANGLES)
def test_rotation_matrix_is_get_rotation_matrix_2d(shape, angle):
    ref = cv2.getRotationMatrix2D((shape[0] / 2, shape[1] / 2), angle, 1)  # evaluate.py:109, centre (rows/2, cols/2)
    assert np.array_equal(rp.rotation_matrix(shape, angle), ref)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("channels", [1, 3, 18, 30])
@pytest.mark.parametrize("angle", ANGLES)
def test_warp_equals_cv2_bit_for_bit(shape, channels, angle):
    rng = np.random.default_rng(hash((shape, channels, angle)) & 0xffff)
    src = rng.standard_normal(shape + ((channels,) if channels > 1 else ()), dtype=np.float32)
    M = rp.rotation_matrix(shape, angle)
    ref = cv2.warpAffine(src, M, (0, 0))
    got = rp.warp_affine_linear(src, M)
    assert got.shape == ref.shape and got.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_warp_with_nans_equals_cv2():
    """cv2's fixed-point path multiplies every in-map tap by its weight, so a NaN tap poisons the pixel even at weight
    0; taps outside the map read the border value 0.  The port does the same, payloads included."""
    rng = np.random.default_rng(11)
    src = rng.random((64, 80, 3), dtype=np.float32)
    src[10, 20, 1] = src[0, 0, 0] = src[63, 79, 2] = np.nan
    src[30, 40, 0] = np.inf
    for angle in (22.5, -5.0, 90.0):
        M = rp.rotation_matrix(src.shape[:2], angle)
        ref = cv2.warpAffine(src, M, (0, 0))
        got = rp.warp_affine_linear(src, M)
        assert np.isnan(ref).any() and np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_warp_at_angle_zero_is_the_identity():
    src = np.random.default_rng(3).random((33, 47, 2), dtype=np.float32)
    assert np.array_equal(rp.warp_affine_linear(src, rp.rotation_matrix(src.shape[:2], 0.0)), src)


@pytest.mark.parametrize("angle", [5.0, -37.3, 90.0])
def test_post_network_item_equals_the_reference_lines_with_cv2(angle):
    """evaluate.py:108-158 for one (scale, angle) item written out with cv2 vs the port."""
    rng = np.random.default_rng(17)
    n_paf, n_heat = skeleton.NUM_LIMBS, skeleton.NUM_PARTS + 2
    n_layers = n_paf + n_heat
    stride, h, w = 4, 48, 64
    padded_shape, pad, image_shape = (192, 256), [0, 0, 7, 12], (370, 488)
    out = rng.random((2, n_layers, h, w), dtype=np.float32)

    rotate_matrix_reverse = cv2.getRotationMatrix2D((padded_shape[0] / 2, padded_shape[1] / 2), -angle, 1)
    blob, blob_flip = out[0].transpose(1, 2, 0), out[1].transpose(1, 2, 0)
    b0, b1 = blob[:, :, :n_paf], blob[:, :, n_paf:n_layers]
    f0, f1 = blob_flip[:, :, :n_paf], blob_flip[:, :, n_paf:n_layers]
    b0_avg = (b0 + f0[:, ::-1, :][:, :, list(skeleton.FLIP_PAF_ORD)]) / 2
    b1_avg = (b1 + f1[:, ::-1, :][:, :, list(skeleton.FLIP_HEAT_ORD)]) / 2
    ref = []
    for m in (b1_avg, b0_avg):
        up = cv2.resize(m, (0, 0), fx=stride, fy=stride, interpolation=cv2.INTER_CUBIC)
        up = cv2.warpAffine(up, rotate_matrix_reverse, (0, 0))
        up = up[pad[0]:padded_shape[0] - pad[2], pad[1]:padded_shape[1] - pad[3], :]
        ref.append(cv2.resize(up, (image_shape[1], image_shape[0]), interpolation=cv2.INTER_CUBIC))

    got = rp.post_network_scale(out, stride, padded_shape, pad, image_shape, n_paf, n_layers, skeleton.FLIP_PAF_ORD,
                                skeleton.FLIP_HEAT_ORD, angle=angle)
    for r, g in zip(ref, got):
        assert g.shape == r.shape
        assert np.abs(pp.accumulate(np.zeros(r.shape), g, 1) - r).max() <= 1e-4  # the resize's tolerance (IPP)
    # with the same resize routine on both sides the rest of the item is exact
    same = rp.post_network_scale(out, stride, padded_shape, pad, image_shape, n_paf, n_layers, skeleton.FLIP_PAF_ORD,
                                 skeleton.FLIP_HEAT_ORD, angle=angle,
                                 resize=lambda m, dsize, fx=0.0, fy=0.0: cv2.resize(m, dsize or (0, 0), fx=fx, fy=fy,
                                                                                    interpolation=cv2.INTER_CUBIC))
    assert all(np.array_equal(r, s) for r, s in zip(ref, same))


def test_angle_zero_is_the_existing_path():
    rng = np.random.default_rng(5)
    out = rng.random((2, 50, 12, 16), dtype=np.float32)
    args = (out, 4, (48, 64), [0, 0, 3, 5], (40, 50), 30, 48, skeleton.FLIP_PAF_ORD, skeleton.FLIP_HEAT_ORD[:18])
    a, b = rp.post_network_scale(*args, angle=0.0), pp.post_network_scale(*args)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
