"""TEST INFRASTRUCTURE -- CPU restatement of the reference's pre-network stage, numpy only.

What ``evaluate.py:98-116`` hands to the network for one ``(scale, angle)`` item of ``predict()``'s loop:

    imageToTest        = cv2.resize(image, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)   # uint8 BGR
    imageToTest_padded = util.padRightDownCorner(imageToTest, max_downsample, padValue)
    input_img          = np.float32(imageToTest_padded / 255)
    input_img          = cv2.warpAffine(input_img, getRotationMatrix2D((Hp / 2, Wp / 2), angle, 1), (0, 0))  # angle != 0
    pair               = [input_img, input_img[:, ::-1]]

``resize_cubic_u8`` follows OpenCV's generic 8-bit ``INTER_CUBIC`` path (``modules/imgproc/src/resize.cpp``) without IPP:

* ``dsize = (rint(w fx), rint(h fy))`` in float64, round half to even; ``dsize == ssize`` is a plain copy;
* per destination index ``d`` of an axis: ``f = (float)((d + 0.5) (1 / fx) - 0.5)``, ``s = floor(f)``, the weights
  ``interpolateCubic(f - s)`` (float32, ``A = -0.75``, ``oracle.postnet_port.cubic_coeffs``) converted to
  ``saturate_cast<short>(c 2048)`` (rint of the float32 product); taps ``s - 1 .. s + 2`` clamped to the axis;
* horizontal pass: exact int32 sums of ``u8 x short``;
* vertical pass (``VResizeCubicVec_32s8u``): float32, ``b_k = (float)beta_k (1 / 2048^2)``,
  ``S0 b0 + (S1 b1 + (S2 b2 + S3 b3))`` with every product and sum rounded (no FMA), ``rint`` (half to even),
  saturated to ``[0, 255]``.  The last ``(width cn) mod VEC_LANES`` values of each row, which the vector loop does not
  reach, take the scalar integer form ``(S0 beta0 + S1 beta1 + S2 beta2 + S3 beta3 + 2^21) >> 22``, saturated.

It equals ``cv2.resize`` with ``cv2.ipp.setUseIPP(False)`` bit for bit and default cv2 (IPP on) within 1
(``tests/test_prenet_port.py``).  The rotation is ``rotation_port.warp_affine_linear`` on the float image (border 0)
with the forward matrix.  Nothing under ``improved_body_parts_b200/`` imports this file.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np

import rotation_port as rp
from oracle import postnet_port as pp

_F = np.float32
#: int16 lanes of OpenCV's baseline 128-bit vector width: the vertical pass's vector loop covers whole groups of 8 values
VEC_LANES = 8
#: ``np.float32(u8 / 255)``: the float64 quotient rounded to float32
DIV255 = (np.arange(256, dtype=np.float64) / 255).astype(_F)


def resized_size(h: int, w: int, scale: float) -> Tuple[int, int]:
    """``cv2.resize(..., fx=scale, fy=scale)``'s output ``(rows, cols)``: ``saturate_cast<int>`` of the float64 product."""
    return int(np.rint(h * float(scale))), int(np.rint(w * float(scale)))


def padded_size(h: int, w: int, max_downsample: int) -> Tuple[int, int]:
    """``util.padRightDownCorner``: the next multiples of ``max_downsample``."""
    return h + (-h) % max_downsample, w + (-w) % max_downsample


def _axis(n_dst: int, n_src: int, scale: float) -> Tuple[np.ndarray, np.ndarray]:
    """Per destination index: the four clamped source indices and the fixed-point weights (int64 holding shorts)."""
    d = np.arange(n_dst, dtype=np.float64)
    f = ((d + 0.5) * (1.0 / scale) - 0.5).astype(_F)
    s = np.floor(f).astype(np.int64)
    frac = (f - s.astype(_F)).astype(_F)
    idx = np.clip(s[:, None] + np.arange(-1, 3)[None, :], 0, n_src - 1)
    coef = np.rint(pp.cubic_coeffs(frac) * _F(2048)).astype(np.int64)  # saturate_cast<short>(cbuf[k] * 2048)
    return idx, coef


def resize_cubic_u8(src: np.ndarray, scale: float) -> np.ndarray:
    """``cv2.resize(src, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)`` without IPP, uint8 ``[h, w, C]``."""
    a = np.asarray(src)
    assert a.dtype == np.uint8 and a.ndim == 3
    h, w, cn = a.shape
    H, W = resized_size(h, w, scale)
    if (H, W) == (h, w):
        return a.copy()
    ix, ax = _axis(W, w, scale)
    iy, ay = _axis(H, h, scale)
    ai = a.astype(np.int64)
    S = sum(ai[:, ix[:, k], :] * ax[None, :, k, None] for k in range(4))  # [h, W, cn], exact
    rows = [S[iy[:, k]] for k in range(4)]                                 # [H, W, cn] per tap
    # float form (the vector loop)
    b = (ay.astype(_F) * _F(1.0 / (2048 * 2048))).astype(_F)
    f = [r.astype(_F) * b[:, k, None, None] for k, r in enumerate(rows)]
    vf = f[0] + (f[1] + (f[2] + f[3]))
    out_f = np.clip(np.rint(vf), 0, 255)
    # integer form (the scalar tail of each row)
    vi = sum(r * ay[:, k, None, None] for k, r in enumerate(rows))
    out_i = np.clip((vi + (1 << 21)) >> 22, 0, 255)
    flat = np.arange(W * cn).reshape(W, cn)
    tail = flat >= (W * cn) // VEC_LANES * VEC_LANES
    return np.where(tail[None], out_i, out_f).astype(np.uint8)


def pad_right_down(img: np.ndarray, max_downsample: int, pad_value: int) -> Tuple[np.ndarray, list]:
    """``util.padRightDownCorner`` (utils/util.py:44-64): ``(padded, pad)`` with ``pad = [up, left, down, right]``."""
    h, w = img.shape[:2]
    Hp, Wp = padded_size(h, w, max_downsample)
    return np.pad(img, ((0, Hp - h), (0, Wp - w), (0, 0)), constant_values=pad_value), [0, 0, Hp - h, Wp - w]


def network_input(image: np.ndarray, scale: float, angle: float = 0.0, max_downsample: int = 64, pad_value: int = 128,
                  resize=resize_cubic_u8):
    """One item of ``evaluate.py:98-116``: ``(pair [2, Hp, Wp, 3] float32, (crop_h, crop_w), pad)``.

    ``pair[0]`` is the scaled, padded image over 255 (rotated by ``angle`` about the reference's swapped centre),
    ``pair[1]`` its mirror; ``(crop_h, crop_w)`` is ``imageToTest``'s size, what ``spg_postnet`` crops to."""
    resized = resize(image, scale)
    padded, pad = pad_right_down(resized, max_downsample, pad_value)
    x = DIV255[padded]
    if float(angle) != 0.0:
        x = rp.warp_affine_linear(x, rp.rotation_matrix(x.shape[:2], float(angle)))
    return np.stack([x, x[:, ::-1]]), resized.shape[:2], pad


def network_inputs(image: np.ndarray, scale: float, angles: Sequence[float], max_downsample: int = 64,
                   pad_value: int = 128) -> Tuple[np.ndarray, Tuple[int, int]]:
    """Every angle of one scale, as ``spg_prenet`` writes them: ``([n_angles, 2, Hp, Wp, 3], (crop_h, crop_w))``."""
    items = [network_input(image, scale, a, max_downsample, pad_value) for a in angles]
    return np.stack([p for p, _, _ in items]), items[0][1]
