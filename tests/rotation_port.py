"""TEST INFRASTRUCTURE -- CPU restatement of the rotation search of the reference's post-network stage, numpy only.

Extends ``oracle/postnet_port.py`` (the scale loop at angle 0) with the two ``cv2.warpAffine`` calls the reference makes
when ``rotation_search`` has a non-zero angle (``evaluate.py:108-111`` on the network input, ``:144-146`` and
``:153-155`` on the up-sampled maps).  Nothing under ``improved_body_parts_b200/`` imports this file.

``warp_affine_linear`` follows OpenCV's generic fixed-point path (``modules/imgproc/src/imgwarp.cpp``: ``warpAffine``
with ``INTER_LINEAR``, ``BORDER_CONSTANT``, value 0, and ``remapBilinear`` on float32), step for step:

* the 2x3 matrix is inverted in float64 as ``warpAffine`` does without ``WARP_INVERSE_MAP``;
* source coordinates are fixed point with ``AB_BITS = 10`` and ``INTER_BITS = 5``: ``adelta[x] = rint(M0 x 1024)``,
  ``X0(y) = rint((M1 y + M2) 1024) + 16``, ``X = (X0 + adelta) >> 5`` (round half to even, arithmetic shifts), and
  the same for y with ``M3, M4, M5``;
* the integer tap is ``(Y >> 5, X >> 5)``; the weights are the float32 products of the table entries ``1 - t`` and
  ``t`` with ``t = (Y & 31) / 32`` and ``(X & 31) / 32``;
* the value is ``p00 w00 + p01 w01 + p10 w10 + p11 w11`` in float32, left to right; taps outside the map read 0.

It equals ``cv2.warpAffine`` bit for bit (``tests/test_postnet_rotation_port.py``), NaNs included: a NaN anywhere among
a pixel's four in-map taps makes that pixel NaN, whatever its weight; taps outside the map never contribute one.
"""
from __future__ import annotations

import math
from typing import Sequence, Tuple

import numpy as np

from oracle import postnet_port as pp

_F = np.float32


def rotation_matrix(padded_hw: Tuple[int, int], angle: float) -> np.ndarray:
    """``cv2.getRotationMatrix2D((rows / 2, cols / 2), angle, 1)`` as the reference calls it (``evaluate.py:109``).

    The centre is the padded image's ``(rows / 2, cols / 2)`` passed as ``(x, y)``: the reference swaps the two, and
    so does this.  OpenCV takes the centre as a ``Point2f`` and computes in float64 with libm's ``cos`` / ``sin``."""
    cx, cy = float(_F(padded_hw[0] / 2)), float(_F(padded_hw[1] / 2))
    a = float(angle) * (math.pi / 180)
    alpha, beta = math.cos(a), math.sin(a)
    return np.array([[alpha, beta, (1 - alpha) * cx - beta * cy],
                     [-beta, alpha, beta * cx + (1 - alpha) * cy]], np.float64)


def invert_affine(M: np.ndarray) -> Tuple[float, float, float, float, float, float]:
    """The inversion ``warpAffine`` applies to its matrix (no ``WARP_INVERSE_MAP``): destination -> source map."""
    m = [float(v) for v in np.asarray(M, np.float64).reshape(6)]
    D = m[0] * m[4] - m[1] * m[3]
    D = 1.0 / D if D != 0 else 0.0
    a11, a22 = m[4] * D, m[0] * D
    m[0], m[4] = a11, a22
    m[1] *= -D
    m[3] *= -D
    b1 = -m[0] * m[2] - m[1] * m[5]
    b2 = -m[3] * m[2] - m[4] * m[5]
    m[2], m[5] = b1, b2
    return tuple(m)


def warp_taps(M: np.ndarray, dst_hw: Tuple[int, int]):
    """Per destination pixel: integer tap ``(sy, sx)`` and fraction indices ``(fy, fx)`` in 0..31, each ``[H, W]``."""
    H, W = dst_hw
    m = invert_affine(M)
    x = np.arange(W, dtype=np.float64)
    y = np.arange(H, dtype=np.float64)
    adelta = np.rint(m[0] * x * 1024).astype(np.int64)
    bdelta = np.rint(m[3] * x * 1024).astype(np.int64)
    X0 = np.rint((m[1] * y + m[2]) * 1024).astype(np.int64) + 16
    Y0 = np.rint((m[4] * y + m[5]) * 1024).astype(np.int64) + 16
    X = (X0[:, None] + adelta[None, :]) >> 5
    Y = (Y0[:, None] + bdelta[None, :]) >> 5
    return Y >> 5, X >> 5, Y & 31, X & 31


def bilinear_weights(fy: np.ndarray, fx: np.ndarray):
    """The float32 table of ``initInterTab2D(INTER_LINEAR)``: ``(w00, w01, w10, w11)`` for fraction indices 0..31."""
    ty, tx = fy.astype(_F) * _F(1 / 32), fx.astype(_F) * _F(1 / 32)
    uy, ux = _F(1) - ty, _F(1) - tx
    return uy * ux, uy * tx, ty * ux, ty * tx


def warp_affine_linear(src: np.ndarray, M: np.ndarray) -> np.ndarray:
    """``cv2.warpAffine(src, M, (0, 0))`` (``INTER_LINEAR``, ``BORDER_CONSTANT`` 0) for float32 ``[h, w]`` / ``[h, w, C]``."""
    a = np.asarray(src, _F)
    squeeze = a.ndim == 2
    if squeeze:
        a = a[:, :, None]
    h, w = a.shape[:2]
    sy, sx, fy, fx = warp_taps(M, (h, w))
    weights = bilinear_weights(fy, fx)
    out = None
    for (dy, dx), wt in zip(((0, 0), (0, 1), (1, 0), (1, 1)), weights):
        yy, xx = sy + dy, sx + dx
        inside = (yy >= 0) & (yy < h) & (xx >= 0) & (xx < w)
        tap = np.where(inside[:, :, None], a[np.clip(yy, 0, h - 1), np.clip(xx, 0, w - 1)], _F(0))
        with np.errstate(invalid="ignore"):  # inf * 0 -> NaN, as in OpenCV
            term = tap * wt[:, :, None]
        out = term if out is None else out + term
    out = out.astype(_F)
    return out[:, :, 0] if squeeze else out


def post_network_scale(out_pair: np.ndarray, stride: int, padded_shape: Tuple[int, int], pad: Sequence[int],
                       image_shape: Tuple[int, int], n_paf: int, n_layers: int, flip_paf_ord: Sequence[int],
                       flip_heat_ord: Sequence[int], angle: float = 0.0, resize=pp.resize_cubic):
    """One item ``(scale, angle)`` of the loop after the forward pass (``evaluate.py:126-158``).

    Angle 0 is ``oracle.postnet_port.post_network_scale`` itself.  Otherwise the up-sampled maps are warped with the
    reverse rotation over the whole padded image before the crop (``:144-146``, ``:153-155``).  Returns
    ``(heatmap, paf)`` at image size."""
    if float(angle) == 0.0:
        return pp.post_network_scale(out_pair, stride, padded_shape, pad, image_shape, n_paf, n_layers, flip_paf_ord,
                                     flip_heat_ord, resize=resize)
    M_rev = rotation_matrix(padded_shape, -float(angle))
    paf_avg, heat_avg = pp.flip_ensemble(out_pair, n_paf, n_layers, flip_paf_ord, flip_heat_ord)
    outs = []
    for m in (heat_avg, paf_avg):
        up = resize(np.ascontiguousarray(m, np.float32), None, fx=stride, fy=stride)
        up = warp_affine_linear(up, M_rev)
        up = up[pad[0]:padded_shape[0] - pad[2], pad[1]:padded_shape[1] - pad[3], :]
        outs.append(resize(np.ascontiguousarray(up), (image_shape[1], image_shape[0])))
    return outs[0], outs[1]
