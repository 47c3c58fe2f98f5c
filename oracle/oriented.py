"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the oriented boxes of mask regions and the affine crop warp
(``prepost.mask_components_oriented`` / ``prepost.warp_crops``, DESIGN.md section 6b).

Restates in numpy / Python what the device computes:

* ``moments``   -- the int64 raw moments n, Sx, Sy, Sxx, Sxy, Syy of one region (``cv2.moments(binaryImage=True)``'s
  m00, m10, m01, m20, m11, m02, which are exact integers for such planes);
* ``principal_axis`` -- the unit eigenvector e1 of the larger eigenvalue of the frame-space covariance, with no
  transcendental function: exact integer covariances, one rounding to float64 each, then correctly rounded
  + - * / sqrt only (Python floats and numpy float64 arrays never contract into FMA);
* ``oriented_rows`` -- moments and ``obox = (e1x, e1y, umin, umax, vmin, vmax)`` of the selected rows of a plane;
* ``warp_affine`` -- ``cv2.warpAffine(src, M, (w, h), flags=INTER_LINEAR | WARP_INVERSE_MAP,
  borderMode=BORDER_REPLICATE)`` for uint8 RGB frames: OpenCV's fixed-point coordinates (AB_BITS = 10,
  INTER_BITS = 5) and 5-bit bilinear weights.

The device results must equal these bit for bit (tests/test_oriented.py); the tests pin ``moments`` and
``warp_affine`` to OpenCV and ``principal_axis`` to ``np.linalg.eigh``.  Nothing in the product path imports this
module.
"""
from __future__ import annotations

import numpy as np


def moments(xs: np.ndarray, ys: np.ndarray):
    """Pixel coordinates of one region -> (n, Sx, Sy, Sxx, Sxy, Syy) as Python ints."""
    x = xs.astype(np.int64)
    y = ys.astype(np.int64)
    return (int(x.size), int(x.sum()), int(y.sum()), int((x * x).sum()), int((x * y).sum()), int((y * y).sum()))


def principal_axis(mom, sx: float = 1.0, sy: float = 1.0):
    """(e1x, e1y) of the raw moments ``mom`` of a region whose mask pixel (x, y) sits at frame point
    ((x + 0.5) sx - 0.5, (y + 0.5) sy - 0.5)."""
    n, Sx, Sy, Sxx, Sxy, Syy = (int(v) for v in mom)
    cxx = float(n * Sxx - Sx * Sx)          # exact integers, one correctly rounded conversion each
    cxy = float(n * Sxy - Sx * Sy)
    cyy = float(n * Syy - Sy * Sy)
    sx, sy = float(sx), float(sy)
    a = (sx * sx) * cxx
    b = (sx * sy) * cxy
    c = (sy * sy) * cyy
    if b == 0.0:
        return (1.0, 0.0) if a >= c else (0.0, 1.0)
    amc = a - c
    d = float(np.sqrt(amc * amc + 4.0 * (b * b)))
    if a >= c:
        vx, vy = amc + d, 2.0 * b
    else:
        vx, vy = 2.0 * b, (c - a) + d
    nrm = float(np.sqrt(vx * vx + vy * vy))
    ex, ey = vx / nrm, vy / nrm
    if ex < 0.0 or (ex == 0.0 and ey < 0.0):
        ex, ey = -ex, -ey
    return ex, ey


def extents(xs: np.ndarray, ys: np.ndarray, e1, sx: float = 1.0, sy: float = 1.0):
    """(umin, umax, vmin, vmax) of the region's frame points projected on e1 and e2 = (-e1y, e1x)."""
    X = (xs.astype(np.float64) + 0.5) * float(sx) - 0.5
    Y = (ys.astype(np.float64) + 0.5) * float(sy) - 0.5
    e1x, e1y = e1
    e2x, e2y = -e1y, e1x
    u = X * e1x + Y * e1y
    v = X * e2x + Y * e2y
    return float(u.min()), float(u.max()), float(v.min()), float(v.max())


def oriented_rows(labels: np.ndarray, comps: np.ndarray, scale=(1.0, 1.0)):
    """Label plane (``scipy.ndimage.label``) + its component rows int32 [K, 6] (label in column 5, 0 = unused)
    -> (moments int64 [K, 6], obox float64 [K, 6]); unused rows are zeros."""
    k = comps.shape[0]
    mom = np.zeros((k, 6), np.int64)
    obox = np.zeros((k, 6), np.float64)
    sx, sy = scale
    for r in range(k):
        lab = int(comps[r, 5])
        if lab == 0:
            continue
        ys, xs = np.nonzero(labels == lab)
        m = moments(xs, ys)
        e1 = principal_axis(m, sx, sy)
        mom[r] = m
        obox[r] = (*e1, *extents(xs, ys, e1, sx, sy))
    return mom, obox


def _rint(a: np.ndarray) -> np.ndarray:
    """cvRound of doubles: round half to even (np.rint), as int64."""
    return np.rint(a).astype(np.int64)


def warp_affine(src: np.ndarray, M, out_w: int, out_h: int) -> np.ndarray:
    """uint8 [H, W, C] -> uint8 [out_h, out_w, C]: output pixel (j, i) samples src at
    (M00 j + M01 i + M02, M10 j + M11 i + M12), bilinear, replicated border -- OpenCV's fixed point:

        X = (rint((M01 i + M02) * 1024) + 16 + rint((M00 j) * 1024)) >> 5    (Y likewise)
        integer part X >> 5, fraction X & 31, weights (32 - fx)(32 - fy), fx (32 - fy), (32 - fx) fy, fx fy,
        each tap clamped into the frame, result (sum w p + 512) >> 10."""
    M = np.asarray(M, np.float64).reshape(2, 3)
    h, w = src.shape[:2]
    j = np.arange(out_w, dtype=np.float64)
    i = np.arange(out_h, dtype=np.float64)
    ax = _rint((M[0, 0] * j) * 1024.0)
    ay = _rint((M[1, 0] * j) * 1024.0)
    rx = _rint((M[0, 1] * i + M[0, 2]) * 1024.0) + 16
    ry = _rint((M[1, 1] * i + M[1, 2]) * 1024.0) + 16
    X = (rx[:, None] + ax[None, :]) >> 5
    Y = (ry[:, None] + ay[None, :]) >> 5
    x0, fx = X >> 5, X & 31
    y0, fy = Y >> 5, Y & 31
    xa, xb = np.clip(x0, 0, w - 1), np.clip(x0 + 1, 0, w - 1)
    ya, yb = np.clip(y0, 0, h - 1), np.clip(y0 + 1, 0, h - 1)
    s = src.astype(np.int64)
    w00 = ((32 - fx) * (32 - fy))[..., None]
    w01 = (fx * (32 - fy))[..., None]
    w10 = ((32 - fx) * fy)[..., None]
    w11 = (fx * fy)[..., None]
    acc = w00 * s[ya, xa] + w01 * s[ya, xb] + w10 * s[yb, xa] + w11 * s[yb, xb]
    return ((acc + 512) >> 10).astype(np.uint8)
