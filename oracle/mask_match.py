"""Host restatement of ``unetb200_mask_match`` (DESIGN.md 6b, "Region matching"), bit for bit.

Regions are ``scipy.ndimage.label`` components (4-connectivity: ``generate_binary_structure(2, 1)``; 8:
``np.ones((3, 3))``).  Every overlapping (pred, gt) region pair and its intersection come from the unique codes
``pred_label * (n_gt + 1) + gt_label`` of the pixels set in both.  A pred region with fewer than ``min_pixels``
pixels is ignored; a pair matches when ``I > t * U`` in float64 (one correctly rounded product of exact integers).
``iou_sum`` adds the correctly rounded ``I / U`` of the matched pairs in the device's order: partial sum ``j`` of
256 takes pred labels ``j + 1, j + 257, ...`` in ascending order from 0.0, then a pairwise tree
(``s[j] += s[j + half]``, half = 128 .. 1) combines them."""
from __future__ import annotations

import numpy as np
from scipy import ndimage

FIELDS = ("px_tp", "px_fp", "px_fn", "n_pred", "n_gt", "tp", "sum_inter", "sum_union")
SUM_THREADS = 256


def structure(connectivity: int) -> np.ndarray:
    if connectivity == 4:
        return ndimage.generate_binary_structure(2, 1)
    if connectivity == 8:
        return np.ones((3, 3), bool)
    raise ValueError("connectivity must be 4 or 8")


def check_threshold(iou: float) -> float:
    t = float(iou)
    if not (np.isfinite(t) and 0.5 <= t < 1.0):
        raise ValueError("iou must be in [0.5, 1)")
    return t


def tree_sum(partial: np.ndarray) -> float:
    """The device's combination of the 256 partial sums."""
    s = np.array(partial, np.float64)
    half = SUM_THREADS // 2
    while half > 0:
        s[:half] = s[:half] + s[half:2 * half]
        half //= 2
    return float(s[0])


def ordered_iou_sum(pred_ids: np.ndarray, quotients: np.ndarray) -> float:
    """Sum of ``quotients`` (one per matched pair, ``pred_ids`` = 0-based pred label) in the device's order.  Rows of
    256 consecutive ids are added one after another (an id without a pair adds +0.0, which changes no sum)."""
    n = int(pred_ids.max()) + 1 if pred_ids.size else 0
    dense = np.zeros(-(-n // SUM_THREADS) * SUM_THREADS, np.float64)
    dense[pred_ids] = quotients
    partial = np.zeros(SUM_THREADS, np.float64)
    for row in dense.reshape(-1, SUM_THREADS):
        partial = partial + row
    return tree_sum(partial)


def match_plane(pred: np.ndarray, gt: np.ndarray, connectivity: int = 8, min_pixels: int = 1, iou: float = 0.5):
    """One plane pair (any dtype, non-zero = set) -> (int64 [8] counts, float iou_sum)."""
    t = check_threshold(iou)
    if min_pixels < 1:
        raise ValueError("min_pixels must be >= 1")
    p, g = np.asarray(pred) != 0, np.asarray(gt) != 0
    st = structure(connectivity)
    lp, n_p = ndimage.label(p, st)
    lg, n_g = ndimage.label(g, st)
    size_p = np.bincount(lp.ravel(), minlength=n_p + 1)
    size_g = np.bincount(lg.ravel(), minlength=n_g + 1)
    both = p & g
    codes = lp[both].astype(np.int64) * (n_g + 1) + lg[both]
    pairs, inter = np.unique(codes, return_counts=True)
    a, b = pairs // (n_g + 1), pairs % (n_g + 1)
    inter = inter.astype(np.int64)
    union = size_p[a].astype(np.int64) + size_g[b] - inter
    keep = size_p[a] >= min_pixels
    hit = keep & (inter.astype(np.float64) > t * union.astype(np.float64))
    counts = np.array([both.sum(), (p & ~g).sum(), (~p & g).sum(), int((size_p[1:] >= min_pixels).sum()), n_g,
                       int(hit.sum()), int(inter[hit].sum()), int(union[hit].sum())], np.int64)
    q = inter[hit].astype(np.float64) / union[hit].astype(np.float64)
    return counts, ordered_iou_sum(a[hit] - 1, q)


def mask_match(pred: np.ndarray, gt: np.ndarray, connectivity: int = 8, min_pixels: int = 1, iou: float = 0.5):
    """Stacks ``[..., H, W]`` -> (int64 ``[..., 8]``, float64 ``[...]``), as ``prepost.mask_match`` returns them."""
    pred, gt = np.asarray(pred), np.asarray(gt)
    if pred.shape != gt.shape or pred.ndim < 2:
        raise ValueError(f"pred {pred.shape} and gt {gt.shape} must be stacks of planes of one shape")
    lead = pred.shape[:-2]
    counts = np.zeros(lead + (8,), np.int64)
    sums = np.zeros(lead, np.float64)
    for idx in np.ndindex(*lead):
        counts[idx], sums[idx] = match_plane(pred[idx], gt[idx], connectivity, min_pixels, iou)
    return counts, sums
