"""GPU pre/post-processing around the forward (SURVEY.md 8f ranks 1-2), via ``libunetb200.so``:

* ``resize_u8``  -- ``PIL.Image.resize((512, 512))`` of reference inference.py:35,63 for uint8
  frames already on the device, bit-identical to Pillow's 8-bit bicubic resample;
* ``mask_bbox``  -- the ``np.where(mask)`` min/max of reference inference.py:85-93 as 5 ints per
  (image, class) instead of a 512x512 mask;
* ``mask_components`` -- connected components of the masks (``scipy.ndimage.label`` labels, the boxes and sizes
  of the largest regions of each plane), where ``mask_bbox`` gives one box over all set pixels;
* ``mask_components_oriented`` -- the same plus the moments and the oriented box (principal axis and extents in
  frame coordinates) of every listed region;
* ``warp_crops`` -- a ragged batch of affine crops of device frames, bit-identical to ``cv2.warpAffine``
  (``INTER_LINEAR | WARP_INVERSE_MAP``, ``BORDER_REPLICATE``), with the byte sum of each crop.
"""
from __future__ import annotations

import threading
from typing import Dict, Tuple

import numpy as np
import torch

from . import _native as nat

_table_cache: Dict[Tuple[int, int, str], Tuple[torch.Tensor, torch.Tensor, int]] = {}
_lock = threading.Lock()


def resize_tables_host(in_size: int, out_size: int):
    """Pillow's fixed-point coefficient table of one axis: (kk int32 [out, ksize], bounds int32 [out, 2])."""
    lib = nat.lib()
    ks = lib.unetb200_resize_ksize(in_size, out_size)
    if ks <= 0:
        raise ValueError(f"bad resize {in_size} -> {out_size}")
    kk = np.zeros((out_size, ks), dtype=np.int32)
    bounds = np.zeros((out_size, 2), dtype=np.int32)
    nat.check(lib.unetb200_resize_coeffs(in_size, out_size, kk.ctypes.data, bounds.ctypes.data))
    return kk, bounds


def _tables(in_size: int, out_size: int, device: torch.device):
    key = (in_size, out_size, str(device))
    with _lock:
        t = _table_cache.get(key)
        if t is None:
            kk, bounds = resize_tables_host(in_size, out_size)
            t = (torch.from_numpy(kk).to(device), torch.from_numpy(bounds).to(device), kk.shape[1])
            if len(_table_cache) > 64:
                _table_cache.clear()
            _table_cache[key] = t
    return t


def resize_u8(frames: torch.Tensor, oh: int, ow: int, out: torch.Tensor = None, channels: int = None) -> torch.Tensor:
    """uint8 ``[N, H, W, C]`` on a CUDA device -> uint8 ``[N, oh, ow, C]``, bit-identical to
    ``PIL.Image.resize((ow, oh))`` (default BICUBIC) of each frame.  Enqueued on the current stream.
    ``out``: optional contiguous destination (e.g. a slot of a batch tensor).  ``channels`` < C reads only
    the leading channels of every pixel (``channels=3`` of a ``[N, H, W, 4]`` RGBX frame, Pillow's own storage
    of an RGB image) and returns ``[N, oh, ow, channels]``."""
    if frames.dtype != torch.uint8 or frames.dim() != 4 or not frames.is_cuda:
        raise RuntimeError("resize_u8 expects a CUDA uint8 [N,H,W,C] tensor")
    frames = frames.contiguous()
    n, h, w, ps = frames.shape
    c = ps if channels is None else int(channels)
    if not (1 <= c <= ps):
        raise RuntimeError(f"resize_u8: channels={c} of a {ps}-byte pixel")
    dev = frames.device
    if out is None:
        out = torch.empty((n, oh, ow, c), dtype=torch.uint8, device=dev)
    elif (out.dtype != torch.uint8 or tuple(out.shape) != (n, oh, ow, c) or out.device != dev
          or not out.is_contiguous()):
        raise RuntimeError("resize_u8: out must be a contiguous uint8 [N,oh,ow,C] tensor on the same device")
    if ow == w and c != ps:          # no horizontal pass to drop the padding byte in: repack first
        frames, ps = frames[..., :c].contiguous(), c
    if oh == h and ow == w:
        out.copy_(frames)
        return out
    kx = bx = ky = by = tmp = None
    ksx = ksy = 0
    if ow != w:
        kx, bx, ksx = _tables(w, ow, dev)
    if oh != h:
        ky, by, ksy = _tables(h, oh, dev)
    if ow != w and oh != h:
        tmp = torch.empty((n, h, ow, c), dtype=torch.uint8, device=dev)
    p = lambda t: None if t is None else t.data_ptr()
    with torch.cuda.device(dev):
        nat.check(nat.lib().unetb200_resize_bicubic_u8_ps(
            frames.data_ptr(), n, h, w, c, ps, p(kx), p(bx), ksx, p(ky), p(by), ksy, p(tmp), out.data_ptr(),
            oh, ow, torch.cuda.current_stream(dev).cuda_stream))
    return out


def mask_bbox(mask: torch.Tensor) -> torch.Tensor:
    """uint8 ``[N, C, H, W]`` (non-zero = set) -> int32 ``[N, C, 5]`` = xmin, xmax, ymin, ymax, count
    (empty plane: W, -1, H, -1, 0).  Enqueued on the current stream."""
    if mask.dtype != torch.uint8 or mask.dim() != 4 or not mask.is_cuda:
        raise RuntimeError("mask_bbox expects a CUDA uint8 [N,C,H,W] tensor")
    mask = mask.contiguous()
    n, c, h, w = mask.shape
    out = torch.empty((n, c, 5), dtype=torch.int32, device=mask.device)
    with torch.cuda.device(mask.device):
        nat.check(nat.lib().unetb200_mask_bbox(mask.data_ptr(), n * c, h, w, out.data_ptr(),
                                               torch.cuda.current_stream(mask.device).cuda_stream))
    return out


def mask_bbox_bits(bits: torch.Tensor) -> torch.Tensor:
    """Bit-packed masks uint8 ``[N, C, H, W/8]`` (``Engine.run(mask_bits=True)``) -> int32 ``[N, C, 5]`` as
    :func:`mask_bbox`.  ``W`` must be a multiple of 32.  Enqueued on the current stream."""
    if bits.dtype != torch.uint8 or bits.dim() != 4 or not bits.is_cuda:
        raise RuntimeError("mask_bbox_bits expects a CUDA uint8 [N,C,H,W/8] tensor")
    bits = bits.contiguous()
    n, c, h, wb = bits.shape
    if wb % 4:
        raise RuntimeError("mask_bbox_bits needs a mask width that is a multiple of 32")
    out = torch.empty((n, c, 5), dtype=torch.int32, device=bits.device)
    with torch.cuda.device(bits.device):
        nat.check(nat.lib().unetb200_mask_bbox_bits(bits.data_ptr(), n * c, h, wb * 8, out.data_ptr(),
                                                    torch.cuda.current_stream(bits.device).cuda_stream))
    return out


def mask_components(mask: torch.Tensor, *, packed: bool = False, connectivity: int = 8, max_components: int = 8,
                    labels: bool = False):
    """Connected components of every plane of uint8 ``[N, C, H, W]`` masks (non-zero = set), or of bit-packed
    ``[N, C, H, W/8]`` masks with ``packed=True`` (``Engine.run(mask_bits=True)``; ``W`` a multiple of 32).

    Returns ``(comps, n)``: int32 ``[N, C, K, 6]`` = xmin, xmax, ymin, ymax, count, label of the
    ``K = max_components`` (1..16) largest components of each plane (count descending, then label ascending;
    unused rows W, -1, H, -1, 0, 0) and int32 ``[N, C]`` = number of components per plane.  With ``labels=True``
    also int32 ``[N, C, H, W]``, equal to ``scipy.ndimage.label`` of each plane (4-connectivity:
    ``generate_binary_structure(2, 1)``; 8: ``np.ones((3, 3))``).  Enqueued on the current stream."""
    if mask.dtype != torch.uint8 or mask.dim() != 4 or not mask.is_cuda:
        raise RuntimeError("mask_components expects a CUDA uint8 [N,C,H,W] (or [N,C,H,W/8] bit-packed) tensor")
    mask = mask.contiguous()
    n, c, h, wm = mask.shape
    w = wm * 8 if packed else wm
    lib = nat.lib()
    ws_bytes = lib.unetb200_components_workspace_bytes(n * c, h, w)
    if ws_bytes == 0:
        raise RuntimeError(f"mask_components: bad mask shape {tuple(mask.shape)}")
    dev = mask.device
    comps = torch.empty((n, c, max(int(max_components), 1), 6), dtype=torch.int32, device=dev)
    counts = torch.empty((n, c), dtype=torch.int32, device=dev)
    lab = torch.empty((n, c, h, w), dtype=torch.int32, device=dev) if labels else None
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        nat.check(lib.unetb200_mask_components(
            mask.data_ptr(), int(bool(packed)), n * c, h, w, int(connectivity), int(max_components),
            None if lab is None else lab.data_ptr(), comps.data_ptr(), counts.data_ptr(), ws.data_ptr(), ws_bytes,
            torch.cuda.current_stream(dev).cuda_stream))
    return (comps, counts, lab) if labels else (comps, counts)


def _plane_scale(scale, n: int, c: int, dev) -> torch.Tensor:
    """``scale`` of :func:`mask_components_oriented` -> float64 ``[n, c, 2]`` on ``dev`` (``None`` stays ``None``)."""
    if scale is None:
        return None
    arr = np.asarray(scale.detach().cpu() if torch.is_tensor(scale) else scale, dtype=np.float64)
    if arr.shape == (2,):
        arr = np.broadcast_to(arr, (n, c, 2))
    elif arr.shape == (n, 2):
        arr = np.broadcast_to(arr[:, None], (n, c, 2))
    elif arr.shape != (n, c, 2):
        raise ValueError(f"scale must be (sx, sy), [N, 2] or [N, C, 2]; got shape {arr.shape}")
    if not (np.isfinite(arr).all() and (arr > 0).all()):
        raise ValueError("scale factors must be positive and finite")
    return torch.from_numpy(np.ascontiguousarray(arr)).to(dev)


def mask_components_oriented(mask: torch.Tensor, *, packed: bool = False, connectivity: int = 8,
                             max_components: int = 8, scale=None, labels: bool = False):
    """:func:`mask_components` plus the oriented box of each listed component (DESIGN.md 6b).

    ``scale``: ``(sx, sy)`` for every plane, or per image ``[N, 2]`` / per plane ``[N, C, 2]`` (default 1, 1): the
    size of a mask pixel in frame pixels, ``(frame_w / W, frame_h / H)`` for masks of a resized frame.  Mask pixel
    ``(x, y)`` stands for the frame point ``((x + 0.5) sx - 0.5, (y + 0.5) sy - 0.5)``.

    Returns ``(comps, n, moments, obox)`` (and the labels last with ``labels=True``): ``comps`` and ``n`` exactly as
    :func:`mask_components`; int64 ``[N, C, K, 6]`` = n, Sx, Sy, Sxx, Sxy, Syy, the raw moments of each row's mask
    pixels; float64 ``[N, C, K, 6]`` = e1x, e1y, umin, umax, vmin, vmax: the unit principal axis ``e1`` of the
    frame-space covariance (``e1x > 0``, or ``e1x == 0`` and ``e1y > 0``) and the extents of the frame points
    projected on ``e1`` and ``e2 = (-e1y, e1x)``.  Unused rows are zeros.  Planes up to 32767 pixels on a side.
    Enqueued on the current stream."""
    if mask.dtype != torch.uint8 or mask.dim() != 4 or not mask.is_cuda:
        raise RuntimeError("mask_components_oriented expects a CUDA uint8 [N,C,H,W] (or [N,C,H,W/8] bit-packed) "
                           "tensor")
    mask = mask.contiguous()
    n, c, h, wm = mask.shape
    w = wm * 8 if packed else wm
    lib = nat.lib()
    ws_bytes = lib.unetb200_components_oriented_workspace_bytes(n * c, h, w)
    if ws_bytes == 0:
        raise RuntimeError(f"mask_components_oriented: bad mask shape {tuple(mask.shape)}")
    dev = mask.device
    sc = _plane_scale(scale, n, c, dev)
    k = max(int(max_components), 1)
    comps = torch.empty((n, c, k, 6), dtype=torch.int32, device=dev)
    counts = torch.empty((n, c), dtype=torch.int32, device=dev)
    mom = torch.empty((n, c, k, 6), dtype=torch.int64, device=dev)
    obox = torch.empty((n, c, k, 6), dtype=torch.float64, device=dev)
    lab = torch.empty((n, c, h, w), dtype=torch.int32, device=dev) if labels else None
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        nat.check(lib.unetb200_mask_components_oriented(
            mask.data_ptr(), int(bool(packed)), n * c, h, w, int(connectivity), int(max_components),
            None if sc is None else sc.data_ptr(), None if lab is None else lab.data_ptr(), comps.data_ptr(),
            counts.data_ptr(), mom.data_ptr(), obox.data_ptr(), ws.data_ptr(), ws_bytes,
            torch.cuda.current_stream(dev).cuda_stream))
    return (comps, counts, mom, obox, lab) if labels else (comps, counts, mom, obox)


def _warp_batch(frames, mats, sizes):
    """Validated batch of :func:`warp_crops` -> (buffer uint8 [total], byte offsets, (out_w, out_h) sizes, sums)."""
    n = len(sizes)
    if isinstance(frames, torch.Tensor):
        frames = [frames] * n
    frames = list(frames)
    mats = np.asarray(mats, dtype=np.float64)
    if len(frames) != n or mats.shape != (n, 2, 3):
        raise ValueError(f"warp_crops: {len(frames)} frames, matrices of shape {mats.shape} and {n} sizes do not "
                         "describe the same crops (one frame, one 2x3 matrix and one (w, h) per crop)")
    if n == 0:
        raise ValueError("warp_crops: no crops")
    dev = frames[0].device
    for f in frames:
        if (f.dtype != torch.uint8 or f.dim() != 3 or f.shape[2] not in (3, 4) or not f.is_cuda
                or not f.is_contiguous() or f.device != dev):
            raise RuntimeError("warp_crops expects contiguous CUDA uint8 [H,W,3] or [H,W,4] frames on one device")
    table = (nat.WarpCrop * n)()
    offs, total = [], 0
    for t, f, m, (ow, oh) in zip(table, frames, mats, sizes):
        ow, oh = int(ow), int(oh)
        t.src, t.src_h, t.src_w = f.data_ptr(), int(f.shape[0]), int(f.shape[1])
        t.src_stride, t.src_pixel_bytes = int(f.shape[1]), int(f.shape[2])
        t.m[:] = [float(v) for v in m.reshape(-1)]
        t.out_w, t.out_h, t.out_off = ow, oh, total
        offs.append(total)
        total += 3 * max(ow, 0) * max(oh, 0)
    buf = torch.empty((max(total, 1),), dtype=torch.uint8, device=dev)
    sums = torch.empty((n,), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        d_tab = torch.frombuffer(bytearray(table), dtype=torch.uint8).to(dev)
        nat.check(nat.lib().unetb200_warp_crops(table, d_tab.data_ptr(), n, buf.data_ptr(), sums.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream))
    return buf, offs, [(int(w), int(h)) for w, h in sizes], sums


def warp_crops(frames, mats, sizes):
    """Ragged batch of upright (or any affine) crops of frames already on the device.

    ``frames``: one contiguous CUDA uint8 ``[H, W, 3]`` (RGB) or ``[H, W, 4]`` (RGBX) frame for all crops, or a
    sequence with one per crop; ``mats``: per crop the inverse 2x3 map ``M`` (output pixel ``(j, i)`` samples the
    frame at ``M @ (j, i, 1)``); ``sizes``: per crop ``(out_w, out_h)``.  Each crop equals
    ``cv2.warpAffine(frame_rgb, M, (out_w, out_h), flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP,
    borderMode=cv2.BORDER_REPLICATE)`` bit for bit.

    Returns ``(crops, sums)``: uint8 ``[out_h, out_w, 3]`` views into one device buffer, and int64 ``[n]`` byte sums
    on the device (a crop is near-black when ``sum < 3 * 3 * out_w * out_h``).  Enqueued on the current stream."""
    buf, offs, sz, sums = _warp_batch(frames, mats, sizes)
    return [buf[o:o + 3 * w * h].view(h, w, 3) for o, (w, h) in zip(offs, sz)], sums


def box_sums(frame: torch.Tensor, rects, channels: int = None) -> torch.Tensor:
    """uint8 ``[H, W, C]`` frame on a CUDA device + up to 16 half-open rectangles ``(x1, y1, x2, y2)``
    -> int64 ``[n]`` byte sums on the device (the ``np.array(crop).mean() < 3`` test of reference
    inference.py:121-125 becomes ``sum < 3 * area * channels``).  ``channels=3`` on a ``[H, W, 4]`` RGBX frame
    leaves the padding byte out.  Enqueued on the current stream."""
    if frame.dtype != torch.uint8 or frame.dim() != 3 or not frame.is_cuda or not frame.is_contiguous():
        raise RuntimeError("box_sums expects a contiguous CUDA uint8 [H,W,C] tensor")
    import ctypes as C
    h, w, c = frame.shape
    used = c if channels is None else int(channels)
    n = len(rects)
    flat = (C.c_int32 * (4 * n))(*[int(v) for r in rects for v in r])
    out = torch.empty((n,), dtype=torch.int64, device=frame.device)
    with torch.cuda.device(frame.device):
        nat.check(nat.lib().unetb200_box_sums_ps(frame.data_ptr(), h, w, c, used, flat, n, out.data_ptr(),
                                                 torch.cuda.current_stream(frame.device).cuda_stream))
    return out
