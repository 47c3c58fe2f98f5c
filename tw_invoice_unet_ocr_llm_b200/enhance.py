"""OCR crop enhancement on the GPU (SURVEY.md 8f rank 4) -- drop-ins for the two helpers the
Streamlit app applies to every ``run_unet`` crop before OCR:

* ``enhance_for_ocrspace(pil_crop, mode="text")``  (reference app_camera.py:572-598)
* ``enhance_for_date_ocr(pil_crop)``               (reference app_camera.py:685-705)

Same names, arguments and return values (``None`` in, ``None`` out; otherwise a mode-"L" PIL image
four times the crop size).  The reference runs cv2.cvtColor -> cv2.resize(4x, INTER_CUBIC) ->
[filter2D sharpen] -> CLAHE -> [GaussianBlur] -> [Otsu] per crop on the host; here a whole ragged
batch of crops goes through ``libunetb200.so`` (``csrc/enhance.cuh``) with one upload and one
download, bit-identical to OpenCV's own code path.  ``enhance_batch`` is the batched entry point
(new, additive).  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np
import torch
from PIL import Image

from . import _native as nat

SHARPEN, BLUR, OTSU = 1, 2, 4
# kind -> (flags, CLAHE clipLimit): app_camera.py:586-598 and :693-703
KINDS = {
    "text": (SHARPEN | OTSU, 4.0),
    "amount": (SHARPEN, 4.0),
    "date": (BLUR | OTSU, 3.0),
}


def _pinned(nbytes: int) -> torch.Tensor:
    """Pinned host buffer from torch's caching host allocator: a block is recycled only after every
    tensor / numpy view of it is gone and the copies queued on it have completed, so results can be
    handed out as views (no extra host copy) and staging buffers need no bookkeeping here."""
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, pin_memory=True)


def _as_rgb_array(crop) -> np.ndarray:
    if isinstance(crop, Image.Image):
        crop = np.asarray(crop.convert("RGB"))            # app_camera.py:581 / :689
    arr = np.ascontiguousarray(crop)
    if arr.dtype != np.uint8 or arr.ndim != 3 or arr.shape[2] != 3:
        raise ValueError(f"expected a uint8 (h, w, 3) crop, got {arr.dtype} {arr.shape}")
    if arr.shape[0] == 0 or arr.shape[1] == 0:
        raise ValueError(f"empty crop {arr.shape}")
    return arr


def _recipe(kind):
    """"text" | "amount" | "date", or an explicit ``(flags, clip_limit)`` pair."""
    if isinstance(kind, str):
        if kind not in KINDS:
            raise ValueError(f"unknown enhancement kind {kind!r} (expected one of {sorted(KINDS)})")
        return KINDS[kind]
    flags, clip = kind
    return int(flags), float(clip)


def plan(sizes: Sequence[tuple], kinds: Sequence):
    """Host-side plan of a batch: (ctypes table, src_bytes, out_bytes, workspace_bytes)."""
    n = len(sizes)
    table = (nat.EnhCrop * n)()
    for i, ((h, w), kind) in enumerate(zip(sizes, kinds)):
        flags, clip = _recipe(kind)
        table[i].h, table[i].w, table[i].flags, table[i].clip = int(h), int(w), flags, clip
    sb, ob, wb = C.c_uint64(), C.c_uint64(), C.c_uint64()
    nat.check(nat.lib().unetb200_enhance_plan(table, n, C.byref(sb), C.byref(ob), C.byref(wb)))
    return table, sb.value, ob.value, wb.value


def _execute(table, n: int, table_dev_ptr: int, src_ptr: int, out_bytes: int, ws_bytes: int, dev, keep) -> list:
    """Run the five kernels on the current stream and bring the results back: list of uint8 (4h, 4w)."""
    stream = torch.cuda.current_stream(dev)
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device=dev)
    d_ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    nat.check(nat.lib().unetb200_enhance_run(table, table_dev_ptr, n, src_ptr, d_out.data_ptr(), d_ws.data_ptr(),
                                             stream.cuda_stream))
    down = _pinned(out_bytes)
    down[:out_bytes].copy_(d_out, non_blocking=True)
    stream.synchronize()
    del keep                                   # inputs stay referenced until the stream has drained
    res = down.numpy()                         # the views below keep the pinned block alive
    return [res[t.out_off: t.out_off + 16 * t.h * t.w].reshape(4 * t.h, 4 * t.w) for t in table]


def enhance_batch(crops: Sequence, kinds: Sequence, device=None) -> List[Optional[np.ndarray]]:
    """Enhance many crops at once.  ``crops``: PIL images or uint8 (h, w, 3) RGB arrays (``None``
    entries pass through); ``kinds``: "text" | "amount" | "date" per crop (or an explicit
    ``(flags, clip_limit)`` pair).  Returns uint8 (4h, 4w) arrays.  One H2D copy (table + pixels),
    five kernels, one D2H copy."""
    if len(crops) != len(kinds):
        raise ValueError("crops and kinds differ in length")
    if not torch.cuda.is_available():
        raise RuntimeError("enhance_batch needs a CUDA (B200, sm_100a) device: there is no CPU path "
                           "(the CPU oracle lives in oracle/ and is test-only)")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    live = [i for i, c in enumerate(crops) if c is not None]
    out: List[Optional[np.ndarray]] = [None] * len(crops)
    if not live:
        return out
    arrays = [_as_rgb_array(crops[i]) for i in live]
    table, src_bytes, out_bytes, ws_bytes = plan([a.shape[:2] for a in arrays], [kinds[i] for i in live])
    tab_bytes = (C.sizeof(table) + 15) & ~15
    stage = _pinned(tab_bytes + src_bytes)
    host = stage.numpy()
    host[:C.sizeof(table)] = np.frombuffer(table, dtype=np.uint8)
    for a, t in zip(arrays, table):
        host[tab_bytes + t.src_off: tab_bytes + t.src_off + a.size] = a.reshape(-1)
    with torch.cuda.device(dev):
        d_in = torch.empty(tab_bytes + src_bytes, dtype=torch.uint8, device=dev)
        d_in.copy_(stage[:tab_bytes + src_bytes], non_blocking=True)
        res = _execute(table, len(live), d_in.data_ptr(), d_in.data_ptr() + tab_bytes, out_bytes, ws_bytes, dev, d_in)
    for i, r in zip(live, res):
        out[i] = r
    return out


def enhance_windows(frame: torch.Tensor, rects: Sequence[tuple], kinds: Sequence) -> List[np.ndarray]:
    """Enhance rectangles ``(x1, y1, x2, y2)`` (half-open) of a uint8 ``[H, W, 3]`` RGB (or ``[H, W, 4]``
    RGBX) frame that is already on the device -- the crops ``run_unet`` cuts from the frame it uploaded --
    without packing or re-uploading them: only the 80-byte descriptors go up."""
    if frame.dtype != torch.uint8 or frame.dim() != 3 or frame.shape[2] not in (3, 4) or not frame.is_cuda \
            or not frame.is_contiguous():
        raise RuntimeError("enhance_windows expects a contiguous CUDA uint8 [H,W,3] or [H,W,4] frame")
    if len(rects) != len(kinds):
        raise ValueError("rects and kinds differ in length")
    if not rects:
        return []
    fh, fw, pb = int(frame.shape[0]), int(frame.shape[1]), int(frame.shape[2])
    n = len(rects)
    table = (nat.EnhCrop * n)()
    for t, (x1, y1, x2, y2), kind in zip(table, rects, kinds):
        x1, y1, x2, y2 = int(x1), int(y1), int(x2), int(y2)
        if not (0 <= x1 < x2 <= fw and 0 <= y1 < y2 <= fh):
            raise ValueError(f"rectangle {(x1, y1, x2, y2)} outside the {fw}x{fh} frame")
        t.flags, t.clip = _recipe(kind)
        t.h, t.w, t.src_stride, t.src_pixel_bytes, t.src_off = y2 - y1, x2 - x1, fw, pb, (y1 * fw + x1) * pb
    sb, ob, wb = C.c_uint64(), C.c_uint64(), C.c_uint64()
    nat.check(nat.lib().unetb200_enhance_plan(table, n, C.byref(sb), C.byref(ob), C.byref(wb)))
    dev = frame.device
    with torch.cuda.device(dev):
        d_tab = torch.frombuffer(bytearray(table), dtype=torch.uint8).to(dev)
        return _execute(table, n, d_tab.data_ptr(), frame.data_ptr(), ob.value, wb.value, dev, (d_tab, frame))


def enhance_packed(buf: torch.Tensor, offsets: Sequence[int], sizes: Sequence[tuple], kinds: Sequence
                   ) -> List[np.ndarray]:
    """Enhance packed uint8 ``[h][w][3]`` RGB crops that are already in the device buffer ``buf`` (1-D uint8) at byte
    ``offsets`` -- the upright crops of ``prepost.warp_crops`` -- in place: only the descriptors go up.  ``sizes``:
    ``(w, h)`` per crop.  Same results as :func:`enhance_batch` of the same crops."""
    if buf.dtype != torch.uint8 or buf.dim() != 1 or not buf.is_cuda or not buf.is_contiguous():
        raise RuntimeError("enhance_packed expects a contiguous CUDA uint8 1-D buffer")
    if not (len(offsets) == len(sizes) == len(kinds)):
        raise ValueError("offsets, sizes and kinds differ in length")
    if not offsets:
        return []
    n = len(offsets)
    table = (nat.EnhCrop * n)()
    for t, off, (w, h), kind in zip(table, offsets, sizes, kinds):
        off, w, h = int(off), int(w), int(h)
        if off < 0 or w <= 0 or h <= 0 or off + 3 * w * h > buf.numel():
            raise ValueError(f"crop of {w}x{h} at byte {off} outside the {buf.numel()}-byte buffer")
        t.flags, t.clip = _recipe(kind)
        t.h, t.w, t.src_stride, t.src_pixel_bytes, t.src_off = h, w, w, 3, off
    sb, ob, wb = C.c_uint64(), C.c_uint64(), C.c_uint64()
    nat.check(nat.lib().unetb200_enhance_plan(table, n, C.byref(sb), C.byref(ob), C.byref(wb)))
    dev = buf.device
    with torch.cuda.device(dev):
        d_tab = torch.frombuffer(bytearray(table), dtype=torch.uint8).to(dev)
        return _execute(table, n, d_tab.data_ptr(), buf.data_ptr(), ob.value, wb.value, dev, (d_tab, buf))


def enhance_for_ocrspace(pil_crop, mode: str = "text"):
    """Reference app_camera.py:572-598: ``mode="text"`` binarises (invoice number, date), any other
    mode returns the contrast-enhanced gray image (total amount)."""
    if pil_crop is None:
        return None
    return Image.fromarray(enhance_batch([pil_crop], ["text" if mode == "text" else "amount"])[0])


def enhance_for_date_ocr(pil_crop):
    """Reference app_camera.py:685-705."""
    if pil_crop is None:
        return None
    return Image.fromarray(enhance_batch([pil_crop], ["date"])[0])
