"""Drop-in for the reference ``inference.py`` (reference inference.py:1-130).

Same names, argument order and return types -- ``DEVICE``, ``IMG_SIZE``,
``FIELDS``, ``load_model(checkpoint_path)``, ``preprocess(pil_img)``,
``run_unet(pil_img, checkpoint_path) -> (masks, crops)`` -- so ``app_camera.py:16,787``
keeps working unmodified.  Differences, all internal:

* ``load_model`` caches the packed model per (checkpoint file, device) instead of
  rebuilding it on every ``run_unet`` call (reference inference.py:58).
* ``run_unet`` ships the resized uint8 frame to the GPU (0.79 MB instead of 3.1 MB
  of float32); the ``/255`` of ``preprocess`` happens in the first CUDA kernel and
  the sigmoid + per-class threshold (reference :72-79) in the last one, in logit
  space, so only three uint8 masks come back.
* For plain RGB inputs the 512x512 resize itself runs on the GPU (``prepost.resize_u8``,
  bit-identical to Pillow's bicubic resample) and the mask -> bounding box reduction of :85-93
  too (``prepost.mask_bbox``); other PIL modes take the reference's PIL calls on the host.
* ``run_unet_batch`` (new, additive) does the same for a list of images in one
  batched forward.
* ``run_unet_instances`` (new, additive) returns one crop per connected region of each field mask
  (``prepost.mask_components``) instead of one crop over all of its set pixels; with ``deskew=True`` each crop
  is cut upright along the region's principal axis (``prepost.mask_components_oriented`` +
  ``prepost.warp_crops``), and ``enhance=True`` adds the OCR enhancement of each crop.
"""
from __future__ import annotations

import math
import os
import threading
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
from PIL import Image

from .unet_model import UNet

# ---------------------------------------------------------------- constants (reference :9-12)
DEVICE = "cuda" if torch.cuda.is_available() else "cpu"
IMG_SIZE = 512
FIELDS = ["invoice_no", "date", "total_amount"]
# sigmoid-probability thresholds per field (reference :75-79)
THRESHOLDS = {"invoice_no": 0.25, "date": 0.40, "total_amount": 0.30}
MAX_CHUNK = 64            # images per forward in the batched entry points

_model_cache: Dict[tuple, UNet] = {}
_engine_cache: Dict[tuple, object] = {}     # same key -> the packed replica of that cached model
_cache_lock = threading.Lock()


def load_model(checkpoint_path: str):
    """Build ``UNet(3, 3)``, strictly load the state_dict, ``eval()`` (reference :17-24).

    The result is cached per (real path, mtime, size, device): the reference re-reads the
    124 MB checkpoint on every call, which costs ~1 s.  Unlike the reference, which returns a fresh
    module per call, the returned instance is therefore SHARED with later ``run_unet`` calls of the same
    checkpoint: treat it as read-only (``copy.deepcopy`` it before fine-tuning or weight surgery; the packed
    replica is never copied along).
    """
    st = os.stat(checkpoint_path)
    key = (os.path.realpath(checkpoint_path), st.st_mtime_ns, st.st_size, DEVICE)
    with _cache_lock:
        model = _model_cache.get(key)
        if model is None:
            model = UNet(n_channels=3, n_classes=3).to(DEVICE)
            state = torch.load(checkpoint_path, map_location=DEVICE)
            model.load_state_dict(state)
            model.eval()
            _model_cache.clear()          # keep one checkpoint resident
            _engine_cache.clear()
            _model_cache[key] = model
    return model


def _cached_engine(checkpoint_path: str):
    """(model, engine) of the cached checkpoint.  ``UNet.engine()`` re-validates its packed replica
    against all 136 tensors on every call (0.9 ms); the cached model is private to this module, so
    its replica is looked up by the checkpoint key instead."""
    model = load_model(checkpoint_path)
    with _cache_lock:
        key = next((k for k, m in _model_cache.items() if m is model), None)
        eng = _engine_cache.get(key)
        if eng is None:
            eng = model.engine(DEVICE)
            if key is not None:
                _engine_cache[key] = eng
    return model, eng


def _resized_rgb_u8(pil_img: Image.Image) -> np.ndarray:
    """``convert("RGB").resize((512, 512))`` -> uint8 (512, 512, 3)  (reference :35)."""
    img = pil_img.convert("RGB").resize((IMG_SIZE, IMG_SIZE))
    arr = np.array(img)              # writable copy, uint8 HWC
    if arr.ndim != 3 or arr.shape[2] != 3:
        raise ValueError(f"Invalid image shape: {arr.shape}")
    return arr


def preprocess(pil_img: Image.Image):
    """PIL image -> float32 tensor ``[1, 3, 512, 512]`` in [0, 1] on ``DEVICE`` (reference :30-44).

    Plain RGB images on a CUDA device take the GPU resize (bit-identical to Pillow's) and the ``/ 255.0``
    there too (IEEE float32 division, the same values as numpy's); everything else follows the reference's
    PIL / numpy calls on the host.  Same tensor either way."""
    if DEVICE == "cuda" and _gpu_resizable(pil_img):
        from . import prepost
        w, h = pil_img.size
        if h <= 0 or w <= 0:
            raise ValueError(f"Invalid image shape: {(h, w, 3)}")
        x = prepost.resize_u8(_upload_rgb(pil_img), IMG_SIZE, IMG_SIZE, channels=3)   # uint8 [1, 512, 512, 3]
        # a device-tensor divisor keeps this a true IEEE division (torch turns `/ python_scalar` into a
        # multiplication by the reciprocal on CUDA, which is 1 ulp off numpy's `/ 255.0` for some k)
        out = (x.permute(0, 3, 1, 2).to(torch.float32) / torch.full((), 255.0, device=x.device)).contiguous()
        torch.cuda.current_stream().synchronize()            # the pinned staging buffer is reusable again
        return out
    arr = _resized_rgb_u8(pil_img).astype(np.float32) / 255.0
    arr = arr.transpose(2, 0, 1)
    return torch.from_numpy(np.ascontiguousarray(arr)).unsqueeze(0).to(DEVICE)


def _crop_rect(size, extent):
    """Mask extent (xmin, xmax, ymin, ymax in 512-space, or None) -> crop rectangle (x1, y1, x2, y2) in
    the ORIGINAL image (reference :95-116): scale by (orig / 512) with ``int()`` truncation, grow by
    15 % of the box size, clamp to the image; ``None`` for an empty mask or an empty rectangle."""
    if extent is None:
        return None
    ow, oh = size
    sx, sy = ow / IMG_SIZE, oh / IMG_SIZE
    mx1, mx2, my1, my2 = extent
    x1, x2 = int(mx1 * sx), int(mx2 * sx)
    y1, y2 = int(my1 * sy), int(my2 * sy)
    px, py = int((x2 - x1) * 0.15), int((y2 - y1) * 0.15)
    x1, y1 = max(0, x1 - px), max(0, y1 - py)
    x2, y2 = min(ow, x2 + px), min(oh, y2 + py)
    if x2 <= x1 or y2 <= y1:
        return None
    return x1, y1, x2, y2


def _oriented_crop(obox, scale) -> dict:
    """Oriented box of a region (``obox`` = e1x, e1y, umin, umax, vmin, vmax from
    ``prepost.mask_components_oriented``; ``scale`` = (sx, sy) frame pixels per mask pixel) -> its upright crop
    (DESIGN.md 6b):

    * ``"size"`` ``(L, Wd)``: the extents along e1 and e2 = (-e1y, e1x), widened by one mask pixel block
      (half sizes ``hu = (|e1x| sx + |e1y| sy) / 2``, ``hv = (|e2x| sx + |e2y| sy) / 2`` on each side);
    * ``"out_size"`` ``(out_w, out_h) = (max(1, ceil(1.3 L)), max(1, ceil(1.3 Wd)))``: the reference's 15 % growth on
      each side, one output pixel per frame pixel;
    * ``"M"``: the inverse 2x3 map, output pixel (j, i) samples frame point ``o + j e1 + i e2``, where ``o`` puts the
      box centre ``c = (umin + umax) / 2 e1 + (vmin + vmax) / 2 e2`` in the middle of the crop;
    * ``"quad"``: the crop's four outer corners in the frame (top-left, top-right, bottom-right, bottom-left of the
      crop), ``"angle"``: ``degrees(atan2(e1y, e1x))`` in (-90, 90], for reporting.

    A 180 degree turn cannot be told from the masks: upside-down text stays upside down."""
    e1x, e1y, umin, umax, vmin, vmax = (float(v) for v in obox)
    sx, sy = float(scale[0]), float(scale[1])
    e2x, e2y = -e1y, e1x
    hu = 0.5 * (abs(e1x) * sx + abs(e1y) * sy)
    hv = 0.5 * (abs(e2x) * sx + abs(e2y) * sy)
    length = umax - umin + 2.0 * hu
    width = vmax - vmin + 2.0 * hv
    out_w = max(1, math.ceil(1.3 * length))
    out_h = max(1, math.ceil(1.3 * width))
    cu, cv = 0.5 * (umin + umax), 0.5 * (vmin + vmax)
    cx, cy = cu * e1x + cv * e2x, cu * e1y + cv * e2y
    ox = cx - 0.5 * (out_w - 1) * e1x - 0.5 * (out_h - 1) * e2x
    oy = cy - 0.5 * (out_w - 1) * e1y - 0.5 * (out_h - 1) * e2y
    quad = tuple((ox + j * e1x + i * e2x, oy + j * e1y + i * e2y)
                 for j, i in ((-0.5, -0.5), (out_w - 0.5, -0.5), (out_w - 0.5, out_h - 0.5), (-0.5, out_h - 0.5)))
    return {"M": np.array([[e1x, e2x, ox], [e1y, e2y, oy]], np.float64), "out_size": (out_w, out_h),
            "size": (length, width), "quad": quad, "angle": math.degrees(math.atan2(e1y, e1x))}


def _crop_from_extent(pil_img: Image.Image, extent) -> Optional[Image.Image]:
    """Extent -> crop of the original image, or ``None`` for an empty box or a near-black crop
    (``np.array(crop).mean() < 3``, reference :118-125), entirely on the host."""
    rect = _crop_rect(pil_img.size, extent)
    if rect is None:
        return None
    crop = pil_img.crop(rect)
    arr = np.array(crop)
    return None if (arr.size == 0 or arr.mean() < 3) else crop


def masks_to_crops(pil_img: Image.Image, masks: Dict[str, np.ndarray]) -> Dict[str, Optional[Image.Image]]:
    """Mask -> bounding box (min/max of the set pixels, reference :85-93) -> crop (reference :95-127)."""
    crops: Dict[str, Optional[Image.Image]] = {}
    for key, mask in masks.items():
        rows = np.flatnonzero(mask.any(axis=1))
        cols = np.flatnonzero(mask.any(axis=0))
        extent = None if (rows.size == 0 or cols.size == 0) else (int(cols[0]), int(cols[-1]), int(rows[0]), int(rows[-1]))
        crops[key] = _crop_from_extent(pil_img, extent)
    return crops


def _extent(box) -> Optional[tuple]:
    xmin, xmax, ymin, ymax, count = (int(v) for v in box)
    return None if count == 0 else (xmin, xmax, ymin, ymax)


def boxes_to_crops(pil_img: Image.Image, boxes: np.ndarray, frame_dev=None, rects_out: Optional[dict] = None
                   ) -> Dict[str, Optional[Image.Image]]:
    """Same, from the GPU reduction ``prepost.mask_bbox``: ``boxes`` int32 [3, 5] = xmin, xmax, ymin,
    ymax, count per field.  With ``frame_dev`` (the uint8 [H, W, 3] or RGBX [H, W, 4] frame on the device) the
    near-black test runs there as well: ``mean < 3`` is the integer test ``sum < 3 * bytes`` (exact: the
    float64 mean of fewer than 2^52 bytes cannot round across 3), so only accepted crops are cut."""
    if frame_dev is None:
        return {key: _crop_from_extent(pil_img, _extent(boxes[i])) for i, key in enumerate(FIELDS)}
    from . import prepost
    rects = [_crop_rect(pil_img.size, _extent(boxes[i])) for i in range(len(FIELDS))]
    live = [r for r in rects if r is not None]
    sums = prepost.box_sums(frame_dev, live, channels=3).cpu().tolist() if live else []
    crops: Dict[str, Optional[Image.Image]] = {}
    channels = 3                    # R, G, B count (an RGBX frame's padding byte does not)
    keep = []
    for key, r in zip(FIELDS, rects):
        crops[key] = None
        if r is None:
            continue
        total = sums.pop(0)
        if total >= 3 * (r[2] - r[0]) * (r[3] - r[1]) * channels:
            keep.append((key, r))
            if rects_out is not None:
                rects_out[key] = r
    # Large crops (a field mask that spans most of a 1080p frame is 8 MB of pixels) are cut side by side on the
    # host threads: PIL.Image.crop copies under the GIL, _crop_fast copies without it.
    big = [kr for kr in keep if (kr[1][2] - kr[1][0]) * (kr[1][3] - kr[1][1]) >= (1 << 18)]
    if len(big) >= 2 and pil_img.mode == "RGB":
        view = _rgb_host_view(pil_img)
        futs = {key: _worker_pool().submit(_crop_fast, pil_img, view, r, False) for key, r in big}
        for key, r in keep:
            crops[key] = futs[key].result() if key in futs else pil_img.crop(r)
    else:
        for key, r in keep:
            crops[key] = pil_img.crop(r)
    return crops


def _require_cuda():
    if DEVICE != "cuda":
        raise RuntimeError("run_unet needs a CUDA (B200, sm_100a) device: there is no CPU path "
                           "(the CPU oracle lives in oracle/ and is test-only)")


_staging: Dict[tuple, torch.Tensor] = {}


try:
    import pyarrow as _pa
    _HAVE_ARROW = True
except Exception:
    _pa = None
    _HAVE_ARROW = False


def _rgb_host_view(pil_img: Image.Image) -> np.ndarray:
    """uint8 view of an RGB image's pixels: ``(H, W, 4)`` RGBX straight out of Pillow's own buffer when it can
    be exported without a copy (Pillow >= 11.1 Arrow interface + pyarrow; the packed ``np.asarray`` costs
    1.2 ms for a 1080p frame), else the packed ``(H, W, 3)`` array."""
    if _HAVE_ARROW and hasattr(pil_img, "__arrow_c_array__"):
        try:
            flat = _pa.array(pil_img).flatten().to_numpy(zero_copy_only=True)
            w, h = pil_img.size
            if flat.dtype == np.uint8 and flat.size == h * w * 4:
                return flat.reshape(h, w, 4)
        except Exception:          # any export problem: the packed path below is always right
            pass
    return np.asarray(pil_img)


def _upload_rgb(pil_img: Image.Image, wait: bool = False) -> torch.Tensor:
    """RGB PIL image -> uint8 [1, H, W, 3] (packed) or [1, H, W, 4] (Pillow's RGBX storage; the fourth byte
    is padding and is never read) on DEVICE through a cached pinned staging buffer.
    Callers synchronise (``.cpu()``) before the next call, so the buffer is free to reuse; with
    ``wait`` the copy is awaited here (several uploads back to back)."""
    arr = _rgb_host_view(pil_img)
    key = (threading.get_ident(), arr.shape)
    buf = _staging.get(key)
    if buf is None:
        if len(_staging) > 8:
            _staging.clear()
        buf = _staging[key] = torch.empty(arr.shape, dtype=torch.uint8).pin_memory()
    buf.numpy()[...] = arr
    dev = buf.to(DEVICE, non_blocking=True)[None]
    if wait:
        torch.cuda.current_stream().synchronize()
    return dev


def _gpu_resizable(pil_img: Image.Image) -> bool:
    """Plain 8-bit RGB: the two PIL calls of the reference (:63 resize, :35 convert + resize) reduce
    to one bicubic resample of the uint8 HWC frame, which prepost.resize_u8 reproduces bit for bit."""
    return pil_img.mode == "RGB" and pil_img.size[0] > 0 and pil_img.size[1] > 0


_pool = None
_batch_state: Dict[tuple, dict] = {}      # (thread, device) -> staging ring + side streams of the batched entry point
_TRACE = None             # set to a list to collect (label, seconds since call start) marks of the batched entry point
PIPE_GROUP = 16           # images per pipeline stage of the batched entry point (one forward each)
STAGE_SLOTS = 3           # pinned staging buffers in flight (fill / upload / reuse)


def _worker_pool():
    """Host threads for the byte work of the batched entry point (staging copies, PIL crops); both release
    the GIL, so a few threads keep one GPU fed."""
    global _pool
    if _pool is None:
        from concurrent.futures import ThreadPoolExecutor
        _pool = ThreadPoolExecutor(max_workers=max(2, min(8, (os.cpu_count() or 4) // 2)),
                                   thread_name_prefix="unetb200-host")
    return _pool


def _batch_ctx(dev_index: int) -> dict:
    key = (threading.get_ident(), dev_index)
    ctx = _batch_state.get(key)
    if ctx is None:
        if len(_batch_state) > 8:
            _batch_state.clear()
        ctx = _batch_state[key] = {
            "up": torch.cuda.Stream(dev_index),        # host -> device copies + resize
            "post": torch.cuda.Stream(dev_index),      # near-black sums of finished groups
            "slots": [{"buf": None, "free": None} for _ in range(STAGE_SLOTS)],
        }
    return ctx


def _crop_fast(pil_img: Image.Image, view: Optional[np.ndarray], r, share: bool) -> Image.Image:
    """``pil_img.crop(r)`` for an RGB image whose pixels are visible as ``view`` (the zero-copy ``(H, W, 4)``
    RGBX export of :func:`_rgb_host_view`): same mode, size and pixels, built without holding the GIL --
    ``PIL.Image.crop`` copies under the GIL, which serialises the host threads of the batched entry point.
    ``share=False``: numpy copies the window (GIL released) and Pillow maps the copy; ``share=True``: Pillow
    maps the window of the SOURCE image in place (no copy; the crop is read-only and aliases ``pil_img``).
    Anything unexpected falls back to ``pil_img.crop``."""
    try:
        if view is None or view.ndim != 3 or view.shape[2] != 4 or pil_img.mode != "RGB":
            return pil_img.crop(r)
        x1, y1, x2, y2 = r
        h, w = view.shape[:2]
        if share and not (y2 == h and x1 > 0):       # (the mapped window must end inside the buffer)
            buf, off, stride = view.reshape(-1), (y1 * w + x1) * 4, w * 4
        else:
            buf, off, stride = np.ascontiguousarray(view[y1:y2, x1:x2]).reshape(-1), 0, (x2 - x1) * 4
        core = Image.core.map_buffer(buf, (x2 - x1, y2 - y1), "raw", off, ("RGB", stride, 1))
        im = Image.new("RGB", (0, 0))._new(core)
        im.readonly = 1                                # Pillow copies on the first write
        return im
    except Exception:
        return pil_img.crop(r)


def _segment_images(eng, pil_imgs: Sequence[Image.Image], crop_views: bool = False):
    """Images -> (uint8 0/1 masks (B, 3, 512, 512) on the host, per-image crops), as a pipeline of groups of
    ``PIPE_GROUP`` images (at most ``MAX_CHUNK`` per forward):

    * host threads copy each group's frames (Pillow's own RGBX buffers where they can be exported without a
      repack) into one of ``STAGE_SLOTS`` pinned staging buffers -- a buffer is refilled as soon as the uploads
      that read it have completed;
    * an upload stream moves every frame to the device and resizes it on the GPU straight into its slot of the
      group's batch tensor (other PIL modes: the reference's PIL calls on the host), so the copies of group g+1
      overlap the forward of group g on the caller's stream; masks and their boxes come back asynchronously
      into pinned memory;
    * as soon as a group's boxes have landed, a host thread computes the crop rectangles (reference :95-112),
      runs the near-black test of ALL its rectangles on the device frames (a side stream, one sync) and fans the
      ``PIL.crop`` calls out to the pool.

    The caller's thread never waits for the GPU before the last group is enqueued."""
    from . import prepost
    _require_cuda()
    thr = [THRESHOLDS[f] for f in FIELDS]
    n_img = len(pil_imgs)
    group = max(1, min(MAX_CHUNK, PIPE_GROUP))
    dev_index = torch.cuda.current_device()
    ctx = _batch_ctx(dev_index)
    up, post = ctx["up"], ctx["post"]
    masks = torch.empty((n_img, len(FIELDS), IMG_SIZE, IMG_SIZE), dtype=torch.uint8, pin_memory=True)
    boxes_host = torch.empty((n_img, len(FIELDS), 5), dtype=torch.int32, pin_memory=True)
    bx_all = boxes_host.numpy()
    pool = _worker_pool()
    main = torch.cuda.current_stream()
    spans = [(lo, min(lo + group, n_img)) for lo in range(0, n_img, group)]
    import time as _time
    _t0 = _time.perf_counter()

    def mark(label):
        if _TRACE is not None:
            _TRACE.append((label, _time.perf_counter() - _t0))
    views = [_rgb_host_view(im) if _gpu_resizable(im) else None for im in pil_imgs]
    mark("views")

    def plan(g):
        lo, hi = spans[g]
        offs, total = [], 0
        for v in views[lo:hi]:
            offs.append(total)
            if v is not None:
                total += (v.size + 255) & ~255
        return offs, total

    def fill_one(g, i, off, flat_np):
        v = views[spans[g][0] + i]
        np.copyto(flat_np[off:off + v.size].reshape(v.shape), v)

    def start_fill(g):
        """Reserve group g's slot (worker thread waits for it to be free), then one copy task per frame."""
        def reserve():
            offs, total = plan(g)
            slot = ctx["slots"][g % STAGE_SLOTS]
            if slot["free"] is not None:
                slot["free"].synchronize()
            if slot["buf"] is None or slot["buf"].numel() < total:
                slot["buf"] = torch.empty(max(total, 1 << 20), dtype=torch.uint8, pin_memory=True)
            flat_np = slot["buf"].numpy()
            lo, hi = spans[g]
            futs = [pool.submit(fill_one, g, i, offs[i], flat_np) if views[lo + i] is not None else None
                    for i in range(hi - lo)]
            return slot, offs, futs
        return pool.submit(reserve)

    def cut(idx, rects, tot):
        im, view = pil_imgs[idx], views[idx]
        out = {}
        for key, r in zip(FIELDS, rects):
            if r is None:
                out[key] = None
            elif tot is None:                          # frame not on the device: the host test of the reference
                c = im.crop(r)
                arr = np.array(c)
                out[key] = None if (arr.size == 0 or arr.mean() < 3) else c
            else:
                total = tot.pop(0)
                out[key] = None if total < 3 * (r[2] - r[0]) * (r[3] - r[1]) * 3 else _crop_fast(im, view, r, crop_views)
        return out

    def finish(g, frames, done):
        """(worker thread) boxes of group g -> rectangles -> near-black sums on the device -> crop tasks."""
        torch.cuda.set_device(dev_index)
        lo, hi = spans[g]
        done.synchronize()
        rects = [[_crop_rect(pil_imgs[i].size, _extent(bx_all[i, k])) for k in range(len(FIELDS))]
                 for i in range(lo, hi)]
        with torch.cuda.stream(post):
            sums = []
            for f, rs in zip(frames, rects):
                live = [r for r in rs if r is not None]
                sums.append(prepost.box_sums(f, live, channels=3) if (f is not None and live) else None)
            sums_host = [None if t is None else t.cpu().tolist() for t in sums]
        return [pool.submit(cut, lo + i, rects[i], sums_host[i]) for i in range(hi - lo)]

    fills = {g: start_fill(g) for g in range(min(STAGE_SLOTS, len(spans)))}
    posts = []
    for g, (lo, hi) in enumerate(spans):
        slot, offs, futs = fills.pop(g).result()
        mark(f"g{g} reserved")
        flat = slot["buf"]
        x = torch.empty((hi - lo, IMG_SIZE, IMG_SIZE, 3), dtype=torch.uint8, device=DEVICE)
        frames = []
        up.wait_stream(main)                           # x's memory is free on the caller's stream
        with torch.cuda.stream(up):
            for i in range(hi - lo):
                im, v = pil_imgs[lo + i], views[lo + i]
                if v is not None:
                    futs[i].result()
                    f = flat[offs[i]:offs[i] + v.size].view(v.shape).to(DEVICE, non_blocking=True)
                    prepost.resize_u8(f[None], IMG_SIZE, IMG_SIZE, out=x[i:i + 1], channels=3)
                    frames.append(f)
                else:
                    x[i].copy_(torch.from_numpy(_resized_rgb_u8(im.resize((IMG_SIZE, IMG_SIZE)))))
                    frames.append(None)
            slot["free"] = torch.cuda.Event()
            slot["free"].record(up)
        mark(f"g{g} uploaded")
        if g + STAGE_SLOTS < len(spans):
            fills[g + STAGE_SLOTS] = start_fill(g + STAGE_SLOTS)
        main.wait_stream(up)
        _, mask = eng.run(x, want_logits=False, thresholds=thr)
        masks[lo:hi].copy_(mask, non_blocking=True)
        boxes_host[lo:hi].copy_(prepost.mask_bbox(mask), non_blocking=True)
        done = torch.cuda.Event()
        done.record(main)
        posts.append(pool.submit(finish, g, frames, done))
        del frames
        mark(f"g{g} enqueued")
    crops: list = []
    for g, p_ in enumerate(posts):
        futs = p_.result()
        mark(f"g{g} boxes+sums")
        crops += [f.result() for f in futs]
        mark(f"g{g} crops")
    main.synchronize()
    mark("done")
    return masks.numpy(), crops


def run_unet(pil_img: Image.Image, checkpoint_path: str):
    """One image -> ``(masks, crops)`` exactly as the reference returns them (reference :50-129).

    ``masks``: dict field -> ``np.bool_`` (512, 512); ``crops``: dict field -> ``PIL.Image`` or
    ``None``; key order = ``FIELDS``.
    """
    from . import prepost
    frame, mask = _segment_one(pil_img, checkpoint_path)
    boxes = prepost.mask_bbox(mask)
    m = mask[0].cpu().numpy()
    masks = {f: m[i] != 0 for i, f in enumerate(FIELDS)}
    crops = boxes_to_crops(pil_img, boxes[0].cpu().numpy(), frame)
    return masks, crops


def _segment_one(pil_img: Image.Image, checkpoint_path: str):
    """The device half of ``run_unet``: ``(frame, mask)`` = the uploaded uint8 [H, W, 3 or 4] frame (``None`` for
    other PIL modes, which are resized on the host) and the uint8 [1, 3, 512, 512] masks, both on the GPU."""
    from . import prepost
    _require_cuda()
    _, eng = _cached_engine(checkpoint_path)
    thr = [THRESHOLDS[f] for f in FIELDS]
    frame = None
    # the reference resizes twice (:63 then :35); the second resize is the identity
    if _gpu_resizable(pil_img):
        frame = _upload_rgb(pil_img)                       # uint8 [1, H, W, 3 or 4]; stays on the GPU
        x = prepost.resize_u8(frame, IMG_SIZE, IMG_SIZE, channels=3)   # the resized frame never leaves the GPU
        frame = frame[0]
    else:
        x = torch.from_numpy(_resized_rgb_u8(pil_img.resize((IMG_SIZE, IMG_SIZE)))[None]).to(DEVICE)
    _, mask = eng.run(x, want_logits=False, thresholds=thr)
    return frame, mask


def run_unet_instances(pil_img: Image.Image, checkpoint_path: str, max_instances: int = 4, min_pixels: int = 1,
                       connectivity: int = 8, deskew: bool = False, enhance: bool = False):
    """``run_unet`` with one crop per connected region of each field mask instead of one crop over all of its set
    pixels (new, additive; ``run_unet`` itself is unchanged).  Returns ``(masks, instances)``: ``masks`` exactly as
    ``run_unet`` returns them; ``instances[field]`` = list, largest region first, of ``{"box": (x1, y1, x2, y2),
    "pixels": count, "crop": PIL.Image}`` for the ``max_instances`` (1..16) largest regions (``connectivity`` 4 or
    8) of at least ``min_pixels`` pixels.  Each box is the reference's crop rectangle of the region's extent
    (scaled to the original size, grown by 15 %, clamped); empty rectangles and near-black crops are dropped, so a
    field may list fewer regions than it has.

    ``deskew=True``: each ``"crop"`` is instead the upright RGB crop of the region along its principal axis
    (:func:`_oriented_crop`), sampled on the GPU from the uploaded frame (``prepost.warp_crops``, equal to
    ``cv2.warpAffine`` with bilinear sampling; the frame's edge pixels repeat where the crop reaches past it), and
    each instance gains ``"quad"`` (the crop's four corners in the frame), ``"angle"`` (degrees, in (-90, 90]) and
    ``"size"`` (the region's length and width in frame pixels).  The near-black test applies to the upright crop.
    ``enhance=True`` adds ``"enhanced"``: the mode-"L" OCR enhancement (four times the crop size) of the crop, with
    the field's ``ENHANCE_KINDS`` recipe, computed on the device from the crop's pixels there."""
    from . import prepost
    frame, mask = _segment_one(pil_img, checkpoint_path)
    m_cpu = None
    if not deskew:
        comps, _ = prepost.mask_components(mask, connectivity=connectivity, max_components=max_instances)
        m_cpu = mask[0].cpu().numpy()
        inst = components_to_instances(pil_img, comps[0].cpu().numpy(), frame, min_pixels)
        if enhance:
            _enhance_instances(inst, frame)
    else:
        scale = (pil_img.size[0] / IMG_SIZE, pil_img.size[1] / IMG_SIZE)
        comps, _, _, obox = prepost.mask_components_oriented(mask, connectivity=connectivity,
                                                             max_components=max_instances, scale=scale)
        m_cpu = mask[0].cpu().numpy()
        if frame is None:                              # other PIL modes: the RGB conversion goes up for the warp
            frame = _upload_rgb(pil_img.convert("RGB"))[0]
        inst = _deskewed_instances(pil_img, comps[0].cpu().numpy(), obox[0].cpu().numpy(), frame, scale,
                                   min_pixels, enhance)
    masks = {f: m_cpu[i] != 0 for i, f in enumerate(FIELDS)}
    return masks, inst


def _deskewed_instances(pil_img: Image.Image, comps: np.ndarray, obox: np.ndarray, frame_dev: torch.Tensor, scale,
                        min_pixels: int, enhance: bool) -> Dict[str, List[dict]]:
    """Rows of ``prepost.mask_components_oriented`` for one image -> instances with upright crops: the rows
    :func:`components_to_instances` would keep, each warped from the device frame in one batch; near-black upright
    crops are dropped on their device sums; with ``enhance`` the enhancement reads the warped buffer in place."""
    from . import prepost
    cands = []                                       # (field, rectangle, pixels, oriented crop)
    for i, key in enumerate(FIELDS):
        for row, ob in zip(comps[i], obox[i]):
            xmin, xmax, ymin, ymax, count = (int(v) for v in row[:5])
            if count == 0 or count < min_pixels:
                continue
            r = _crop_rect(pil_img.size, (xmin, xmax, ymin, ymax))
            if r is not None:
                cands.append((key, r, count, _oriented_crop(ob, scale)))
    out: Dict[str, List[dict]] = {key: [] for key in FIELDS}
    if not cands:
        return out
    buf, offs, sizes, sums = prepost._warp_batch(frame_dev, [c[3]["M"] for c in cands],
                                                 [c[3]["out_size"] for c in cands])
    keep = [k for k, t in enumerate(sums.cpu().tolist()) if t >= 3 * 3 * sizes[k][0] * sizes[k][1]]
    if not keep:
        return out
    host = buf.cpu().numpy()
    enh = None
    if enhance:
        from . import enhance as enh_mod
        enh = enh_mod.enhance_packed(buf, [offs[k] for k in keep], [sizes[k] for k in keep],
                                     [ENHANCE_KINDS[cands[k][0]] for k in keep])
    for n_kept, k in enumerate(keep):
        key, r, count, oc = cands[k]
        w, h = sizes[k]
        d = {"box": r, "pixels": count, "crop": Image.fromarray(host[offs[k]:offs[k] + 3 * w * h].reshape(h, w, 3)),
             "quad": oc["quad"], "angle": oc["angle"], "size": oc["size"]}
        if enh is not None:
            d["enhanced"] = Image.fromarray(enh[n_kept])
        out[key].append(d)
    return out


def _enhance_instances(inst: Dict[str, List[dict]], frame_dev=None) -> None:
    """Adds ``"enhanced"`` to every instance of :func:`components_to_instances`: the enhancement kernels read the
    boxes straight from the device frame when there is one (as ``run_unet_enhanced`` does), else the host crops."""
    from . import enhance
    items = [(key, d) for key, lst in inst.items() for d in lst]
    if not items:
        return
    kinds = [ENHANCE_KINDS[key] for key, _ in items]
    if frame_dev is not None:
        arrs = enhance.enhance_windows(frame_dev, [d["box"] for _, d in items], kinds)
    else:
        arrs = enhance.enhance_batch([d["crop"] for _, d in items], kinds)
    for (_, d), a in zip(items, arrs):
        d["enhanced"] = Image.fromarray(a)


def components_to_instances(pil_img: Image.Image, comps: np.ndarray, frame_dev=None, min_pixels: int = 1
                            ) -> Dict[str, List[dict]]:
    """Component table int32 [3, K, 6] (``prepost.mask_components`` of one image's masks, rows largest first) ->
    ``{field: [{"box", "pixels", "crop"}, ...]}``.  Rows with fewer than ``min_pixels`` pixels (or none) are left
    out; the rest go through ``_crop_rect`` and the near-black test of :func:`boxes_to_crops` -- on the device
    frame ``frame_dev`` when given (``prepost.box_sums``, 16 rectangles per call), else on the host."""
    cands = []                                       # (field, rectangle, pixels, extent)
    for i, key in enumerate(FIELDS):
        for row in comps[i]:
            xmin, xmax, ymin, ymax, count = (int(v) for v in row[:5])
            if count == 0 or count < min_pixels:
                continue
            r = _crop_rect(pil_img.size, (xmin, xmax, ymin, ymax))
            if r is not None:
                cands.append((key, r, count, (xmin, xmax, ymin, ymax)))
    out: Dict[str, List[dict]] = {key: [] for key in FIELDS}
    if frame_dev is None:
        for key, r, count, ext in cands:
            crop = _crop_from_extent(pil_img, ext)
            if crop is not None:
                out[key].append({"box": r, "pixels": count, "crop": crop})
        return out
    from . import prepost
    sums = [prepost.box_sums(frame_dev, [c[1] for c in cands[lo:lo + 16]], channels=3)
            for lo in range(0, len(cands), 16)]
    totals = torch.cat(sums).cpu().tolist() if sums else []
    for (key, r, count, _), total in zip(cands, totals):
        if total >= 3 * (r[2] - r[0]) * (r[3] - r[1]) * 3:
            out[key].append({"box": r, "pixels": count, "crop": pil_img.crop(r)})
    return out


# which enhancement the app applies to which field before OCR.space (reference app_camera.py:800-811)
ENHANCE_KINDS = {"invoice_no": "text", "date": "text", "total_amount": "amount"}


def run_unet_enhanced(pil_img: Image.Image, checkpoint_path: str):
    """``run_unet`` plus the crop enhancement the app applies next (reference app_camera.py:787-811:
    ``enhance_for_ocrspace(crop, "text")`` for invoice number and date, ``"amount"`` for the total), as
    one device pipeline: the frame is uploaded once, resized, segmented, reduced to boxes, tested for
    near-black crops and enhanced from the same device buffer.  New, additive.

    Returns ``(masks, crops, enhanced)``; ``enhanced``: dict field -> mode-"L" ``PIL.Image`` (four times
    the crop size) or ``None``, equal to what the reference's helpers return for ``crops[field]``."""
    from . import enhance, prepost
    _require_cuda()
    _, eng = _cached_engine(checkpoint_path)
    thr = [THRESHOLDS[f] for f in FIELDS]
    if not _gpu_resizable(pil_img):
        masks, crops = run_unet(pil_img, checkpoint_path)
        live = [f for f in FIELDS if crops[f] is not None]
        arrs = enhance.enhance_batch([crops[f] for f in live], [ENHANCE_KINDS[f] for f in live])
        done = dict(zip(live, arrs))
        return masks, crops, {f: Image.fromarray(done[f]) if f in done else None for f in FIELDS}
    frame = _upload_rgb(pil_img)
    x = prepost.resize_u8(frame, IMG_SIZE, IMG_SIZE, channels=3)
    _, mask = eng.run(x, want_logits=False, thresholds=thr)
    boxes = prepost.mask_bbox(mask)
    m = mask[0].cpu().numpy()
    masks = {f: m[i] != 0 for i, f in enumerate(FIELDS)}
    rects: dict = {}
    crops = boxes_to_crops(pil_img, boxes[0].cpu().numpy(), frame[0], rects)
    live = [f for f in FIELDS if f in rects]
    arrs = enhance.enhance_windows(frame[0], [rects[f] for f in live], [ENHANCE_KINDS[f] for f in live])
    done = dict(zip(live, arrs))
    return masks, crops, {f: Image.fromarray(done[f]) if f in done else None for f in FIELDS}


def run_unet_batch(pil_imgs: Sequence[Image.Image], checkpoint_path: str, crop_views: bool = False
                   ) -> List[Tuple[Dict[str, np.ndarray], Dict[str, Optional[Image.Image]]]]:
    """``run_unet`` for many images as one pipeline (new entry point): ``[(masks, crops), ...]`` in input order,
    each pair exactly what ``run_unet`` returns for that image.  ``crop_views=True`` returns the crops of RGB
    inputs as read-only windows INTO the input images (no pixel copy; they alias ``pil_imgs[i]`` and keep it
    alive) instead of independent copies."""
    if len(pil_imgs) == 0:
        return []
    _require_cuda()
    _, eng = _cached_engine(checkpoint_path)
    m, crops = _segment_images(eng, list(pil_imgs), crop_views=crop_views)
    mb = m.view(np.bool_)          # the kernel writes exactly 0 / 1: the boolean planes without another pass
    return [({f: mb[b, i] for i, f in enumerate(FIELDS)}, crops[b]) for b in range(len(pil_imgs))]
