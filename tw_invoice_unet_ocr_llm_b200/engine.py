"""Host-side driver of the B200 U-Net forward: weight fold/pack, workspace, launch.

PyTorch is used for device memory, streams and nothing else; every arithmetic op
of the forward runs inside ``libunetb200.so``.  ``Engine`` is what
``unet_model.UNet.forward`` (eval mode, CUDA input) and ``inference.run_unet``
delegate to.
"""
from __future__ import annotations

import ctypes as C
import math
import threading
from typing import Mapping, Optional, Sequence

import torch

from . import _native as nat

BN_EPS = 1e-5  # nn.BatchNorm2d default, reference unet_model.py:11,15


def logit_thresholds(probs: Sequence[float]) -> list[float]:
    """sigmoid(z) > t  <=>  z > ln(t / (1 - t))   (reference inference.py:72-79)."""
    return [math.log(t / (1.0 - t)) for t in probs]


def unpack_mask_bits(bits, width: Optional[int] = None):
    """Bit-packed masks (``Engine.run(mask_bits=True)``: uint8 ``[..., H, W/8]``, LSB first) -> uint8 0/1
    ``[..., H, W]``.  Accepts a numpy array or a (CPU or CUDA) tensor and returns the same kind."""
    if isinstance(bits, torch.Tensor):
        shifts = torch.arange(8, dtype=torch.uint8, device=bits.device)
        out = ((bits.unsqueeze(-1) >> shifts) & 1).reshape(*bits.shape[:-1], bits.shape[-1] * 8)
        return out if width is None else out[..., :width]
    import numpy as np
    out = np.unpackbits(np.ascontiguousarray(bits), axis=-1, bitorder="little")
    return out if width is None else out[..., :width]


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# float input dtype -> (NCHW format, NHWC format) of the C ABI (include/unetb200.h UNETB200_X_*)
_FLOAT_FORMATS = {
    torch.float32: (nat.X_F32_NCHW, nat.X_F32_NHWC),
    torch.float16: (nat.X_F16_NCHW, nat.X_F16_NHWC),
    torch.bfloat16: (nat.X_BF16_NCHW, nat.X_BF16_NHWC),
}
# logits dtype -> UNETB200_LOGITS_*
LOGITS_TYPES = {torch.float32: nat.LOGITS_F32, torch.float16: nat.LOGITS_F16, torch.bfloat16: nat.LOGITS_BF16}


def input_format(x: torch.Tensor):
    """``(fmt, x_for_kernel)``: the C-ABI input format of ``x`` and the tensor whose storage the forward reads.

    uint8 is ``[N,H,W,C]`` raw pixels (``X_U8_NHWC``).  float32 / float16 / bfloat16 are ``[N,C,H,W]``: NCHW when
    ``x`` is contiguous (also when it is channels-last contiguous as well, as with C = 1 or H = W = 1); NHWC, read in
    place with no copy, when ``x`` is channels-last contiguous (``x.to(memory_format=torch.channels_last)``);
    otherwise ``x.contiguous()`` as NCHW.  Every other dtype raises ``RuntimeError``."""
    if x.dtype == torch.uint8:
        return nat.X_U8_NHWC, x.contiguous()
    fmts = _FLOAT_FORMATS.get(x.dtype)
    if fmts is None:
        raise RuntimeError(f"input dtype must be float32, float16, bfloat16 ([N,C,H,W]) or uint8 ([N,H,W,C]), "
                           f"got {x.dtype}")
    if x.is_contiguous():
        return fmts[0], x
    if x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last):
        return fmts[1], x
    return fmts[0], x.contiguous()


class Engine:
    """One packed model replica on one GPU."""

    def __init__(self, state: Mapping[str, torch.Tensor], device, n_channels: int = 3,
                 n_classes: int = 3, bn_eps: float = BN_EPS):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("tw_invoice_unet_ocr_llm_b200.Engine needs a CUDA (sm_100) device; "
                               "there is no CPU path")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = nat.lib()
        self.arch = nat.Arch(n_channels, n_classes, 64)
        self.layers = nat.layer_table(self.arch)
        self.n_channels, self.n_classes = n_channels, n_classes
        self._lock = threading.Lock()
        # one scratch region PER CUDA STREAM: forwards enqueued on different streams may overlap on the
        # device, so they must never share activations (the lock below only serialises the enqueue)
        self._ws: "dict[int, torch.Tensor]" = {}
        self._handle = C.c_void_p()
        with torch.cuda.device(self.device):
            nbytes = int(self._lib.unetb200_packed_bytes(C.byref(self.arch)))
            self.blob = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            self._pack(state, bn_eps)
            nat.check(self._lib.unetb200_create(C.byref(self.arch), self.blob.data_ptr(), nbytes,
                                                self.device.index, C.byref(self._handle)))

    # ------------------------------------------------------------------ weights
    def _pack(self, state: Mapping[str, torch.Tensor], bn_eps: float) -> None:
        stream = torch.cuda.current_stream(self.device).cuda_stream
        keep = []

        def dev(name: str) -> torch.Tensor:
            if name not in state:
                raise KeyError(f"state_dict is missing {name!r}")
            t = state[name].detach().to(self.device, torch.float32).contiguous()
            keep.append(t)
            return t

        for i, l in enumerate(self.layers):
            name = l.name.decode()
            bn = l.bn_name.decode()
            w = dev(name + ".weight")
            b = dev(name + ".bias") if (name + ".bias") in state else None
            expect = {
                nat.STEM: (l.cout, l.cin, 3, 3), nat.CONV3X3: (l.cout, l.cin, 3, 3),
                nat.CONVT2X2: (l.cin, l.cout, 2, 2), nat.HEAD: (l.cout, l.cin, 1, 1),
            }[l.kind]
            if tuple(w.shape) != expect:
                raise RuntimeError(f"{name}.weight has shape {tuple(w.shape)}, expected {expect}")
            g = be = mu = var = None
            if bn:
                g, be = dev(bn + ".weight"), dev(bn + ".bias")
                mu, var = dev(bn + ".running_mean"), dev(bn + ".running_var")
            nat.check(self._lib.unetb200_pack_layer(
                C.byref(self.arch), i, _ptr(w), _ptr(b), _ptr(g), _ptr(be), _ptr(mu), _ptr(var),
                bn_eps, self.blob.data_ptr(), stream))
        # decoder levels with the up-conv folded into the following 3x3 conv (csrc/conv_phase.cuh,
        # reference unet_model.py:38-51): composite weights from the fp32 tensors of up{j} and conv{j}.net.0/.1
        for j in (4, 3, 2, 1):
            up, cv, bn = f"up{j}", f"conv{j}.net.0", f"conv{j}.net.1"
            nat.check(self._lib.unetb200_pack_fused_up(
                C.byref(self.arch), j, _ptr(dev(up + ".weight")),
                _ptr(dev(up + ".bias")) if (up + ".bias") in state else None,
                _ptr(dev(cv + ".weight")), _ptr(dev(cv + ".bias")) if (cv + ".bias") in state else None,
                _ptr(dev(bn + ".weight")), _ptr(dev(bn + ".bias")), _ptr(dev(bn + ".running_mean")),
                _ptr(dev(bn + ".running_var")), bn_eps, self.blob.data_ptr(), stream))
        torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------ options
    def set_option(self, key: str, value: int) -> None:
        nat.check(self._lib.unetb200_set_option(self._handle, key.encode(), int(value)))

    def get_option(self, key: str) -> int:
        v = C.c_int()
        nat.check(self._lib.unetb200_get_option(self._handle, key.encode(), C.byref(v)))
        return v.value

    def workspace_bytes(self, n: int, h: int, w: int) -> int:
        return int(self._lib.unetb200_workspace_bytes(self._handle, n, h, w))

    MAX_STREAM_WORKSPACES = 4

    def _workspace(self, n: int, h: int, w: int, stream: int):
        """(pointer, bytes) of a 1024-byte aligned scratch region big enough for this shape, private to
        the CUDA stream ``stream`` (the raw ``cudaStream_t`` value).  A region is allocated, grown and
        dropped only while its own stream is current, so torch's stream-ordered caching allocator never
        hands its memory to work that could overlap a forward still running on it."""
        need = self.workspace_bytes(n, h, w)
        ws = self._ws.get(stream)
        if ws is None or ws.numel() < need + 1024:
            self._ws.pop(stream, None)
            ws = None                                        # release before growing
            if len(self._ws) >= self.MAX_STREAM_WORKSPACES:  # oldest stream's region goes back to ITS pool
                self._ws.pop(next(iter(self._ws)))
            ws = self._ws[stream] = torch.empty(need + 1024, dtype=torch.uint8, device=self.device)
        ptr = (ws.data_ptr() + 1023) & ~1023                 # small torch blocks are only 512-byte aligned
        return ptr, ws.numel() - (ptr - ws.data_ptr())

    def _check_out(self, t: torch.Tensor, what: str, shape, dtype) -> None:
        if not isinstance(t, torch.Tensor) or t.device != self.device or t.dtype != dtype \
                or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise RuntimeError(f"{what} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {self.device}, "
                               f"got {getattr(t, 'dtype', type(t))} {tuple(getattr(t, 'shape', ()))} on "
                               f"{getattr(t, 'device', None)} (contiguous={getattr(t, 'is_contiguous', lambda: None)()})")

    # ------------------------------------------------------------------ forward
    def run(self, x: torch.Tensor, *, want_logits: bool = True,
            thresholds: Optional[Sequence[float]] = None,
            logits_out: Optional[torch.Tensor] = None, mask_out: Optional[torch.Tensor] = None,
            mask_bits: bool = False, logits_dtype: Optional[torch.dtype] = None):
        """Enqueue one forward on the current stream.

        ``x``: float32 / float16 / bfloat16 ``[N,C,H,W]`` (values as ``inference.preprocess`` makes them),
        contiguous or channels-last (read in place), or uint8 ``[N,H,W,C]`` raw pixels (:func:`input_format`).
        A 16-bit input gives the same results as ``x.float()``.  Returns ``(logits | None, mask | None)``;
        ``logits`` is ``[N,n_classes,H,W]`` NCHW-contiguous of ``logits_dtype`` (float32, float16 or bfloat16;
        default: the dtype of a float input, float32 for uint8), 16-bit logits being the float32 logits rounded to
        nearest-even.  ``mask`` is uint8 ``[N,n_classes,H,W]`` with 1 where ``sigmoid(logit) > thresholds[c]``
        (decided on the float32 logits), or, with ``mask_bits``, the same booleans packed eight to a byte: uint8
        ``[N,n_classes,H,W/8]``, pixel ``x`` = bit ``x & 7`` (LSB first) of byte ``x >> 3``
        (:func:`unpack_mask_bits` / ``np.unpackbits(bitorder="little")``).
        """
        if x.device != self.device:
            raise RuntimeError(f"input is on {x.device}, engine is on {self.device}")
        if x.dim() != 4:
            raise RuntimeError(f"expected a 4-D input, got shape {tuple(x.shape)}")
        fmt, x = input_format(x)
        if fmt == nat.X_U8_NHWC:
            n, h, w, c = x.shape
        else:
            n, c, h, w = x.shape
        if logits_dtype is None:
            logits_dtype = torch.float32 if x.dtype == torch.uint8 else x.dtype
        if logits_dtype not in LOGITS_TYPES:
            raise RuntimeError(f"logits_dtype must be torch.float32, torch.float16 or torch.bfloat16, got {logits_dtype}")
        if c != self.n_channels:
            raise RuntimeError(f"expected {self.n_channels} input channels, got {c}")
        if h % 16 or w % 16:
            # the reference raises RuntimeError from torch.cat for such sizes (unet_model.py:71)
            raise RuntimeError(f"H and W must be divisible by 16, got {h}x{w}")
        thr = None
        out_shape = (n, self.n_classes, h, w)
        mask_shape = (n, self.n_classes, h, w // 8) if mask_bits else out_shape
        if logits_out is not None:
            self._check_out(logits_out, "logits_out", out_shape, logits_dtype)
        if mask_out is not None:
            self._check_out(mask_out, "mask_out", mask_shape, torch.uint8)
        with self._lock, torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            ws_ptr, ws_bytes = self._workspace(n, h, w, stream)
            logits = None
            if want_logits:
                logits = logits_out if logits_out is not None else torch.empty(
                    out_shape, dtype=logits_dtype, device=self.device)
            mask = None
            if thresholds is not None:
                if len(thresholds) != self.n_classes:
                    raise RuntimeError("one threshold per class is required")
                thr = (C.c_float * self.n_classes)(*logit_thresholds(thresholds))
                mask = mask_out if mask_out is not None else torch.empty(
                    mask_shape, dtype=torch.uint8, device=self.device)
            nat.check(self._lib.unetb200_forward_typed(
                self._handle, x.data_ptr(), fmt, n, h, w, ws_ptr, ws_bytes,
                _ptr(logits), LOGITS_TYPES[logits_dtype], _ptr(mask), 1 if mask_bits else 0, thr, stream))
        return logits, mask

    def layer_times_ms(self) -> list[float]:
        buf = (C.c_float * len(self.layers))()
        nat.check(self._lib.unetb200_layer_times(self._handle, buf, len(self.layers)))
        return list(buf)

    def last_launch_count(self) -> int:
        return int(self._lib.unetb200_last_launch_count(self._handle))

    def close(self) -> None:
        if self._handle:
            self._lib.unetb200_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):  # best effort
        try:
            self.close()
        except Exception:
            pass
