"""Drop-in for the reference ``unet_model.py`` (reference unet_model.py:6-86).

Same public surface -- ``DoubleConv(in_ch, out_ch)`` with attribute ``.net``
(parameters at Sequential indices 0, 1, 3, 4) and ``UNet(n_channels=3,
n_classes=3)`` with sub-modules ``down1..4, pool, bottleneck, up4..1, conv4..1,
out_conv`` -- so ``checkpoints/best_unet_model.pth`` loads unchanged with a strict
``load_state_dict`` (136 keys).

What changed is where the arithmetic runs.  In eval mode ``UNet.forward`` does
not execute any ``torch.nn`` op: it hands the input to the sm_100a CUDA library
(``engine.Engine`` -> ``libunetb200.so``), which runs the 23 layers as
hand-written tcgen05/TMA kernels with BatchNorm folded into the weights, and
returns NCHW logits on the same device, like the reference.  It accepts float32,
float16 and bfloat16 inputs, contiguous or channels-last, and returns logits in
the input's dtype (``m.half().eval(); m(x.half())`` gives float16 logits): a 16-bit
input is widened exactly to float32 where it is read, the network computes in
bf16 / fp32 as for float32 input, and 16-bit logits are the float32 logits
rounded to nearest-even.  Eval mode has no CPU path: a CPU tensor raises.

Training mode (``train.py:103,137`` instantiates this same class) still runs the
``torch.nn`` graph -- batch statistics and autograd are not part of the
inference hot path this package replaces.
"""
from __future__ import annotations

import itertools

import torch
import torch.nn as nn

from .engine import Engine

_WIDTHS = (64, 128, 256, 512, 1024)


def _conv_bn_relu(cin: int, cout: int):
    return [nn.Conv2d(cin, cout, kernel_size=3, padding=1), nn.BatchNorm2d(cout), nn.ReLU(inplace=True)]


class DoubleConv(nn.Module):
    """(Conv3x3 pad 1 -> BatchNorm -> ReLU) x 2, reference unet_model.py:6-20."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.net = nn.Sequential(*_conv_bn_relu(in_ch, out_ch), *_conv_bn_relu(out_ch, out_ch))

    def forward(self, x):
        return self.net(x)


class UNet(nn.Module):
    """4-level U-Net, reference unet_model.py:23-86."""

    def __init__(self, n_channels=3, n_classes=3):
        super().__init__()
        self.n_channels = n_channels
        self.n_classes = n_classes
        w = _WIDTHS
        # registration order below fixes the state_dict key order (reference :29-50)
        for i in range(4):
            setattr(self, f"down{i + 1}", DoubleConv(n_channels if i == 0 else w[i - 1], w[i]))
        self.pool = nn.MaxPool2d(2)
        self.bottleneck = DoubleConv(w[3], w[4])
        for i in (4, 3, 2, 1):
            setattr(self, f"up{i}", nn.ConvTranspose2d(w[i], w[i - 1], 2, stride=2))
            setattr(self, f"conv{i}", DoubleConv(w[i], w[i - 1]))
        self.out_conv = nn.Conv2d(w[0], n_classes, kernel_size=1)
        nn.init.constant_(self.out_conv.bias, -4)   # reference :53
        self._engine = None          # packed replica, built lazily on the first eval forward
        self._engine_key = None

    # ---- engine cache: anything that can change weights or placement drops it
    def _drop_engine(self):
        object.__setattr__(self, "_engine", None)
        object.__setattr__(self, "_engine_key", None)

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self._drop_engine()
        return out

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._drop_engine()
        return out

    def train(self, mode: bool = True):
        if mode:
            self._drop_engine()
        return super().train(mode)

    def __getstate__(self):
        # the packed replica holds device pointers and a ctypes handle: never pickled / deep-copied
        state = self.__dict__.copy()
        state["_engine"] = None
        state["_engine_key"] = None
        return state

    def invalidate_engine(self):
        """Drop the packed replica so that the next eval forward re-folds and re-packs the weights.

        The replica is rebuilt automatically after ``load_state_dict``, ``.to()`` / ``.cuda()`` / ``.half()``,
        ``train()`` and any in-place update autograd can see (the key below tracks every tensor's storage
        pointer and version counter).  Writes that bypass the version counter -- ``param.data.copy_()``,
        EMA updates through ``.data``, manual weight surgery on ``.data`` -- are invisible to it: call this
        method after them."""
        self._drop_engine()

    def _weights_key(self):
        return tuple((t.data_ptr(), t._version) for t in itertools.chain(self.parameters(), self.buffers()))

    def engine(self, device=None) -> Engine:
        """The packed B200 replica of the current weights (built on first use)."""
        p = self.out_conv.weight
        device = torch.device(device) if device is not None else p.device
        key = (str(device), self._weights_key())
        if self._engine is None or self._engine_key != key:
            eng = Engine(self.state_dict(), device, self.n_channels, self.n_classes)
            object.__setattr__(self, "_engine", eng)
            object.__setattr__(self, "_engine_key", key)
        return self._engine

    # ---- forward
    def forward(self, x):
        if self.training:
            return self._forward_train(x)
        if not x.is_cuda:
            raise RuntimeError(
                "tw_invoice_unet_ocr_llm_b200.UNet runs its eval forward on a B200 (sm_100a) GPU only; "
                "got a CPU tensor and there is no CPU path")
        if x.dtype not in (torch.float32, torch.float16, torch.bfloat16):
            raise RuntimeError(f"expected a float32, float16 or bfloat16 input, got {x.dtype}")
        logits, _ = self.engine(x.device).run(x, want_logits=True)
        return logits

    def _forward_train(self, x):
        skips = []
        for i in range(4):
            x = getattr(self, f"down{i + 1}")(x)
            skips.append(x)
            x = self.pool(x)
        x = self.bottleneck(x)
        for i in (4, 3, 2, 1):
            x = getattr(self, f"up{i}")(x)
            x = torch.cat([x, skips[i - 1]], dim=1)   # upsampled channels first, then the skip
            x = getattr(self, f"conv{i}")(x)
        return self.out_conv(x)
