"""CPU-side checks: the C-ABI library loads and exports every symbol include/unetb200.h
declares, argument validation works without a GPU, the drop-in modules keep the reference's
surface, and the package never imports the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def nat():
    import __graft_entry__ as g
    g.build()
    from tw_invoice_unet_ocr_llm_b200 import _native
    return _native


def test_header_symbols_exported_at_abi_version_2(nat):
    """Every symbol of include/unetb200.h is bound and exported, and the library and the ctypes bindings agree on
    ABI version 2 (unetb200_enh_crop.clip became a double: 80-byte descriptors)."""
    hdr = open(os.path.join(ROOT, "include", "unetb200.h")).read()
    declared = set(re.findall(r"\b(unetb200_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(nat.SYMBOLS), declared ^ set(nat.SYMBOLS)
    lib = nat.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.unetb200_abi_version() == nat.ABI_VERSION == 2


def test_layer_table_and_blob_layout(nat):
    arch = nat.Arch(3, 3, 64)
    layers = nat.layer_table(arch)
    assert len(layers) == 23
    names = [l.name.decode() for l in layers]
    assert names[0] == "down1.net.0" and names[-1] == "out_conv" and names[10] == "up4"
    # every conv of the reference module appears exactly once, in forward order
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    convs = [n for n, m in UNet().named_modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.ConvTranspose2d))]
    assert sorted(convs) == sorted(names)
    end = 0
    for l in layers:
        assert l.w_off >= end and l.w_off % 256 == 0 and l.b_off >= l.w_off + l.w_bytes and l.b_off % 256 == 0
        end = l.b_off + l.b_bytes
    assert nat.lib().unetb200_packed_bytes(C.byref(arch)) >= end
    total_w = sum(l.w_bytes for l in layers)
    assert 62_000_000 < total_w < 62_300_000        # 31.04 M weights in bf16 (SURVEY.md 8e: "62 MB")


def test_argument_validation_without_gpu(nat):
    lib = nat.lib()
    bad = nat.Arch(3, 3, 32)
    assert lib.unetb200_num_layers(C.byref(bad)) == -1
    assert "base_width" in nat.last_error()
    assert lib.unetb200_packed_bytes(C.byref(nat.Arch(2, 3, 64))) == 0
    l = nat.Layer()
    assert lib.unetb200_layer_info(C.byref(nat.Arch(3, 3, 64)), 99, C.byref(l)) == nat.EINVAL
    assert lib.unetb200_forward(None, None, 0, 1, 64, 64, None, 0, None, None, None, None) == nat.EINVAL
    assert lib.unetb200_workspace_bytes(None, 1, 64, 64) == 0
    if not torch.cuda.is_available():
        h = C.c_void_p()
        rc = lib.unetb200_create(C.byref(nat.Arch(3, 3, 64)), C.c_void_p(16), 1 << 30, 0, C.byref(h))
        assert rc in (nat.ECUDA, nat.EARCH) and nat.last_error()      # no device: loud failure, no fallback


def test_module_surface_matches_reference(fixture_state):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.unet_model import DoubleConv, UNet
    m = UNet()
    assert (m.n_channels, m.n_classes) == (3, 3)
    assert [n for n, _ in m.named_children()] == ["down1", "down2", "down3", "down4", "pool", "bottleneck",
                                                  "up4", "conv4", "up3", "conv3", "up2", "conv2", "up1",
                                                  "conv1", "out_conv"]
    assert isinstance(m.down1, DoubleConv) and len(m.down1.net) == 6
    assert float(m.out_conv.bias.detach()[0]) == -4.0                    # reference unet_model.py:53
    res = m.load_state_dict(fixture_state, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert list(m.state_dict()) == list(fixture_state)
    assert inf.IMG_SIZE == 512 and inf.FIELDS == ["invoice_no", "date", "total_amount"]
    assert inf.DEVICE in ("cuda", "cpu")
    for fn in ("load_model", "preprocess", "run_unet", "run_unet_batch"):
        assert callable(getattr(inf, fn))


def test_eval_forward_has_no_cpu_path(fixture_state):
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    m = UNet().eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(1, 3, 32, 32))


def test_train_mode_forward_is_the_reference_graph(fixture_state):
    """train.py:103,137 uses the same class in train mode: batch statistics + autograd keep working
    and match the oracle when BatchNorm is frozen to running statistics."""
    from oracle.unet_oracle import oracle_forward
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    m = UNet()
    m.load_state_dict(fixture_state)
    m.train()
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eval()
    x = synthetic_invoices(1, 32, 32, seed=1).requires_grad_(True)
    z = m(x)
    assert torch.allclose(z, oracle_forward(fixture_state, x.detach()), atol=1e-5)
    z.sum().backward()
    assert x.grad is not None and m.down1.net[0].weight.grad is not None


def test_logit_thresholds():
    from tw_invoice_unet_ocr_llm_b200.engine import logit_thresholds
    thr = logit_thresholds([0.25, 0.40, 0.30])
    assert np.allclose(thr, [-1.0986123, -0.4054651, -0.8472979], atol=1e-6)     # SURVEY.md section 7
    z = torch.linspace(-3, 3, 20001)
    for t, lt in zip([0.25, 0.40, 0.30], thr):
        a = (torch.sigmoid(z) > t)
        b = z > np.float32(lt)
        assert int((a != b).sum()) <= 1


def test_package_does_not_import_oracle():
    pkg = os.path.join(ROOT, "tw_invoice_unet_ocr_llm_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f


def test_shims_expose_the_reference_module_names():
    """shims/ first on sys.path makes `from inference import run_unet` / `from unet_model import UNet`
    (reference app_camera.py:16, inference.py:4, train.py:12) resolve to this package."""
    import importlib
    import sys
    shim_dir = os.path.join(ROOT, "shims")
    saved = {k: sys.modules.pop(k, None) for k in ("inference", "unet_model")}
    sys.path.insert(0, shim_dir)
    try:
        inf = importlib.import_module("inference")
        um = importlib.import_module("unet_model")
        from tw_invoice_unet_ocr_llm_b200 import inference as pkg_inf
        from tw_invoice_unet_ocr_llm_b200 import unet_model as pkg_um
        assert inf.run_unet is pkg_inf.run_unet and inf.load_model is pkg_inf.load_model
        assert inf.preprocess is pkg_inf.preprocess and inf.IMG_SIZE == 512
        assert um.UNet is pkg_um.UNet and um.DoubleConv is pkg_um.DoubleConv
    finally:
        sys.path.remove(shim_dir)
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v


def test_module_copies_and_pickles_without_the_engine(fixture_state):
    """copy.deepcopy / pickle (torch.save(model)) must not try to serialise the packed GPU replica."""
    import copy
    import io
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    m = UNet()
    m.load_state_dict(fixture_state)
    object.__setattr__(m, "_engine", object())          # stand-in for a live engine
    m2 = copy.deepcopy(m)
    assert m2._engine is None and list(m2.state_dict()) == list(m.state_dict())
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    m3 = torch.load(buf, weights_only=False)
    assert m3._engine is None and torch.equal(m3.down1.net[0].weight, m.down1.net[0].weight)


def test_enhance_surface_matches_reference_and_has_no_cpu_path():
    """enhance_for_ocrspace / enhance_for_date_ocr keep the reference's signatures (app_camera.py:572, 685);
    None passes through without touching the GPU; without a CUDA device the batched entry raises."""
    import inspect
    import numpy as np
    from tw_invoice_unet_ocr_llm_b200 import enhance, inference as inf
    sig = inspect.signature(enhance.enhance_for_ocrspace)
    assert list(sig.parameters) == ["pil_crop", "mode"] and sig.parameters["mode"].default == "text"
    assert list(inspect.signature(enhance.enhance_for_date_ocr).parameters) == ["pil_crop"]
    assert enhance.enhance_for_ocrspace(None) is None and enhance.enhance_for_ocrspace(None, mode="amount") is None
    assert enhance.enhance_for_date_ocr(None) is None
    assert set(inf.ENHANCE_KINDS) == set(inf.FIELDS) and set(inf.ENHANCE_KINDS.values()) <= set(enhance.KINDS)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU path"):
            enhance.enhance_batch([np.zeros((4, 4, 3), np.uint8)], ["text"])
        with pytest.raises(RuntimeError, match="no CPU path"):
            from PIL import Image
            inf.run_unet_enhanced(Image.new("RGB", (32, 32)), "missing.pth")


def test_fastdiv_magic_numbers(nat):
    """The conv kernels divide tile indices by launch constants with multiply-high + shift; the magic numbers
    must give floor(x / d) for every dividend below 2^31 (edge values, powers of two, and random pairs)."""
    import random
    lib = nat.lib()
    rnd = random.Random(7)
    ds = [1, 2, 3, 4, 5, 6, 7, 9, 10, 31, 32, 33, 63, 64, 65, 127, 128, 148, 255, 256, 1000, 4096, 4097, 65535, 65536,
          131072, 999983, 2 ** 20 + 1, 2 ** 30, 2 ** 31 - 1] + [rnd.randrange(1, 2 ** 31) for _ in range(60)]
    for d in ds:
        xs = [0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, 2 ** 31 - 1, 2 ** 31 - 2, (2 ** 31 - 1) // d * d,
              max((2 ** 31 - 1) // d * d - 1, 0)] + [rnd.randrange(0, 2 ** 31) for _ in range(200)]
        for x in xs:
            if 0 <= x < 2 ** 31:
                assert lib.unetb200_test_fastdiv(d, x) == x // d, (d, x)


def test_integration_doc_names_every_symbol():
    """INTEGRATION.md maps every entry point of include/unetb200.h to the reference code it replaces."""
    hdr = open(os.path.join(ROOT, "include", "unetb200.h")).read()
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    declared = set(re.findall(r"\b(unetb200_[a-z0-9_]+)\s*\(", hdr))
    assert not [d for d in sorted(declared) if d not in doc]


def test_trained_fixture_generator_produces_the_checkpoint_format():
    """synthetic.train_fixture_state (tools/make_fixture_checkpoint.py --trained): two steps on the CPU give a
    state_dict in the checkpoint's exact format (136 keys, fp32 + int64 counters) that loads strictly."""
    from tw_invoice_unet_ocr_llm_b200.synthetic import invoice_loss, marked_invoices, train_fixture_state
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    x, m = marked_invoices(2, 64, seed=5)
    assert x.shape == (2, 3, 64, 64) and m.shape == (2, 3, 64, 64) and set(m.unique().tolist()) <= {0.0, 1.0}
    assert torch.equal(x, torch.round(x * 255) / 255)                  # values k/255, like preprocess output
    assert 0.0 < float(invoice_loss(torch.zeros(2, 3, 64, 64), m)) < 2.0
    state, loss = train_fixture_state("cpu", steps=2)
    assert len(state) == 136 and loss == loss
    res = UNet().load_state_dict(state, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert all(v.dtype in (torch.float32, torch.int64) for v in state.values())
