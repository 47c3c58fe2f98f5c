"""fp16 / bf16 and channels-last inputs, and logits in the input's dtype.

A 16-bit element is exact in fp32 and an NHWC element is the same value read from another address, so every new
input format must give the bits of the fp32 NCHW path on ``x.float().contiguous()``; 16-bit logits are the fp32
logits rounded to nearest-even, i.e. ``z.to(dtype)`` bit for bit.  Everything here is compared with ``torch.equal``,
except one oracle check of the drop-in fp16 path.
"""
import copy
import ctypes as C

import pytest
import torch

gpu = pytest.mark.gpu

F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
THR = [0.25, 0.40, 0.30]
# (dtype, channels_last): every new way in -- all but the fp32 NCHW path, which is the reference
CASES = [(dt, cl) for dt in (F16, BF16, F32) for cl in (False, True) if (dt, cl) != (F32, False)]
CASE_IDS = [f"{str(dt)[6:]}-{'cl' if cl else 'nchw'}" for dt, cl in CASES]


def _nat():
    from tw_invoice_unet_ocr_llm_b200 import _native as nat
    return nat


def _as(x, dt, channels_last):
    y = x.to(dt)
    return y.to(memory_format=torch.channels_last) if channels_last else y.contiguous()


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("dt", [F32, F16, BF16])
def test_input_format_mapping(dt):
    from tw_invoice_unet_ocr_llm_b200.engine import input_format
    nat = _nat()
    nchw, nhwc = {F32: (nat.X_F32_NCHW, nat.X_F32_NHWC), F16: (nat.X_F16_NCHW, nat.X_F16_NHWC),
                  BF16: (nat.X_BF16_NCHW, nat.X_BF16_NHWC)}[dt]
    x = torch.rand(2, 3, 16, 32).to(dt)
    fmt, y = input_format(x)
    assert fmt == nchw and y is x
    xc = x.to(memory_format=torch.channels_last)
    fmt, y = input_format(xc)
    assert fmt == nhwc and y is xc                              # read in place: no copy
    # C = 1: contiguous and channels-last contiguous at once -> NCHW
    x1 = torch.rand(2, 1, 16, 16).to(dt).to(memory_format=torch.channels_last)
    assert x1.is_contiguous() and x1.is_contiguous(memory_format=torch.channels_last)
    assert input_format(x1)[0] == nchw
    # neither layout: copied to NCHW
    xt = torch.rand(2, 3, 16, 16).to(dt).transpose(2, 3)
    assert not xt.is_contiguous() and not xt.is_contiguous(memory_format=torch.channels_last)
    fmt, y = input_format(xt)
    assert fmt == nchw and y.is_contiguous() and torch.equal(y, xt) and y.data_ptr() != xt.data_ptr()


def test_input_format_uint8_and_rejected_dtypes():
    from tw_invoice_unet_ocr_llm_b200.engine import input_format
    nat = _nat()
    u8 = torch.zeros(2, 16, 16, 3, dtype=torch.uint8)
    assert input_format(u8)[0] == nat.X_U8_NHWC
    for dt in (torch.float64, torch.int32):
        with pytest.raises(RuntimeError):
            input_format(torch.zeros(1, 3, 16, 16, dtype=dt))


def test_forward_typed_null_handle_without_device():
    import __graft_entry__ as g
    g.build()
    nat = _nat()
    lib = nat.lib()
    assert lib.unetb200_forward_typed(None, None, nat.X_F16_NCHW, 1, 64, 64, None, 0, None, nat.LOGITS_F16,
                                      None, 0, None, None) == nat.EINVAL
    assert "handle" in nat.last_error()


def test_half_model_has_no_cpu_path():
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    m = UNet().half().eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(1, 3, 32, 32, dtype=F16))


# ---------------------------------------------------------------------------------------------------- GPU
def _model(state, dev, n_channels=3, n_classes=3):
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    m = UNet(n_channels=n_channels, n_classes=n_classes)
    m.load_state_dict(state)
    return m.to(dev).eval()


@pytest.fixture(scope="module")
def model(fixture_state, cuda_dev):
    return _model(fixture_state, cuda_dev)


@pytest.fixture(scope="module")
def eng(model, cuda_dev):
    return model.engine(cuda_dev)


def _outputs(e, x, **kw):
    """(logits, byte masks, bit-packed masks) of one input, synchronised."""
    thr = (THR + [0.35] * 8)[:e.n_classes]
    z, m = e.run(x, thresholds=thr, **kw)
    _, b = e.run(x, want_logits=False, thresholds=thr, mask_bits=True, **kw)
    torch.cuda.synchronize()
    return z, m, b


def _assert_same(got, ref, what):
    for name, a, b in zip(("logits", "masks", "bit masks"), got, ref):
        assert a.dtype == b.dtype and torch.equal(a, b), f"{what}: {name} differ"


@gpu
@pytest.mark.parametrize("dt,cl", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("n,h,w", [(2, 64, 64), (1, 32, 48), (3, 16, 16), (1, 96, 80), (2, 512, 512)])
def test_ingest_is_exact(eng, cuda_dev, dt, cl, n, h, w):
    """Tensor-core stem (n_channels = 3): every input format equals the fp32 NCHW path on x.float()."""
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    x = _as(synthetic_invoices(n, h, w, seed=70 + h).to(cuda_dev), dt, cl)
    ref = _outputs(eng, x.float().contiguous())
    got = _outputs(eng, x, logits_dtype=F32)
    _assert_same(got, ref, f"{dt} channels_last={cl} {n}x{h}x{w}")


def _small_model(n_channels, n_classes, dev):
    """As test_forward_parity.test_other_channel_and_class_counts builds it."""
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    torch.manual_seed(7 + n_channels + n_classes)
    m = UNet(n_channels=n_channels, n_classes=n_classes)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.normal_(0, 0.1)
                mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.8, 1.6)
                mod.bias.normal_(0, 0.1)
        m.out_conv.weight.mul_(8.0)
    return m.to(dev).eval()


@gpu
@pytest.mark.parametrize("n_channels,n_classes,stem_tc", [(1, 2, 1), (4, 5, 1), (3, 3, 0)],
                         ids=["1ch-tensor-core-stem", "4ch-cuda-core-stem", "3ch-stem_tc0"])
def test_ingest_is_exact_other_stems(cuda_dev, n_channels, n_classes, stem_tc):
    m = _small_model(n_channels, n_classes, cuda_dev)
    e = m.engine(cuda_dev)
    e.set_option("stem_tc", stem_tc)
    g = torch.Generator(device="cpu").manual_seed(n_channels)
    for n, h, w in [(2, 32, 48), (1, 64, 96)]:
        x0 = torch.rand((n, n_channels, h, w), generator=g).to(cuda_dev)
        for dt, cl in CASES:
            x = _as(x0, dt, cl)
            _assert_same(_outputs(e, x, logits_dtype=F32), _outputs(e, x.float().contiguous()),
                         f"n_channels={n_channels} stem_tc={stem_tc} {dt} channels_last={cl} {n}x{h}x{w}")


# options that put conv1.net.3 + out_conv on each head kernel
HEAD_VARIANTS = {
    "ps64-head": {},                                  # default: phase-stacked kernel (conv_ps64.cuh)
    "generic-head-pair": {"ps64": 1, "pair": 1},      # conv_tc.cuh head, CTA pairs
    "generic-head-single": {"ps64": 1, "pair": 0},    # conv_tc.cuh head, one CTA
    "row-head": {"ps64": 0, "row64": 1},              # conv_row.cuh head
    "ps64-head-pair0": {"pair": 0},
}


@gpu
@pytest.mark.parametrize("variant", list(HEAD_VARIANTS))
@pytest.mark.parametrize("dt", [F16, BF16])
def test_16bit_logits_are_rounded_fp32_logits(eng, cuda_dev, variant, dt):
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    opts = HEAD_VARIANTS[variant]
    saved = {k: eng.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            eng.set_option(k, v)
        for n, h, w in [(2, 64, 64), (1, 96, 80)]:
            x = synthetic_invoices(n, h, w, seed=80 + w).to(cuda_dev)
            for xin in (x, x.to(dt)):
                z32, m32, b32 = _outputs(eng, xin, logits_dtype=F32)
                z16, m16, b16 = _outputs(eng, xin, logits_dtype=dt)
                assert z16.dtype == dt and z16.is_contiguous()
                assert torch.equal(z16, z32.to(dt)), f"{variant}: {dt} logits != fp32 logits rounded"
                assert torch.equal(m16, m32) and torch.equal(b16, b32), f"{variant}: masks depend on the logits type"
            # a 16-bit input defaults to logits of its own dtype
            assert eng.run(x.to(dt))[0].dtype == dt
    finally:
        for k, v in saved.items():
            eng.set_option(k, v)


# ---- single-kernel hooks
def _pack_stem(nat, cin, dev, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    wt = (torch.randn((64, cin, 3, 3), generator=g) / 5.0).to(dev)
    b = torch.randn((64,), generator=g).to(dev)
    arch = nat.Arch(cin, 3, 64)
    layers = nat.layer_table(arch)
    blob = torch.zeros(int(nat.lib().unetb200_packed_bytes(C.byref(arch))), dtype=torch.uint8, device=dev)
    nat.check(nat.lib().unetb200_pack_layer(C.byref(arch), 0, wt.data_ptr(), b.data_ptr(), None, None, None, None,
                                            1e-5, blob.data_ptr(), None))
    return blob, layers[0]


def _formats(nat):
    return {nat.X_F16_NCHW: (F16, False), nat.X_BF16_NCHW: (BF16, False), nat.X_F32_NHWC: (F32, True),
            nat.X_F16_NHWC: (F16, True), nat.X_BF16_NHWC: (BF16, True)}


def _storage(x, nhwc):
    return x.permute(0, 2, 3, 1).contiguous() if nhwc else x.contiguous()


@gpu
@pytest.mark.parametrize("kernel,cin", [("stem_tc", 1), ("stem_tc", 3), ("stem", 1), ("stem", 3), ("stem", 4)])
@pytest.mark.parametrize("n,h,w", [(2, 40, 48), (1, 16, 16), (3, 4, 16), (1, 20, 144)])
def test_stem_hooks_new_formats(cuda_dev, kernel, cin, n, h, w):
    """unetb200_stem_tc (im2col tensor-core stem) and unetb200_stem (CUDA-core stem): each new format equals the
    fp32 NCHW result on the same values."""
    nat = _nat()
    lib = nat.lib()
    blob, l0 = _pack_stem(nat, cin, cuda_dev, 17 + cin)
    bias = blob.data_ptr() + l0.b_off
    g = torch.Generator(device="cpu").manual_seed(h * w + cin)
    x0 = torch.rand((n, cin, h, w), generator=g).to(cuda_dev)

    def run(src, fmt):
        out = torch.full((n, h, w, 64), float("nan"), dtype=torch.bfloat16, device=cuda_dev)
        if kernel == "stem_tc":
            wp = blob.data_ptr() + l0.w_off + int(lib.unetb200_stem_tc_offset(cin))
            nat.check(lib.unetb200_stem_tc(src.data_ptr(), fmt, cin, wp, bias, n, h, w, out.data_ptr(), None))
        else:
            nat.check(lib.unetb200_stem(src.data_ptr(), fmt, cin, blob.data_ptr() + l0.w_off, bias, n, h, w,
                                        out.data_ptr(), None))
        torch.cuda.synchronize()
        return out

    for fmt, (dt, nhwc) in _formats(nat).items():
        xd = x0.to(dt)
        ref = run(xd.float().contiguous(), nat.X_F32_NCHW)
        assert not torch.isnan(ref.float()).any()
        assert torch.equal(run(_storage(xd, nhwc), fmt), ref), f"{kernel} cin={cin} format {fmt}"


A_PS64 = 7


@gpu
@pytest.mark.parametrize("amode,pair", [(0, 0), (1, 0), (2, 0), (2, 1), (5, 0), (A_PS64, 1)],
                         ids=["tap", "col3", "halo", "halo-pair", "row", "ps64"])
@pytest.mark.parametrize("dt", [F16, BF16])
def test_conv3x3_head_logits_type(cuda_dev, amode, pair, dt):
    """unetb200_conv3x3_head with wstat bits 3-4 = the logits type: the fp32 logits rounded, masks unchanged."""
    nat = _nat()
    if amode == 1 and not nat.has_test_variants():
        pytest.skip("variant not compiled in (build with UNETB200_TEST_VARIANTS=1)")
    lt = {F16: nat.LOGITS_F16, BF16: nat.LOGITS_BF16}[dt]
    n, h, w, ncls = (2, 32, 32, 3) if amode != 5 else (2, 24, 176, 3)
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn((n, 64, h, w), generator=g).to(cuda_dev)
    wt = (torch.randn((64, 64, 3, 3), generator=g) / 24.0).to(cuda_dev)
    b = torch.randn((64,), generator=g).to(cuda_dev)
    hw = torch.randn((ncls, 64), generator=g).to(cuda_dev) / 4.0
    hb = torch.randn((ncls,), generator=g).to(cuda_dev)
    xb = x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    wb = wt.permute(2, 3, 0, 1).reshape(9, 64, 64).contiguous().to(torch.bfloat16)
    thr = (C.c_float * ncls)(-0.5, 0.0, 0.7)
    flags = 1 | (pair << 1)
    res = {}
    for t, ltype in ((F32, 0), (dt, lt)):
        logits = torch.full((n, ncls, h, w), float("nan"), dtype=t, device=cuda_dev)
        mask = torch.full((n, ncls, h, w), 7, dtype=torch.uint8, device=cuda_dev)
        nat.check(nat.lib().unetb200_conv3x3_head(xb.data_ptr(), 64, wb.data_ptr(), b.data_ptr(), hw.data_ptr(),
                                                  hb.data_ptr(), ncls, n, h, w, logits.data_ptr(), mask.data_ptr(),
                                                  thr, amode, flags | (ltype << 3), None))
        torch.cuda.synchronize()
        res[t] = (logits, mask)
    assert not torch.isnan(res[F32][0]).any()
    assert torch.equal(res[dt][0], res[F32][0].to(dt))
    assert torch.equal(res[dt][1], res[F32][1])
    # logits type 3 does not exist
    assert nat.lib().unetb200_conv3x3_head(xb.data_ptr(), 64, wb.data_ptr(), b.data_ptr(), hw.data_ptr(),
                                           hb.data_ptr(), ncls, n, h, w, res[dt][0].data_ptr(), None, None, amode,
                                           flags | (3 << 3), None) == nat.EINVAL


# ---- the drop-in module
def _rounded_state(state, dt):
    return {k: (v.to(dt).float() if v.is_floating_point() else v) for k, v in state.items()}


@gpu
@pytest.mark.parametrize("dt", [F16, BF16])
def test_half_and_bfloat16_modules(fixture_state, cuda_dev, dt):
    """m.half().eval(); m(x.half()) -> fp16 logits on the GPU (likewise bf16), equal to the fp32 module on the
    same (16-bit-representable) weights and input values, rounded."""
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    model = _model(_rounded_state(fixture_state, dt), cuda_dev)
    m16 = copy.deepcopy(model)
    m16 = m16.half() if dt == F16 else m16.bfloat16()
    m16.eval()
    x = synthetic_invoices(2, 64, 96, seed=91).to(cuda_dev)
    with torch.no_grad():
        z = m16(x.to(dt))
        ref = model(x.to(dt).float()).to(dt)
    assert z.dtype == dt and z.is_cuda and z.shape == (2, 3, 64, 96) and z.is_contiguous()
    assert torch.equal(z, ref)


@gpu
def test_channels_last_module_input(model, cuda_dev):
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    x = synthetic_invoices(2, 64, 96, seed=92).to(cuda_dev)
    with torch.no_grad():
        z = model(x)
        zc = model(x.to(memory_format=torch.channels_last))
    assert zc.is_contiguous() and zc.dtype == F32 and torch.equal(zc, z)


def _check(rep, min_agree):
    # the stated tolerance of tests/test_forward_parity.py
    assert rep["max_abs"] <= 0.25, rep
    assert rep["max_abs_over_std"] <= 0.19, rep
    assert rep["mean_abs"] <= 0.025, rep
    assert rep["agreement"] >= min_agree, rep
    assert rep["agreement_outside_0.25"] == 1.0, rep
    assert min(rep["iou"]) >= 0.95, rep


@gpu
def test_fp16_input_against_oracle_512(model, fixture_state, cuda_dev):
    from oracle.unet_oracle import oracle_forward, parity_report
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    x = synthetic_invoices(1, 512, 512, seed=42).half()
    with torch.no_grad():
        z = model(x.to(cuda_dev))
    assert z.dtype == F16
    rep = parity_report(oracle_forward(fixture_state, x.float()), z.float())
    print(f"parity fp16 1x512x512: {rep}")
    _check(rep, 0.999)


# ---- plan and graph cache
@gpu
def test_plan_cache_keys_on_formats_and_logits_type(model, fixture_state, cuda_dev):
    """fp16 / bf16 views of ONE input buffer and fp32 / fp16 logits in ONE output buffer, each combination run
    three times (graph replay from the second use): every result equals the same forward on a fresh engine."""
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    eng = model.engine(cuda_dev)
    shape = (2, 3, 64, 64)
    x = synthetic_invoices(*shape[:1], 64, 64, seed=93).to(cuda_dev)
    raw = torch.empty(x.numel() * 2, dtype=torch.uint8, device=cuda_dev)
    inputs = {F16: raw.view(F16).view(shape), BF16: raw.view(BF16).view(shape)}
    out_raw = torch.empty(x.numel() * 4, dtype=torch.uint8, device=cuda_dev)
    outs = {F32: out_raw.view(F32).view(shape), F16: out_raw[:x.numel() * 2].view(F16).view(shape)}
    mask = torch.empty(shape, dtype=torch.uint8, device=cuda_dev)
    combos = [(di, dl) for di in (F16, BF16) for dl in (F32, F16)]
    fresh = Engine(fixture_state, cuda_dev)
    ref = {}
    for di, dl in combos:
        z, m = fresh.run(x.to(di), thresholds=THR, logits_dtype=dl)
        torch.cuda.synchronize()
        ref[(di, dl)] = (z, m)
    for it in range(3):
        for di, dl in combos:
            inputs[di].copy_(x.to(di))
            z, m = eng.run(inputs[di], thresholds=THR, logits_dtype=dl, logits_out=outs[dl], mask_out=mask)
            torch.cuda.synchronize()
            assert z.data_ptr() == out_raw.data_ptr()
            assert torch.equal(z, ref[(di, dl)][0]) and torch.equal(m, ref[(di, dl)][1]), (it, di, dl)
    fresh.close()


# ---- errors
@gpu
def test_errors_raised_before_launch(eng, cuda_dev):
    nat = _nat()
    for dt in (torch.float64, torch.int32):
        with pytest.raises(RuntimeError):
            eng.run(torch.zeros(1, 3, 64, 64, dtype=dt, device=cuda_dev))
    shape = (1, 3, 64, 64)
    numel = 3 * 64 * 64
    for dt in (F16, BF16):
        buf = torch.zeros(numel + 8, dtype=dt, device=cuda_dev)
        x = buf[1:1 + numel].view(shape)                          # 2 bytes past a 16-byte boundary
        assert x.is_contiguous() and x.data_ptr() % 16 == 2
        with pytest.raises(RuntimeError, match="aligned"):
            eng.run(x)
    with pytest.raises(RuntimeError):
        eng.run(torch.zeros(shape, device=cuda_dev), logits_dtype=torch.float64)
    with pytest.raises(RuntimeError):
        eng.run(torch.zeros(shape, device=cuda_dev), logits_out=torch.empty(shape, dtype=F16, device=cuda_dev))
    if nat.has_test_variants():
        saved = eng.get_option("stem_tc")
        eng.set_option("stem_tc", 2)
        try:
            with pytest.raises(RuntimeError, match="patch stem"):
                eng.run(torch.zeros(shape, dtype=F16, device=cuda_dev))
        finally:
            eng.set_option("stem_tc", saved)
    # nothing was launched: the context is healthy and the next forward runs
    z, _ = eng.run(torch.zeros(shape, dtype=F16, device=cuda_dev))
    torch.cuda.synchronize()
    assert z.dtype == F16 and torch.isfinite(z.float()).all()
