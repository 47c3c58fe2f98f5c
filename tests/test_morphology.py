"""Mask clean-up (unetb200_mask_morph / prepost.mask_morphology / prepost.fill_holes / run_unet_instances(clean=)).
The oracles are cv2.erode / cv2.dilate / cv2.morphologyEx and scipy.ndimage.binary_fill_holes, run in this process;
every result is bits, so the bar is np.array_equal.  A numpy window model of the rules (DESIGN 6b, "Mask clean-up")
pins the semantics to both libraries on the CPU."""

import cv2
import numpy as np
import pytest
import torch
from numpy.lib.stride_tricks import sliding_window_view
from PIL import Image
from scipy import ndimage

KS = [1, 2, 3, 4, 5, 7, 8, 15, 16, 31, 32, 33, 62, 63]
# every size of KS as kw and as kh, square and with kw != kh
KPAIRS = [(k, k) for k in KS] + [(1, 63), (63, 1), (2, 33), (33, 2), (15, 4), (4, 15), (62, 7), (8, 31), (16, 5),
                                 (32, 3), (3, 32), (5, 16), (7, 62), (31, 8)]
OPS = ["erode", "dilate", "open", "close"]
SHAPES = [(h, w) for h in (1, 2, 63, 512) for w in (1, 31, 32, 33, 64, 100, 512, 1000)] + [(1080, 1920)]


# ---------------------------------------------------------------- the window model and the oracles

def model_rect(m, kw, kh, dilate):
    """AND (OR) over the window x - kw//2 .. x + kw - 1 - kw//2, y - kh//2 .. y + kh - 1 - kh//2, clipped to
    the plane: the outside is padded with the identity of the operation."""
    ax, ay = kw // 2, kh // 2
    p = np.pad(m != 0, ((ay, kh - 1 - ay), (ax, kw - 1 - ax)), constant_values=not dilate)
    win = sliding_window_view(p, (kh, kw))
    return (win.any(axis=(2, 3)) if dilate else win.all(axis=(2, 3))).astype(np.uint8)


def model_op(m, op, kw, kh):
    if op in ("erode", "dilate"):
        return model_rect(m, kw, kh, op == "dilate")
    first = op == "close"                               # close dilates first, open erodes first
    return model_rect(model_rect(m, kw, kh, first), kw, kh, not first)


def model_fill_holes(m):
    """m | the 4-connected background components that touch no border pixel."""
    bg = m == 0
    lab, _ = ndimage.label(bg, ndimage.generate_binary_structure(2, 1))
    border = np.unique(np.concatenate([lab[0], lab[-1], lab[:, 0], lab[:, -1]]))
    return ((m != 0) | (bg & ~np.isin(lab, border))).astype(np.uint8)


CV_OPS = {"open": cv2.MORPH_OPEN, "close": cv2.MORPH_CLOSE}


def cv_op(m, op, kw, kh):
    el = np.ones((kh, kw), np.uint8)
    m = np.ascontiguousarray(m, np.uint8)
    if op == "erode":
        return cv2.erode(m, el)
    if op == "dilate":
        return cv2.dilate(m, el)
    return cv2.morphologyEx(m, CV_OPS[op], el)


def sp_fill(m):
    return ndimage.binary_fill_holes(m != 0).astype(np.uint8)


def patterns(h, w, seed=0):
    rng = np.random.default_rng(seed * 7919 + h * 1009 + w)
    yy, xx = np.mgrid[:h, :w]
    out = {f"rand{d}": (rng.random((h, w)) < d).astype(np.uint8) for d in (0.05, 0.5, 0.95)}
    out["zeros"] = np.zeros((h, w), np.uint8)
    out["ones"] = np.ones((h, w), np.uint8)
    for name, (y, x) in {"c00": (0, 0), "c01": (0, w - 1), "c10": (h - 1, 0), "c11": (h - 1, w - 1)}.items():
        c = np.zeros((h, w), np.uint8)
        c[y, x] = 1
        out[name] = c
    out["stripes_v"] = (xx % 3 == 1).astype(np.uint8)
    out["stripes_h"] = (yy % 2 == 0).astype(np.uint8)
    out["checker"] = ((xx + yy) % 2 == 0).astype(np.uint8)
    return out


def hole_patterns():
    """64 x 96 planes with known holes."""
    h, w = 64, 96
    out = {}
    rings = np.zeros((h, w), np.uint8)              # nested rings: the ring gaps and the centre are holes
    for r in (28, 22, 16, 10, 4):                   # outermost first
        rings[32 - r:32 + r, 40 - r:40 + r] = (r // 6) % 2 == 0
    rings[30:34, 38:42] = 0
    out["rings"] = rings
    edge = np.zeros((h, w), np.uint8)                # a square open to the left border: no hole
    edge[10:30, 0:20] = 1
    edge[15:25, 0:15] = 0
    edge[40:60, 50:90] = 1                           # a closed square: a hole
    edge[45:55, 55:85] = 0
    out["border_hole"] = edge
    diag = np.zeros((h, w), np.uint8)                # a box whose only gap is a diagonal step: still a hole (4-conn.)
    diag[10:30, 10:30] = 1
    diag[12:28, 12:28] = 0
    diag[10, 20] = 0                                 # a gap in the top wall, joined to the inside only diagonally
    diag[11, 20] = 1
    diag[12, 20] = 1
    diag[11, 19] = 0
    out["diagonal_gap"] = diag
    yy, xx = np.mgrid[:h, :w]
    out["checker"] = ((xx + yy) % 2 == 0).astype(np.uint8)
    out["zeros"] = np.zeros((h, w), np.uint8)
    out["ones"] = np.ones((h, w), np.uint8)
    rng = np.random.default_rng(5)
    for d in (0.3, 0.5, 0.7):
        out[f"rand{d}"] = (rng.random((h, w)) < d).astype(np.uint8)
    return out


def expected_rows(plane, k, conn=8):
    """scipy labels and the K largest rows (xmin, xmax, ymin, ymax, count, label) as mask_components orders them."""
    h, w = plane.shape
    lab, n = ndimage.label(plane, ndimage.generate_binary_structure(2, 1) if conn == 4 else np.ones((3, 3), bool))
    counts = np.bincount(lab.ravel(), minlength=n + 1)[1:]
    order = np.lexsort((np.arange(1, n + 1), -counts))[:k]
    objs = ndimage.find_objects(lab)
    rows = [(objs[i][1].start, objs[i][1].stop - 1, objs[i][0].start, objs[i][0].stop - 1, counts[i], i + 1)
            for i in order]
    rows += [(w, -1, h, -1, 0, 0)] * (k - len(rows))
    return lab, np.array(rows, np.int32)


def pack_bits(m):
    return np.packbits(np.ascontiguousarray(m).astype(np.uint8), axis=-1, bitorder="little")


def unpack_bits(b):
    return np.unpackbits(b, axis=-1, bitorder="little")


# ---------------------------------------------------------------- CPU: the model against cv2 and scipy

def test_model_matches_cv2():
    rng = np.random.default_rng(1)
    for h, w in [(1, 1), (1, 40), (37, 1), (23, 45), (64, 70)]:
        planes = list(patterns(h, w).values()) + [(rng.random((h, w)) < 0.3).astype(np.uint8) * 255]
        for kw, kh in KPAIRS:
            for op in OPS:
                for m in planes:
                    assert np.array_equal(model_op(m, op, kw, kh), cv_op(m != 0, op, kw, kh)), (h, w, kw, kh, op)


def test_model_fill_holes_matches_scipy():
    for name, m in list(hole_patterns().items()) + list(patterns(40, 33).items()):
        assert np.array_equal(model_fill_holes(m), sp_fill(m)), name
    hp = hole_patterns()
    assert sp_fill(hp["border_hole"])[20, 5] == 0 and sp_fill(hp["border_hole"])[50, 70] == 1
    assert sp_fill(hp["diagonal_gap"])[20, 20] == 1 and sp_fill(hp["diagonal_gap"])[11, 19] == 1


def test_even_element_window_is_opencvs():
    """Even sizes: dilation uses the erosion window (OpenCV), not the reflected one (scipy.ndimage)."""
    m = np.zeros((9, 9), np.uint8)
    m[4, 4] = 1
    d = cv_op(m, "dilate", 2, 2)
    assert d[4:6, 4:6].all() and d.sum() == 4                  # window x - 1 .. x: the dot spreads down-right
    assert np.array_equal(d, model_rect(m, 2, 2, True))
    s = ndimage.binary_dilation(m, np.ones((2, 2), bool)).astype(np.uint8)
    assert not np.array_equal(s, d)


@pytest.fixture(scope="module")
def nat():
    import __graft_entry__ as g
    g.build()
    from tw_invoice_unet_ocr_llm_b200 import _native
    return _native


def test_workspace_query(nat):
    q = nat.lib().unetb200_morph_workspace_bytes
    for h, w in [(1, 1), (63, 33), (512, 512), (1080, 1920)]:
        for p in (1, 192):
            words = p * h * ((w + 31) // 32)
            for op in range(4):
                assert q(p, h, w, op) == 2 * ((4 * words + 15) // 16 * 16)
            assert q(p, h, w, nat.MORPH_FILL_HOLES) == nat.lib().unetb200_components_workspace_bytes(p, h, w)
    assert q(192, 512, 512, nat.MORPH_OPEN) == 2 * 6_291_456        # two bit planes of 64 x 3 x 512^2
    assert q(0, 16, 16, 0) == 0 and q(1, 0, 16, 0) == 0 and q(1, 16, -1, 0) == 0 and q(1, 1 << 16, 1 << 15, 0) == 0
    assert q(1, 16, 16, 5) == 0 and q(1, 16, 16, -1) == 0


def test_c_abi_errors(nat):
    lib = nat.lib()
    dev = 1 << 20                                   # never dereferenced: every call below fails validation

    def call(inp=dev, inp_packed=0, out=dev + (1 << 16), out_packed=0, planes=2, h=64, w=64, op=nat.MORPH_OPEN,
             kw=3, kh=3, ws=dev + (1 << 18), ws_bytes=None):
        if ws_bytes is None:
            ws_bytes = lib.unetb200_morph_workspace_bytes(2, 64, 64, op if 0 <= op <= 4 else 0)
        return lib.unetb200_mask_morph(inp, inp_packed, out, out_packed, planes, h, w, op, kw, kh, ws, ws_bytes, None)

    cases = [(dict(inp=None), "null pointer"), (dict(out=None), "null pointer"), (dict(ws=None), "null pointer"),
             (dict(op=-1), "op"), (dict(op=5), "op"),
             (dict(kw=0), "kw and kh"), (dict(kh=0), "kw and kh"), (dict(kw=64), "kw and kh"),
             (dict(kh=64), "kw and kh"), (dict(kw=-3), "kw and kh"),
             (dict(inp_packed=2), "0 or 1"), (dict(out_packed=-1), "0 or 1"),
             (dict(planes=0), "bad size"), (dict(h=0), "bad size"), (dict(w=-3), "bad size"),
             (dict(h=1 << 16, w=1 << 15), "bad size"),
             (dict(inp_packed=1, w=48), "w % 32"), (dict(out_packed=1, w=100), "w % 32"),
             (dict(op=nat.MORPH_FILL_HOLES, inp_packed=1, w=33), "w % 32"),
             (dict(inp_packed=1, inp=dev + 2), "misaligned"), (dict(out_packed=1, out=dev + 1), "misaligned"),
             (dict(ws=dev + (1 << 18) + 8), "misaligned")]
    for kw, msg in cases:
        assert call(**kw) == nat.EINVAL, kw
        err = nat.last_error()
        assert err.startswith("mask_morph: ") and msg in err, (kw, err)
    # byte planes at any alignment, and k ignored for fill holes: these pass validation up to the workspace check
    for op in range(5):
        need = lib.unetb200_morph_workspace_bytes(2, 64, 64, op)
        for kw in (dict(), dict(inp=dev + 1, out=dev + 3)) + ((dict(kw=0, kh=99),) if op == 4 else ()):
            assert call(op=op, ws_bytes=need - 1, **kw) == nat.ENOMEM, (op, kw)
            assert "workspace smaller than unetb200_morph_workspace_bytes" in nat.last_error()


def test_python_errors_without_gpu(tmp_path):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200 import prepost
    m = torch.zeros((1, 1, 32, 32), dtype=torch.uint8)
    for bad in (dict(op="opening"), dict(op="fill_holes"), dict(op="open", ksize=(0, 3)),
                dict(op="open", ksize=(3, 64)), dict(op="open", ksize=3), dict(op="open", ksize=(3.0, 3)),
                dict(op="open", ksize=(True, 3)), dict(op="open", ksize=(3, 3, 3))):
        with pytest.raises(ValueError):
            prepost.mask_morphology(m, **bad)
    with pytest.raises(RuntimeError):
        prepost.mask_morphology(m, "open")                      # CPU tensor
    with pytest.raises(RuntimeError):
        prepost.fill_holes(m)
    pil = Image.fromarray(np.zeros((64, 64, 3), np.uint8))
    missing = str(tmp_path / "no_such_checkpoint.pth")          # never opened: the steps fail first
    for clean in ("open", [("open",)], [("open", 3)], [("opening", (3, 3))], [("open", (3, 0))], ["fill"],
                  [("fill_holes", (3, 3))], [None], [("close", (9, 3)), "fill_holes", ("open", (64, 3))], 5,
                  [["dilate", [3, 3], 1]]):
        with pytest.raises(ValueError):
            inf.run_unet_instances(pil, missing, clean=clean)
    assert inf._clean_steps([("close", (9, 3)), "fill_holes", ["open", [3, 3]]]) == [
        ("close", (9, 3)), ("fill_holes", None), ("open", (3, 3))]
    assert inf._clean_steps(None) == [] and inf._clean_steps([]) == []


# ---------------------------------------------------------------- GPU: every op against cv2

def run_morph(batch, dev, op, k=(3, 3), packed=False, out_packed=False):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    src = torch.from_numpy(pack_bits(batch) if packed else batch).to(dev)
    if op == "fill_holes":
        out = prepost.fill_holes(src, packed=packed, out_packed=out_packed)
    else:
        out = prepost.mask_morphology(src, op, k, packed=packed, out_packed=out_packed)
    out = out.cpu().numpy()
    return unpack_bits(out)[..., :batch.shape[-1]] if out_packed else out


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SHAPES)
def test_ops_match_cv2(cuda_dev, h, w):
    pats = patterns(h, w)
    batch = np.stack(list(pats.values()))[None]                 # [1, P, h, w]
    bad = []
    for kw, kh in KPAIRS:
        for op in OPS:
            got = run_morph(batch, cuda_dev, op, (kw, kh))
            for j, name in enumerate(pats):
                if not np.array_equal(got[0, j], cv_op(batch[0, j], op, kw, kh)):
                    bad.append((op, kw, kh, name))
    assert bad == [], bad[:20]


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(1, 1), (1, 40), (2, 33), (64, 96), (63, 100), (512, 512), (1080, 1920)])
def test_fill_holes_matches_scipy(cuda_dev, h, w):
    pats = patterns(h, w, seed=1)
    if (h, w) == (64, 96):
        pats.update({f"holes_{k}": v for k, v in hole_patterns().items()})
    batch = np.stack(list(pats.values()))[None]
    got = run_morph(batch, cuda_dev, "fill_holes")
    bad = [name for j, name in enumerate(pats) if not np.array_equal(got[0, j], sp_fill(batch[0, j]))]
    assert bad == []
    if (h, w) == (64, 96):
        names = list(pats)
        assert got[0, names.index("holes_diagonal_gap"), 20, 20] == 1
        assert got[0, names.index("holes_border_hole"), 20, 5] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(1, 32), (63, 64), (100, 96), (512, 512), (33, 1024)])
def test_byte_and_packed_sides_agree(cuda_dev, h, w):
    batch = np.stack(list(patterns(h, w, seed=2).values()))[None]
    for op, k in [("erode", (5, 3)), ("dilate", (2, 7)), ("open", (3, 3)), ("close", (33, 4)), ("fill_holes", None)]:
        ref = run_morph(batch, cuda_dev, op, k)
        for packed in (False, True):
            for out_packed in (False, True):
                got = run_morph(batch, cuda_dev, op, k, packed, out_packed)
                assert np.array_equal(got, ref), (op, packed, out_packed)
        want = np.stack([sp_fill(p) if op == "fill_holes" else cv_op(p, op, *k) for p in batch[0]])
        assert np.array_equal(ref[0], want), op


@pytest.mark.gpu
def test_batch_independence_and_determinism(cuda_dev):
    rng = np.random.default_rng(9)
    batch = (rng.random((64, 3, 40, 100)) < rng.random((64, 3, 1, 1))).astype(np.uint8)
    for op, k in [("open", (3, 3)), ("close", (9, 3)), ("erode", (16, 2)), ("dilate", (63, 63)), ("fill_holes", None)]:
        full = run_morph(batch, cuda_dev, op, k)
        assert np.array_equal(run_morph(batch, cuda_dev, op, k), full), op
        for idx in [(0, 0), (17, 2), (63, 1), (40, 0)]:
            alone = run_morph(batch[idx][None, None], cuda_dev, op, k)
            assert np.array_equal(alone[0, 0], full[idx]), (op, idx)
        want = sp_fill(batch[5, 1]) if op == "fill_holes" else cv_op(batch[5, 1], op, *k)
        assert np.array_equal(full[5, 1], want), op


@pytest.mark.gpu
def test_in_place_and_out(cuda_dev):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    batch = np.stack(list(patterns(64, 96, seed=3).values()))[None]
    for packed in (False, True):
        for op, k in [("erode", (3, 5)), ("close", (9, 3)), ("fill_holes", None)]:
            t = torch.from_numpy(pack_bits(batch) if packed else batch).to(cuda_dev)
            if op == "fill_holes":
                r = prepost.fill_holes(t, packed=packed, out=t)
            else:
                r = prepost.mask_morphology(t, op, k, packed=packed, out=t)
            assert r.data_ptr() == t.data_ptr()
            got = t.cpu().numpy()
            got = unpack_bits(got) if packed else got
            want = np.stack([sp_fill(p) if op == "fill_holes" else cv_op(p, op, *k) for p in batch[0]])
            assert np.array_equal(got[0], want), (op, packed)
    with pytest.raises(RuntimeError):
        prepost.mask_morphology(t, "open", out=torch.empty((1, 1, 64, 12), dtype=torch.uint8, device=cuda_dev),
                                packed=True)


@pytest.mark.gpu
def test_fixture_forward_masks_cleaned_in_place(cuda_dev, fixture_state):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    eng = Engine(fixture_state, cuda_dev)
    x = torch.from_numpy(synthetic_invoices_u8(8, 512, 512, seed=31)).to(cuda_dev)
    _, bits = eng.run(x, want_logits=False, thresholds=[0.25, 0.40, 0.30], mask_bits=True)
    m = unpack_bits(bits.cpu().numpy())
    assert m.any()
    prepost.mask_morphology(bits, "close", (9, 3), packed=True, out=bits)
    prepost.fill_holes(bits, packed=True, out=bits)
    prepost.mask_morphology(bits, "open", (3, 3), packed=True, out=bits)
    got = unpack_bits(bits.cpu().numpy())
    for idx in np.ndindex(m.shape[:2]):
        want = cv_op(sp_fill(cv_op(m[idx], "close", 9, 3)), "open", 3, 3)
        assert np.array_equal(got[idx], want), idx
    # the specks go: fewer components after the clean-up
    _, n0 = prepost.mask_components(torch.from_numpy(pack_bits(m)).to(cuda_dev), packed=True)
    _, n1 = prepost.mask_components(bits, packed=True)
    assert int(n1.sum()) < int(n0.sum())


# ---------------------------------------------------------------- GPU: run_unet_instances(clean=...)

@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory, fixture_state):
    import os
    path = os.path.join(tmp_path_factory.mktemp("ckpt"), "best_unet_model.pth")
    torch.save(fixture_state, path)
    return path


def host_clean(m, steps):
    for step in steps:
        m = sp_fill(m) if step == "fill_holes" else cv_op(m, step[0], *step[1])
    return m


def host_instances(pil, masks, steps, k, deskew):
    """cv2 / scipy clean-up -> scipy.ndimage.label -> the crop rule of _crop_rect (and _oriented_crop with
    cv2.warpAffine) -> the near-black test, on the host."""
    from oracle import oriented as orc
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    rgb = np.asarray(pil.convert("RGB"))
    scale = (pil.size[0] / 512, pil.size[1] / 512)
    out = {}
    for f in inf.FIELDS:
        lab, rows = expected_rows(host_clean(masks[f].astype(np.uint8), steps), k)
        obox = orc.oriented_rows(lab, rows, scale)[1]
        lst = []
        for row, ob in zip(rows, obox):
            if row[4] == 0:
                continue
            box = inf._crop_rect(pil.size, tuple(int(v) for v in row[:4]))
            if box is None:
                continue
            if deskew:
                oc = inf._oriented_crop(ob, scale)
                crop = cv2.warpAffine(rgb, np.asarray(oc["M"], np.float64), tuple(oc["out_size"]),
                                      flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP, borderMode=cv2.BORDER_REPLICATE)
            else:
                x1, y1, x2, y2 = box
                crop = rgb[y1:y2, x1:x2]
            if crop.mean() < 3:
                continue
            d = {"box": box, "pixels": int(row[4]), "crop": crop}
            if deskew:
                d.update(quad=oc["quad"], angle=oc["angle"], size=oc["size"])
            lst.append(d)
        out[f] = lst
    return out


def assert_same(got, want):
    assert list(got) == list(want)
    for f in want:
        assert [(d["box"], d["pixels"]) for d in got[f]] == [(d["box"], d["pixels"]) for d in want[f]], f
        for g, w in zip(got[f], want[f]):
            assert set(g) == set(w) and np.array_equal(np.asarray(g["crop"]), w["crop"]), f
            for key in ("quad", "angle", "size"):
                assert g.get(key) == w.get(key), (f, key)


@pytest.mark.gpu
@pytest.mark.parametrize("deskew", [False, True])
def test_run_unet_instances_clean(cuda_dev, checkpoint, deskew):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    pil = Image.fromarray(synthetic_invoices_u8(1, 720, 1280, seed=77)[0])
    masks0, _ = inf.run_unet(pil, checkpoint)
    # clean=None: today's behaviour, against the recomputation without clean-up
    masks, inst = inf.run_unet_instances(pil, checkpoint, max_instances=8, deskew=deskew)
    assert all(np.array_equal(masks[f], masks0[f]) for f in inf.FIELDS)
    assert_same(inst, host_instances(pil, masks0, [], 8, deskew))
    for steps in ([("close", (9, 3)), "fill_holes", ("open", (3, 3))], [("open", (3, 3))],
                  [("dilate", (15, 1)), ("erode", (2, 2))], ["fill_holes"]):
        masks, inst = inf.run_unet_instances(pil, checkpoint, max_instances=8, deskew=deskew, clean=steps)
        assert all(np.array_equal(masks[f], masks0[f]) for f in inf.FIELDS)      # the masks stay run_unet's
        want = host_instances(pil, masks0, steps, 8, deskew)
        assert sum(len(v) for v in want.values()) > 0
        assert_same(inst, want)
