"""Connected components of the field masks (unetb200_mask_components / prepost.mask_components /
inference.run_unet_instances).  The oracle is scipy.ndimage.label, run in this process: labels, counts and
extents are integer results, so the bar is bit-exact."""

import numpy as np
import pytest
import torch
from PIL import Image
from scipy import ndimage

SHAPES = [(16, 16), (33, 50), (512, 512), (1024, 768), (16, 1024), (1024, 16)]


def structure(conn):
    return ndimage.generate_binary_structure(2, 1) if conn == 4 else np.ones((3, 3), bool)


def serpentine(h, w):
    """One-pixel-wide path: every even row full, odd rows joined at alternating ends."""
    m = np.zeros((h, w), bool)
    m[0::2] = True
    m[1::4, w - 1] = True
    m[3::4, 0] = True
    return m


def patterns(h, w):
    rng = np.random.default_rng(h * 1009 + w)
    yy, xx = np.mgrid[:h, :w]
    out = {f"rand{d}": rng.random((h, w)) < d for d in (0.02, 0.4, 0.6, 0.95)}
    out["checker"] = (yy + xx) % 2 == 0
    out["zeros"] = np.zeros((h, w), bool)
    out["ones"] = np.ones((h, w), bool)
    corners = np.zeros((h, w), bool)
    corners[0, 0] = corners[0, -1] = corners[-1, 0] = corners[-1, -1] = True
    out["corners"] = corners
    out["serpentine"] = serpentine(h, w)
    out["serpentine_t"] = serpentine(w, h).T
    out["diagonal"] = (xx - yy) % 4 == 0            # staircases: joined only under 8-connectivity
    out["antidiagonal"] = (xx + yy) % 5 == 0
    out["stripes_v"] = xx % 3 == 1
    out["stripes_h"] = yy % 2 == 0
    return out


def expected(plane, conn, k):
    """(labels, n, comps [k, 6]) of one plane from scipy and numpy."""
    h, w = plane.shape
    lab, n = ndimage.label(plane, structure(conn))
    counts = np.bincount(lab.ravel(), minlength=n + 1)[1:]
    order = np.lexsort((np.arange(1, n + 1), -counts))[:k]           # count descending, then label ascending
    objs = ndimage.find_objects(lab)
    rows = []
    for i in order:
        sy, sx = objs[i]
        rows.append((sx.start, sx.stop - 1, sy.start, sy.stop - 1, counts[i], i + 1))
    rows += [(w, -1, h, -1, 0, 0)] * (k - len(rows))
    return lab.astype(np.int32), n, np.array(rows, np.int32)


def pack_bits(m):
    return np.packbits(np.ascontiguousarray(m).astype(np.uint8), axis=-1, bitorder="little")


def run(mask_np, dev, packed=False, **kw):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    src = pack_bits(mask_np) if packed else mask_np.astype(np.uint8)
    out = prepost.mask_components(torch.from_numpy(src).to(dev), packed=packed, **kw)
    return tuple(t.cpu().numpy() for t in out)


# ---------------------------------------------------------------- CPU: ABI validation and workspace bound

@pytest.fixture(scope="module")
def nat():
    import __graft_entry__ as g
    g.build()
    from tw_invoice_unet_ocr_llm_b200 import _native
    return _native


def test_workspace_bound(nat):
    q = nat.lib().unetb200_components_workspace_bytes
    for h, w in SHAPES + [(3, 3), (1, 4096), (4096, 1), (480, 640)]:
        for p in (1, 3, 192):
            assert 0 < q(p, h, w) <= 16 * p * h * w, (p, h, w)
    assert q(64 * 3, 512, 512) <= 805_306_368
    assert q(0, 16, 16) == 0 and q(1, 0, 16) == 0 and q(1, 16, -1) == 0 and q(1, 1 << 16, 1 << 15) == 0


def test_c_abi_errors(nat):
    lib = nat.lib()
    ws_need = lib.unetb200_components_workspace_bytes(2, 64, 64)
    dev = 1 << 20                                   # never dereferenced: every call below fails validation

    def call(mask=dev, packed=0, planes=2, h=64, w=64, conn=8, k=4, labels=None, comps=dev, n=dev, ws=dev,
             ws_bytes=ws_need):
        return lib.unetb200_mask_components(mask, packed, planes, h, w, conn, k, labels, comps, n, ws, ws_bytes, None)

    for kw in (dict(mask=None), dict(comps=None), dict(n=None), dict(ws=None), dict(conn=6), dict(conn=0),
               dict(k=0), dict(k=17), dict(planes=0), dict(h=0), dict(w=-3), dict(h=1 << 16, w=1 << 15),
               dict(packed=1, w=48), dict(packed=2), dict(packed=1, mask=dev + 2), dict(labels=dev + 1),
               dict(comps=dev + 2), dict(n=dev + 1), dict(ws=dev + 4)):
        assert call(**kw) == nat.EINVAL, kw
        assert nat.last_error().startswith("mask_components"), kw
    assert call(ws_bytes=ws_need - 1) == nat.ENOMEM
    assert "workspace" in nat.last_error()


def test_python_errors_without_gpu():
    from tw_invoice_unet_ocr_llm_b200 import prepost
    with pytest.raises(RuntimeError):
        prepost.mask_components(torch.zeros((1, 1, 16, 16), dtype=torch.uint8))          # CPU tensor
    with pytest.raises(RuntimeError):
        prepost.mask_components(torch.zeros((1, 1, 16, 16), dtype=torch.int32))
    with pytest.raises(RuntimeError):
        prepost.mask_components(torch.zeros((16, 16), dtype=torch.uint8))


def test_scipy_oracle_conventions():
    """The oracle's own conventions: raster numbering, the tie rule and the empty rows."""
    m = np.zeros((6, 8), bool)
    m[4, 1:3] = True          # label 3, 2 px
    m[0, 5] = True            # label 1, 1 px
    m[1, 0:2] = True          # label 2, 2 px
    lab, n, rows = expected(m, 4, 4)
    assert n == 3 and lab[0, 5] == 1 and lab[1, 0] == 2 and lab[4, 1] == 3
    assert rows.tolist() == [[0, 1, 1, 1, 2, 2], [1, 2, 4, 4, 2, 3], [5, 5, 0, 0, 1, 1], [8, -1, 6, -1, 0, 0]]


# ---------------------------------------------------------------- CPU: components -> instances

def _fake_box_sums(calls):
    def box_sums(frame, rects, channels=None):
        assert 1 <= len(rects) <= 16
        calls.append(len(rects))
        return torch.tensor([int(frame[y1:y2, x1:x2, :channels].astype(np.int64).sum()) for x1, y1, x2, y2 in rects])
    return box_sums


def test_components_to_instances_mapping(monkeypatch):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200 import prepost
    frame = np.full((1024, 2048, 3), 200, np.uint8)
    frame[:256, :256] = 0                                   # near-black top-left corner
    pil = Image.fromarray(frame)
    k = 8
    comps = np.tile(np.array([256, -1, 256, -1, 0, 0], np.int32), (3, k, 1))
    # field 0, largest first: a live region, one on the black corner, a single pixel (an empty rectangle, as
    # in the reference), a small live region
    comps[0, 0] = (300, 400, 300, 350, 900, 5)
    comps[0, 1] = (10, 50, 10, 50, 400, 1)                  # inside the black corner -> dropped
    comps[0, 2] = (100, 100, 300, 300, 1, 3)                # x1 == x2 after scaling -> dropped before the sums
    comps[0, 3] = (450, 470, 40, 50, 30, 4)
    # field 1: eight live regions, field 2: empty
    for j in range(k):
        comps[1, j] = (300 + 20 * j, 310 + 20 * j, 200, 260, 100 - j, j + 1)
    calls = []
    monkeypatch.setattr(prepost, "box_sums", _fake_box_sums(calls))
    out = inf.components_to_instances(pil, comps, frame, min_pixels=1)
    assert calls == [11]                                    # 3 + 8 + 0 rectangles, one call
    assert list(out) == inf.FIELDS and out["total_amount"] == []
    boxes0 = [d["box"] for d in out["invoice_no"]]
    assert boxes0 == [inf._crop_rect(pil.size, (300, 400, 300, 350)),
                      inf._crop_rect(pil.size, (450, 470, 40, 50))]
    assert [d["pixels"] for d in out["invoice_no"]] == [900, 30]
    assert [d["pixels"] for d in out["date"]] == [100 - j for j in range(k)]
    for lst in out.values():
        for d in lst:
            assert np.array_equal(np.asarray(d["crop"]), frame[d["box"][1]:d["box"][3], d["box"][0]:d["box"][2]])
    # min_pixels filters; the same table without a device frame takes the host test and agrees
    calls.clear()
    out2 = inf.components_to_instances(pil, comps, frame, min_pixels=31)
    assert [d["pixels"] for d in out2["invoice_no"]] == [900] and len(out2["date"]) == k
    host = inf.components_to_instances(pil, comps, None, min_pixels=31)
    assert {f: [d["box"] for d in v] for f, v in host.items()} == {f: [d["box"] for d in v] for f, v in out2.items()}
    # more than 16 rectangles: groups of 16
    comps3 = np.concatenate([comps[1:2]] * 3)               # 24 live rectangles
    calls.clear()
    out3 = inf.components_to_instances(pil, comps3, frame)
    assert calls == [16, 8] and all(len(v) == k for v in out3.values())
    # a region whose rectangle is empty after scaling (1-row-high image) is dropped before the sums
    flat = Image.fromarray(np.full((1, 600, 3), 200, np.uint8))
    comps4 = comps[:, :1].copy()
    comps4[:] = (10, 20, 0, 0, 11, 1)
    calls.clear()
    assert all(v == [] for v in inf.components_to_instances(flat, comps4, np.asarray(flat)).values())
    assert calls == []


# ---------------------------------------------------------------- GPU: labels and statistics

@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("h,w", SHAPES)
def test_labels_and_stats_match_scipy(cuda_dev, h, w, conn):
    pats = patterns(h, w)
    batch = np.stack(list(pats.values()))[None]             # [1, P, h, w]
    k = 16
    comps, n, lab = run(batch, cuda_dev, connectivity=conn, max_components=k, labels=True)
    for j, name in enumerate(pats):
        ref_lab, ref_n, ref_rows = expected(batch[0, j], conn, k)
        assert n[0, j] == ref_n, (name, n[0, j], ref_n)
        assert np.array_equal(lab[0, j], ref_lab), (name, int((lab[0, j] != ref_lab).sum()))
        assert np.array_equal(comps[0, j], ref_rows), (name, comps[0, j], ref_rows)
    names = list(pats)
    assert n[0, names.index("checker")] == ((h * w + 1) // 2 if conn == 4 else 1)
    if w % 32 == 0:
        comps_b, n_b, lab_b = run(batch, cuda_dev, packed=True, connectivity=conn, max_components=k, labels=True)
        assert np.array_equal(comps_b, comps) and np.array_equal(n_b, n) and np.array_equal(lab_b, lab)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_k1_bbox_consistency_batch_independence(cuda_dev, conn):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    pats = patterns(33, 50)
    batch = np.stack(list(pats.values())).reshape(2, -1, 33, 50)
    comps1, n1 = run(batch, cuda_dev, connectivity=conn, max_components=1)
    for idx in np.ndindex(batch.shape[:2]):
        _, ref_n, ref_rows = expected(batch[idx], conn, 1)
        assert np.array_equal(comps1[idx], ref_rows) and n1[idx] == ref_n
    # K >= n: the listed boxes cover exactly what mask_bbox reports
    comps, n, lab = run(batch, cuda_dev, connectivity=conn, max_components=16, labels=True)
    bb = prepost.mask_bbox(torch.from_numpy(batch.astype(np.uint8)).to(cuda_dev)).cpu().numpy()
    for idx in np.ndindex(batch.shape[:2]):
        if n[idx] > 16:
            continue
        rows = comps[idx][: n[idx]]
        got = (rows[:, 0].min(initial=50), rows[:, 1].max(initial=-1), rows[:, 2].min(initial=33),
               rows[:, 3].max(initial=-1), rows[:, 4].sum())
        assert got == tuple(bb[idx]), (idx, got, bb[idx])
    # each plane alone gives the same bits; a second run too
    for idx in np.ndindex(batch.shape[:2]):
        c1, m1, l1 = run(batch[idx][None, None], cuda_dev, connectivity=conn, max_components=16, labels=True)
        assert np.array_equal(c1[0, 0], comps[idx]) and m1[0, 0] == n[idx] and np.array_equal(l1[0, 0], lab[idx])
    again = run(batch, cuda_dev, connectivity=conn, max_components=16, labels=True)
    assert all(np.array_equal(a, b) for a, b in zip(again, (comps, n, lab)))


@pytest.mark.gpu
def test_python_argument_errors(cuda_dev):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    m = torch.zeros((1, 1, 32, 32), dtype=torch.uint8, device=cuda_dev)
    for kw in (dict(connectivity=6), dict(max_components=0), dict(max_components=17)):
        with pytest.raises(RuntimeError):
            prepost.mask_components(m, **kw)
    with pytest.raises(RuntimeError):
        prepost.mask_components(m.float())
    with pytest.raises(RuntimeError):
        prepost.mask_components(m[0])
    with pytest.raises(RuntimeError):
        prepost.mask_components(m[..., :3], packed=True)      # 24-pixel rows


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_fixture_forward_masks_match_scipy(cuda_dev, fixture_state, conn):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    eng = Engine(fixture_state, cuda_dev)
    x = torch.from_numpy(synthetic_invoices_u8(8, 512, 512, seed=31)).to(cuda_dev)
    _, mask = eng.run(x, want_logits=False, thresholds=[0.25, 0.40, 0.30])
    _, bits = eng.run(x, want_logits=False, thresholds=[0.25, 0.40, 0.30], mask_bits=True)
    comps, n, lab = (t.cpu().numpy() for t in prepost.mask_components(mask, connectivity=conn, max_components=8,
                                                                      labels=True))
    packed = tuple(t.cpu().numpy() for t in prepost.mask_components(bits, packed=True, connectivity=conn,
                                                                    max_components=8, labels=True))
    m = mask.cpu().numpy() != 0
    assert m.any()
    for idx in np.ndindex(m.shape[:2]):
        ref_lab, ref_n, ref_rows = expected(m[idx], conn, 8)
        assert n[idx] == ref_n and np.array_equal(lab[idx], ref_lab) and np.array_equal(comps[idx], ref_rows), idx
    assert all(np.array_equal(a, b) for a, b in zip(packed, (comps, n, lab)))


# ---------------------------------------------------------------- GPU: run_unet_instances

@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory, fixture_state):
    import os
    path = os.path.join(tmp_path_factory.mktemp("ckpt"), "best_unet_model.pth")
    torch.save(fixture_state, path)
    return path


@pytest.mark.gpu
def test_run_unet_instances_on_fixture_masks(cuda_dev, checkpoint):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    pil = Image.fromarray(synthetic_invoices_u8(1, 720, 1280, seed=77)[0])
    masks0, _ = inf.run_unet(pil, checkpoint)
    for conn in (4, 8):
        masks, inst = inf.run_unet_instances(pil, checkpoint, max_instances=16, connectivity=conn)
        assert list(masks) == inf.FIELDS and all(np.array_equal(masks[f], masks0[f]) for f in inf.FIELDS)
        for f in inf.FIELDS:
            _, n, rows = expected(masks[f], conn, 16)
            want = [(inf._crop_rect(pil.size, tuple(int(v) for v in r[:4])), int(r[4])) for r in rows if r[4] > 0]
            got = [(d["box"], d["pixels"]) for d in inst[f]]
            assert all(g in want for g in got), (f, got, want)
            assert [p for _, p in got] == sorted((p for _, p in got), reverse=True)
            for d in inst[f]:
                x1, y1, x2, y2 = d["box"]
                assert np.array_equal(np.asarray(d["crop"]), np.asarray(pil)[y1:y2, x1:x2])
                assert np.asarray(d["crop"]).mean() >= 3
    _, few = inf.run_unet_instances(pil, checkpoint, max_instances=1, min_pixels=50)
    assert all(len(v) <= 1 and all(d["pixels"] >= 50 for d in v) for v in few.values())


@pytest.mark.gpu
def test_run_unet_instances_constructed_masks(cuda_dev, checkpoint, monkeypatch):
    """Masks with known regions (one region, two regions, none) through both entry points: a one-region field's
    single instance is run_unet's crop; two regions give two crops instead of one spanning both."""
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    pil = Image.fromarray(synthetic_invoices_u8(1, 600, 900, seed=12)[0])
    m = torch.zeros((1, 3, 512, 512), dtype=torch.uint8, device=cuda_dev)
    m[0, 0, 100:140, 60:300] = 1
    m[0, 1, 20:40, 30:90] = 1
    m[0, 1, 400:450, 300:480] = 1
    real = inf._segment_one

    def fake(img, ckpt):
        frame, _ = real(img, ckpt)
        return frame, m.clone()
    monkeypatch.setattr(inf, "_segment_one", fake)
    masks0, crops0 = inf.run_unet(pil, checkpoint)
    masks, inst = inf.run_unet_instances(pil, checkpoint)
    assert all(np.array_equal(masks[f], masks0[f]) for f in inf.FIELDS)
    (one,) = inst["invoice_no"]
    assert one["pixels"] == 40 * 240 and np.array_equal(np.asarray(one["crop"]), np.asarray(crops0["invoice_no"]))
    two = inst["date"]
    assert [d["pixels"] for d in two] == [50 * 180, 20 * 60]
    assert [d["box"] for d in two] == [inf._crop_rect(pil.size, (300, 479, 400, 449)),
                                       inf._crop_rect(pil.size, (30, 89, 20, 39))]
    assert inst["total_amount"] == [] and crops0["total_amount"] is None
