"""Scoring masks against ground truth (unetb200_mask_match / prepost.mask_match / inference.evaluate_masks).  The
oracle is oracle/mask_match.py (scipy.ndimage.label, pair codes, the same float64 operations and summation order);
on the CPU it is checked against a brute-force loop over all region pairs, and on the GPU every integer output and
iou_sum must be np.array_equal with it."""

import math
import os

import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import mask_match as om


# ---------------------------------------------------------------- helpers

def brute_force(pred, gt, conn=8, min_pixels=1, iou=0.5):
    """Every (pred region, gt region) pair by a Python loop; iou_sum in the device's order."""
    st = om.structure(conn)
    lp, n_p = ndimage.label(pred != 0, st)
    lg, n_g = ndimage.label(gt != 0, st)
    p, g = pred != 0, gt != 0
    tp = sum_i = sum_u = kept = 0
    ids, qs = [], []
    for a in range(1, n_p + 1):
        ma = lp == a
        na = int(ma.sum())
        if na < min_pixels:
            continue
        kept += 1
        partners = []
        for b in range(1, n_g + 1):
            mb = lg == b
            i = int((ma & mb).sum())
            u = na + int(mb.sum()) - i
            if i > 0 and float(i) > iou * float(u):
                partners.append((i, u))
        assert len(partners) <= 1
        for i, u in partners:
            tp, sum_i, sum_u = tp + 1, sum_i + i, sum_u + u
            ids.append(a - 1)
            qs.append(i / u)
    counts = np.array([(p & g).sum(), (p & ~g).sum(), (~p & g).sum(), kept, n_g, tp, sum_i, sum_u], np.int64)
    partial = np.zeros(256)
    for a, q in sorted(zip(ids, qs)):
        partial[a % 256] += q
    return counts, om.tree_sum(partial)


def pack_bits(m):
    return np.packbits(np.ascontiguousarray(m).astype(np.uint8), axis=-1, bitorder="little")


def blobs(rng, h, w, n, rmax=6):
    m = np.zeros((h, w), np.uint8)
    for _ in range(n):
        cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(1, rmax + 1)
        yy, xx = np.ogrid[:h, :w]
        m[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 1
    return m


def checker(h, w, conn):
    yy, xx = np.mgrid[:h, :w]
    if conn == 8:                      # isolated pixels on a 2-pixel grid: the most 8-connected regions
        return ((yy % 2 == 0) & (xx % 2 == 0)).astype(np.uint8)
    return ((xx + yy) % 2 == 0).astype(np.uint8)      # every pixel its own 4-connected region


def pair_set(h, w, seed):
    """(name, pred, gt) plane pairs of one shape."""
    rng = np.random.default_rng(seed * 7919 + h * 131 + w)
    out = []
    b = blobs(rng, h, w, max(1, h * w // 200))
    out.append(("blobs", b, blobs(rng, h, w, max(1, h * w // 200))))
    out.append(("blobs_shifted", b, np.roll(b, 1, axis=1)))
    out.append(("same", b, b.copy()))
    out.append(("noise", (rng.random((h, w)) < 0.5).astype(np.uint8), (rng.random((h, w)) < 0.5).astype(np.uint8)))
    out.append(("checker4", checker(h, w, 4), (rng.random((h, w)) < 0.5).astype(np.uint8)))
    out.append(("checker8", checker(h, w, 8), np.roll(checker(h, w, 8), 1, axis=0)))
    out.append(("empty_pred", np.zeros((h, w), np.uint8), b))
    out.append(("empty_gt", b, np.zeros((h, w), np.uint8)))
    return out


# ---------------------------------------------------------------- CPU: the oracle

@pytest.mark.parametrize("conn", [4, 8])
def test_oracle_matches_brute_force(conn):
    rng = np.random.default_rng(conn)
    for trial in range(40):
        h, w = int(rng.integers(1, 24)), int(rng.integers(1, 24))
        d = rng.random()
        pred = (rng.random((h, w)) < d).astype(np.uint8)
        gt = pred.copy() if trial % 5 == 0 else (rng.random((h, w)) < rng.random()).astype(np.uint8)
        if trial % 3 == 0:
            gt = blobs(rng, h, w, 3, 4)
        for iou in (0.5, 0.75, 0.999):
            for mp in (1, 3):
                c, s = om.match_plane(pred, gt, conn, mp, iou)
                bc, bs = brute_force(pred, gt, conn, mp, iou)
                assert np.array_equal(c, bc) and s == bs, (trial, iou, mp)


def plane(h, w, *rects):
    m = np.zeros((h, w), np.uint8)
    for y0, y1, x0, x1 in rects:
        m[y0:y1, x0:x1] = 1
    return m


def test_oracle_edge_cases():
    # IoU exactly t does not match: a 2-pixel gt region holding a 1-pixel pred region is 0.5
    c, s = om.match_plane(plane(4, 8, (1, 2, 1, 2)), plane(4, 8, (1, 2, 1, 3)), iou=0.5)
    assert c.tolist() == [1, 0, 1, 1, 1, 0, 0, 0] and s == 0.0
    # IoU 3/4 against t = 0.75 (no match) and one ulp below it (match)
    pred, gt = plane(4, 8, (1, 2, 1, 4)), plane(4, 8, (1, 2, 1, 5))
    assert om.match_plane(pred, gt, iou=0.75)[0][5] == 0
    c, s = om.match_plane(pred, gt, iou=float(np.nextafter(0.75, 0.0)))
    assert c.tolist() == [3, 0, 1, 1, 1, 1, 3, 4] and s == 0.75
    # one pred region over two gt regions (and the reverse): at most one partner, the one holding > half
    big, two = plane(3, 12, (1, 2, 0, 12)), plane(3, 12, (1, 2, 0, 8), (1, 2, 9, 12))
    c, s = om.match_plane(big, two)
    assert c.tolist() == [11, 1, 0, 1, 2, 1, 8, 12] and s == 8 / 12
    c, s = om.match_plane(two, big)
    assert c.tolist() == [11, 0, 1, 2, 1, 1, 8, 12] and s == 8 / 12
    # min_pixels at the size of a region keeps it, one above drops it (and only the pred side)
    pred = plane(4, 8, (0, 2, 0, 2), (3, 4, 6, 8))
    assert om.match_plane(pred, pred, min_pixels=4)[0].tolist() == [6, 0, 0, 1, 2, 1, 4, 4]
    assert om.match_plane(pred, pred, min_pixels=5)[0].tolist() == [6, 0, 0, 0, 2, 0, 0, 0]
    # empty planes on either side
    z = np.zeros((5, 5), np.uint8)
    assert om.match_plane(z, z)[0].tolist() == [0] * 8
    assert om.match_plane(pred[:, :5], z[:4])[0].tolist() == [0, 4, 0, 1, 0, 0, 0, 0]
    assert om.match_plane(z[:4], pred[:, :5])[0].tolist() == [0, 0, 4, 0, 1, 0, 0, 0]
    # t = 0.999: only a near-identical region matches
    a, b = plane(40, 40, (0, 40, 0, 40)), plane(40, 40, (0, 40, 0, 40))
    b[0, 0] = 0
    assert om.match_plane(a, b, iou=0.999)[0][5] == 1          # 1599 / 1600 = 0.999375
    b[0, 1] = 0
    assert om.match_plane(a, b, iou=0.999)[0][5] == 0          # 1598 / 1600 = 0.99875
    for bad in (0.49, 1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            om.match_plane(a, a, iou=bad)


def test_oracle_iou_sum_order():
    """The device's order: partial sum j of ids j, j + 256, ..., then the pairwise tree; pred == gt sums to tp."""
    m = checker(64, 64, 8)                                          # 1024 one-pixel regions
    c, s = om.match_plane(m, m)
    assert c[5] == 1024 and s == 1024.0
    ids = np.arange(700)
    q = 1.0 / (ids + 3.0)
    partial = np.zeros(256)
    for a in ids:
        partial[a % 256] = partial[a % 256] + q[a]
    assert om.ordered_iou_sum(ids, q) == om.tree_sum(partial)
    assert om.ordered_iou_sum(ids[::-1].copy(), q[::-1].copy()) == om.tree_sum(partial)


# ---------------------------------------------------------------- CPU: the C ABI without a GPU

@pytest.fixture(scope="module")
def nat():
    import __graft_entry__ as g
    g.build()
    from tw_invoice_unet_ocr_llm_b200 import _native
    return _native


def test_workspace_query(nat):
    lib = nat.lib()
    for p, h, w in [(1, 1, 1), (3, 63, 33), (192, 512, 512), (1, 1080, 1920)]:
        cw = lib.unetb200_components_workspace_bytes(p, h, w)
        rows = p * ((h * w + 1) // 2)
        assert lib.unetb200_match_workspace_bytes(p, h, w) == 2 * ((cw + 15) // 16 * 16) + 12 * rows + 8 * p
    q = lib.unetb200_match_workspace_bytes
    assert q(0, 16, 16) == 0 and q(1, 0, 16) == 0 and q(1, 16, -1) == 0 and q(1, 1 << 16, 1 << 15) == 0


def test_c_abi_errors(nat):
    lib = nat.lib()
    dev = 1 << 20                                   # never dereferenced: every call below fails validation

    def call(pred=dev, pp=0, gt=dev + (1 << 16), gp=0, planes=2, h=64, w=64, conn=8, mp=1, t=0.5,
             counts=dev + (1 << 17), sums=dev + (1 << 17) + 4096, ws=dev + (1 << 18), ws_bytes=None):
        if ws_bytes is None:
            ws_bytes = lib.unetb200_match_workspace_bytes(2, 64, 64)
        return lib.unetb200_mask_match(pred, pp, gt, gp, planes, h, w, conn, mp, t, counts, sums, ws, ws_bytes, None)

    cases = [(dict(pred=None), "null pointer"), (dict(gt=None), "null pointer"), (dict(counts=None), "null pointer"),
             (dict(sums=None), "null pointer"), (dict(ws=None), "null pointer"),
             (dict(pp=2), "0 or 1"), (dict(gp=-1), "0 or 1"),
             (dict(conn=6), "connectivity"), (dict(conn=0), "connectivity"),
             (dict(mp=0), "min_pixels"), (dict(mp=-5), "min_pixels"),
             (dict(t=0.4999999), "iou_threshold"), (dict(t=1.0), "iou_threshold"), (dict(t=-0.5), "iou_threshold"),
             (dict(t=float("nan")), "iou_threshold"), (dict(t=float("inf")), "iou_threshold"),
             (dict(planes=0), "bad size"), (dict(h=0), "bad size"), (dict(w=-3), "bad size"),
             (dict(h=1 << 16, w=1 << 15), "bad size"),
             (dict(pp=1, w=48), "w % 32"), (dict(gp=1, w=100), "w % 32"),
             (dict(pp=1, pred=dev + 2), "misaligned"), (dict(gp=1, gt=dev + 1), "misaligned"),
             (dict(counts=dev + (1 << 17) + 4), "misaligned"), (dict(sums=dev + (1 << 17) + 4100), "misaligned"),
             (dict(ws=dev + (1 << 18) + 8), "misaligned")]
    for kw, msg in cases:
        assert call(**kw) == nat.EINVAL, kw
        err = nat.last_error()
        assert err.startswith("mask_match: ") and msg in err, (kw, err)
    need = lib.unetb200_match_workspace_bytes(2, 64, 64)
    # byte planes at any alignment, every flag combination and the threshold range: these reach the workspace check
    for kw in (dict(), dict(pred=dev + 1, gt=dev + 3), dict(pp=1, gp=1), dict(pp=1), dict(gp=1, conn=4),
               dict(t=0.999), dict(t=float(np.nextafter(1.0, 0.0))), dict(mp=1 << 30)):
        assert call(ws_bytes=need - 1, **kw) == nat.ENOMEM, kw
        assert "workspace smaller than unetb200_match_workspace_bytes" in nat.last_error()


def test_python_errors_without_gpu(tmp_path):
    from PIL import Image  # noqa: F401
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200 import prepost
    m = torch.zeros((1, 1, 32, 32), dtype=torch.uint8)
    with pytest.raises(RuntimeError):
        prepost.mask_match(m, m)                                    # CPU tensors
    missing = str(tmp_path / "no_such_checkpoint.pth")              # never opened: the steps fail first
    x = torch.zeros((1, 3, 32, 32))
    for clean in ("open", [("open", 3)], [("opening", (3, 3))], ["fill"], [("open", (3, 64))]):
        with pytest.raises(ValueError):
            inf.evaluate_masks(missing, x, x, clean=clean)


def test_match_metrics():
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    c = dict(px_tp=6, px_fp=2, px_fn=4, n_pred=4, n_gt=3, tp=2, sum_inter=5, sum_union=7)
    r = inf._match_metrics(c, 1.5)
    assert r["pixel_iou"] == 6 / 12 and r["dice"] == 12 / 18 and r["pixel_precision"] == 6 / 8
    assert r["pixel_recall"] == 6 / 10 and r["precision"] == 2 / 4 and r["recall"] == 2 / 3
    assert r["f1"] == 4 / 7 and r["sq"] == 0.75 and r["rq"] == 2 / 3.5 and r["pq"] == 1.5 / 3.5
    assert r["iou_sum"] == 1.5 and all(r[k] == v for k, v in c.items())
    z = inf._match_metrics(dict.fromkeys(c, 0), 0.0)
    assert all(z[k] is None for k in ("pixel_iou", "dice", "pixel_precision", "pixel_recall", "precision", "recall",
                                      "f1", "sq", "rq", "pq"))
    r = inf._match_metrics(dict(c, tp=0, sum_inter=0, sum_union=0), 0.0)
    assert r["sq"] is None and r["pq"] == 0.0 and r["rq"] == 0.0


# ---------------------------------------------------------------- GPU: against the oracle

def run_match(pred, gt, dev, pred_packed=False, gt_packed=False, **kw):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    p = torch.from_numpy(pack_bits(pred) if pred_packed else pred).to(dev)
    g = torch.from_numpy(pack_bits(gt) if gt_packed else gt).to(dev)
    c, s = prepost.mask_match(p, g, pred_packed=pred_packed, gt_packed=gt_packed, **kw)
    return c.cpu().numpy(), s.cpu().numpy()


def check_batch(pred, gt, dev, conn=8, mp=1, iou=0.5, combos=((False, False),)):
    want_c, want_s = om.mask_match(pred, gt, conn, mp, iou)
    for pp, gp in combos:
        c, s = run_match(pred, gt, dev, pp, gp, connectivity=conn, min_pixels=mp, iou=iou)
        bad = [idx for idx in np.ndindex(pred.shape[:2])
               if not (np.array_equal(c[idx], want_c[idx]) and np.array_equal(s[idx], want_s[idx]))]
        assert bad == [], (pp, gp, conn, mp, iou, bad[:5], c[bad[0]] if bad else None,
                           want_c[bad[0]] if bad else None)
    return want_c, want_s


ALL_COMBOS = ((False, False), (True, False), (False, True), (True, True))


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(1, 1), (1, 33), (1, 4097), (7, 5), (31, 100), (64, 64), (96, 160), (512, 512),
                                 (1080, 1920)])
def test_matches_oracle(cuda_dev, h, w):
    pairs = pair_set(h, w, seed=1)
    pred = np.stack([p for _, p, _ in pairs])[None]
    gt = np.stack([g for _, _, g in pairs])[None]
    combos = ALL_COMBOS if w % 32 == 0 else ((False, False),)
    for conn in (4, 8):
        for iou in (0.5, 0.75, 0.999):
            for mp in (1, 50):
                want_c, _ = check_batch(pred, gt, cuda_dev, conn, mp, iou,
                                        combos if (iou, mp) == (0.5, 1) else ((False, False),))
    names = [n for n, _, _ in pairs]
    c, s = run_match(pred, gt, cuda_dev)
    same = names.index("same")
    assert c[0, same, 5] == c[0, same, 3] == c[0, same, 4] and s[0, same] == c[0, same, 5]
    if h * w >= 64:
        assert c[0, :, 5].sum() > 0


@pytest.mark.gpu
def test_checkerboards_every_region(cuda_dev):
    """The most regions a plane can have, matched one by one: pred == gt and gt shifted by one pixel."""
    for conn in (4, 8):
        m = checker(512, 512, conn)
        pred = np.stack([m, m, m])[None]
        gt = np.stack([m, np.roll(m, 1, axis=1), np.roll(m, 1, axis=0)])[None]
        want_c, want_s = check_batch(pred, gt, cuda_dev, conn, combos=ALL_COMBOS)
        assert want_c[0, 0, 5] == want_c[0, 0, 3] and want_s[0, 0] == want_c[0, 0, 5]
        assert want_c[0, 0, 3] == (512 * 512 // 2 if conn == 4 else 256 * 256)


@pytest.mark.gpu
def test_past_one_megapixel(cuda_dev):
    """One 1100 x 1024 plane: more than 1024 root-count segments, so the segment scan takes several rounds."""
    rng = np.random.default_rng(3)
    b = blobs(rng, 1100, 1024, 3000, 9)
    g = np.roll(b, 2, axis=0)
    g[rng.random(g.shape) < 0.02] ^= 1
    pred = np.stack([b, (rng.random(b.shape) < 0.5).astype(np.uint8)])[None]
    gt = np.stack([g, (rng.random(b.shape) < 0.5).astype(np.uint8)])[None]
    for conn in (4, 8):
        for iou in (0.5, 0.75):
            check_batch(pred, gt, cuda_dev, conn, 1, iou, ALL_COMBOS if iou == 0.5 else ((False, False),))


@pytest.mark.gpu
def test_edge_cases_on_device(cuda_dev):
    cases = [(plane(4, 8, (1, 2, 1, 2)), plane(4, 8, (1, 2, 1, 3)), 0.5),
             (plane(4, 8, (1, 2, 1, 4)), plane(4, 8, (1, 2, 1, 5)), 0.75),
             (plane(4, 8, (1, 2, 1, 4)), plane(4, 8, (1, 2, 1, 5)), float(np.nextafter(0.75, 0.0))),
             (plane(3, 12, (1, 2, 0, 12)), plane(3, 12, (1, 2, 0, 8), (1, 2, 9, 12)), 0.5),
             (plane(3, 12, (1, 2, 0, 8), (1, 2, 9, 12)), plane(3, 12, (1, 2, 0, 12)), 0.5)]
    for pred, gt, t in cases:
        check_batch(pred[None, None], gt[None, None], cuda_dev, 8, 1, t)
    pred = plane(4, 8, (0, 2, 0, 2), (3, 4, 6, 8))
    for mp in (4, 5):
        check_batch(pred[None, None], pred[None, None], cuda_dev, 8, mp, 0.5)


@pytest.mark.gpu
def test_batch_independence_and_determinism(cuda_dev):
    rng = np.random.default_rng(9)
    pred = np.stack([np.stack([blobs(rng, 40, 100, int(rng.integers(1, 40))) for _ in range(3)])
                     for _ in range(64)])
    gt = np.stack([np.stack([np.roll(pred[i, c], int(rng.integers(-2, 3)), axis=c % 2) for c in range(3)])
                   for i in range(64)])
    gt[rng.random(gt.shape) < 0.01] ^= 1
    c0, s0 = run_match(pred, gt, cuda_dev)
    c1, s1 = run_match(pred, gt, cuda_dev)
    assert np.array_equal(c0, c1) and np.array_equal(s0, s1)
    for idx in [(0, 0), (17, 2), (63, 1), (40, 0)]:
        c, s = run_match(pred[idx][None, None], gt[idx][None, None], cuda_dev)
        assert np.array_equal(c[0, 0], c0[idx]) and np.array_equal(s[0, 0], s0[idx]), idx
    want_c, want_s = om.mask_match(pred, gt)
    assert np.array_equal(c0, want_c) and np.array_equal(s0, want_s)


# ---------------------------------------------------------------- GPU: evaluate_masks on the trained stand-in

@pytest.fixture(scope="module")
def trained(cuda_dev, tmp_path_factory):
    from tw_invoice_unet_ocr_llm_b200.synthetic import train_fixture_state
    state, _ = train_fixture_state(cuda_dev, steps=300, seed=0)
    path = os.path.join(tmp_path_factory.mktemp("ckpt"), "trained.pth")
    torch.save(state, path)
    return state, path


def host_clean(m, steps):
    import cv2
    ops = {"open": cv2.MORPH_OPEN, "close": cv2.MORPH_CLOSE, "erode": cv2.MORPH_ERODE, "dilate": cv2.MORPH_DILATE}
    for step in steps:
        if step == "fill_holes":
            m = ndimage.binary_fill_holes(m != 0).astype(np.uint8)
        else:
            kw, kh = step[1]
            m = cv2.morphologyEx(np.ascontiguousarray(m, np.uint8), ops[step[0]], np.ones((kh, kw), np.uint8))
    return m


def host_scores(masks, gt, steps, conn, mp, iou):
    """Host masks -> cv2 / scipy clean-up -> the oracle -> what evaluate_masks returns."""
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    n = masks.shape[0]
    cleaned = np.stack([np.stack([host_clean(masks[i, c], steps) for c in range(3)]) for i in range(n)])
    c, s = om.mask_match(cleaned, gt, conn, mp, iou)
    return {f: inf._match_metrics(dict(zip(om.FIELDS, c[:, k].sum(axis=0).tolist())), math.fsum(s[:, k].tolist()))
            for k, f in enumerate(inf.FIELDS)}


@pytest.mark.gpu
def test_evaluate_masks_matches_oracle(cuda_dev, trained):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import marked_invoices
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    state, path = trained
    x, gt = marked_invoices(70, 512, seed=311)                      # two chunks: 64 + 6
    gt_u8 = gt.numpy().astype(np.uint8)
    thr = [inf.THRESHOLDS[f] for f in inf.FIELDS]
    eng = Engine(state, cuda_dev)
    _, m = eng.run(x.to(cuda_dev), want_logits=False, thresholds=thr)
    masks = m.cpu().numpy()
    model = UNet(3, 3)
    model.load_state_dict(state)
    model = model.to(cuda_dev).eval()
    x_u8 = torch.round(x * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    steps_list = [None, [("open", (3, 3))], [("close", (9, 3)), "fill_holes", ("open", (3, 3))]]
    for steps in steps_list:
        for conn, mp, iou in ((8, 1, 0.5), (4, 20, 0.75)):
            want = host_scores(masks, gt_u8, steps or [], conn, mp, iou)
            got = inf.evaluate_masks(model, x, gt, clean=steps, connectivity=conn, min_pixels=mp, iou=iou)
            assert got == want, (steps, conn, mp, iou)
            if steps is None and conn == 8:
                assert all(got[f]["tp"] > 0 for f in inf.FIELDS)
                # uint8 NHWC frames with the same values, and the checkpoint path, give the same result
                assert inf.evaluate_masks(model, x_u8, gt, connectivity=conn, min_pixels=mp, iou=iou) == got
                assert inf.evaluate_masks(path, x.to(cuda_dev), gt.to(cuda_dev), connectivity=conn,
                                          min_pixels=mp, iou=iou) == got
    # other thresholds, as a dict and as a list
    t2 = {"invoice_no": 0.5, "date": 0.6, "total_amount": 0.2}
    _, m2 = eng.run(x.to(cuda_dev), want_logits=False, thresholds=[t2[f] for f in inf.FIELDS])
    want = host_scores(m2.cpu().numpy(), gt_u8, [], 8, 1, 0.5)
    assert inf.evaluate_masks(model, x, gt, thresholds=t2) == want
    assert inf.evaluate_masks(model, x, gt, thresholds=[t2[f] for f in inf.FIELDS]) == want


@pytest.mark.gpu
def test_evaluate_masks_bad_clean_before_gpu_work(cuda_dev, trained):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    _, path = trained
    x = torch.zeros((2, 3, 64, 64), device=cuda_dev)
    torch.cuda.synchronize()
    for clean in ([("open", (3, 0))], [("fill_holes", (3, 3))], "fill_holes"):
        with pytest.raises(ValueError):
            inf.evaluate_masks(path, x, x, clean=clean)
