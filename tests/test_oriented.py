"""Oriented boxes of the mask regions and upright crops (unetb200_mask_components_oriented / unetb200_warp_crops /
prepost.mask_components_oriented / prepost.warp_crops / inference.run_unet_instances(deskew=True)).

The oracle (oracle/oriented.py) restates the geometry and the warp in numpy; the CPU tests pin it to OpenCV
(moments, warpAffine) and to np.linalg.eigh (axis), and the device must equal it bit for bit."""

import math

import cv2
import numpy as np
import pytest
import torch
from PIL import Image
from scipy import ndimage

from oracle import oriented as orc
from test_components import SHAPES, expected, patterns

FRAME_SCALE = (1920 / 512, 1080 / 512)


def rotated_bar(h, w, cx, cy, length, width, angle_deg, scale=(1.0, 1.0)):
    """Mask pixels whose frame point ((x + 0.5) sx - 0.5, (y + 0.5) sy - 0.5) lies in the rotated rectangle."""
    sx, sy = scale
    yy, xx = np.mgrid[:h, :w]
    X = (xx + 0.5) * sx - 0.5 - cx
    Y = (yy + 0.5) * sy - 0.5 - cy
    t = math.radians(angle_deg)
    u = X * math.cos(t) + Y * math.sin(t)
    v = -X * math.sin(t) + Y * math.cos(t)
    return (np.abs(u) <= length / 2) & (np.abs(v) <= width / 2)


def extra_patterns(h, w):
    """Bars at angles -85..85, lines (horizontal, vertical, 45 degrees: the a == c case), single pixels, empty."""
    out = {}
    for a in range(-85, 90, 17):
        out[f"bar{a}"] = rotated_bar(h, w, w / 2, h / 2, 0.8 * min(h, w), 0.08 * min(h, w) + 1, a)
    hl = np.zeros((h, w), bool)
    hl[h // 3, 1: w - 1] = True
    out["hline"] = hl
    vl = np.zeros((h, w), bool)
    vl[1: h - 1, w // 4] = True
    out["vline"] = vl
    n = min(h, w)
    d = np.zeros((h, w), bool)
    d[np.arange(n), np.arange(n)] = True
    out["diag45"] = d
    p = np.zeros((h, w), bool)
    p[0, 0] = p[h // 2, w // 2] = p[-1, -1] = True
    out["pixels"] = p
    out["empty"] = np.zeros((h, w), bool)
    return out


# ---------------------------------------------------------------- CPU: the oracle against OpenCV and numpy

def test_oracle_moments_match_cv2():
    rng = np.random.default_rng(5)
    for shape in [(33, 50), (200, 300), (512, 512)]:
        lab, n = ndimage.label(rng.random(shape) < 0.45, np.ones((3, 3), bool))
        for i in range(1, min(n, 40) + 1):
            plane = lab == i
            ys, xs = np.nonzero(plane)
            got = orc.moments(xs, ys)
            m = cv2.moments(plane.astype(np.uint8), binaryImage=True)
            want = (m["m00"], m["m10"], m["m01"], m["m20"], m["m11"], m["m02"])
            assert all(float(g) == w for g, w in zip(got, want)), (shape, i, got, want)
    big = np.ones((1024, 768), np.uint8)
    ys, xs = np.nonzero(big)
    m = cv2.moments(big, binaryImage=True)
    assert orc.moments(xs, ys) == tuple(int(m[k]) for k in ("m00", "m10", "m01", "m20", "m11", "m02"))


def _eigh_axis(mom, sx, sy):
    n, Sx, Sy, Sxx, Sxy, Syy = mom
    a = sx * sx * float(n * Sxx - Sx * Sx)
    b = sx * sy * float(n * Sxy - Sx * Sy)
    c = sy * sy * float(n * Syy - Sy * Sy)
    w, v = np.linalg.eigh(np.array([[a, b], [b, c]]))
    e = v[:, 1]
    if e[0] < 0 or (e[0] == 0 and e[1] < 0):
        e = -e
    return e, w


def test_oracle_axis_matches_eigh():
    h, w = 512, 512
    for scale in [(1.0, 1.0), FRAME_SCALE]:
        for ang in list(range(-89, 91, 7)) + [0, 45, -45, 90]:
            m = rotated_bar(h, w, 960 if scale != (1.0, 1.0) else 256, 540 if scale != (1.0, 1.0) else 256,
                            400, 40, ang, scale)
            ys, xs = np.nonzero(m)
            mom = orc.moments(xs, ys)
            e1 = orc.principal_axis(mom, *scale)
            ref, ev = _eigh_axis(mom, *scale)
            assert ev[1] > 2 * ev[0]
            assert abs(math.hypot(*e1) - 1) < 1e-15
            assert e1[0] > 0 or (e1[0] == 0 and e1[1] > 0)
            assert np.abs(np.array(e1) - ref).max() < 1e-12, (scale, ang, e1, ref)
    # b == 0: the larger diagonal entry wins, ties go to x
    assert orc.principal_axis((3, 3, 0, 5, 0, 0)) == (1.0, 0.0)            # horizontal segment x = 0..2
    assert orc.principal_axis((3, 0, 3, 0, 0, 5)) == (0.0, 1.0)            # vertical
    assert orc.principal_axis((1, 7, 9, 49, 63, 81)) == (1.0, 0.0)         # a single pixel
    # a == c, b != 0: a 45 degree line
    ys = xs = np.arange(10)
    e = orc.principal_axis(orc.moments(xs, ys))
    assert abs(e[0] - math.sqrt(0.5)) < 1e-15 and e[0] == e[1]
    e = orc.principal_axis(orc.moments(xs, 9 - ys))
    assert abs(e[0] - math.sqrt(0.5)) < 1e-15 and e[1] == -e[0]


def _warp_cv2(src, M, w, h):
    return cv2.warpAffine(src, np.asarray(M, np.float64), (w, h), flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP,
                          borderMode=cv2.BORDER_REPLICATE)


def warp_cases(fh, fw, seed):
    """(M, out_w, out_h) of crops at angles -89..90, sub-pixel and integer offsets, inside, across the edges and
    corners, and wholly outside a fw x fh frame."""
    rng = np.random.default_rng(seed)
    out = []
    angles = [-89, -60, -33.3, -10, -1, 0, 0.5, 7, 30, 45, 71.2, 89, 90]
    origins = [(10.3, 20.7), (50, 60), (-40.25, -30.5), (fw - 20.5, fh - 10.125), (fw * 0.5, -25), (-300, fh / 2),
               (fw + 40, fh + 40)]
    for k, ang in enumerate(angles):
        t = math.radians(ang)
        c, s = math.cos(t), math.sin(t)
        for ox, oy in origins:
            w, h = int(rng.integers(1, 160)), int(rng.integers(1, 60))
            out.append((np.array([[c, -s, ox], [s, c, oy]]), w, h))
    return out


def test_oracle_warp_matches_cv2():
    rng = np.random.default_rng(9)
    src = rng.integers(0, 256, (180, 260, 3), dtype=np.uint8)
    src[40:120, 60:200] = np.linspace(0, 255, 140, dtype=np.uint8)[None, :, None]      # smooth ramp too
    diff = total = 0
    for M, w, h in warp_cases(180, 260, 1) + [(np.array([[1.0, 0, 17], [0, 1.0, 23]]), 64, 32)]:
        got = orc.warp_affine(src, M, w, h)
        ref = _warp_cv2(src, M, w, h)
        diff += int((got != ref).sum())
        total += got.size
    assert diff == 0 and total > 100_000
    M = np.array([[1.0, 0.0, 17.0], [0.0, 1.0, 23.0]])                      # integer translation == slicing
    assert np.array_equal(orc.warp_affine(src, M, 64, 32), src[23:55, 17:81])


# ---------------------------------------------------------------- CPU: the crop rule

def test_oriented_crop_rule():
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    r = inf._oriented_crop((1.0, 0.0, 10.0, 109.0, 20.0, 29.0), (1.0, 1.0))
    assert r["size"] == (100.0, 10.0) and r["out_size"] == (130, 13) and r["angle"] == 0.0
    assert np.array_equal(r["M"], [[1.0, -0.0, -5.0], [0.0, 1.0, 18.5]])
    assert r["quad"] == ((-5.5, 18.0), (124.5, 18.0), (124.5, 31.0), (-5.5, 31.0))
    # vertical axis, anisotropic scale: the pixel block is sy long along e1 and sx wide across
    r = inf._oriented_crop((0.0, 1.0, 0.0, 40.0, -30.0, -10.0), (2.0, 3.0))
    assert r["angle"] == 90.0 and r["size"] == (43.0, 22.0) and r["out_size"] == (56, 29)
    M = r["M"]
    centre = M @ np.array([(56 - 1) / 2, (29 - 1) / 2, 1.0])
    assert np.allclose(centre, (20.0, 20.0))                                 # c = 20 e1 + (-20) e2, e2 = (-1, 0)
    # 45 degrees: the crop's centre maps to the box centre; corners half a pixel outside the sample grid
    e = math.sqrt(0.5)
    r = inf._oriented_crop((e, e, 100.0, 300.0, -5.0, 5.0), FRAME_SCALE)
    hu = 0.5 * (e * FRAME_SCALE[0] + e * FRAME_SCALE[1])
    assert r["size"] == (200.0 + 2 * hu, 10.0 + 2 * hu)
    assert r["out_size"] == (math.ceil(1.3 * (200 + 2 * hu)), math.ceil(1.3 * (10 + 2 * hu)))
    ow, oh = r["out_size"]
    assert np.allclose(r["M"] @ np.array([(ow - 1) / 2, (oh - 1) / 2, 1.0]), (200 * e + 0 * -e, 200 * e))
    assert abs(r["angle"] - 45.0) < 1e-12
    q = np.array(r["quad"])
    assert np.allclose(q[1] - q[0], np.array([e, e]) * ow) and np.allclose(q[3] - q[0], np.array([-e, e]) * oh)
    # an empty row (count 0: all zeros) still gives a 1 x 1 crop
    assert inf._oriented_crop((0.0,) * 6, (1.0, 1.0))["out_size"] == (1, 1)


# ---------------------------------------------------------------- CPU: C ABI argument errors

@pytest.fixture(scope="module")
def nat():
    import __graft_entry__ as g
    g.build()
    from tw_invoice_unet_ocr_llm_b200 import _native
    return _native


def test_oriented_workspace_query(nat):
    lib = nat.lib()
    for h, w in SHAPES + [(3, 3), (32767, 1)]:
        for p in (1, 3, 192):
            base = lib.unetb200_components_workspace_bytes(p, h, w)
            got = lib.unetb200_components_oriented_workspace_bytes(p, h, w)
            assert base + 512 * p <= got <= base + 15 + 512 * p, (p, h, w)
    q = lib.unetb200_components_oriented_workspace_bytes
    assert q(1, 32768, 16) == 0 and q(1, 16, 32768) == 0 and q(65536, 16, 16) == 0 and q(0, 16, 16) == 0


def test_c_abi_errors_oriented(nat):
    lib = nat.lib()
    need = lib.unetb200_components_oriented_workspace_bytes(2, 64, 64)
    dev = 1 << 20                                   # never dereferenced: every call below fails validation

    def call(mask=dev, packed=0, planes=2, h=64, w=64, conn=8, k=4, scale=None, labels=None, comps=dev, n=dev,
             mom=dev, obox=dev, ws=dev, ws_bytes=need):
        return lib.unetb200_mask_components_oriented(mask, packed, planes, h, w, conn, k, scale, labels, comps, n,
                                                     mom, obox, ws, ws_bytes, None)

    for kw in (dict(mask=None), dict(comps=None), dict(n=None), dict(ws=None), dict(mom=None), dict(obox=None),
               dict(conn=6), dict(k=0), dict(k=17), dict(planes=0), dict(h=0), dict(w=-3), dict(h=32768),
               dict(w=32768), dict(planes=65536), dict(packed=1, w=48), dict(packed=2), dict(labels=dev + 1),
               dict(comps=dev + 2), dict(ws=dev + 4), dict(mom=dev + 4), dict(obox=dev + 4), dict(scale=dev + 4)):
        assert call(**kw) == nat.EINVAL, kw
        assert nat.last_error().startswith("mask_components_oriented:"), kw
    assert call(ws_bytes=need - 1) == nat.ENOMEM
    assert "oriented_workspace" in nat.last_error()
    # the plain entry point's workspace is too small for the oriented call
    assert call(ws_bytes=lib.unetb200_components_workspace_bytes(2, 64, 64)) == nat.ENOMEM


def _desc(nat, **kw):
    t = nat.WarpCrop()
    t.src, t.src_h, t.src_w, t.src_stride, t.src_pixel_bytes = 1 << 20, 1080, 1920, 1920, 3
    t.m[:] = [1.0, 0.0, 10.0, 0.0, 1.0, 20.0]
    t.out_w, t.out_h, t.out_off = 100, 30, 0
    for k, v in kw.items():
        if k == "m":
            t.m[:] = v
        else:
            setattr(t, k, v)
    return t


def test_c_abi_errors_warp(nat):
    lib = nat.lib()
    dev = 1 << 20

    def call(descs, table_dev=dev, n=None, out=dev, sums=dev):
        tab = (nat.WarpCrop * len(descs))(*descs)
        return lib.unetb200_warp_crops(tab, table_dev, len(descs) if n is None else n, out, sums, None)

    ok = _desc(nat)
    for args in (dict(table_dev=None), dict(out=None), dict(sums=None), dict(n=0), dict(n=-1), dict(n=65536),
                 dict(table_dev=dev + 4), dict(sums=dev + 4)):
        assert call([ok], **args) == nat.EINVAL, args
        assert nat.last_error().startswith("warp_crops:"), args
    assert lib.unetb200_warp_crops(None, dev, 1, dev, dev, None) == nat.EINVAL
    nan, big = float("nan"), float(1 << 19)
    for kw in (dict(src=0), dict(src_h=0), dict(src_w=0), dict(src_w=32768, src_stride=32768), dict(src_stride=1919),
               dict(src_pixel_bytes=1), dict(src_pixel_bytes=2), dict(out_w=0), dict(out_h=-1), dict(out_w=32768),
               dict(m=[1.0, 0.0, big, 0.0, 1.0, 0.0]), dict(m=[1.0, 0.0, 0.0, 0.0, 1.0, -big]),
               dict(m=[600.0, 0.0, 0.0, 0.0, 1.0, 0.0], out_w=1000), dict(m=[1.0, 0.0, 0.0, 0.0, 1e4, 0.0], out_h=60),
               dict(m=[nan, 0.0, 0.0, 0.0, 1.0, 0.0]), dict(m=[1.0, 0.0, float("inf"), 0.0, 1.0, 0.0])):
        assert call([ok, _desc(nat, out_off=9000, **kw)]) == nat.EINVAL, kw
        assert nat.last_error().startswith("warp_crops: crop 1:"), (kw, nat.last_error())
    # the second crop may not start inside the first (100 x 30 x 3 = 9000 bytes)
    assert call([ok, _desc(nat, out_off=8999)]) == nat.EINVAL and "overlaps" in nat.last_error()


def test_python_errors_without_gpu():
    from tw_invoice_unet_ocr_llm_b200 import prepost
    with pytest.raises(RuntimeError):
        prepost.mask_components_oriented(torch.zeros((1, 1, 16, 16), dtype=torch.uint8))          # CPU tensor
    with pytest.raises(RuntimeError):
        prepost.mask_components_oriented(torch.zeros((16, 16), dtype=torch.uint8))
    with pytest.raises(RuntimeError):
        prepost.warp_crops(torch.zeros((16, 16, 3), dtype=torch.uint8), [np.eye(2, 3)], [(4, 4)])  # CPU frame
    with pytest.raises(ValueError):
        prepost.warp_crops(torch.zeros((16, 16, 3), dtype=torch.uint8), [np.eye(2, 3)] * 2, [(4, 4)])


# ---------------------------------------------------------------- GPU: oriented boxes

def run_oriented(batch, dev, scale=None, **kw):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    m = torch.from_numpy(batch.astype(np.uint8)).to(dev)
    return tuple(t.cpu().numpy() for t in prepost.mask_components_oriented(m, scale=scale, labels=True, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("h,w", SHAPES)
def test_oriented_matches_components_and_oracle(cuda_dev, h, w, conn):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    pats = {**patterns(h, w), **extra_patterns(h, w)}
    batch = np.stack(list(pats.values()))[None]
    k = 16
    m = torch.from_numpy(batch.astype(np.uint8)).to(cuda_dev)
    c0, n0, l0 = prepost.mask_components(m, connectivity=conn, max_components=k, labels=True)
    for scale in [None, FRAME_SCALE]:
        c1, n1, mom, obox, l1 = prepost.mask_components_oriented(m, connectivity=conn, max_components=k, scale=scale,
                                                                 labels=True)
        assert torch.equal(c0, c1) and torch.equal(n0, n1) and torch.equal(l0, l1)
        mom, obox, comps, lab = mom.cpu().numpy(), obox.cpu().numpy(), c1.cpu().numpy(), l1.cpu().numpy()
        for j, name in enumerate(pats):
            ref_m, ref_o = orc.oriented_rows(lab[0, j], comps[0, j], scale or (1.0, 1.0))
            assert np.array_equal(mom[0, j], ref_m), (name, scale)
            assert np.array_equal(obox[0, j], ref_o), (name, scale, obox[0, j], ref_o)
            assert np.array_equal(mom[0, j, :, 0], comps[0, j, :, 4])          # n == the component's count
    # the packed input gives the same bits
    if w % 32 == 0:
        bits = torch.from_numpy(np.packbits(batch.astype(np.uint8), axis=-1, bitorder="little")).to(cuda_dev)
        a = prepost.mask_components_oriented(m, connectivity=conn, max_components=k, scale=FRAME_SCALE)
        b = prepost.mask_components_oriented(bits, packed=True, connectivity=conn, max_components=k,
                                             scale=FRAME_SCALE)
        assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.gpu
def test_bar_recovery(cuda_dev):
    """A rasterised 600 x 60 bar in a 1920 x 1080 frame, seen through 512 x 512 masks: angle within 0.5 degrees,
    length and width within two mask pixel blocks."""
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    sx, sy = FRAME_SCALE
    angles = [-88, -60, -40, -20, -5, 0, 3, 10, 30, 45, 60, 75, 88, 90]
    batch = np.stack([rotated_bar(512, 512, 960, 540, 600, 60, a, FRAME_SCALE) for a in angles])[None]
    comps, n, mom, obox, lab = run_oriented(batch, cuda_dev, scale=FRAME_SCALE, max_components=1)
    tol = 2 * max(sx, sy)
    for j, a in enumerate(angles):
        assert n[0, j] == 1
        r = inf._oriented_crop(obox[0, j, 0], FRAME_SCALE)
        err = (r["angle"] - a + 90) % 180 - 90
        assert abs(err) < 0.5, (a, r["angle"])
        assert abs(r["size"][0] - 600) <= tol and abs(r["size"][1] - 60) <= tol, (a, r["size"])


@pytest.mark.gpu
def test_oriented_batch_independence_and_determinism(cuda_dev):
    pats = {**patterns(33, 50), **extra_patterns(33, 50)}
    batch = np.stack(list(pats.values()))
    batch = batch[: batch.shape[0] // 2 * 2].reshape(2, -1, 33, 50)
    scales = np.array([[3.75, 2.1], [1.5, 0.75]])
    full = run_oriented(batch, cuda_dev, scale=scales, max_components=16)
    again = run_oriented(batch, cuda_dev, scale=scales, max_components=16)
    assert all(np.array_equal(a, b) for a, b in zip(full, again))
    for idx in np.ndindex(batch.shape[:2]):
        one = run_oriented(batch[idx][None, None], cuda_dev, scale=tuple(scales[idx[0]]), max_components=16)
        assert all(np.array_equal(o[0, 0], f[idx]) for o, f in zip(one, full)), idx


# ---------------------------------------------------------------- GPU: warp

def _frames(n, seed, h=1080, w=1920):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        f = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        f[100:900, 200:1700] = (np.arange(1500, dtype=np.uint16)[None, :, None] % 256).astype(np.uint8)
        out.append(f)
    return out


@pytest.mark.gpu
def test_warp_matches_oracle_ragged_batch(cuda_dev):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    hosts = _frames(3, 4)
    dev_rgb = [torch.from_numpy(f).to(cuda_dev) for f in hosts]
    rgbx = [np.concatenate([f, np.full(f.shape[:2] + (1,), 77, np.uint8)], axis=2) for f in hosts]
    dev_rgbx = [torch.from_numpy(f).to(cuda_dev) for f in rgbx]
    cases = warp_cases(1080, 1920, 2)
    rng = np.random.default_rng(6)
    for k in range(20):                                     # larger crops inside the frame
        t = math.radians(rng.uniform(-89, 90))
        M = np.array([[math.cos(t), -math.sin(t), rng.uniform(300, 1500)],
                      [math.sin(t), math.cos(t), rng.uniform(200, 800)]])
        cases.append((M, int(rng.integers(100, 700)), int(rng.integers(20, 120))))
    assert len(cases) >= 64
    which = [k % 3 for k in range(len(cases))]
    for frames in (dev_rgb, dev_rgbx):
        crops, sums = prepost.warp_crops([frames[i] for i in which], [c[0] for c in cases],
                                         [(c[1], c[2]) for c in cases])
        sums = sums.cpu().numpy()
        for k, ((M, w, h), crop) in enumerate(zip(cases, crops)):
            ref = orc.warp_affine(hosts[which[k]], M, w, h)
            got = crop.cpu().numpy()
            assert got.shape == (h, w, 3) and np.array_equal(got, ref), (k, int((got != ref).sum()))
            assert sums[k] == int(ref.astype(np.int64).sum())
        # a crop alone gives the same bits
        one, s1 = prepost.warp_crops(frames[which[5]], [cases[5][0]], [cases[5][1:]])
        assert torch.equal(one[0], crops[5]) and int(s1[0]) == sums[5]
        again, s2 = prepost.warp_crops([frames[i] for i in which], [c[0] for c in cases], [(c[1], c[2]) for c in cases])
        assert all(torch.equal(a, b) for a, b in zip(again, crops)) and np.array_equal(s2.cpu().numpy(), sums)
    # integer translation == slicing; against OpenCV itself too
    M = np.array([[1.0, 0.0, 333.0], [0.0, 1.0, 222.0]])
    (c,), _ = prepost.warp_crops(dev_rgbx[1], [M], [(400, 50)])
    assert np.array_equal(c.cpu().numpy(), hosts[1][222:272, 333:733])
    M, w, h = cases[-1]
    (c,), _ = prepost.warp_crops(dev_rgb[0], [M], [(w, h)])
    assert np.array_equal(c.cpu().numpy(), _warp_cv2(hosts[0], M, w, h))


@pytest.mark.gpu
def test_python_argument_errors(cuda_dev):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200._native import UnetB200Error
    m = torch.zeros((2, 3, 32, 32), dtype=torch.uint8, device=cuda_dev)
    for kw in (dict(connectivity=6), dict(max_components=0), dict(max_components=17)):
        with pytest.raises(RuntimeError):
            prepost.mask_components_oriented(m, **kw)
    for sc in ((1.0,), (1.0, 0.0), (-1.0, 1.0), (float("nan"), 1.0), np.ones((3, 2)), np.ones((2, 2, 2))):
        with pytest.raises(ValueError):
            prepost.mask_components_oriented(m, scale=sc)
    with pytest.raises(RuntimeError):
        prepost.mask_components_oriented(torch.zeros((1, 1, 32768, 1), dtype=torch.uint8, device=cuda_dev))
    f = torch.zeros((64, 64, 3), dtype=torch.uint8, device=cuda_dev)
    eye = np.array([[1.0, 0, 0], [0, 1.0, 0]])
    with pytest.raises(ValueError):
        prepost.warp_crops(f, [eye], [(4, 4), (4, 4)])
    with pytest.raises(ValueError):
        prepost.warp_crops(f, [], [])
    with pytest.raises(RuntimeError):
        prepost.warp_crops(f.float(), [eye], [(4, 4)])
    with pytest.raises(RuntimeError):
        prepost.warp_crops(f[:, :, :2].contiguous(), [eye], [(4, 4)])
    with pytest.raises(UnetB200Error):
        prepost.warp_crops(f, [eye], [(0, 4)])
    with pytest.raises(UnetB200Error):
        prepost.warp_crops(f, [[[1.0, 0, 6e5], [0, 1.0, 0]]], [(4, 4)])


# ---------------------------------------------------------------- GPU: run_unet_instances(deskew=True)

@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory, fixture_state):
    import os
    path = os.path.join(tmp_path_factory.mktemp("ckpt"), "best_unet_model.pth")
    torch.save(fixture_state, path)
    return path


def host_instances(pil, masks, k, conn=8, min_pixels=1):
    """Host recomputation of run_unet_instances(deskew=True): scipy labels, oracle geometry, the crop rule,
    cv2.warpAffine on the PIL frame and the near-black test."""
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    scale = (pil.size[0] / 512, pil.size[1] / 512)
    rgb = np.asarray(pil.convert("RGB"))
    out = {}
    for f in inf.FIELDS:
        lab, _, rows = expected(masks[f], conn, k)
        _, obox = orc.oriented_rows(lab, rows, scale)
        lst = []
        for row, ob in zip(rows, obox):
            if row[4] == 0 or row[4] < min_pixels:
                continue
            box = inf._crop_rect(pil.size, tuple(int(v) for v in row[:4]))
            if box is None:
                continue
            oc = inf._oriented_crop(ob, scale)
            crop = _warp_cv2(rgb, oc["M"], *oc["out_size"])
            if crop.mean() < 3:
                continue
            lst.append({"box": box, "pixels": int(row[4]), "crop": crop, "quad": oc["quad"], "angle": oc["angle"],
                        "size": oc["size"]})
        out[f] = lst
    return out


def assert_same_instances(got, want):
    assert list(got) == list(want)
    for f in want:
        assert len(got[f]) == len(want[f]), f
        for g, w in zip(got[f], want[f]):
            assert g["box"] == w["box"] and g["pixels"] == w["pixels"]
            assert g["quad"] == w["quad"] and g["angle"] == w["angle"] and g["size"] == w["size"]
            assert g["crop"].mode == "RGB" and np.array_equal(np.asarray(g["crop"]), w["crop"]), f


def assert_enhanced(inst):
    from tw_invoice_unet_ocr_llm_b200 import enhance, inference as inf
    items = [(f, d) for f, lst in inst.items() for d in lst]
    ref = enhance.enhance_batch([d["crop"] for _, d in items], [inf.ENHANCE_KINDS[f] for f, _ in items])
    for (_, d), r in zip(items, ref):
        assert d["enhanced"].mode == "L" and np.array_equal(np.asarray(d["enhanced"]), r)


@pytest.mark.gpu
def test_run_unet_instances_deskew_on_fixture(cuda_dev, checkpoint):
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    pil = Image.fromarray(synthetic_invoices_u8(1, 1080, 1920, seed=77)[0])
    masks0, inst0 = inf.run_unet_instances(pil, checkpoint, max_instances=8)
    masks1, inst1 = inf.run_unet_instances(pil, checkpoint, max_instances=8, deskew=False, enhance=False)
    assert all(np.array_equal(masks0[f], masks1[f]) for f in inf.FIELDS)
    for f in inf.FIELDS:
        assert [(d["box"], d["pixels"]) for d in inst0[f]] == [(d["box"], d["pixels"]) for d in inst1[f]]
        assert all(np.array_equal(np.asarray(a["crop"]), np.asarray(b["crop"])) for a, b in zip(inst0[f], inst1[f]))
        assert all(set(d) == {"box", "pixels", "crop"} for d in inst1[f])
    masks, inst = inf.run_unet_instances(pil, checkpoint, max_instances=8, deskew=True, enhance=True)
    assert all(np.array_equal(masks[f], masks0[f]) for f in inf.FIELDS)
    assert sum(len(v) for v in inst.values()) > 0
    assert_same_instances(inst, host_instances(pil, masks, 8))
    assert_enhanced(inst)
    # enhancement of the axis-aligned crops reads the frame windows
    _, inst_e = inf.run_unet_instances(pil, checkpoint, max_instances=8, enhance=True)
    assert_enhanced(inst_e)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["RGB", "L"])
def test_run_unet_instances_deskew_constructed(cuda_dev, checkpoint, monkeypatch, mode):
    """Tilted bars with known angles through run_unet_instances(deskew=True): the host recomputation, the angles,
    and upright crops of a frame with a tilted printed strip."""
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    pil = Image.fromarray(synthetic_invoices_u8(1, 1080, 1920, seed=12)[0]).convert(mode)
    sc = (1920 / 512, 1080 / 512)
    m = np.zeros((1, 3, 512, 512), np.uint8)
    m[0, 0] = rotated_bar(512, 512, 600, 300, 600, 60, 10, sc)
    m[0, 1] = rotated_bar(512, 512, 1400, 700, 400, 50, -25, sc) | rotated_bar(512, 512, 400, 800, 300, 40, 80, sc)
    md = torch.from_numpy(m).to(cuda_dev)
    real = inf._segment_one

    def fake(img, ckpt):
        frame, _ = real(img, ckpt)
        return frame, md.clone()
    monkeypatch.setattr(inf, "_segment_one", fake)
    masks, inst = inf.run_unet_instances(pil, checkpoint, deskew=True, enhance=True)
    assert_same_instances(inst, host_instances(pil, masks, 4))
    assert_enhanced(inst)
    assert len(inst["invoice_no"]) == 1 and abs(inst["invoice_no"][0]["angle"] - 10) < 0.5
    assert sorted(round(d["angle"]) for d in inst["date"]) == [-25, 80]
    assert inst["total_amount"] == []
    (one,) = inst["invoice_no"]
    assert abs(one["size"][0] - 600) < 8 and abs(one["size"][1] - 60) < 8
    assert len(one["quad"]) == 4
    masks0, inst0 = inf.run_unet_instances(pil, checkpoint)
    assert [(d["box"], d["pixels"]) for d in inst0["invoice_no"]] == [(one["box"], one["pixels"])]
