"""Labelling and oriented boxes past one megapixel (unetb200_mask_components / _oriented, DESIGN.md 6b).

Two parts of csrc/components.cu only do real work on large planes:

* cc_scan_kernel scans the per-plane root counts of the 1024-pixel segments in rounds of 1024 segments and carries
  the running total from round to round; a second round starts above 2^20 pixels per plane, and cc_number_kernel
  numbers the roots from that carry;
* i128_to_double_rn converts a covariance of 2^63 or more by keeping its top 63 bits and a sticky bit; that takes a
  component of about 2200 x 2200 pixels.  A wrong rounding shows only through the principal axis, and only where
  the axis is sensitive to the last bit of the covariance.

The CPU part restates the segment model and the conversion, and checks that the shapes and the literal table of
single-component planes below reach every edge and rounding class, each with a sensitive axis.  The GPU part compares
the device with scipy.ndimage.label and oracle/oriented.py bit for bit.  Run this file as a script with --search to
look for more table entries."""

import math
import sys

import numpy as np
import pytest
import torch

from oracle import oriented as orc
from test_components import expected, pack_bits, patterns
from test_oriented import FRAME_SCALE

SEG = 1024                  # raster pixels per root-count segment (kSeg)
SCAN = 1024                 # segments per scan round (cc_scan_kernel's block)
MAX_SIDE = 32767            # the oriented call's limit on either side

# w = 1024 puts nseg = h; the others add a one-pixel last segment, an odd pixel count, a 1080p plane, 16 rounds and
# the oriented call's longest side (two rounds)
SCAN_SHAPES = [(1023, 1024), (1024, 1024), (1025, 1024), (2048, 1024), (2049, 1024), (1, 1048577), (1025, 1025),
               (1080, 1920), (4096, 4096), (32767, 64), (64, 32767)]
SCAN_PATTERNS = ("rand0.4", "rand0.6", "checker", "serpentine", "ones", "corners", "late", "early")
BIG = (4096, 4096)
BIG_PATTERNS = ("rand0.4", "serpentine", "ones", "corners", "late")


def segments(h, w):
    """(nseg, rounds, cap) of an h x w plane, as plane_of and cc_scan_kernel compute them."""
    n = h * w
    nseg = -(-n // SEG)
    return nseg, -(-nseg // SCAN), -(-n // 2)


def scan_edges(h, w):
    """Edges of the segment scan that an h x w plane reaches."""
    n = h * w
    nseg, rounds, cap = segments(h, w)
    out = set()
    if nseg == SCAN:
        out.add("one full round")
    if nseg == SCAN + 1:
        out.add("nseg = 1025")
    if nseg == 2 * SCAN:
        out.add("two full rounds")
    if nseg == 2 * SCAN + 1:
        out.add("nseg = 2049")
    if rounds >= 16:
        out.add(">= 16 rounds")
    if n % SEG == 1:
        out.add("one-pixel last segment")
    if n % 2 == 1:
        out.add("odd n: 4-connected checkerboard has cap components")
    return out


SCAN_EDGES = {"one full round", "nseg = 1025", "two full rounds", "nseg = 2049", ">= 16 rounds",
              "one-pixel last segment", "odd n: 4-connected checkerboard has cap components"}


# ---------------------------------------------------------------- the int128 -> fp64 conversion

def i128_to_double_model(v):
    """i128_to_double_rn restated on Python ints: below 2^63 one correctly rounded conversion; otherwise the top 63
    bits of |v| with a sticky bit for what was cut, rounded half to even to 53 bits, scaled by 2^s."""
    m = abs(v)
    if m >> 63 == 0:
        return float(v)
    s = m.bit_length() - 63
    t = m >> s
    if m & ((1 << s) - 1):
        t |= 1
    q, r = t >> 10, t & 0x3ff                       # 63 - 53 = 10 bits below the kept significand
    if r > 0x200 or (r == 0x200 and q & 1):
        q += 1
    d = math.ldexp(float(q), s + 10)                # q <= 2^53: exact
    return -d if v < 0 else d


def covariance_class(m):
    """(magnitude, rounding) classes of an exact covariance with |m| >= 2^63, else None.  t = the kept 63 bits,
    "cut" = the bits below them."""
    a = abs(m)
    if a >> 63 == 0:
        return None
    s = a.bit_length() - 63
    cut, t = a & ((1 << s) - 1), a >> s
    mag = ("negative" if m < 0 else "positive, 2^63 <= m < 2^64" if a >> 64 == 0 else
           "positive, 2^64 <= m < 2^65" if a >> 65 == 0 else "positive, m >= 2^65")
    low = t & 0x3ff
    if cut == 0 and low == 0x200:
        rnd = "exact tie"
    elif cut and low == 0x200:
        rnd = "sticky tie, even" if not t & 0x400 else "sticky tie, odd"
    elif cut and low == 0x1ff:
        rnd = "0x1ff + sticky"
    elif cut == 0:
        rnd = "cut zero"
    else:
        rnd = "sticky"
    return mag, rnd


# ---------------------------------------------------------------- single components with covariances >= 2^63

def band_x0(h, p, q, s):
    """Left edge of each row of a sheared band: floor(s y p / q), shifted so that its minimum is 0."""
    x0 = (s * np.arange(h, dtype=np.int64) * p) // q
    return x0 - x0.min()


def band_moments(W, H, p, q, s):
    """Exact raw moments (n, Sx, Sy, Sxx, Sxy, Syy) of the band of H rows of W pixels from band_x0, and its width."""
    x0 = band_x0(H, p, q, s)
    y = np.arange(H, dtype=np.int64)
    sx0, sx02, syx0 = (int(v) for v in (x0.sum(), (x0 * x0).sum(), (y * x0).sum()))
    t1, t2 = W * (W - 1) // 2, (W - 1) * W * (2 * W - 1) // 6
    n = W * H
    Sx = W * sx0 + H * t1
    Sy = W * (H * (H - 1) // 2)
    Sxx = W * sx02 + 2 * t1 * sx0 + H * t2
    Sxy = W * syx0 + t1 * (H * (H - 1) // 2)
    Syy = W * ((H - 1) * H * (2 * H - 1) // 6)
    return (n, Sx, Sy, Sxx, Sxy, Syy), int(x0.max()) + W


def covariances(mom):
    n, Sx, Sy, Sxx, Sxy, Syy = mom
    return n * Sxx - Sx * Sx, n * Sxy - Sx * Sy, n * Syy - Sy * Sy


def sensitive(cov, i):
    """True when replacing covariance i's fp64 value by either neighbour changes principal_axis at scale (1, 1).
    The covariances go in as (n, Sx, Sy) = (1, 0, 0), so the oracle converts exactly the integers given."""
    f = [float(c) for c in cov]

    def axis(vals):
        return orc.principal_axis((1, 0, 0, int(vals[0]), int(vals[1]), int(vals[2])))
    base = axis(f)
    for direction in (math.inf, -math.inf):
        g = list(f)
        g[i] = math.nextafter(f[i], direction)
        if axis(g) == base:
            return False
    return True


NAMES = ("Cxx", "Cxy", "Cyy")

# (W, H, p, q, s): H rows of W pixels from band_x0(H, p, q, s); found by search_class_table
BANDS = [
    (2469, 2023, 1, 2, 1),      # Cxx 2^63 <= m < 2^64, cut zero
    (2372, 2517, 2, 3, -1),     # Cxx and Cyy in [2^64, 2^65), cut zero
    (2155, 2176, 3, 4, 1),      # Cxx < 2^64, exact tie
    (2562, 2272, 1, 2, 1),      # Cxx in [2^64, 2^65), exact tie
    (2398, 2317, 1, 3, -1),     # Cxx < 2^64, sticky tie on an even significand
    (2559, 2334, 1, 3, 1),      # Cxx in [2^64, 2^65), sticky tie on an even significand
    (2022, 2175, 3, 4, 1),      # Cxx < 2^64, sticky
    (2571, 2379, 1, 3, 1),      # Cxx in [2^64, 2^65), sticky
    (2321, 2587, 2, 4, -1),     # Cxy negative, sticky tie on an even significand
    (2544, 2296, 2, 3, -1),     # Cxy negative, exact tie
    (2589, 2511, 2, 4, -1),     # Cxx in [2^64, 2^65), low bits 0x1ff and sticky
    (2565, 2490, 1, 2, 1),      # Cyy in [2^64, 2^65), sticky tie on an even significand
    (3362, 2809, 1, 4, 1),      # Cxx >= 2^65, sticky tie on an even significand
    (2162, 3264, 1, 3, 1),      # Cyy >= 2^65, exact tie
    (2990, 2695, 2, 5, 1),      # Cxx >= 2^65, sticky
]

# filled W x H rectangles with every covariance >= 2^63: b == 0 and a >= c at those magnitudes
RECTS = [(3600, 2400), (2400, 3600), (2400, 2400)]

# m >= 2^64 is split at 2^65: below it, a shift of 1 instead of 2 keeps all of m's bits and rounds the same
REQUIRED_CLASSES = {"positive, 2^63 <= m < 2^64", "positive, 2^64 <= m < 2^65", "positive, m >= 2^65", "negative",
                    "cut zero", "exact tie", "sticky tie, even", "sticky"}


def class_rows():
    """(case, covariance name, magnitude class, rounding class, sensitive) of every covariance >= 2^63 of BANDS."""
    rows = []
    for case in BANDS:
        mom, _ = band_moments(*case)
        cov = covariances(mom)
        for i, name in enumerate(NAMES):
            c = covariance_class(cov[i])
            if c is not None:
                rows.append((case, name, c[0], c[1], sensitive(cov, i)))
    return rows


def band_plane(W, H, p, q, s):
    """The band at the top left of a plane (H + 4 rows), and below it, two blank rows away, a 2 x 3 block and a
    diagonal pixel pair (one component under 8-connectivity): with K = 4 one row stays unused."""
    x0 = band_x0(H, p, q, s)
    width = int(x0.max()) + W
    xx = np.arange(width)[None, :]
    m = np.zeros((H + 4, width), bool)
    m[:H] = (xx >= x0[:, None]) & (xx < x0[:, None] + W)
    m[H + 2:H + 4, 1:4] = True
    m[H + 2, width - 2] = m[H + 3, width - 1] = True
    return m


def rect_plane(W, H):
    m = np.zeros((H + 4, W + 8), bool)
    m[:H, 2:W + 2] = True
    m[H + 2:H + 4, W + 3:W + 6] = True
    m[H + 2, 0] = m[H + 3, 1] = True
    return m


def search_class_table(seconds=120.0, seed=1):
    """Random search over the band family for a sensitive case of every (covariance, class) pair; prints the first
    case found for each.  Not part of the test run: `python tests/test_components_large.py --search`."""
    import time
    rng = np.random.default_rng(seed)
    found = {}
    t0 = time.time()
    while time.time() - t0 < seconds:
        q = int(rng.integers(1, 7))
        case = (int(rng.integers(1600, 4000)), int(rng.integers(1600, 4000)), int(rng.integers(1, q + 1)), q,
                int(rng.choice([-1, 1])))
        mom, width = band_moments(*case)
        if width > 4096:
            continue
        cov = covariances(mom)
        for i, name in enumerate(NAMES):
            c = covariance_class(cov[i])
            if c is not None and (name, *c) not in found and sensitive(cov, i):
                found[(name, *c)] = case
                print(name, c, case, flush=True)
    return found


# ---------------------------------------------------------------- CPU: shape cover, class table, conversion

def test_scan_shape_cover():
    reached = set()
    print(f"{'h x w':>12s} {'nseg':>6s} {'rounds':>6s} {'cap':>8s}  edges")
    for h, w in SCAN_SHAPES:
        nseg, rounds, cap = segments(h, w)
        edges = scan_edges(h, w)
        reached |= edges
        print(f"{h:>5d} x {w:<6d} {nseg:>6d} {rounds:>6d} {cap:>8d}  {', '.join(sorted(edges))}")
        assert h * w <= 4096 * 4096 and (max(h, w) <= 4096 or min(h, w) <= 64), (h, w)
        n_pat = len(BIG_PATTERNS) if (h, w) == BIG else len(SCAN_PATTERNS)
        assert n_pat * h * w <= 1 << 27, (h, w)
    assert reached == SCAN_EDGES, SCAN_EDGES - reached
    # w = 1024 gives nseg = h, and a one-pixel last segment holds raster index n - 1
    assert all(segments(h, 1024)[0] == h for h in (1023, 1024, 1025, 2048, 2049))
    assert segments(1025, 1025) == (1027, 2, 525313) and segments(1, 1048577)[:2] == (1025, 2)
    assert segments(*BIG)[1] == 16 and segments(MAX_SIDE, 64)[1] == segments(64, MAX_SIDE)[1] == 2


def test_class_table_cover():
    rows = class_rows()
    print(f"{'W, H, p, q, s':24s} {'cov':4s} {'magnitude':28s} {'rounding':18s} sensitive")
    for case, name, mag, rnd, sens in rows:
        print(f"{str(case):24s} {name:4s} {mag:28s} {rnd:18s} {'yes' if sens else 'no'}")
    covered = {c for _, _, mag, rnd, sens in rows if sens for c in (mag, rnd)}
    assert REQUIRED_CLASSES <= covered, REQUIRED_CLASSES - covered
    print("0x1ff + sticky:", "covered" if "0x1ff + sticky" in covered else "not found")
    # every listed case adds a sensitive class of its own to some covariance
    assert all(any(r[0] == case and r[4] for r in rows) for case in BANDS)
    # the closed-form moments are those of the planes the GPU test builds; each band fits a 4096 x 4096 plane
    from scipy import ndimage
    for case in BANDS:
        m = band_plane(*case)
        assert m.shape[0] <= 4096 and m.shape[1] <= 4096, case
        lab, n = ndimage.label(m, np.ones((3, 3), bool))
        assert n == 3 and np.count_nonzero(lab == 1) == case[0] * case[1], case
        ys, xs = np.nonzero(lab == 1)
        assert orc.moments(xs, ys) == band_moments(*case)[0], case
    # the rectangles: wider, taller and square, every covariance >= 2^63 and Cxy == 0
    for W, H in RECTS:
        ys, xs = np.nonzero(rect_plane(W, H)[:H])
        cxx, cxy, cyy = covariances(orc.moments(xs, ys))
        assert cxy == 0 and min(cxx, cyy) >= 1 << 63, (W, H)
        print(f"rectangle {W} x {H}: Cxx {covariance_class(cxx)}, Cyy {covariance_class(cyy)}")
    assert {np.sign(W - H) for W, H in RECTS} == {-1, 0, 1}


def test_conversion_model_matches_float():
    vals = [(1 << 63) - 1, -((1 << 63) - 1), 1 << 63, -(1 << 63), (1 << 64) - 1, 1 << 64, (1 << 64) + 1, 1 << 90,
            -(1 << 90), 0, 1, -1, (1 << 53) + 1]
    rng = np.random.default_rng(11)
    ties = 0
    for bits in range(64, 92):
        s = bits - 63
        for low in (0x200, 0x1ff, 0x201, 0x000, 0x3ff):
            for odd in (0, 1):
                sig = (1 << 52) | (int(rng.integers(0, 1 << 51)) << 1) | odd          # 53-bit significand
                t = (sig << 10) | low
                for cut in {0, 1, (1 << s) - 1, int(rng.integers(0, 1 << min(s, 62))) % (1 << s)}:
                    vals += [(t << s) | cut, -((t << s) | cut)]
                    ties += low == 0x200
    for _ in range(100_000):
        bits = int(rng.integers(63, 92))
        v = (1 << (bits - 1)) | int.from_bytes(rng.bytes(12), "little") % (1 << (bits - 1))
        vals.append(-v if rng.integers(0, 2) else v)
    bad = [v for v in vals if i128_to_double_model(v) != float(v)]
    assert not bad, [hex(v) for v in bad[:5]]
    assert ties >= 100 and len(vals) > 100_000


# ---------------------------------------------------------------- GPU: the segment scan against scipy

def scan_patterns(h, w):
    """rand0.4, rand0.6, checker, serpentine, ones and corners of test_components, plus "late" (rand0.4 with the
    whole first scan round empty) and "early" (rand0.4 in the first round only)."""
    base = patterns(h, w)
    out = {k: base[k] for k in SCAN_PATTERNS[:-2]}
    first = (np.arange(h * w) < SCAN * SEG).reshape(h, w)
    out["late"] = base["rand0.4"] & ~first
    out["early"] = base["rand0.4"] & first
    return out


def run_labels(batch, dev, packed, conn, k):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    src = pack_bits(batch) if packed else batch.astype(np.uint8)
    out = prepost.mask_components(torch.from_numpy(src).to(dev), packed=packed, connectivity=conn, max_components=k,
                                  labels=True)
    return tuple(t.cpu().numpy() for t in out)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("h,w", SCAN_SHAPES)
def test_scan_rounds_match_scipy(cuda_dev, h, w, conn):
    pats = scan_patterns(h, w)
    if (h, w) == BIG:
        pats = {k: pats[k] for k in BIG_PATTERNS}
    names = list(pats)
    batch = np.stack(list(pats.values()))[None]
    refs = [expected(batch[0, j], conn, 16) for j in range(len(names))]
    for packed in (False, True) if w % 32 == 0 else (False,):
        for k in (1, 16):
            comps, n, lab = run_labels(batch, cuda_dev, packed, conn, k)
            for j, name in enumerate(names):
                ref_lab, ref_n, ref_rows = refs[j]
                assert n[0, j] == ref_n, (name, packed, k, n[0, j], ref_n)
                assert np.array_equal(lab[0, j], ref_lab), (name, packed, k, int((lab[0, j] != ref_lab).sum()))
                assert np.array_equal(comps[0, j], ref_rows[:k]), (name, packed, k, comps[0, j], ref_rows[:k])
    if "checker" in pats and conn == 4 and h * w % 2:
        cap = segments(h, w)[2]
        assert refs[names.index("checker")][1] == cap and lab[0, names.index("checker"), -1, -1] == cap
    if "serpentine" in pats:
        assert refs[names.index("serpentine")][1] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_batch_of_multi_round_planes(cuda_dev, conn):
    from tw_invoice_unet_ocr_llm_b200 import prepost
    h, w = 1080, 1920
    pats = scan_patterns(h, w)
    names = ["rand0.4", "checker", "late", "serpentine", "rand0.6", "early"]
    batch = np.stack([pats[k] for k in names]).reshape(2, 3, h, w)
    m = torch.from_numpy(batch.astype(np.uint8)).to(cuda_dev)
    comps, n, lab = prepost.mask_components(m, connectivity=conn, max_components=16, labels=True)
    comps0, n0 = prepost.mask_components(m, connectivity=conn, max_components=16)
    assert torch.equal(comps, comps0) and torch.equal(n, n0)
    again = prepost.mask_components(m, connectivity=conn, max_components=16, labels=True)
    assert all(torch.equal(a, b) for a, b in zip(again, (comps, n, lab)))
    comps, n, lab = comps.cpu().numpy(), n.cpu().numpy(), lab.cpu().numpy()
    for idx in np.ndindex(2, 3):
        one = run_labels(batch[idx][None, None], cuda_dev, False, conn, 16)
        assert all(np.array_equal(o[0, 0], f[idx]) for o, f in zip(one, (comps, n, lab))), idx
        ref_lab, ref_n, ref_rows = expected(batch[idx], conn, 16)
        assert n[idx] == ref_n and np.array_equal(comps[idx], ref_rows) and np.array_equal(lab[idx], ref_lab), idx


# ---------------------------------------------------------------- GPU: top-K selection at scale

@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_selection_of_equal_components(cuda_dev, conn):
    """2 x 2 blocks on a pitch of 3 in a 2048 x 2048 plane: 683^2 components of 4 pixels; ties go to the lowest
    labels."""
    yy, xx = np.mgrid[:2048, :2048]
    m = (yy % 3 < 2) & (xx % 3 < 2)
    comps, n, lab = run_labels(m[None, None], cuda_dev, False, conn, 16)
    assert n[0, 0] == 683 * 683
    assert comps[0, 0, :, 5].tolist() == list(range(1, 17)) and (comps[0, 0, :, 4] == 4).all()
    ref_lab, ref_n, ref_rows = expected(m, conn, 16)
    assert n[0, 0] == ref_n and np.array_equal(comps[0, 0], ref_rows) and np.array_equal(lab[0, 0], ref_lab)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_selection_of_last_round_ids(cuda_dev, conn):
    """Bars on every other row of a 4096 x 1024 plane (four scan rounds), their lengths growing in raster order: the
    winners' roots lie in the last round."""
    h, w = 4096, 1024
    m = np.zeros((h, w), bool)
    for k in range(h // 2):
        m[2 * k, : 1 + k * (w - 1) // (h // 2 - 1)] = True
    comps, n, lab = run_labels(m[None, None], cuda_dev, False, conn, 16)
    ref_lab, ref_n, ref_rows = expected(m, conn, 16)
    assert n[0, 0] == ref_n == h // 2
    assert np.array_equal(comps[0, 0], ref_rows) and np.array_equal(lab[0, 0], ref_lab)
    assert (comps[0, 0, :, 2] * w >= 3 * SCAN * SEG).all()           # every winner's root is in round 4


# ---------------------------------------------------------------- GPU: oriented boxes at 128-bit covariances

def check_oriented(plane, dev, conn, k, packed=False):
    """mask_components_oriented of one plane against mask_components, scipy and oracle/oriented.py."""
    from tw_invoice_unet_ocr_llm_b200 import prepost
    src = pack_bits(plane[None, None]) if packed else plane[None, None].astype(np.uint8)
    m = torch.from_numpy(src).to(dev)
    c0, n0, l0 = prepost.mask_components(m, packed=packed, connectivity=conn, max_components=k, labels=True)
    ref_lab, ref_n, ref_rows = expected(plane, conn, k)
    assert n0[0, 0] == ref_n and np.array_equal(c0[0, 0].cpu().numpy(), ref_rows)
    assert np.array_equal(l0[0, 0].cpu().numpy(), ref_lab)
    for scale in (None, FRAME_SCALE):
        c1, n1, mom, obox, l1 = prepost.mask_components_oriented(m, packed=packed, connectivity=conn,
                                                                 max_components=k, scale=scale, labels=True)
        assert torch.equal(c0, c1) and torch.equal(n0, n1) and torch.equal(l0, l1)
        ref_m, ref_o = orc.oriented_rows(ref_lab, ref_rows, scale or (1.0, 1.0))
        mom, obox = mom[0, 0].cpu().numpy(), obox[0, 0].cpu().numpy()
        assert np.array_equal(mom, ref_m), (scale, mom, ref_m)
        assert np.array_equal(obox, ref_o), (scale, obox, ref_o)
        assert np.array_equal(mom[:, 0], ref_rows[:, 4])
    return ref_rows


@pytest.mark.gpu
@pytest.mark.parametrize("case", BANDS + [("rect",) + r for r in RECTS],
                         ids=lambda c: "_".join(map(str, c)))
def test_oriented_at_128bit_covariances(cuda_dev, case):
    plane = rect_plane(*case[1:]) if case[0] == "rect" else band_plane(*case)
    rows = check_oriented(plane, cuda_dev, 8, 4)
    assert rows[:, 4].tolist()[1:] == [6, 2, 0]                      # used and unused rows


# ---------------------------------------------------------------- GPU: the oriented call's longest side

def long_patterns(h, w):
    """A line over the full length, a band sheared across the short side and 40 % noise."""
    tall = h > w
    L, S = (h, w) if tall else (w, h)
    line = np.zeros((L, S), bool)
    line[:, S // 2] = True
    x0 = band_x0(L, S - 16, L - 1, 1)
    xx = np.arange(S)[None, :]
    band = (xx >= x0[:, None]) & (xx < x0[:, None] + 16)
    rand = np.random.default_rng(L + S).random((L, S)) < 0.4
    out = {"line": line, "band": band, "rand0.4": rand}
    return out if tall else {k: v.T.copy() for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,packed", [(MAX_SIDE, 64, False), (MAX_SIDE, 64, True), (64, MAX_SIDE, False)])
def test_oriented_at_the_longest_side(cuda_dev, h, w, packed):
    for name, plane in long_patterns(h, w).items():
        for conn in (4, 8):
            rows = check_oriented(plane, cuda_dev, conn, 16, packed)
            if name != "rand0.4":
                assert rows[0, 4] == plane.sum() and rows[1, 4] == 0, (name, conn)


if __name__ == "__main__" and "--search" in sys.argv:
    search_class_table()
