"""The OCR crop enhancement at the edges of its host plan and of its kernels.

CPU: ``unetb200_enhance_plan`` restated in Python and compared field by field; the CLAHE clip limit computed in
double precision, as ``cv::createCLAHE(double clipLimit)`` does, over a sweep of clips and tile areas; clip limits
that are out of range, side and batch limits, every argument check of ``unetb200_enhance_plan``, the checks
``unetb200_enhance_run`` makes before any CUDA call, and the ctypes mirror of ``unetb200_enh_crop``.

GPU: clip limits float32 cannot represent and huge clip limits, persistent upscale runs that span whole crops, every
residue of the 32 x 32 block grid, CLAHE tile geometries, the longest sides and the spans of the Otsu binarize pass,
each compared with ``oracle/opencv_enhance.py`` (and cv2 for CLAHE alone) with ``np.array_equal``.
"""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import opencv_enhance as oe

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TILES, BLOCK, SPAN, MAX_SIDE = 8, 32, 16384, 8192       # kEnhTiles, kEnhBlock, kEnhBinSpan, kMaxSide
SHARPEN, BLUR, OTSU = 1, 2, 4
DBL_MAX = sys.float_info.max
HUGE_CLIPS = [256.0, 1e4, 1e9, 1e30, 1e300, DBL_MAX]
# (h, w, clip): the rounding of clip to float32 moves (int)(clip * tile_area / 256) to another integer.  The
# first three share the tile area 2560 (20 x 128, 32 x 80, 40 x 64); the others are the smallest tile areas a
# search over h < 100, w < 200 and the clips k / 100 finds for their clip.
F32_CASES = [(38, 255, 0.7), (62, 159, 0.7), (78, 127, 0.7), (1, 198, 5.12), (2, 199, 2.56), (6, 159, 5.6),
             (6, 199, 1.28), (14, 159, 2.8), (14, 199, 0.64), (30, 159, 1.4)]


@pytest.fixture(scope="module")
def nat():
    import __graft_entry__ as g
    g.build()
    from tw_invoice_unet_ocr_llm_b200 import _native
    return _native


# ------------------------------------------------------------------ the plan, restated
def _tiles(h, w):
    """CLAHE_Impl::apply on the 4x image: both sides are padded to the 8 x 8 grid unless both divide it."""
    H, W = 4 * h, 4 * w
    if H % TILES or W % TILES:
        H, W = H + TILES - H % TILES, W + TILES - W % TILES
    return H // TILES, W // TILES


def _clip_count(clip, area):
    """The oracle's clip limit, clamped at the tile area: no bin holds more than the area, so a limit at or
    above it clips nothing, like any larger one (this also covers products that overflow to inf)."""
    if clip * area / 256 >= area:
        return area
    return oe.clahe_clip_limit(clip, area)


def _ceil16(x):
    return (x + 15) // 16 * 16


def _restate_plan(crops):
    """unetb200_enhance_plan in Python: the planned fields of each crop, and the (src, out, workspace) sizes."""
    so = oo = wo = blocks = 0
    rows = []
    for c in crops:
        h, w = c["h"], c["w"]
        th, tw = _tiles(h, w)
        bx = -(-4 * w // BLOCK)
        nb = bx * -(-4 * h // BLOCK)
        r = dict(tile_h=th, tile_w=tw, clip_count=_clip_count(c["clip"], th * tw), blocks_x=bx, n_blocks=nb,
                 first_block=blocks, src_pixel_bytes=c.get("src_pixel_bytes", 0) or 3, out_off=oo, ws_off=wo)
        if c.get("src_stride", 0) == 0:            # packed: placed back to back at 16-byte aligned offsets
            r.update(src_stride=w, src_off=so)
            so += _ceil16(3 * h * w)
        else:                                      # a window of a frame keeps its own offset
            r.update(src_stride=c["src_stride"], src_off=c["src_off"])
        blocks += nb
        oo += _ceil16(16 * h * w)
        wo += _ceil16(16 * h * w) + TILES * TILES * 256 + 256 * 4 + 16     # image, 64 LUTs, histogram + threshold
        rows.append(r)
    return rows, (so, oo, wo)


def _table(nat, crops):
    t = (nat.EnhCrop * len(crops))()
    for row, c in zip(t, crops):
        for k, v in c.items():
            setattr(row, k, v)
    return t


def _plan(nat, table, n=None):
    sizes = [C.c_uint64() for _ in range(3)]
    code = nat.lib().unetb200_enhance_plan(table, len(table) if n is None else n, *[C.byref(s) for s in sizes])
    return code, tuple(s.value for s in sizes)


BOUNDARY_SIDES = [1, 2, 3, 4, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 4095, 4096, 4097, 8191,
                  8192]


def _random_clip(rng):
    pick = int(rng.integers(7))
    if pick == 0:
        return float(rng.choice([4.0, 3.0]))                  # the recipes
    if pick == 1:
        return int(rng.integers(1, 1001)) / 100
    if pick == 2:
        return float(rng.uniform(0.0, 300.0)) or 1.0
    if pick == 3:
        return float(10.0 ** rng.uniform(-300, 300))
    return float(rng.choice([5e-324, 0.7, 256.0, np.nextafter(256.0, 0.0), 1e30, DBL_MAX]))


def _random_crops(rng, n):
    crops = []
    for _ in range(n):
        h, w = (int(rng.choice(BOUNDARY_SIDES)) if rng.random() < 0.4 else int(np.exp(rng.uniform(0, np.log(8192))))
                for _ in range(2))
        c = dict(h=h, w=w, flags=int(rng.integers(8)), clip=_random_clip(rng))
        if rng.random() < 0.5:                      # packed RGB, src_pixel_bytes 0 (= 3) or 3
            c["src_pixel_bytes"] = int(rng.choice([0, 3]))
        else:                                       # a window of a 3- or 4-byte frame
            c.update(src_stride=w + int(rng.integers(0, 5000)), src_pixel_bytes=int(rng.choice([0, 3, 4])),
                     src_off=int(rng.integers(0, 1 << 40)))
        crops.append(c)
    return crops


# ------------------------------------------------------------------ CPU
def test_plan_fields_equal_a_python_restatement(nat):
    """Every field unetb200_enhance_plan writes, on 4000 random and boundary crops, packed crops and windows
    mixed; the input fields are left as they were."""
    rng = np.random.default_rng(1)
    for rep in range(16):
        crops = _random_crops(rng, 250)
        t = _table(nat, crops)
        code, sizes = _plan(nat, t)
        assert code == nat.OK, nat.last_error()
        rows, want_sizes = _restate_plan(crops)
        assert sizes == want_sizes, rep
        for i, (row, c, r) in enumerate(zip(t, crops, rows)):
            assert (row.h, row.w, row.flags, row.clip) == (c["h"], c["w"], c["flags"], c["clip"]), (rep, i)
            assert {k: getattr(row, k) for k in r} == r, (rep, i, c)
            assert (row.tile_h, row.tile_w) == oe.clahe_geometry(4 * c["h"], 4 * c["w"])[2:]
            if c.get("src_stride", 0) == 0:
                assert row.src_off % 16 == 0
            assert row.out_off % 16 == 0 and row.ws_off % 16 == 0


def test_plan_tile_quirk_and_block_grid(nat):
    """Both sides are padded when either does not divide the grid: a side that divides gains a whole tile row."""
    cases = [  # (h, w) -> (tile_h, tile_w, blocks_x, n_blocks)
        ((2, 2), (1, 1, 1, 1)), ((2, 3), (2, 2, 1, 1)), ((3, 2), (2, 2, 1, 1)), ((1, 1), (1, 1, 1, 1)),
        ((38, 255), (20, 128, 32, 160)), ((62, 159), (32, 80, 20, 160)), ((78, 127), (40, 64, 16, 160)),
        ((64, 64), (32, 32, 8, 64)), ((64, 63), (33, 32, 8, 64)), ((8192, 8192), (4096, 4096, 1024, 1 << 20)),
        ((8192, 1), (4097, 1, 1, 1024)), ((1, 8192), (1, 4097, 1024, 1024)),
    ]
    t = _table(nat, [dict(h=h, w=w, flags=0, clip=4.0) for (h, w), _ in cases])
    assert _plan(nat, t)[0] == nat.OK, nat.last_error()
    for row, ((h, w), want) in zip(t, cases):
        assert (row.tile_h, row.tile_w, row.blocks_x, row.n_blocks) == want, (h, w)
        assert (row.tile_h, row.tile_w) == _tiles(h, w)


def _sweep_clips():
    clips = [k / 100 for k in range(1, 1001)]
    clips += [0.7, 0.1, 0.3, 1 / 3, 2 / 3, 1.1, 2.2, 2.3, 3.3, 4.4, 5.55, 0.07, 1e-5, math.pi, math.e, math.sqrt(2),
              2.9999999, 3.0000001, 4.0000001, 255.99, 256.01]
    clips += [float(np.nextafter(v, d)) for v in (3.0, 4.0, 256.0) for d in (0.0, 1e3)]
    clips += [float(c) for c in np.random.default_rng(2).uniform(0.0, 300.0, 200) if c > 0]
    return clips


SWEEP_SIDES = [1, 2, 3, 5, 8, 13, 38, 62, 78, 127, 159, 198, 199, 255, 1000, 4097, 8192]


def test_clip_count_is_computed_in_double_over_a_sweep(nat):
    """clip_count equals the oracle's (int)(clip * area / 256) in double for every clip k / 100, k = 1..1000, and
    values float32 cannot represent, on a grid of tile areas; many of these limits would truncate to another
    integer with the clip rounded to float32."""
    clips = _sweep_clips()
    f32_moves = 0
    for h in SWEEP_SIDES:
        for w in SWEEP_SIDES:
            t = _table(nat, [dict(h=h, w=w, flags=0, clip=c) for c in clips])
            assert _plan(nat, t)[0] == nat.OK, nat.last_error()
            th, tw = _tiles(h, w)
            area = th * tw
            got = [row.clip_count for row in t]
            want = [_clip_count(c, area) for c in clips]
            bad = [(c, g, x) for c, g, x in zip(clips, got, want) if g != x]
            assert not bad, f"{h}x{w} (tile area {area}): (clip, plan, oracle) {bad[:5]} of {len(bad)}"
            f32_moves += sum(_clip_count(float(np.float32(c)), area) != x for c, x in zip(clips, want))
    assert f32_moves > 1000, f32_moves


def test_out_of_range_clips(nat):
    """Clips whose limit reaches the tile area (up to DBL_MAX, whose product overflows to inf) clip nothing:
    clip_count is the area.  The smallest positive clips give 1.  Non-finite and non-positive clips are EINVAL."""
    sizes = [(1, 1), (38, 255), (2, 199), (8192, 8192), (8192, 1)]
    for clip in HUGE_CLIPS:
        t = _table(nat, [dict(h=h, w=w, flags=0, clip=clip) for h, w in sizes])
        assert _plan(nat, t)[0] == nat.OK, (clip, nat.last_error())
        for row in t:
            assert row.clip_count == row.tile_h * row.tile_w, (clip, row.h, row.w, row.clip_count)
    for clip in (5e-324, sys.float_info.min, 1e-300):
        t = _table(nat, [dict(h=h, w=w, flags=0, clip=clip) for h, w in sizes])
        assert _plan(nat, t)[0] == nat.OK
        assert [row.clip_count for row in t] == [1] * len(sizes)
    good = dict(h=4, w=4, flags=0, clip=4.0)
    for clip in (math.inf, -math.inf, math.nan, 0.0, -0.0, -1.0, -5e-324, -DBL_MAX):
        t = _table(nat, [good, good, dict(good, clip=clip)])
        assert _plan(nat, t)[0] == nat.EINVAL, clip
        assert "enhance_plan: crop 2 invalid" in nat.last_error(), (clip, nat.last_error())


def test_side_flag_and_layout_limits(nat):
    def one(**kw):
        code = _plan(nat, _table(nat, [dict(dict(h=10, w=20, flags=0, clip=4.0), **kw)]))[0]
        if code != nat.OK:
            assert "enhance_plan: crop 0 invalid" in nat.last_error()
        return code

    for h, w in [(MAX_SIDE, 1), (1, MAX_SIDE), (MAX_SIDE, MAX_SIDE)]:
        assert one(h=h, w=w) == nat.OK, (h, w)
    for h, w in [(MAX_SIDE + 1, 1), (1, MAX_SIDE + 1), (MAX_SIDE + 1, MAX_SIDE + 1), (0, 4), (4, 0), (-1, 4),
                 (4, -1), (-(1 << 31), 4)]:
        assert one(h=h, w=w) == nat.EINVAL, (h, w)
    for flags in range(8):
        assert one(flags=flags) == nat.OK
    for flags in (8, 9, 16, 1 << 30, -1, -(1 << 31)):
        assert one(flags=flags) == nat.EINVAL, flags
    for stride in (20, 21, 1 << 20):
        assert one(src_stride=stride) == nat.OK, stride
    for stride in (19, 1, -1, -20):                                          # src_stride < w
        assert one(src_stride=stride) == nat.EINVAL, stride
    for pb in (0, 3):
        assert one(src_pixel_bytes=pb) == nat.OK and one(src_stride=30, src_pixel_bytes=pb) == nat.OK
    assert one(src_stride=30, src_pixel_bytes=4) == nat.OK
    assert one(src_pixel_bytes=4) == nat.EINVAL                              # packed crops are RGB
    for pb in (1, 2, 5, 6, 8, -1, -3):
        assert one(src_pixel_bytes=pb) == nat.EINVAL and one(src_stride=30, src_pixel_bytes=pb) == nat.EINVAL, pb
    # the argument list itself
    t = _table(nat, [dict(h=4, w=4, flags=0, clip=4.0)])
    s = C.c_uint64()
    lib = nat.lib()
    for args in [(t, 0, C.byref(s), C.byref(s), C.byref(s)), (t, -1, C.byref(s), C.byref(s), C.byref(s)),
                 (None, 1, C.byref(s), C.byref(s), C.byref(s)), (t, 1, None, C.byref(s), C.byref(s)),
                 (t, 1, C.byref(s), None, C.byref(s)), (t, 1, C.byref(s), C.byref(s), None)]:
        assert lib.unetb200_enhance_plan(*args) == nat.EINVAL
        assert "enhance_plan: bad argument" in nat.last_error()


def test_batch_block_limit(nat):
    """Block indices are int32: 2047 crops of 8192 x 8192 (2^20 blocks each) fit, 2048 do not."""
    big = dict(h=MAX_SIDE, w=MAX_SIDE, flags=OTSU, clip=4.0)
    t = _table(nat, [big] * 2047)
    code, sizes = _plan(nat, t)
    assert code == nat.OK, nat.last_error()
    assert t[2046].first_block == 2046 << 20 and t[2046].n_blocks == 1 << 20
    img = 16 * MAX_SIDE * MAX_SIDE
    assert sizes == (2047 * 3 * MAX_SIDE * MAX_SIDE, 2047 * img, 2047 * (img + 64 * 256 + 1024 + 16))
    assert t[2046].src_off == 2046 * 3 * MAX_SIDE * MAX_SIDE and t[2046].out_off == 2046 * img
    t = _table(nat, [big] * 2048)
    assert _plan(nat, t)[0] == nat.EINVAL
    assert "enhance_plan: batch too large" in nat.last_error()


# unetb200_enhance_run with tables that did not come out of the plan.  Each call must fail its checks before any
# CUDA call; the cases run in a child process that sees no CUDA device, so that a check that let a table through
# could not launch a kernel on made-up device addresses.
_RUN_CASES = [  # (name, crop index, field, new value or a function of the planned value, expected message part)
    ("first_block +1", 0, "first_block", lambda v: v + 1, "crop 0: first_block"),
    ("first_block -1", 3, "first_block", lambda v: v - 1, "crop 3: first_block"),
    ("blocks_x +1", 2, "blocks_x", lambda v: v + 1, "crop 2: blocks_x / n_blocks"),
    ("n_blocks +1", 2, "n_blocks", lambda v: v + 1, "crop 2: blocks_x / n_blocks"),
    ("n_blocks -1", 4, "n_blocks", lambda v: v - 1, "crop 4: blocks_x / n_blocks"),
    ("n_blocks 0", 1, "n_blocks", 0, "crop 1: blocks_x / n_blocks"),
    ("out_off +16", 4, "out_off", lambda v: v + 16, "crop 4: out_off"),
    ("out_off 0", 1, "out_off", 0, "crop 1: out_off"),
    ("ws_off +16", 1, "ws_off", lambda v: v + 16, "crop 1: ws_off"),
    ("tile_h 0", 2, "tile_h", 0, "crop 2: tile_h / tile_w"),
    ("tile_w 0", 2, "tile_w", 0, "crop 2: tile_h / tile_w"),
    ("tile_h +1", 3, "tile_h", lambda v: v + 1, "crop 3: tile_h / tile_w"),
    ("tile_w -1", 0, "tile_w", lambda v: v - 1, "crop 0: tile_h / tile_w"),
    ("clip_count +1", 2, "clip_count", lambda v: v + 1, "crop 2: clip_count"),
    ("clip_count 0", 1, "clip_count", 0, "crop 1: clip_count"),
    ("clip 3 -> 6", 2, "clip", 6.0, "crop 2: clip_count"),
    ("clip inf", 3, "clip", math.inf, "crop 3: h, w, flags, clip"),
    ("clip nan", 2, "clip", math.nan, "crop 2: h, w, flags, clip"),
    ("clip 0", 0, "clip", 0.0, "crop 0: h, w, flags, clip"),
    ("flags 8", 2, "flags", 8, "crop 2: h, w, flags, clip"),
    ("h 8193", 2, "h", MAX_SIDE + 1, "crop 2: h, w, flags, clip"),
    ("h +1", 2, "h", lambda v: v + 1, "crop 2: "),
    ("w -1", 4, "w", lambda v: v - 1, "crop 4: "),
    ("src_stride < w", 1, "src_stride", 8, "crop 1: h, w, flags, clip"),
    ("src_stride 0", 0, "src_stride", 0, "crop 0: src_stride / src_pixel_bytes"),
    ("src_pixel_bytes 0", 3, "src_pixel_bytes", 0, "crop 3: src_stride / src_pixel_bytes"),
    ("src_pixel_bytes 2", 3, "src_pixel_bytes", 2, "crop 3: h, w, flags, clip"),
]
_RUN_CROPS = [dict(h=10, w=20, flags=5, clip=4.0), dict(h=7, w=9, flags=6, clip=0.7, src_stride=640,
              src_pixel_bytes=4, src_off=4 * 12345), dict(h=33, w=41, flags=1, clip=3.0),
              dict(h=3, w=70, flags=2, clip=1e30), dict(h=16, w=16, flags=7, clip=2.5, src_stride=100, src_off=999)]


def _run_validation_results(nat):
    """[(name, return code, message)] of unetb200_enhance_run over _RUN_CASES and the pointer checks."""
    lib = nat.lib()
    planned = _table(nat, _RUN_CROPS)
    assert _plan(nat, planned)[0] == nat.OK, nat.last_error()
    n = len(_RUN_CROPS)
    dev = [C.c_void_p(a) for a in (1 << 20, 1 << 21, 1 << 22, 1 << 23)]       # 16-byte aligned, never dereferenced
    out = []
    for name, k, field, value, _ in _RUN_CASES:
        t = (nat.EnhCrop * n)()
        C.memmove(t, planned, C.sizeof(planned))
        setattr(t[k], field, value(getattr(t[k], field)) if callable(value) else value)
        out.append((name, lib.unetb200_enhance_run(t, dev[0], n, dev[1], dev[2], dev[3], None), nat.last_error()))
    off = [C.c_void_p(a) for a in ((1 << 20) + 8, (1 << 21) + 4, (1 << 22) + 1)]
    for name, args in [("table_dev misaligned", (off[0], n, dev[1], dev[2], dev[3])),
                       ("out misaligned", (dev[0], n, dev[1], off[1], dev[3])),
                       ("workspace misaligned", (dev[0], n, dev[1], dev[2], off[2])),
                       ("table_dev null", (None, n, dev[1], dev[2], dev[3])),
                       ("src null", (dev[0], n, None, dev[2], dev[3])),
                       ("out null", (dev[0], n, dev[1], None, dev[3])),
                       ("workspace null", (dev[0], n, dev[1], dev[2], None)),
                       ("n 0", (dev[0], 0, dev[1], dev[2], dev[3])),
                       ("n -1", (dev[0], -1, dev[1], dev[2], dev[3]))]:
        out.append((name, lib.unetb200_enhance_run(planned, *args, None), nat.last_error()))
    out.append(("table_host null", lib.unetb200_enhance_run(None, dev[0], n, dev[1], dev[2], dev[3], None),
                nat.last_error()))
    return out


def test_enhance_run_rejects_tables_not_from_the_plan(nat):
    """A planned table with one field changed, misaligned device buffers and missing arguments: each is EINVAL,
    and the message names the crop and the field."""
    child = ("import json, sys; sys.path[:0] = sys.argv[1:3]; import test_enhance_edges as m; "
             "from tw_invoice_unet_ocr_llm_b200 import _native; print(json.dumps(m._run_validation_results(_native)))")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="-1")
    res = subprocess.run([sys.executable, "-c", child, ROOT, os.path.dirname(os.path.abspath(__file__))],
                         env=env, capture_output=True, text=True, check=True)
    results = {name: (code, msg) for name, code, msg in json.loads(res.stdout.strip().splitlines()[-1])}
    for name, _, _, _, part in _RUN_CASES:
        code, msg = results[name]
        assert code == nat.EINVAL and part in msg and "not produced by unetb200_enhance_plan" in msg, (name, code, msg)
    for name in ("table_dev misaligned", "out misaligned", "workspace misaligned"):
        assert results[name] == (nat.EINVAL, "enhance_run: device buffers must be 16-byte aligned"), name
    for name in ("table_dev null", "src null", "out null", "workspace null", "n 0", "n -1", "table_host null"):
        assert results[name] == (nat.EINVAL, "enhance_run: bad argument"), name


def test_enh_crop_layout_matches_the_header(nat, tmp_path):
    """ctypes.sizeof(EnhCrop) and every field offset equal those a C compiler gives unetb200_enh_crop."""
    from tw_invoice_unet_ocr_llm_b200 import build
    names = [f for f, _ in nat.EnhCrop._fields_]
    src = tmp_path / "layout.c"
    src.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"unetb200.h\"\nint main(void) {\n"
                   "    printf(\"sizeof %zu\\n\", sizeof(unetb200_enh_crop));\n"
                   "    printf(\"version %d\\n\", UNETB200_ABI_VERSION);\n" +
                   "".join(f"    printf(\"{f} %zu\\n\", offsetof(unetb200_enh_crop, {f}));\n" for f in names) +
                   "    return 0;\n}\n")
    exe = str(tmp_path / "layout")
    subprocess.run([build._nvcc(), "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)], check=True,
                   capture_output=True)
    got = dict(line.split() for line in subprocess.run([exe], check=True, capture_output=True,
                                                       text=True).stdout.splitlines())
    assert int(got.pop("sizeof")) == C.sizeof(nat.EnhCrop) == 80
    assert int(got.pop("version")) == nat.ABI_VERSION == nat.lib().unetb200_abi_version()
    assert {f: int(v) for f, v in got.items()} == {f: getattr(nat.EnhCrop, f).offset for f in names}
    assert nat.EnhCrop.clip.size == 8


# ------------------------------------------------------------------ GPU
def _recipe(kind):
    return oe.MODES[kind] if isinstance(kind, str) else kind


def _oracle(rgb, kind):
    """oe.enhance.  Every clip from 256 up gives a limit at or above the tile area, i.e. no clipping; the oracle's
    int64 histogram arithmetic overflows past about 1e15, so larger clips run at 1e9
    (test_huge_clip_limits_clip_nothing shows 256 and 1e9 agree)."""
    flags, clip = _recipe(kind)
    return oe.enhance(rgb, flags, min(clip, 1e9))


def _check(got, want, what):
    assert got.shape == want.shape and got.dtype == np.uint8, (what, got.shape, want.shape)
    bad = int((got != want).sum())
    assert bad == 0, f"{what}: {bad} of {want.size} pixels differ"


def _enhance(crops, kinds):
    from tw_invoice_unet_ocr_llm_b200 import enhance
    return enhance.enhance_batch(crops, kinds)


def _upscaled(rgb, flags):
    """The oracle's stage in front of CLAHE."""
    g = oe.resize_cubic_x4(oe.rgb_to_gray(rgb))
    return oe.sharpen(g) if flags & SHARPEN else g


@pytest.mark.gpu
def test_clip_limits_float32_cannot_represent(cuda_dev, nat):
    """The crops of F32_CASES under all 8 flag combinations against the oracle; with flags 0 and SHARPEN the
    result is CLAHE alone, also compared with cv2.createCLAHE on the oracle's upscaled stage."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(70)
    crops, kinds, want = [], [], []
    for h, w, clip in F32_CASES:
        th, tw = _tiles(h, w)
        assert _clip_count(clip, th * tw) != _clip_count(float(np.float32(clip)), th * tw), (h, w, clip)
        rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        up = _upscaled(rgb, 0)
        clahe = oe.clahe(up, clip)
        # the float32-rounded clip gives other LUTs on this crop, and cv2 agrees with the oracle's CLAHE
        assert not np.array_equal(clahe, oe.clahe(up, float(np.float32(clip)))), (h, w, clip)
        assert np.array_equal(clahe, cv2.createCLAHE(clip, (8, 8)).apply(up)), (h, w, clip)
        for flags in range(8):
            crops.append(rgb)
            kinds.append((flags, clip))
            want.append(oe.enhance(rgb, flags, clip))
    got = _enhance(crops, kinds)
    for i, (g, x, k) in enumerate(zip(got, want, kinds)):
        _check(g, x, f"crop {i} {crops[i].shape} {k}")
        if k[0] in (0, SHARPEN):
            assert np.array_equal(g, cv2.createCLAHE(k[1], (8, 8)).apply(_upscaled(crops[i], k[0]))), (i, k)


@pytest.mark.gpu
def test_huge_clip_limits_clip_nothing(cuda_dev, nat):
    """Clips from 256 to DBL_MAX against the oracle (at 1e9, where its arithmetic holds; 256 gives the same), and
    against cv2 where cv2's (int)(clip * area / 256) stays below 2^31."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(71)
    crops, kinds, want, areas = [], [], [], []
    for h, w in [(2, 2), (5, 7), (2, 199), (38, 255), (64, 64)]:
        rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        th, tw = _tiles(h, w)
        up = _upscaled(rgb, 0)
        # without the clamp a huge limit became 1, the strongest clipping, which differs where a tile has 2 px
        assert th * tw == 1 or not np.array_equal(oe.clahe(up, 1e9), oe.clahe(up, 1e-9)), (h, w)
        for flags in range(8):
            ref = oe.enhance(rgb, flags, 1e9)
            assert np.array_equal(ref, oe.enhance(rgb, flags, 256.0)), (h, w, flags)
            for clip in HUGE_CLIPS:
                crops.append(rgb)
                kinds.append((flags, clip))
                want.append(ref)
                areas.append(th * tw)
    got = _enhance(crops, kinds)
    n_cv2 = 0
    for i, (g, x, (flags, clip), area) in enumerate(zip(got, want, kinds, areas)):
        _check(g, x, f"crop {i} {crops[i].shape} {(flags, clip)}")
        if flags in (0, SHARPEN) and clip * area / 256 < 2 ** 31:
            assert np.array_equal(g, cv2.createCLAHE(clip, (8, 8)).apply(_upscaled(crops[i], flags))), (i, clip)
            n_cv2 += 1
    assert n_cv2 >= 20


TINY_KINDS = ["text", "amount", "date", (0, 0.7), (3, 1.1), (6, 2.3), (7, 40.0), (5, 1e30)]


@pytest.fixture(scope="module")
def persistent_batch():
    """An RGBX frame: a 720p synthetic invoice over 40 rows of noise; one crop is the whole invoice (14 400 output
    blocks), 3000 are windows of at most 8 x 8 px (one block each), half of them in the noise."""
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    rng = np.random.default_rng(80)
    fh, fw = 760, 1280
    frame = np.empty((fh, fw, 4), np.uint8)
    frame[:720, :, :3] = synthetic_invoices_u8(1, 720, fw, seed=81)[0]
    frame[720:, :, :3] = rng.integers(0, 256, (fh - 720, fw, 3), dtype=np.uint8)
    frame[..., 3] = rng.integers(0, 256, (fh, fw), dtype=np.uint8)       # ignored byte of every pixel
    rects, kinds = [(0, 0, fw, 720)], ["text"]
    for i in range(3000):
        h, w = int(rng.integers(1, 9)), int(rng.integers(1, 9))
        y = int(rng.integers(720, fh - h + 1)) if i % 2 else int(rng.integers(0, fh - h + 1))
        x = int(rng.integers(0, fw - w + 1))
        rects.append((x, y, x + w, y + h))
        kinds.append(TINY_KINDS[i % len(TINY_KINDS)])
    crops = [np.ascontiguousarray(frame[y1:y2, x1:x2, :3]) for x1, y1, x2, y2 in rects]
    want = [_oracle(c, k) for c, k in zip(crops, kinds)]
    return frame, rects, kinds, crops, want


@pytest.mark.gpu
def test_persistent_upscale_runs_span_whole_crops(cuda_dev, persistent_batch):
    """More than 148 x 16 x 4 output blocks, so every CTA of the persistent upscale grid walks at least 4 blocks
    whatever the occupancy (at most 16 CTAs of 128 threads per SM), and most runs and prefetches cross crops;
    big crop first, tiny crops first and the big crop among them, packed and as windows of the RGBX frame."""
    import torch
    from tw_invoice_unet_ocr_llm_b200 import enhance
    frame, rects, kinds, crops, want = persistent_batch
    table = enhance.plan([c.shape[:2] for c in crops], kinds)[0]
    assert all(t.n_blocks == 1 for t in table[1:]) and table[0].n_blocks == 90 * 160
    sms = torch.cuda.get_device_properties(cuda_dev).multi_processor_count
    assert sum(t.n_blocks for t in table) > sms * 16 * 4
    n = len(crops)
    orders = {"big first": list(range(n)), "tiny first": list(range(1, n)) + [0],
              "big among the tiny": list(range(1, n // 2)) + [0] + list(range(n // 2, n))}
    d_frame = torch.from_numpy(frame).to(cuda_dev)
    for what, order in orders.items():
        ks = [kinds[i] for i in order]
        packed = enhance.enhance_batch([crops[i] for i in order], ks)
        windows = enhance.enhance_windows(d_frame, [rects[i] for i in order], ks)
        for j, i in enumerate(order):
            _check(packed[j], want[i], f"{what}, packed crop {i} {rects[i]} {kinds[i]}")
            _check(windows[j], want[i], f"{what}, window {i} {rects[i]} {kinds[i]}")
    _check(enhance.enhance_batch([crops[0]], [kinds[0]])[0], want[0], "the big crop alone")
    for i in range(1, n, 97):
        _check(enhance.enhance_batch([crops[i]], [kinds[i]])[0], want[i], f"crop {i} alone")
        _check(enhance.enhance_windows(d_frame, [rects[i]], [kinds[i]])[0], want[i], f"window {i} alone")


@pytest.mark.gpu
def test_block_grid_residues(cuda_dev):
    """Every (4w mod 32, 4h mod 32) with at least 2 blocks per axis: the last block is 4..32 px wide and tall, so
    the sharpen's REFLECT_101 halo row / column lands at every position of the block, the blur's halo at every
    clamp, and odd widths end in the integer tail of the vertical pass."""
    sizes = [(h, w) for h in range(9, 17) for w in range(9, 17)]
    assert {(4 * w % 32, 4 * h % 32) for h, w in sizes} == {(a, b) for a in range(0, 32, 4) for b in range(0, 32, 4)}
    rng = np.random.default_rng(90)
    crops = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    for kind in [(SHARPEN, 4.0), (BLUR, 3.0), (SHARPEN | BLUR, 0.7), "text", "date"]:
        got = _enhance(crops, [kind] * len(crops))
        for c, g in zip(crops, got):
            _check(g, _oracle(c, kind), f"{c.shape} {kind}")


def _touches_all_luts(n):
    """Whether one block spanning the 4n px of an axis blends LUT rows 0 and 7 (enh_axis / the oracle's axis)."""
    tile = _tiles(n, n)[0]
    t = np.arange(4 * n).astype(np.float32) * (np.float32(1) / np.float32(tile)) - np.float32(0.5)
    t1 = np.floor(t).astype(np.int64)
    return np.maximum(t1, 0).min() == 0 and np.minimum(t1 + 1, TILES - 1).max() == TILES - 1


@pytest.mark.gpu
def test_clahe_tile_geometry(cuda_dev, nat):
    """1-px tiles; tiles narrower than, as wide as (32, 64) and wider than a block; tile edges on block edges;
    and every crop of one block, among them the smallest whose block touches all 64 LUTs (full LUT cache)."""
    from tw_invoice_unet_ocr_llm_b200 import enhance
    cases = {  # (h, w): (tile_h, tile_w)
        (2, 2): (1, 1), (2, 4): (1, 2), (2, 64): (1, 32), (64, 2): (32, 1), (2, 3): (2, 2),
        (20, 40): (10, 20), (40, 20): (20, 10), (64, 64): (32, 32), (64, 128): (32, 64), (128, 64): (64, 32),
        (128, 128): (64, 64), (100, 200): (50, 100), (256, 96): (128, 48), (128, 192): (64, 96), (65, 70): (33, 36),
    }
    one_block = [(h, w) for h in range(1, 9) for w in range(1, 9)]
    full = [(h, w) for h, w in one_block if _touches_all_luts(h) and _touches_all_luts(w) and h % 2 == w % 2]
    assert (2, 2) in full and (1, 1) not in full
    sizes = list(cases) + one_block
    table = enhance.plan(sizes, ["text"] * len(sizes))[0]
    for (h, w), t in zip(sizes, table):
        if (h, w) in cases:
            assert (t.tile_h, t.tile_w) == cases[(h, w)], (h, w)
        else:
            assert t.n_blocks == 1
    rng = np.random.default_rng(100)
    crops = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    for kind in ("text", "amount", "date", (0, 0.7)):
        got = _enhance(crops, [kind] * len(crops))
        for c, g in zip(crops, got):
            _check(g, _oracle(c, kind), f"{c.shape} {kind}")


@pytest.mark.gpu
def test_longest_sides(cuda_dev, nat):
    """Crops 8192 px long (outputs 32 768 px on a side) under all three recipes; 8193 is refused by the plan,
    before any launch, through every Python entry point."""
    import torch
    from tw_invoice_unet_ocr_llm_b200 import enhance
    rng = np.random.default_rng(110)
    crops = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
             for h, w in [(MAX_SIDE, 1), (1, MAX_SIDE), (MAX_SIDE, 8), (8, MAX_SIDE)]]
    for kind in ("text", "amount", "date"):
        got = _enhance(crops, [kind] * len(crops))
        for c, g in zip(crops, got):
            _check(g, _oracle(c, kind), f"{c.shape} {kind}")
    for h, w in [(MAX_SIDE + 1, 1), (1, MAX_SIDE + 1)]:
        with pytest.raises(nat.UnetB200Error, match="enhance_plan: crop 1 invalid"):
            enhance.enhance_batch([crops[0], np.zeros((h, w, 3), np.uint8)], ["text", "date"])
        frame = torch.zeros((h, w, 4), dtype=torch.uint8, device=cuda_dev)
        with pytest.raises(nat.UnetB200Error, match="enhance_plan: crop 0 invalid"):
            enhance.enhance_windows(frame, [(0, 0, w, h)], ["text"])
        buf = torch.zeros(3 * h * w, dtype=torch.uint8, device=cuda_dev)
        with pytest.raises(nat.UnetB200Error, match="enhance_plan: crop 0 invalid"):
            enhance.enhance_packed(buf, [0], [(w, h)], ["amount"])


@pytest.mark.gpu
def test_otsu_binarize_spans(cuda_dev, nat):
    """The threshold pass walks 16 384-byte spans of the packed output: results that start exactly on a span
    (32 x 32 crops fill one), spans that start inside a crop, and Otsu and non-Otsu crops alternating inside a
    span (4 x 4 crops: 64 per span; 1 x 1 crops: one 16-byte chunk each)."""
    from tw_invoice_unet_ocr_llm_b200 import enhance
    rng = np.random.default_rng(120)
    alternate = ["text", "amount", "date", (0, 0.7), (OTSU, 1e30), (SHARPEN | BLUR, 2.0)]
    batches = {
        "on span boundaries": [(32, 32)] * 6,
        "spans inside crops": [(1, 1)] + [(32, 32)] * 4 + [(40, 50), (33, 31), (1, 3), (64, 64)],
        "alternating in a span": [(4, 4)] * 130 + [(1, 1)] * 600 + [(2, 3), (3, 2)] * 20,
    }
    for what, sizes in batches.items():
        kinds = [alternate[i % len(alternate)] for i in range(len(sizes))]
        table, _, out_bytes, _ = enhance.plan(sizes, kinds)
        starts = [t.out_off for t in table]
        if what == "on span boundaries":
            assert all(s % SPAN == 0 for s in starts)
        elif what == "spans inside crops":
            # results that start off a span boundary and run into the next span
            inside = [t for t in table
                      if t.out_off % SPAN and t.out_off // SPAN != (t.out_off + 16 * t.h * t.w - 1) // SPAN]
            assert len(inside) >= 4
        else:
            span_kinds = {}
            for t, k in zip(table, kinds):
                span_kinds.setdefault(t.out_off // SPAN, set()).add(bool(_recipe(k)[0] & OTSU))
            assert sum(v == {True, False} for v in span_kinds.values()) >= 2
        crops = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
        got = _enhance(crops, kinds)
        for i, (c, g, k) in enumerate(zip(crops, got, kinds)):
            _check(g, _oracle(c, k), f"{what}: crop {i} {c.shape} {k}")
