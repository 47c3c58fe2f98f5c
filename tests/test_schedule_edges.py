"""The forward at the edges of its tile schedule, at every production batch size, and the grid-stride paths of the
warp and resize kernels.

Every tensor-core launch of the forward is persistent: `build_plan` (csrc/unet_b200.cu) turns a shape into U work
units (8 x 16 pixel M tiles, or pairs of them for CTA pairs, times column blocks, times phase groups for the folded
decoder levels), launches min(U, S) CTAs (S = number of SMs, halved for pairs), and each CTA walks units
`u += unit_stride`.  Its mbarrier rings and TMEM accumulator buffers wrap at counts that follow from U and S, so the
walk goes wrong, if anywhere, at its edges: one wave exactly, one unit past it, a CTA with one unit less than its
neighbours, an odd or even number of units per CTA, a CTA pair whose second M tile is missing.  `_schedule` restates
the unit count of every launch of the default plan (as `_ws_layout` of test_layer_audit restates `ws_layout`), and a
greedy cover picks a short list of ordinary shapes that puts every launch on each of those edges it can reach at
production memory.  The profiler proves the model on the hardware (each launch's grid), the per-launch audit of
test_layer_audit is the oracle at those shapes, and batched == per-image forwards is checked bit for bit at every
batch size the batched entry points run (1 .. MAX_CHUNK).

The default plan has no launch of the row kernel (conv_row.cuh): it serves conv1.net.0 only when level 1 is not
folded (`row64` bit 1), and the default plan folds it into the phase-stacked kernel; the model covers the 18 launches
that do run.
"""
import functools
import json
import math
import time

import numpy as np
import pytest
import torch

from test_layer_audit import _failures, _summary, _ws_layout, audit

THR = [0.25, 0.40, 0.30]
NUM_SMS_B200 = 148
SIDES = tuple(range(16, 1025, 16))
MAX_N = 64
CAP_SHAPE = (64, 512, 512)             # production batch: the memory cap of the shape search
MAX_SHAPES = 40

# The launches of the default plan (fold_up = 15, ps64 = 3, row64 = 2, stem_tc = 1, pair = 2, bn_max = 256), in
# launch order: layer name, launch kind, resolution level, input channels, output channels.  A folded level reads the
# low-resolution tensor: its level is that tensor's, its input channels are the low tensor's.
PLAN = [
    ("down1.net.0", "stem", 0, 3, 64),
    ("down1.net.3", "ps64", 0, 64, 64),
    ("down2.net.0", "conv", 1, 64, 128), ("down2.net.3", "conv", 1, 128, 128),
    ("down3.net.0", "conv", 2, 128, 256), ("down3.net.3", "conv", 2, 256, 256),
    ("down4.net.0", "conv", 3, 256, 512), ("down4.net.3", "conv", 3, 512, 512),
    ("bottleneck.net.0", "conv", 4, 512, 1024), ("bottleneck.net.3", "conv", 4, 1024, 1024),
    ("conv4.net.0", "fold", 4, 1024, 512), ("conv4.net.3", "conv", 3, 512, 512),
    ("conv3.net.0", "fold", 3, 512, 256), ("conv3.net.3", "conv", 2, 256, 256),
    ("conv2.net.0", "fold", 2, 256, 128), ("conv2.net.3", "conv", 1, 128, 128),
    ("conv1.net.0", "fold", 1, 128, 64), ("conv1.net.3", "head", 0, 64, 64),
]
CLASSES = ["U=1", "1<U<S", "U=S", "U=S+1", "q>=2 U%S=S-1", "q>=2 U%S=0", "q>=2 U%S=1", "q odd>=3", "q even>=2",
           "pair m_tiles odd", "fill_sms flip"]


# ---------------------------------------------------------------------------------------------------- the model
def _cdiv(a, b):
    return -(-a // b)


def _conv_eff(b):
    return np.where(b == 256, 0.97, np.where(b == 128, 0.95, 0.70))


def _launch(kind, lvl, cin, cout, n, H, W, S, fill_sms):
    """One launch of the plan at (n, H, W) (numpy int64 arrays, element-wise): dict of family, bn, pair, m_tiles,
    units, slots, grid, as build_stem_tc_step / build_ps64_step / build_conv_step / build_phase_step compute them."""
    h, w = H >> lvl, W >> lvl
    ones = np.ones_like(n)
    if kind == "stem":                   # tensor-core stem: unpaired, one 64-column block, 8 x 16 pixel tiles
        m = _cdiv(w, 8) * _cdiv(h, 16) * n
        return dict(family="stem_tc", bn=64 * ones, pair=False, m_tiles=m, units=m, slots=S, grid=np.minimum(m, S))
    if kind in ("ps64", "head"):         # phase-stacked 64 -> 64 kernel: tiles of the 2 x 2 block grid, CTA pairs
        m = _cdiv(w // 2, 8) * _cdiv(h // 2, 16) * n
        u = (m + 1) // 2
        return dict(family="ps64" if kind == "ps64" else "head (ps64)", bn=64 * ones, pair=True, m_tiles=m, units=u,
                    slots=S // 2, grid=2 * np.minimum(u, S // 2))
    m = _cdiv(w, 8) * _cdiv(h, 16) * n
    mu, slots = (m + 1) // 2, S // 2     # every launch below runs as CTA pairs in the default plan
    bn0 = min(256, cout)
    while cout % bn0:
        bn0 >>= 1
    if kind == "conv":
        # build_conv_step: fill_sms narrows the column block while waves x width / efficiency drops by > 3 %
        best = np.full_like(n, bn0)
        if fill_sms:
            def cost(b):
                return _cdiv(mu * (cout // b), slots).astype(np.float64) * b / _conv_eff(b)
            b = bn0 >> 1
            while b >= 64:
                if cout % b == 0:
                    best = np.where(cost(np.full_like(n, b)) < 0.97 * cost(best), b, best)
                b >>= 1
        u = mu * (cout // best)
        return dict(family="conv", bn=best, pair=True, m_tiles=m, units=u, slots=slots, grid=2 * np.minimum(u, slots))
    # build_phase_step: a 256-column level may take 128-column blocks on the same one-phase kernel
    assert kind == "fold"
    bn = np.full_like(n, bn0)
    narrow = np.zeros(n.shape, dtype=bool)
    if fill_sms and bn0 == 256 and cout % 128 == 0:
        def cost(b, eff):
            return _cdiv(mu * 4 * (cout // b), slots).astype(np.float64) * b / eff
        narrow = cost(128, 0.70) < 0.97 * cost(256, 0.985)
        bn = np.where(narrow, 128, bn)
    if bn0 == 256:
        family, nph = "fold 1-phase", np.ones_like(n)
    elif bn0 == 128:
        family, nph = "fold multi-phase", np.full_like(n, 2)
    else:
        family, nph = ("fold stacked" if cout == 64 else "fold multi-phase"), np.full_like(n, 4)
    u = mu * (4 // nph) * (cout // bn)
    return dict(family=family, bn=bn, pair=True, m_tiles=m, units=u, slots=slots, grid=2 * np.minimum(u, slots))


def _schedule(n, H, W, num_sms=NUM_SMS_B200, fill_sms=1):
    """Every launch of the default plan at (n, H, W) (ints or int64 arrays): list of `_launch` dicts with `name`."""
    n, H, W = (np.asarray(v, dtype=np.int64) for v in (n, H, W))
    out = []
    for name, kind, lvl, cin, cout in PLAN:
        d = _launch(kind, lvl, cin, cout, n, H, W, num_sms, fill_sms)
        d.update(name=name, kind=kind, level=lvl, cin=cin, cout=cout)
        out.append(d)
    return out


def _ws_bytes(n, H, W, bw=64):
    """`_ws_layout(...)["total"]`, element-wise over int64 arrays."""
    r = lambda e: (e * 2 + 1023) // 1024 * 1024
    px = lambda k: n * (H >> k) * (W >> k)
    tot = sum(r(px(k) * (bw << k)) for k in range(5))                   # a
    tot = tot + sum(r(px(k) * (bw << k)) for k in range(4))             # c
    tot = tot + sum(r(px(k + 1) * (bw << k)) for k in range(4))         # p
    tot = tot + r(px(4) * (bw << 4))                                    # bt
    tot = tot + sum(r(px(k) * (bw << k)) for k in range(4))             # ca
    return tot + sum(r(px(k) * (bw << k)) for k in range(1, 4))         # cc


def _classes(d, flip):
    """Boolean arrays, one per CLASSES entry, of the launch `d` (and its fill_sms flip array)."""
    U, S = d["units"], d["slots"]
    q = _cdiv(U, S)
    r = U % S
    false = np.zeros(U.shape, dtype=bool)
    return [U == 1, (U > 1) & (U < S), U == S, U == S + 1, (q >= 2) & (r == S - 1), (q >= 2) & (r == 0),
            (q >= 2) & (r == 1), (q >= 3) & (q % 2 == 1), (q >= 2) & (q % 2 == 0),
            (d["m_tiles"] % 2 == 1) if d["pair"] else false, flip]


def _space():
    """The searched shapes (n, H, W), n-fastest, within the workspace of the production batch."""
    H, W, n = np.meshgrid(np.array(SIDES), np.array(SIDES), np.arange(1, MAX_N + 1), indexing="ij")
    n, H, W = n.ravel().astype(np.int64), H.ravel().astype(np.int64), W.ravel().astype(np.int64)
    keep = _ws_bytes(n, H, W) <= _ws_bytes(*(np.int64(v) for v in CAP_SHAPE))
    return n[keep], H[keep], W[keep]


@functools.lru_cache(maxsize=None)
def _cover(num_sms=NUM_SMS_B200):
    """Greedy cover of the reachable (launch, edge class) pairs.  Returns (shapes, flips, table, unreachable):
    `shapes` the chosen (n, H, W) in choice order, a chosen shape's fill_sms flip partner (n + 1, H, W) right after
    it; `flips` the (lower, upper) flip pairs; `table` (launch, class) -> first chosen shape in it; `unreachable`
    (launch, class) -> reason."""
    n, H, W = _space()
    cap = _ws_bytes(*(np.int64(v) for v in CAP_SHAPE))
    at = _schedule(n, H, W, num_sms)
    up = _schedule(np.minimum(n + 1, MAX_N), H, W, num_sms)
    up_ok = (n < MAX_N) & (_ws_bytes(n + 1, H, W) <= cap)
    cols, names = [], []
    for d, e in zip(at, up):
        flip = up_ok & (d["bn"] != e["bn"])
        for c, v in zip(CLASSES, _classes(d, flip)):
            cols.append(v)
            names.append((d["name"], c))
    cov = np.stack(cols, 1)
    reach = cov.any(0)
    pix = n * H * W
    index = {(int(a), int(b), int(c)): i for i, (a, b, c) in enumerate(zip(n, H, W))}
    shapes, flips, table = [], [], {}
    todo = reach.copy()
    flip_cols = [j for j, (_, c) in enumerate(names) if c == "fill_sms flip"]

    def take(i):
        s = (int(n[i]), int(H[i]), int(W[i]))
        if s not in shapes:
            shapes.append(s)
        for j in np.flatnonzero(cov[i] & todo):
            table[names[j]] = s
        todo[cov[i]] = False

    while todo.any():
        cols_left = np.flatnonzero(todo)
        gain = cov[:, cols_left].sum(1, dtype=np.int64)
        i = int(np.argmax(gain * (1 << 40) - pix))             # most new pairs; ties: the fewest pixels, then order
        new_flip = [j for j in flip_cols if cov[i, j] and todo[j]]
        take(i)
        if new_flip:                                           # a flip is a pair of shapes: run the partner too
            s = shapes[-1]
            partner = (s[0] + 1, s[1], s[2])
            flips.append((s, partner))
            take(index[partner])
    unreachable = {}
    for j, (name, c) in enumerate(names):
        if reach[j]:
            continue
        d = at[[p[0] for p in PLAN].index(name)]
        q = _cdiv(d["units"], d["slots"])
        if c == "fill_sms flip":
            why = "bn never changes between n and n + 1"
        elif c == "pair m_tiles odd":
            why = "unpaired launch" if not d["pair"] else "m_tiles always even"
        else:
            why = (f"U in {int(d['units'].min())}..{int(d['units'].max())}, always a multiple of "
                   f"{int(np.gcd.reduce(d['units']))}; q <= {int(q.max())}; S = {int(d['slots'])}")
        unreachable[(name, c)] = why
    return shapes, flips, table, unreachable


def _print_table(table, unreachable):
    w = max(len(c) for c in CLASSES)
    for name, *_ in PLAN:
        print(f"{name}:")
        for c in CLASSES:
            if (name, c) in table:
                print(f"    {c:{w}s}  {'x'.join(map(str, table[(name, c)]))}")
            else:
                print(f"    {c:{w}s}  unreachable: {unreachable[(name, c)]}")


# ---------------------------------------------------------------------------------------------------- CPU tests
def test_ws_model_matches_layout():
    """The vectorised workspace size is test_layer_audit's `_ws_layout` (the restatement of `ws_layout`)."""
    shapes = [(1, 16, 16), (64, 512, 512), (3, 1024, 48), (17, 272, 800), (5, 1008, 16)]
    for s in shapes:
        assert int(_ws_bytes(*(np.int64(v) for v in s))) == _ws_layout(*s)["total"], s


def test_schedule_model_basics():
    """Hand-checked points of the model: a 512^2 batch of 64 keeps the wide blocks and fills every SM; batch 1
    narrows the deep layers (fill_sms) and folded level 4 takes the 128-column one-phase kernel."""
    big = {d["name"]: d for d in _schedule(64, 512, 512)}
    assert int(big["down1.net.0"]["units"]) == 64 * 64 * 32 and int(big["down1.net.0"]["grid"]) == 148
    assert int(big["bottleneck.net.3"]["bn"]) == 256 and int(big["bottleneck.net.3"]["units"]) == 64 * 4 * 2 // 2 * 4
    one = {d["name"]: d for d in _schedule(1, 512, 512)}
    assert int(one["bottleneck.net.3"]["bn"]) == 64 and int(one["bottleneck.net.3"]["units"]) == 4 * 16
    assert int(one["conv4.net.0"]["bn"]) == 128 and one["conv4.net.0"]["family"] == "fold 1-phase"
    off = {d["name"]: d for d in _schedule(1, 512, 512, fill_sms=0)}
    assert int(off["bottleneck.net.3"]["bn"]) == 256 and int(off["conv4.net.0"]["bn"]) == 256
    assert {d["family"] for d in _schedule(1, 64, 64)} == {
        "stem_tc", "ps64", "conv", "fold 1-phase", "fold multi-phase", "fold stacked", "head (ps64)"}


def test_cover_is_complete_short_and_deterministic():
    t0 = time.time()
    shapes, flips, table, unreachable = _cover()
    _print_table(table, unreachable)
    print(f"{len(shapes)} shapes ({len(flips)} fill_sms flip pairs), {len(table)} (launch, class) pairs covered, "
          f"{len(unreachable)} unreachable, {time.time() - t0:.1f} s:")
    print("  " + " ".join("x".join(map(str, s)) for s in shapes))
    assert len(table) + len(unreachable) == len(PLAN) * len(CLASSES)
    assert len(shapes) <= MAX_SHAPES
    cap = _ws_layout(*CAP_SHAPE)["total"]
    for n, h, w in shapes:
        assert 1 <= n <= MAX_N and h in SIDES and w in SIDES and _ws_layout(n, h, w)["total"] <= cap
    # every covered pair really holds at its shape, recomputed one shape at a time
    for (name, c), (n, h, w) in table.items():
        i = [p[0] for p in PLAN].index(name)
        d = _schedule(n, h, w)[i]
        flip = np.array(int(d["bn"]) != int(_schedule(n + 1, h, w)[i]["bn"])) if n < MAX_N else np.array(False)
        assert bool(_classes(d, flip)[CLASSES.index(c)]), (name, c, (n, h, w))
        if c == "fill_sms flip":
            assert ((n, h, w), (n + 1, h, w)) in flips
    again = _cover.__wrapped__()
    assert again == (shapes, flips, table, unreachable)


# ---------------------------------------------------------------------------------------------------- GPU fixtures
@pytest.fixture(scope="module")
def engine(fixture_state, cuda_dev):
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    e = Engine(fixture_state, cuda_dev)
    yield e
    e.close()


@pytest.fixture(scope="module")
def gpu_cover(engine):
    """The cover for the device's SM count, with the default options the model assumes checked on the handle."""
    defaults = dict(fold_up=15, ps64=3, row64=2, stem_tc=1, pair=2, bn_max=256, amode=2, fill_sms=1,
                    fold_stack=1, fold_one_phase=0)
    got = {k: engine.get_option(k) for k in defaults}
    assert got == defaults, got
    assert [l.name.decode() for l in engine.layers][:10] == [p[0] for p in PLAN[:10]]
    return engine.get_option("num_sms"), _cover(engine.get_option("num_sms"))


def _x(n, h, w, seed, u8=False):
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices, synthetic_invoices_u8
    if u8:
        return torch.from_numpy(synthetic_invoices_u8(n, h, w, seed=seed))
    return synthetic_invoices(n, h, w, seed=seed)


def _kernel_grids(engine, x, trace_path):
    """Grids of the library's kernels of one forward on a plan's first use (direct launches), in launch order."""
    from torch.profiler import ProfilerActivity, profile
    engine.set_option("graph", 1)                 # drops the cached plans: the forward below builds and launches
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        engine.run(x, thresholds=THR)
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(trace_path))
    with open(trace_path) as f:
        ev = json.load(f)["traceEvents"]
    ks = [e for e in ev if e.get("cat") == "kernel" and "ub::" in e.get("name", "")]
    ks.sort(key=lambda e: (e["args"].get("correlation", 0), e["ts"]))
    return [(e["name"].split("<")[0].replace("void ", ""), tuple(e["args"]["grid"])) for e in ks]


# ---------------------------------------------------------------------------------------------------- B: the model on the device
@pytest.mark.gpu
def test_profiler_grids_match_model(engine, gpu_cover, tmp_path):
    """Each launch's grid from the profiler trace equals the model's, at every chosen shape (both fill_sms policies
    at the flip shapes).  Below one wave the grid is the unit count itself, so this checks the unit formulas too."""
    num_sms, (shapes, flips, _, _) = gpu_cover
    flip_shapes = {s for p in flips for s in p}
    bad, count = [], 0
    keep = engine.get_option("fill_sms")
    try:
        for s in shapes:
            for fill in ((1, 0) if s in flip_shapes else (1,)):
                engine.set_option("fill_sms", fill)
                got = _kernel_grids(engine, _x(*s, seed=7).to(engine.device), tmp_path / "trace.json")
                want = [(int(d["grid"]), 1, 1) for d in _schedule(*s, num_sms=num_sms, fill_sms=fill)]
                count += len(want)
                if [g for _, g in got] != want:
                    bad.append((s, fill, [(k, g, w) for (k, g), w in zip(got, want) if g != w], len(got)))
    finally:
        engine.set_option("fill_sms", keep)
    print(f"profiler grids: {count} launches over {len(shapes)} shapes compared with the model, {len(bad)} mismatches")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------- C: audit at the edges
@pytest.mark.gpu
def test_audit_at_schedule_edges(engine, gpu_cover):
    """Every launch of the default plan audited (test_layer_audit's gates) at every chosen shape, direct and replayed;
    fp32 NCHW inputs, uint8 NHWC at every fifth shape.  Prints the worst normalised error and mismatch fraction per
    edge class."""
    num_sms, (shapes, _, _, _) = gpu_cover
    worst = {c: [0.0, 0.0] for c in CLASSES}
    fails = []
    t0 = time.time()
    for k, s in enumerate(shapes):
        u8 = k % 5 == 4
        x = _x(*s, seed=500 + k, u8=u8).to(engine.device)
        label = f"edges {'u8' if u8 else 'f32'} {'x'.join(map(str, s))}"
        rows = audit(engine, x, {}, label=label)
        print(f"audit {label}: {_summary(rows)}")
        fails += [(label,) + f for f in _failures(rows)]
        sched = _schedule(*s, num_sms=num_sms)
        nxt = _schedule(s[0] + 1, s[1], s[2], num_sms=num_sms)
        for r in rows:
            d, e = sched[r["launch"]], nxt[r["launch"]]
            assert d["name"] == r["name"], (d["name"], r["name"])
            for c, v in zip(CLASSES, _classes(d, np.array(int(d["bn"]) != int(e["bn"])))):
                if bool(v):
                    worst[c][0] = max(worst[c][0], r["max_norm"])
                    worst[c][1] = max(worst[c][1], r["mismatch"])
    for c, (e, m) in worst.items():
        print(f"edge class {c:14s}: worst normalised error {e:.4f}, worst mismatch fraction {m:.2e}")
    print(f"audit of {len(shapes)} edge shapes: {time.time() - t0:.1f} s")
    assert not fails, fails


@pytest.mark.gpu
def test_fill_sms_flip_bit_identical(engine, gpu_cover):
    """On both sides of every change of the chosen column block, fill_sms = 0 and 1 give the same bits."""
    _, (_, flips, _, _) = gpu_cover
    keep = engine.get_option("fill_sms")
    try:
        for pair in flips:
            for s in pair:
                x = _x(*s, seed=600).to(engine.device)
                out = []
                for fill in (0, 1):
                    engine.set_option("fill_sms", fill)
                    z, m = engine.run(x, thresholds=THR)
                    out.append((z, m))
                torch.cuda.synchronize()
                assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), s
    finally:
        engine.set_option("fill_sms", keep)


# ---------------------------------------------------------------------------------------------------- D: batch invariance
def _first_diff(got, want):
    idx = (got != want).nonzero()[0].tolist()
    return f"first differing element {tuple(idx)}: {got[tuple(idx)].item()} vs {want[tuple(idx)].item()} alone"


def _sweep(engine, images, solo, n_max, seed, **kw):
    """Batches n = 1 .. n_max of images (s_n + j) mod len(images), each run twice (direct, then the graph replay)
    with its outputs refilled in between; every image's outputs must equal its solo outputs bit for bit."""
    g = np.random.default_rng(seed)
    m = images.shape[0]
    for n in range(1, n_max + 1):
        s_n = int(g.integers(m))
        idx = torch.tensor([(s_n + j) % m for j in range(n)], device=images.device)
        x = images[idx].contiguous()
        want = [None if t is None else t[idx] for t in solo]
        outs = [None if t is None else torch.empty_like(t) for t in want]
        for run in ("direct", "replay"):
            if outs[0] is not None:
                outs[0].fill_(float("nan"))
            outs[1].fill_(0xA5)
            engine.run(x, want_logits=outs[0] is not None, thresholds=THR, logits_out=outs[0], mask_out=outs[1], **kw)
            torch.cuda.synchronize()
            for what, got, ref in zip(("logits", "masks"), outs, want):
                if got is None or torch.equal(got, ref):
                    continue
                j = next(j for j in range(n) if not torch.equal(got[j], ref[j]))
                pytest.fail(f"{run} batch n={n}: {what} of position {j} (image {int(idx[j])}) differ from the "
                            f"image alone; {_first_diff(got[j], ref[j])}")


def _solo(engine, images, **kw):
    """Each image's (logits | None, masks) from a forward of its own (n = 1)."""
    z, m = [], []
    want_logits = kw.pop("want_logits", True)
    for i in range(images.shape[0]):
        a, b = engine.run(images[i:i + 1].contiguous(), want_logits=want_logits, thresholds=THR, **kw)
        z.append(a)
        m.append(b)
    torch.cuda.synchronize()
    return (torch.cat(z) if want_logits else None), torch.cat(m)


def _max_chunk():
    from tw_invoice_unet_ocr_llm_b200 import inference, launcher
    assert inference.MAX_CHUNK == launcher.MAX_CHUNK
    return inference.MAX_CHUNK


@pytest.mark.gpu
def test_batch_invariance_u8_every_chunk_size(engine):
    """The uint8 NHWC path of run_unet_batch and MultiGpuSegmenter: logits + byte masks, and bit-packed masks alone,
    at every batch size 1 .. MAX_CHUNK, equal the images' solo outputs."""
    mc = _max_chunk()
    t0 = time.time()
    images = _x(64, 512, 512, seed=900, u8=True).to(engine.device)
    _sweep(engine, images, _solo(engine, images), mc, seed=901)
    _sweep(engine, images, (None, _solo(engine, images, want_logits=False, mask_bits=True)[1]), mc, seed=902,
           mask_bits=True)
    print(f"batch invariance uint8 NHWC, n = 1..{mc}: {time.time() - t0:.1f} s")


@pytest.mark.gpu
def test_batch_invariance_f32_every_chunk_size(engine):
    """The fp32 NCHW path of the drop-in UNet.forward at every batch size 1 .. MAX_CHUNK, and 1024^2 (BASELINE
    configs[3]) at n = 1 .. 16."""
    mc = _max_chunk()
    t0 = time.time()
    images = _x(64, 512, 512, seed=910).to(engine.device)
    _sweep(engine, images, _solo(engine, images), mc, seed=911)
    images = _x(16, 1024, 1024, seed=912).to(engine.device)
    _sweep(engine, images, _solo(engine, images), 16, seed=913)
    print(f"batch invariance fp32 NCHW: {time.time() - t0:.1f} s")


# ---------------------------------------------------------------------------------------------------- E: byte kernels
def _frame(h, w, seed):
    rng = np.random.default_rng(seed)
    f = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    f[h // 8:h - h // 8, w // 8:w - w // 8] = (np.arange(w - 2 * (w // 8), dtype=np.int64)[None, :, None] * 7 % 256
                                               ).astype(np.uint8)
    return f


def _centred(w, h, angle, cx, cy):
    """Inverse map of a w x h crop rotated by `angle` degrees about (cx, cy) of the frame (sub-pixel centre)."""
    t = math.radians(angle)
    c, s = math.cos(t), math.sin(t)
    return np.array([[c, -s, cx - (c * w / 2 - s * h / 2)], [s, c, cy - (s * w / 2 + c * h / 2)]])


@pytest.mark.gpu
def test_warp_crops_grid_stride(cuda_dev):
    """Crops of more than 512 tiles (the kernel's grid.x cap: each block walks several tiles and carries the crop's
    byte sum across them) from a 3840 x 2160 frame, mixed with 1 x 1 and 33 x 9 crops in one call, RGB and RGBX."""
    import cv2
    from oracle import oriented as orc
    from tw_invoice_unet_ocr_llm_b200 import prepost
    host = _frame(2160, 3840, 31)
    cases = []
    for w, h in ((2600, 220), (1500, 900)):
        for ang in (0, 7, -33, 90):
            cases.append((_centred(w, h, ang, 1920.37, 1080.61), w, h))
    cases.insert(3, (_centred(1, 1, 12, 100.5, 200.25), 1, 1))
    cases.insert(6, (_centred(33, 9, -4, 3000.1, 500.9), 33, 9))
    assert max(math.ceil(w / 32) * math.ceil(h / 8) for _, w, h in cases) > 4 * 512
    rgbx = np.concatenate([host, np.full(host.shape[:2] + (1,), 201, np.uint8)], axis=2)
    refs = [orc.warp_affine(host, M, w, h) for M, w, h in cases]
    for frame in (host, rgbx):
        dev = torch.from_numpy(frame).to(cuda_dev)
        crops, sums = prepost.warp_crops(dev, [c[0] for c in cases], [(c[1], c[2]) for c in cases])
        sums = sums.cpu().numpy()
        for k, ((M, w, h), crop, ref) in enumerate(zip(cases, crops, refs)):
            got = crop.cpu().numpy()
            assert got.shape == (h, w, 3) and np.array_equal(got, ref), (frame.shape, k, w, h, int((got != ref).sum()))
            assert int(sums[k]) == int(ref.astype(np.int64).sum()), (frame.shape, k)
    M, w, h = cases[1]
    cv = cv2.warpAffine(host, M, (w, h), flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP, borderMode=cv2.BORDER_REPLICATE)
    assert np.array_equal(refs[1], cv)


@pytest.mark.gpu
def test_resize_u8_launch_split(cuda_dev):
    """unetb200_resize_bicubic_u8_ps runs the horizontal pass as one launch while n * h <= 65535 and one launch per
    image beyond; both sides of the split, per frame against Pillow (3 channels) or the oracle (4 channels)."""
    from PIL import Image
    from oracle.pillow_resample import resize_u8 as oracle_resize
    from tw_invoice_unet_ocr_llm_b200 import prepost
    rng = np.random.default_rng(41)
    pil = lambda f: np.asarray(Image.fromarray(f).resize((512, 512)))
    for n, h, w in ((15, 4369, 64), (16, 4096, 64)):
        frames = rng.integers(0, 256, (n, h, w, 4), dtype=np.uint8)
        frames[:, ::7] = 250
        dev = torch.from_numpy(frames).to(cuda_dev)
        got3 = prepost.resize_u8(dev[..., :3].contiguous(), 512, 512).cpu().numpy()
        gotx = prepost.resize_u8(dev, 512, 512, channels=3).cpu().numpy()
        got4 = prepost.resize_u8(dev, 512, 512).cpu().numpy()
        for i in range(n):
            assert np.array_equal(got3[i], pil(np.ascontiguousarray(frames[i, ..., :3]))), (n, h, i)
        assert np.array_equal(gotx, got3), (n, h)
        for i in (0, n - 1):
            assert np.array_equal(got4[i], oracle_resize(frames[i], 512, 512)), (n, h, i)
    frames = np.stack([_frame(1080, 1920, 50 + i) for i in range(64)])
    dev = torch.from_numpy(frames).to(cuda_dev)
    got = prepost.resize_u8(dev, 512, 512).cpu().numpy()
    for i in range(64):
        assert np.array_equal(got[i], pil(frames[i])), i
    rgbx = torch.cat([dev, torch.full(dev.shape[:3] + (1,), 9, dtype=torch.uint8, device=cuda_dev)], -1)
    assert np.array_equal(prepost.resize_u8(rgbx, 512, 512, channels=3).cpu().numpy(), got)
