"""Per-launch audit of the production forward, and the weight packing against the BatchNorm fold.

The unit tests (test_conv_kernels, test_fused_up) hold one kernel at a time to one bf16 rounding, but at toy shapes;
test_forward_parity runs the real plans at real shapes, but only against the fp32 oracle through loose end-to-end
gates (bf16 storage compounds over 23 layers).  This file closes the gap between them.  After a forward every launch's
operands are still in the caller's workspace (layout: `_ws_layout`, a restatement of `ws_layout` in
csrc/unet_b200.cu) and its packed weights in the blob, so each launch of the real plan is checked against a float64
reference computed from exactly the bf16 / fp32 operands the kernel read.  Errors do not compound across launches
here, and a wrong launch is named, not merely noticed.

Gates, for every element of every audited output:
  1. no NaN is left: the workspace is filled with 0xFF (bf16 NaN), the logits with NaN and the masks with 7
     before the forward, so an unwritten element fails (checked over the whole batch);
  2. |got - ref| <= 2^-7 |ref| + 2^-14 S, with S = conv(|x|, |w|) + |b| in float64: one bf16 output rounding with
     2x margin, plus fp32 accumulation-order noise bounded by the size of the sum.  bf16 keeps 8 significand bits,
     so one rounding to nearest moves a value by up to 2^-8 of it (not 2^-9): a first term of 2^-8 |ref| has no
     margin at all, and the stem (K = 27, so S adds almost nothing) measured 0.97 of that bound.  2^-7 is also the
     unit tests' relative term.  For the fp32 logits the first term is 2^-23 |ref| and S is carried through the
     1x1 head (S_z = S_y |w_head| + |b_head|);
  3. got != bf16_rn(ref) for at most 1 % of a launch's elements (bf16 outputs; accumulation order moves only
     results that sit next to a rounding boundary);
  4. exact relations: pooled outputs == max_pool2d of the stored output, masks == logits > threshold,
     bit-packed masks == byte masks.
The "normalised error" printed per launch is max |got - ref| / (gate 2's bound): the launch passes at <= 1.

What the kernel reads, per launch kind: 3x3 convs the bf16 activations (two sources for the decoder convs) and the
bf16 blob weights [tap][Cout][Cin] + fp32 bias, then ReLU; folded decoder levels `_same_operand_ref` of test_fused_up
with the composite weights and bias9; unfolded up-convs a ConvTranspose over the blob's [(a,b,co)][ci]; the
tensor-core stem the hi/lo split (x_hi = bf16(x), x_lo = bf16(x - x_hi), w_hi (x_hi + x_lo) + w_lo x_hi + the bias
slot at k = 9 Cin); the CUDA-core stem the fp32 [k][64] weights; the head the fp32 accumulator of conv1.net.3 (never
rounded to bf16) and the fp32 out_conv weights.  A plan with an unfolded level k writes the up-conv output u[k]
over a[k]: the launches that write and read a[k] cannot be audited from the workspace there and are listed as
skipped (the default plan audits them).  Each case runs the plan twice: direct launches, then the CUDA-graph replay,
with the NaN fill renewed in between; the replay is audited again (references are reused only where a launch's
inputs are bitwise those of the first run).  At batch > 3 the float64 references cover images {0, one seeded, N-1}
of the full batch-N forward; the NaN and exact-relation gates cover every image.

Measured on one B200 (1000 W power limit), every case of this file, direct and replayed runs alike:
  * gate 2, bf16 outputs: worst normalised error 0.47-0.49 per case, always at the stem (down1.net.0, where one
    bf16 rounding is all there is) or the up-convs; that is one rounding of 2^-8 against the 2^-7 bound;
  * gate 2, fp32 logits: worst 0.0016 (the bound is set by the accumulation term; one fp32 rounding is far below it);
  * gate 3: worst mismatch fraction 2.4e-3 (bottleneck.net.3, K = 9216; 7e-4 to 2.4e-3 across cases) against the
    1 % gate.  It grows with K, as reordered fp32 sums predict; the 1e-4 guessed before measuring was too low;
  * gates 1 and 4: no unwritten element, every exact relation holds;
  * corrupted blob: one zeroed 64-channel K slice of the centre tap of bottleneck.net.3 gives 144x the bound and
    51 % mismatches at that launch alone; +0.05 on bias9's top-edge case at level 2 gives 123x at conv2.net.0 alone.
    The same forwards against the fp32 oracle at 1 x 512^2 (test_forward_parity's gates in brackets):
    max-abs 0.241 / 0.183 (0.25), max-abs / std 0.183 / 0.139 (0.19), mean-abs 0.020 / 0.013 (0.025),
    agreement 99.93 % / 99.95 % (99.9 %), IoU >= 0.975 / 0.981 (0.95).  Both pass every end-to-end gate.
The whole file runs in about 20 s on one B200 (the float64 references are cuBLAS / cuDNN float64 on the device).

The packing audit compares every layer of the blob with the fold computed in torch fp32 (s = gamma / sqrt(var + eps),
w s rounded to bf16; every fp32 operation correctly rounded, as pack.cuh does it): bit for bit for the weights and
the stem's hi/lo rows, and for the folded biases equal to (b - mean) s + beta either unfused or as one FMA (nvcc may
contract it; under cancellation the two differ by more than 1 ulp, so a 1-ulp gate would be wrong), in the layouts
of csrc/pack.cuh.
"""
import contextlib
import ctypes as C
import time

import pytest
import torch
import torch.nn.functional as F

from test_fused_up import EPS, _bias9_ref, _composite_ref, _same_operand_ref

pytestmark = pytest.mark.gpu

THR = [0.25, 0.40, 0.30]
DEFAULT_SHAPES = [(64, 512, 512), (1, 512, 512), (16, 1024, 1024), (1, 1024, 768), (3, 64, 96), (2, 16, 16),
                  (2, 32, 1024), (2, 1024, 32), (5, 48, 272)]
SWEEP_SHAPES = [(3, 64, 96), (2, 512, 512)]
SWEEP = [
    {"pair": 0}, {"ps64": 0, "row64": 0}, {"ps64": 0, "row64": 1}, {"row64": 3},
    {"fold_up": 0}, {"fold_up": 5}, {"fold_up": 10}, {"fold_stack": 0}, {"fold_one_phase": 1}, {"stem_tc": 0},
    {"amode": 0}, {"wstat": 0}, {"bn_max": 64}, {"bn_max": 128}, {"epi2": 2}, {"fill_sms": 0}, {"fill_sms": 2},
    {"pdl": 0},
]
ARCHS = [(1, 2), (4, 5), (3, 8), (3, 1)]
SMALL = (2, 32, 48)


def _nat():
    from tw_invoice_unet_ocr_llm_b200 import _native as nat
    return nat


# ---------------------------------------------------------------------------------------------------- workspace map
def _ws_layout(n, h, w, bw=64):
    """`ws_layout` (csrc/unet_b200.cu): byte offsets of the bf16 NHWC regions, each rounded up to 1024 bytes.
    Level k has (h >> k) x (w >> k) pixels and bw << k channels; u[k] aliases a[k]; cc[0] is not allocated
    (level 0's second decoder conv is fused with the head)."""
    off = 0

    def take(elems):
        nonlocal off
        o = off
        off = (off + elems * 2 + 1023) // 1024 * 1024
        return o

    px = lambda k: n * (h >> k) * (w >> k)
    L = {"a": [take(px(k) * (bw << k)) for k in range(5)]}
    L["c"] = [take(px(k) * (bw << k)) for k in range(4)]
    L["p"] = [take(px(k + 1) * (bw << k)) for k in range(4)]
    L["bt"] = [take(px(4) * (bw << 4))]
    L["u"], L["ca"], L["cc"] = list(L["a"][:4]), [], []
    for k in range(4):
        L["ca"].append(take(px(k) * (bw << k)))
        L["cc"].append(None if k == 0 else take(px(k) * (bw << k)))
    L["total"] = off
    return L


def _region_shape(name, k, bw=64):
    """(level, channels) of a workspace region."""
    if name == "p":
        return k + 1, bw << k
    if name == "bt":
        return 4, bw << 4
    return k, bw << k


def _plan(n_channels, stem_tc, fold):
    """The launches of `build_plan` (csrc/unet_b200.cu) in order: kind, layer-table row, source / output regions.
    `fold` = the decoder levels whose up-conv is folded into the next conv (bit k: level k)."""
    P = []
    stem = "stem_tc" if stem_tc == 1 and n_channels <= 3 else "stem_cc"
    P.append(dict(kind=stem, li=0, src=[], out=("a", 0)))
    P.append(dict(kind="conv", li=1, src=[("a", 0)], out=("c", 0), pool=("p", 0)))
    for k in range(1, 4):
        P.append(dict(kind="conv", li=2 * k, src=[("p", k - 1)], out=("a", k)))
        P.append(dict(kind="conv", li=2 * k + 1, src=[("a", k)], out=("c", k), pool=("p", k)))
    P.append(dict(kind="conv", li=8, src=[("p", 3)], out=("a", 4)))
    P.append(dict(kind="conv", li=9, src=[("a", 4)], out=("bt", 0)))
    prev = ("bt", 0)
    for k in range(3, -1, -1):
        li_up = 10 + 3 * (3 - k)
        if fold >> k & 1:
            P.append(dict(kind="fold", li=li_up + 1, level=k + 1, src=[prev, ("c", k)], out=("ca", k)))
        else:
            # the up-conv output u[k] overwrites a[k]: its writer and its reader are not auditable in this plan
            for q in P:
                if q["out"] == ("a", k) or ("a", k) in q["src"]:
                    q["skip"] = f"a[{k}] overwritten by u[{k}]"
            P.append(dict(kind="convt", li=li_up, src=[prev], out=("u", k)))
            P.append(dict(kind="conv", li=li_up + 1, src=[("u", k), ("c", k)], out=("ca", k)))
        if k > 0:
            P.append(dict(kind="conv", li=li_up + 2, src=[("ca", k)], out=("cc", k)))
            prev = ("cc", k)
        else:
            P.append(dict(kind="head", li=21, src=[("ca", 0)], out=None))
    return P


class _Workspace:
    """A 1024-byte aligned workspace of exactly `unetb200_workspace_bytes`, readable region by region."""

    def __init__(self, engine, n, h, w):
        self.n, self.h, self.w = n, h, w
        self.L = _ws_layout(n, h, w)
        self.bytes = engine.workspace_bytes(n, h, w)
        assert self.bytes == self.L["total"], (n, h, w, self.bytes, self.L["total"])
        self.raw = torch.empty(self.bytes + 1024, dtype=torch.uint8, device=engine.device)
        self.ptr = (self.raw.data_ptr() + 1023) & ~1023
        s = self.ptr - self.raw.data_ptr()
        self.buf = self.raw[s:s + self.bytes]

    def region(self, reg):
        name, k = reg
        lvl, ch = _region_shape(name, k)
        off = self.L[name][k]
        shape = (self.n, self.h >> lvl, self.w >> lvl, ch)
        return self.buf[off:off + 2 * shape[0] * shape[1] * shape[2] * shape[3]].view(torch.bfloat16).view(shape)


# ---------------------------------------------------------------------------------------------------- references
@contextlib.contextmanager
def _default_dtype(dt):
    keep = torch.get_default_dtype()
    torch.set_default_dtype(dt)         # `_same_operand_ref` allocates its output with the default dtype
    try:
        yield
    finally:
        torch.set_default_dtype(keep)


def _conv3x3(x, w9):
    """x [H, W, Cin], w9 [9][Cout][Cin] (tap = ky * 3 + kx), zero padding 1 -> [H, W, Cout], in x's dtype."""
    h, w, cin = x.shape
    xp = F.pad(x, (0, 0, 1, 1, 1, 1))
    out = torch.zeros(h * w, w9.shape[1], dtype=x.dtype, device=x.device)
    for t in range(9):
        ky, kx = divmod(t, 3)
        out.addmm_(xp[ky:ky + h, kx:kx + w].reshape(h * w, cin), w9[t].T)
    return out.view(h, w, -1)


def _blob_bf16(blob, off, nbytes, shape):
    return blob[off:off + nbytes].view(torch.bfloat16).view(shape).double()


def _blob_f32(blob, off, nbytes, shape):
    return blob[off:off + nbytes].view(torch.float32).view(shape).double()


def _input_f32(x):
    """The network input as the kernels see it, fp32 [N, H, W, C]: uint8 is k / 255.0f, 16-bit floats widen exactly."""
    if x.dtype == torch.uint8:
        return (x.cpu().float() / 255.0).to(x.device)
    return x.float().permute(0, 2, 3, 1).contiguous()


class _Refs:
    """float64 (ref, S) of every launch kind, one image at a time, from the operands the kernel read."""

    def __init__(self, engine, blob):
        nat = _nat()
        self.layers, self.blob, self.nat = engine.layers, blob, nat
        self.arch = engine.arch
        self.ops = {}

    def _w(self, li):
        if li not in self.ops:
            l = self.layers[li]
            if l.kind == self.nat.CONV3X3:
                w = _blob_bf16(self.blob, l.w_off, l.w_bytes, (9, l.cout, l.cin))
            elif l.kind == self.nat.CONVT2X2:
                w = _blob_bf16(self.blob, l.w_off, l.w_bytes, (4, l.cout, l.cin))
            else:
                w = None
            self.ops[li] = (w, _blob_f32(self.blob, l.b_off, l.b_bytes, (l.cout,)))
        return self.ops[li]

    def conv(self, li, xs):
        w, b = self._w(li)
        x = torch.cat([t.double() for t in xs], -1)
        return F.relu(_conv3x3(x, w) + b), _conv3x3(x.abs(), w.abs()) + b.abs()

    def convt(self, li, x):
        w, b = self._w(li)
        x = x.double()
        h, wd, cin = x.shape
        ref = torch.empty(h, 2, wd, 2, w.shape[1], dtype=torch.float64, device=x.device)
        s = torch.empty_like(ref)
        xf, xa = x.reshape(-1, cin), x.reshape(-1, cin).abs()
        for a in range(2):
            for bb in range(2):
                ref[:, a, :, bb] = (xf @ w[2 * a + bb].T + b).view(h, wd, -1)
                s[:, a, :, bb] = (xa @ w[2 * a + bb].T.abs() + b.abs()).view(h, wd, -1)
        return ref.view(2 * h, 2 * wd, -1), s.view(2 * h, 2 * wd, -1)

    def fold(self, li, level, low, skip):
        key = ("fold", level)
        if key not in self.ops:
            off = [C.c_uint64() for _ in range(4)]
            self.nat.check(self.nat.lib().unetb200_fused_up_info(C.byref(self.arch), level, *[C.byref(o) for o in off]))
            w_off, w_bytes, b_off, b_bytes = [o.value for o in off]
            l = self.layers[li]
            c = l.cin // 2
            wc = _blob_bf16(self.blob, w_off, w_bytes, (16, l.cout, 2 * c))
            w3 = _blob_bf16(self.blob, l.w_off, l.w_bytes, (3, 3, l.cout, 2 * c))[:, :, :, c:].permute(2, 3, 0, 1)
            b9 = _blob_f32(self.blob, b_off, b_bytes, (9, l.cout))
            self.ops[key] = (wc, w3.contiguous(), b9)
        wc, w3, b9 = self.ops[key]
        lo = low.double().permute(2, 0, 1)[None]
        sk = skip.double().permute(2, 0, 1)[None]
        with _default_dtype(torch.float64):
            ref = _same_operand_ref(lo, sk, wc, w3, b9)
            s = _same_operand_ref(lo.abs(), sk.abs(), wc.abs(), w3.abs(), b9.abs(), relu=False)
        return ref[0].permute(1, 2, 0), s[0].permute(1, 2, 0)

    def stem(self, kind, x):
        """x: fp32 [H, W, Cin] as the kernel sees it."""
        l = self.layers[0]
        cin = l.cin
        if kind == "stem_cc":
            w = _blob_f32(self.blob, l.w_off, 9 * cin * 64 * 4, (9, cin, 64)).permute(0, 2, 1)
            b = _blob_f32(self.blob, l.b_off, l.b_bytes, (64,))
            xd = x.double()
            return F.relu(_conv3x3(xd, w) + b), _conv3x3(xd.abs(), w.abs()) + b.abs()
        off = l.w_off + int(self.nat.lib().unetb200_stem_tc_offset(cin))
        rows = _blob_bf16(self.blob, off, 64 * 128 * 2, (64, 128))
        w_hi = rows[:, :9 * cin].reshape(64, 9, cin).permute(1, 0, 2)
        w_lo = rows[:, 64:64 + 9 * cin].reshape(64, 9, cin).permute(1, 0, 2)
        b = rows[:, 9 * cin] + rows[:, 64 + 9 * cin]
        b_abs = rows[:, 9 * cin].abs() + rows[:, 64 + 9 * cin].abs()
        x_hi = x.to(torch.bfloat16).float()
        x_lo = (x - x_hi).to(torch.bfloat16).double()
        x_hi = x_hi.double()
        ref = _conv3x3(x_hi + x_lo, w_hi) + _conv3x3(x_hi, w_lo) + b
        s = _conv3x3(x_hi.abs() + x_lo.abs(), w_hi.abs()) + _conv3x3(x_hi.abs(), w_lo.abs()) + b_abs
        return F.relu(ref), s

    def head(self, x):
        """conv1.net.3 (fp32 accumulator, ReLU) then out_conv: logits [H, W, ncls] and their S."""
        y, sy = self.conv(21, [x])
        l = self.layers[22]
        hw = _blob_f32(self.blob, l.w_off, l.w_bytes, (l.cout, l.cin))
        hb = _blob_f32(self.blob, l.b_off, l.b_bytes, (l.cout,))
        return y @ hw.T + hb, sy @ hw.abs().T + hb.abs()


def _compare(got, ref, s, bf16_out=True):
    """(max normalised error, elements with got != bf16_rn(ref), elements)."""
    got = got.double()
    d = (got - ref).abs()
    den = (2.0 ** -7 if bf16_out else 2.0 ** -23) * ref.abs() + 2.0 ** -14 * s
    norm = torch.where(den > 0, d / den.clamp_min(1e-300), torch.where(d > 0, float("inf"), 0.0))
    if torch.isnan(got).any():
        norm = torch.full_like(norm, float("inf"))
    mism = int((got != ref.to(torch.bfloat16).double()).sum()) if bf16_out else 0
    return float(norm.max()), mism, got.numel()


def _images(n):
    """Images of a batch the float64 references cover: all up to 3, else the first, the last and one seeded."""
    if n <= 3:
        return list(range(n))
    g = torch.Generator().manual_seed(1000 + n)
    return [0, 1 + int(torch.randint(n - 2, (1,), generator=g)), n - 1]


# ---------------------------------------------------------------------------------------------------- the audit
def _forward(engine, handle, x, ws, logits, mask, mask_bits, thr):
    from tw_invoice_unet_ocr_llm_b200.engine import LOGITS_TYPES, input_format, logit_thresholds
    nat = _nat()
    fmt, xk = input_format(x)
    n, h, w = ws.n, ws.h, ws.w
    t = (C.c_float * len(thr))(*logit_thresholds(thr))
    ptr = lambda a: None if a is None else a.data_ptr()
    nat.check(nat.lib().unetb200_forward_typed(
        handle, xk.data_ptr(), fmt, n, h, w, ws.ptr, ws.bytes, ptr(logits),
        LOGITS_TYPES[torch.float32], ptr(mask), mask_bits, t, torch.cuda.current_stream().cuda_stream))


def _audit_run(engine, refs, plan, x, xf, ws, logits, mask, thr, label, run, cache):
    """Gates 1-4 for every launch of one forward whose results are in `ws` / `logits` / `mask`."""
    rows = []
    n = ws.n
    imgs = _images(n)
    for i, q in enumerate(plan):
        name = engine.layers[q["li"]].name.decode()
        row = dict(case=label, run=run, launch=i, name=name, kind=q["kind"], ok=True, why="")
        out = ws.region(q["out"]) if q["out"] is not None else logits
        # gate 1 over the whole batch (an overwritten output is the up-conv's, audited there)
        if q["out"] is not None and not (q.get("skip") and q["out"][0] == "a"):
            if torch.isnan(out.float()).any():
                row.update(ok=False, why="unwritten (NaN) outputs")
        if "pool" in q:
            c = ws.region(q["out"]).permute(0, 3, 1, 2)
            p = ws.region(q["pool"]).permute(0, 3, 1, 2)
            if not torch.equal(F.max_pool2d(c, 2), p):
                row.update(ok=False, why=row["why"] + " pooled output != max_pool2d(stored output)")
        if q["kind"] == "head":
            t = torch.tensor(_logit_thr(thr), dtype=torch.float32, device=logits.device).view(1, -1, 1, 1)
            if torch.isnan(logits).any():
                row.update(ok=False, why="unwritten (NaN) logits")
            if not torch.equal(mask, (logits > t).to(torch.uint8)):
                row.update(ok=False, why=row["why"] + " masks != logits > thr")
        if q.get("skip"):
            row.update(skipped=q["skip"], max_norm=float("nan"), mismatch=float("nan"))
            rows.append(row)
            continue
        worst, mism, tot = 0.0, 0, 0
        for b in imgs:
            srcs = [ws.region(r)[b] for r in q["src"]]
            key = (i, b)
            hit = cache.get(key)
            if hit is not None and all(torch.equal(u, v) for u, v in zip(hit[0], srcs)) and \
                    (q["kind"] not in ("stem_tc", "stem_cc") or torch.equal(hit[3], xf[b])):
                ref, s = hit[1], hit[2]
            else:
                if q["kind"] == "conv":
                    ref, s = refs.conv(q["li"], srcs)
                elif q["kind"] == "convt":
                    ref, s = refs.convt(q["li"], srcs[0])
                elif q["kind"] == "fold":
                    ref, s = refs.fold(q["li"], q["level"], srcs[0], srcs[1])
                elif q["kind"] == "head":
                    ref, s = refs.head(srcs[0])
                else:
                    ref, s = refs.stem(q["kind"], xf[b])
                cache[key] = ([t.clone() for t in srcs], ref, s, xf[b].clone())
            got = out[b] if q["kind"] != "head" else logits[b].permute(1, 2, 0)
            e, m, t = _compare(got, ref, s, bf16_out=q["kind"] != "head")
            worst, mism, tot = max(worst, e), mism + m, tot + t
        row.update(max_norm=worst, mismatch=mism / tot)
        if not worst <= 1.0:
            row.update(ok=False, why=row["why"] + f" error bound exceeded ({worst:.3g}x)")
        if mism / tot > 0.01:
            row.update(ok=False, why=row["why"] + f" rounding mismatch {mism / tot:.3%}")
        rows.append(row)
    return rows


def _logit_thr(thr):
    from tw_invoice_unet_ocr_llm_b200.engine import logit_thresholds
    return logit_thresholds(thr)


def audit(engine, x, options=None, *, handle=None, label=""):
    """Run the plan of `options` on `x` twice (direct launches, then the graph replay) in a workspace of this
    test's own, and audit every launch of both runs.  `handle` runs the forward on another handle (a corrupted
    blob) while the references keep reading `engine.blob`.  Returns the report rows (one per run and launch)."""
    nat = _nat()
    options = dict(options or {})
    keep = {k: engine.get_option(k) for k in options}
    try:
        for k, v in options.items():
            engine.set_option(k, v)
        engine.set_option("graph", 1)                 # (also drops the cached plans: run 1 is direct launches)
        fold = engine.get_option("fold_up")
        plan = _plan(engine.n_channels, engine.get_option("stem_tc"), fold)
        h = handle if handle is not None else engine._handle
        if x.dtype == torch.uint8:
            n, hh, ww, _ = x.shape
        else:
            n, _, hh, ww = x.shape
        ws = _Workspace(engine, n, hh, ww)
        ncls = engine.n_classes
        thr = (THR * 3)[:ncls]
        logits = torch.empty((n, ncls, hh, ww), dtype=torch.float32, device=engine.device)
        mask = torch.empty((n, ncls, hh, ww), dtype=torch.uint8, device=engine.device)
        xf = _input_f32(x)
        refs = _Refs(engine, engine.blob)
        cache, rows = {}, []
        for run in ("direct", "replay"):
            ws.buf.fill_(0xFF)
            logits.fill_(float("nan"))
            mask.fill_(7)
            _forward(engine, h, x, ws, logits, mask, 0, thr)
            torch.cuda.synchronize()
            count = int(nat.lib().unetb200_last_launch_count(h))
            assert count == 22 - bin(fold).count("1") == len(plan), (label, count, len(plan))
            rows += _audit_run(engine, refs, plan, x, xf, ws, logits, mask, thr, label, run, cache)
        # bit-packed masks (their own plan) == the byte masks of the audited runs
        from tw_invoice_unet_ocr_llm_b200.engine import unpack_mask_bits
        bits = torch.full((n, ncls, hh, ww // 8), 0xA5, dtype=torch.uint8, device=engine.device)
        _forward(engine, h, x, ws, None, bits, 1, thr)
        torch.cuda.synchronize()
        if not torch.equal(unpack_mask_bits(bits), mask):
            rows[-1].update(ok=False, why=rows[-1]["why"] + " bit-packed masks != byte masks")
    finally:
        for k, v in keep.items():
            engine.set_option(k, v)
    for r in rows:
        if r.get("skipped"):
            print(f"audit {label:44s} {r['run']:6s} {r['launch']:2d} {r['name']:17s} skipped: {r['skipped']}"
                  + ("" if r["ok"] else f"  FAIL:{r['why']}"))
        else:
            print(f"audit {label:44s} {r['run']:6s} {r['launch']:2d} {r['name']:17s} {r['kind']:7s} "
                  f"max_norm {r['max_norm']:.4f}  mismatch {r['mismatch']:.2e}" + ("" if r["ok"] else f"  FAIL:{r['why']}"))
    return rows


def _failures(rows):
    return [(r["run"], r["name"], r["why"]) for r in rows if not r["ok"]]


def _summary(rows):
    done = [r for r in rows if not r.get("skipped")]
    w = max(done, key=lambda r: r["max_norm"])
    m = max(done, key=lambda r: r["mismatch"])
    return (f"worst normalised error {w['max_norm']:.4f} ({w['name']}), "
            f"worst mismatch fraction {m['mismatch']:.2e} ({m['name']})")


# ---------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def engine(fixture_state, cuda_dev):
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    e = Engine(fixture_state, cuda_dev)
    yield e
    e.close()


def _random_state(n_channels, n_classes):
    """A random checkpoint with non-trivial BatchNorm, as test_forward_parity's other-architecture test builds."""
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
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


def _x(n, h, w, seed):
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices
    return synthetic_invoices(n, h, w, seed=seed)


# ---------------------------------------------------------------------------------------------------- tests
def test_workspace_map(engine):
    """`_ws_layout` reproduces `unetb200_workspace_bytes` at every shape this file runs, and its regions tile the
    workspace without overlap (u[k] aliasing a[k] aside)."""
    for n, h, w in DEFAULT_SHAPES + SWEEP_SHAPES + [SMALL]:
        L = _ws_layout(n, h, w)
        assert engine.workspace_bytes(n, h, w) == L["total"], (n, h, w)
        spans = []
        for name in ("a", "c", "p", "bt", "ca", "cc"):
            for k, off in enumerate(L[name]):
                if off is None:
                    continue
                lvl, ch = _region_shape(name, k)
                spans.append((off, off + 2 * n * (h >> lvl) * (w >> lvl) * ch))
        spans.sort()
        assert spans[0][0] == 0 and all(a[1] <= b[0] and b[0] % 1024 == 0 for a, b in zip(spans, spans[1:]))
        assert spans[-1][1] <= L["total"] < spans[-1][1] + 1024


@pytest.mark.parametrize("n,h,w", DEFAULT_SHAPES, ids=[f"{n}x{h}x{w}" for n, h, w in DEFAULT_SHAPES])
def test_default_plan(engine, n, h, w):
    """All 18 launches of the default plan, direct and replayed."""
    t0 = time.time()
    rows = audit(engine, _x(n, h, w, seed=300 + n + h + w).to(engine.device), {}, label=f"default {n}x{h}x{w}")
    assert len(rows) == 36 and not any(r.get("skipped") for r in rows)
    print(f"audit default {n}x{h}x{w}: {_summary(rows)}, {time.time() - t0:.1f} s")
    assert not _failures(rows), _failures(rows)


@pytest.mark.parametrize("shape", SWEEP_SHAPES, ids=[f"{n}x{h}x{w}" for n, h, w in SWEEP_SHAPES])
@pytest.mark.parametrize("opts", SWEEP, ids=[",".join(f"{k}={v}" for k, v in o.items()) for o in SWEEP])
def test_option_sweep(engine, opts, shape):
    n, h, w = shape
    t0 = time.time()
    label = f"{n}x{h}x{w} " + ",".join(f"{k}={v}" for k, v in opts.items())
    rows = audit(engine, _x(n, h, w, seed=400 + h).to(engine.device), opts, label=label)
    print(f"audit {label}: {_summary(rows)}, {time.time() - t0:.1f} s")
    assert not _failures(rows), _failures(rows)
    if opts.get("fold_up") == 0:                  # every launch kind of the 22-launch plan was audited
        done = {r["name"] for r in rows if not r.get("skipped")}
        assert {"up4", "up3", "up2", "up1", "conv4.net.0", "conv1.net.0", "bottleneck.net.3"} <= done, done
        assert not any(r["kind"] == "fold" for r in rows)


@pytest.mark.parametrize("fmt", ["f32_nchw", "u8_nhwc", "bf16_nhwc"])
def test_input_formats(engine, fmt):
    """The stems read every input format as the fp32 value the reference computes from (uint8: k / 255.0f)."""
    from tw_invoice_unet_ocr_llm_b200.synthetic import synthetic_invoices_u8
    n, h, w = 3, 64, 96
    if fmt == "u8_nhwc":
        x = torch.from_numpy(synthetic_invoices_u8(n, h, w, seed=61))
    elif fmt == "bf16_nhwc":
        x = _x(n, h, w, seed=62).bfloat16().to(memory_format=torch.channels_last)
    else:
        x = _x(n, h, w, seed=63)
    for stem_tc in (1, 0):
        rows = audit(engine, x.to(engine.device), {"stem_tc": stem_tc}, label=f"{fmt} stem_tc={stem_tc} {n}x{h}x{w}")
        assert not _failures(rows), _failures(rows)


@pytest.mark.parametrize("n_channels,n_classes", ARCHS)
def test_other_architectures(cuda_dev, n_channels, n_classes):
    """1- and 4-channel stems (4 channels: CUDA-core stem) and the generic head, on a random state."""
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    e = Engine(_random_state(n_channels, n_classes), cuda_dev, n_channels, n_classes)
    try:
        g = torch.Generator().manual_seed(70 + n_channels)
        x = torch.rand((SMALL[0], n_channels) + SMALL[1:], generator=g).to(cuda_dev)
        rows = audit(e, x, {}, label=f"arch ({n_channels}, {n_classes}) {'x'.join(map(str, SMALL))}")
        assert not _failures(rows), _failures(rows)
    finally:
        e.close()


# ---------------------------------------------------------------------------------------------------- packing
def _fold(state, l, eps=EPS):
    """The fp32 fold of one layer with correctly rounded fp32 operations, as csrc/pack.cuh computes it
    (`__fsqrt_rn`, `__fdiv_rn`, one multiply): (scaled fp32 weights in the state's layout, folded-bias candidates).
    Each operation is done in float64 and rounded to fp32, which is exact rounding for + - * / sqrt.  (torch's own
    fp32 CPU division / sqrt were measured 1 ulp off the correctly rounded scale on 2 of 64 channels of one random
    state, so they cannot serve as the reference.)  The bias candidates are (b - mean) s + beta evaluated unfused
    and as one FMA: nvcc may contract it, and under cancellation the two differ by more than 1 ulp."""
    r = lambda t: t.float().double()
    name, bn = l.name.decode(), l.bn_name.decode()
    w = r(state[name + ".weight"].cpu())
    b = r(state[name + ".bias"].cpu()) if name + ".bias" in state else torch.zeros(w.shape[0], dtype=torch.float64)
    if not bn:
        return w.float(), [b.float()]
    g, be = r(state[bn + ".weight"].cpu()), r(state[bn + ".bias"].cpu())
    mu, var = r(state[bn + ".running_mean"].cpu()), r(state[bn + ".running_var"].cpu())
    s = r(g / r(torch.sqrt(r(var + r(torch.tensor(eps))))))
    d = r(b - mu)
    return r(w * s[:, None, None, None]).float(), [r(r(d * s) + be).float(), r(d * s + be).float()]


def _bias_ok(got, cands):
    return bool(torch.stack([got == c for c in cands]).any(0).all())


def _split(f):
    hi = f.to(torch.bfloat16)
    return hi, (f - hi.float()).to(torch.bfloat16)


def _check_packing(eng, state):
    nat = _nat()
    blob = eng.blob.cpu()
    for l in eng.layers:
        name = l.name.decode()
        wf, bf = _fold(state, l)
        bits = lambda off, nb, dt: blob[off:off + nb].view(dt)
        b_got = bits(l.b_off, l.b_bytes, torch.float32)
        if l.kind == nat.CONV3X3:
            ref = wf.permute(2, 3, 0, 1).reshape(9, l.cout, l.cin).to(torch.bfloat16).reshape(-1)
            assert torch.equal(bits(l.w_off, l.w_bytes, torch.int16), ref.view(torch.int16)), name
            assert _bias_ok(b_got, bf), name
        elif l.kind == nat.STEM:
            cin = l.cin
            ref = wf.permute(2, 3, 1, 0).reshape(9 * cin * l.cout)          # [k = tap * Cin + ci][64]
            assert torch.equal(bits(l.w_off, 9 * cin * l.cout * 4, torch.float32), ref), name
            assert _bias_ok(b_got, bf), name
            if cin > 3:
                continue                    # the tensor-core stem (9 Cin <= 32 K slots) serves Cin <= 3 only
            off = l.w_off + int(nat.lib().unetb200_stem_tc_offset(cin))
            rows = bits(off, l.cout * 256, torch.int16).view(l.cout, 128)
            hi, lo = _split(wf.permute(0, 2, 3, 1).reshape(l.cout, 9 * cin))   # [co][k]
            exp = torch.zeros(l.cout, 128, dtype=torch.bfloat16)
            exp[:, :9 * cin], exp[:, 32:32 + 9 * cin], exp[:, 64:64 + 9 * cin] = hi, hi, lo
            k = 9 * cin
            assert torch.equal(rows[:, :k], exp[:, :k].view(torch.int16)), name
            assert torch.equal(rows[:, 32:32 + k], exp[:, 32:32 + k].view(torch.int16)), name
            assert torch.equal(rows[:, 64:64 + k], exp[:, 64:64 + k].view(torch.int16)), name
            zero = torch.ones(128, dtype=torch.bool)
            zero[:k + 1], zero[32:32 + k], zero[64:64 + k + 1] = False, False, False
            assert not rows[:, zero].any(), name + ": padding slots"
            # bias slot k = 9 Cin: hi / lo of the folded bias (either evaluation), zero against x_lo
            ok = torch.zeros(l.cout, dtype=torch.bool)
            for cand in bf:
                bh, bl = _split(cand)
                ok |= (rows[:, k] == bh.view(torch.int16)) & (rows[:, 64 + k] == bl.view(torch.int16))
            assert ok.all(), name + ": bias slot"
        elif l.kind == nat.CONVT2X2:
            ref = wf.permute(2, 3, 1, 0).reshape(4, l.cout, l.cin).to(torch.bfloat16).reshape(-1)
            assert torch.equal(bits(l.w_off, l.w_bytes, torch.int16), ref.view(torch.int16)), name
            assert torch.equal(b_got, bf[0]), name
        else:
            assert torch.equal(bits(l.w_off, l.w_bytes, torch.float32), wf.reshape(-1)), name
            assert torch.equal(b_got, bf[0]), name


def test_packing_fixture(engine, fixture_state):
    _check_packing(engine, fixture_state)


@pytest.mark.parametrize("n_channels,n_classes", ARCHS)
def test_packing_random(cuda_dev, n_channels, n_classes):
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    state = _random_state(n_channels, n_classes)
    e = Engine(state, cuda_dev, n_channels, n_classes)
    try:
        _check_packing(e, state)
    finally:
        e.close()


@pytest.mark.parametrize("level", [1, 2, 3, 4])
def test_packing_composites(engine, fixture_state, cuda_dev, level):
    """Composite weights and bias9 of the fixture checkpoint's folded levels, with test_pack_fused_up's gates."""
    nat = _nat()
    S = lambda k: fixture_state[k].float().to(cuda_dev).contiguous()
    p = dict(wT=S(f"up{level}.weight"), bT=S(f"up{level}.bias"), w3=S(f"conv{level}.net.0.weight"),
             b3=S(f"conv{level}.net.0.bias"), gamma=S(f"conv{level}.net.1.weight"), beta=S(f"conv{level}.net.1.bias"),
             mean=S(f"conv{level}.net.1.running_mean"), var=S(f"conv{level}.net.1.running_var"))
    c = 64 << (level - 1)
    off = [C.c_uint64() for _ in range(4)]
    nat.check(nat.lib().unetb200_fused_up_info(C.byref(engine.arch), level, *[C.byref(o) for o in off]))
    w_off, w_bytes, b_off, b_bytes = [o.value for o in off]
    wc = engine.blob[w_off:w_off + w_bytes].view(torch.bfloat16).float().reshape(16, c, 2 * c)
    ref = _composite_ref(p, 2 * c, c, c)
    err = (wc - ref).abs()
    assert float((err - ref.abs() * 2.0 ** -8).max()) <= 1e-6, float(err.max())
    b9 = engine.blob[b_off:b_off + b_bytes].view(torch.float32).reshape(9, c)
    assert torch.allclose(b9, _bias9_ref(p, c, c), rtol=1e-4, atol=1e-4)


# ---------------------------------------------------------------------------------------------------- sensitivity
@pytest.mark.parametrize("case", ["bottleneck_k_slice", "bias9_border"])
def test_audit_names_the_corrupted_launch(engine, fixture_state, case):
    """A corrupted blob: the audit flags exactly the launch that reads the corruption, every other launch passes
    (each is checked from its own inputs).  The end-to-end oracle figures of the same forward are printed: they are
    what the forward-parity gates see of such an error."""
    from oracle.unet_oracle import oracle_forward, parity_report
    nat = _nat()
    bad = engine.blob.clone()
    if case == "bottleneck_k_slice":
        l = engine.layers[9]                                  # bottleneck.net.3: [9][1024][1024]
        w = bad[l.w_off:l.w_off + l.w_bytes].view(torch.int16).view(9, l.cout, l.cin)
        w[4, :, 5 * 64:6 * 64] = 0                            # centre tap, K slice 5
        expect = "bottleneck.net.3"
    else:
        off = [C.c_uint64() for _ in range(4)]
        nat.check(nat.lib().unetb200_fused_up_info(C.byref(engine.arch), 2, *[C.byref(o) for o in off]))
        b9 = bad[off[2].value:off[2].value + off[3].value].view(torch.float32).view(9, -1)
        b9[1] += 0.05                                          # first row, interior columns
        expect = "conv2.net.0"
    h = C.c_void_p()
    nat.check(nat.lib().unetb200_create(C.byref(engine.arch), bad.data_ptr(), bad.numel(),
                                        engine.device.index, C.byref(h)))
    try:
        x = _x(1, 512, 512, seed=42)
        rows = audit(engine, x.to(engine.device), {}, handle=h, label=f"corrupted {case} 1x512x512")
        flagged = {r["name"] for r in rows if not r["ok"]}
        assert flagged == {expect}, _failures(rows)
        z = torch.empty((1, 3, 512, 512), dtype=torch.float32, device=engine.device)
        ws = _Workspace(engine, 1, 512, 512)
        _forward(engine, h, x.to(engine.device), ws, z, None, 0, THR)
        torch.cuda.synchronize()
        print(f"corrupted {case}: parity of the forward vs the oracle: {parity_report(oracle_forward(fixture_state, x), z)}")
    finally:
        nat.lib().unetb200_destroy(h)
