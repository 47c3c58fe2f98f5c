#!/usr/bin/env python
"""Cost of the mask clean-up (prepost.mask_morphology / prepost.fill_holes) at batch 64 x 3 x 512 x 512 on one GPU.

    python tools/morph_bench.py --out DIR [--n 64 --size 512 --steps 10 --rounds 7 --trained-steps 0]

Mask sets: the fixture checkpoint's forward masks of bench.py's synthetic invoices, and 50 % noise.  Variants, each
timed with CUDA events around `--steps` back-to-back calls, alternated within each of `--rounds` rounds (rotated
start) after a warm-up pass, as tools/components_bench.py does:
  * erode / dilate / open / close at 3 x 3, 15 x 3 and 31 x 31, and fill_holes, byte planes in and out;
  * the same at 3 x 3 and fill_holes on the bit-packed forward masks (Engine.run(mask_bits=True)), packed in and out;
  * mask_components (8-connectivity, K = 8) of the masks as they are, of the masks after a 3 x 3 opening, and the
    opening + labelling together.
The medians are reported.  Algorithmic bytes of one call = its input plus its output (1 byte per pixel for byte
planes, 1 bit for packed ones); GB/s = those bytes over the median time.  Components per plane are counted before and
after a 3 x 3 opening and after clean=[("close", (9, 3)), ("open", (3, 3))].  With --trained-steps N > 0 the same
counts are taken on the masks of a checkpoint trained for N steps (synthetic.train_fixture_state, the recipe of
tools/make_fixture_checkpoint.py --trained) in the same process.

Writes DIR/morph_bench.json with the GPU's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.io_formats_bench import THR, gpu_info  # noqa: E402

SIZES = [(3, 3), (15, 3), (31, 31)]
OPS = ["erode", "dilate", "open", "close"]


def component_counts(masks, prepost):
    """Mean / max components per plane (8-connectivity) of byte masks as they are, after a 3 x 3 opening, and after
    clean=[("close", (9, 3)), ("open", (3, 3))]."""
    opened = prepost.mask_morphology(masks, "open", (3, 3))
    cleaned = prepost.mask_morphology(prepost.mask_morphology(masks, "close", (9, 3)), "open", (3, 3))
    out = {}
    for name, m in (("raw", masks), ("open3x3", opened), ("close9x3_open3x3", cleaned)):
        c = prepost.mask_components(m)[1].cpu().float()
        out[name] = {"mean": float(c.mean()), "max": int(c.max())}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--trained-steps", type=int, default=0)
    args = ap.parse_args()

    import torch
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import make_fixture_state, synthetic_invoices_u8
    if not torch.cuda.is_available():
        raise SystemExit("morph_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n, s = args.n, args.size
    eng = Engine(make_fixture_state(), dev)
    x = torch.from_numpy(synthetic_invoices_u8(n, s, s, seed=7)).to(dev)
    fwd_mask = torch.empty((n, 3, s, s), dtype=torch.uint8, device=dev)
    eng.run(x, want_logits=False, thresholds=THR, mask_out=fwd_mask)
    _, fwd_bits = eng.run(x, want_logits=False, thresholds=THR, mask_bits=True)
    gen = torch.Generator(device=dev).manual_seed(3)
    masks = {"fixture": fwd_mask,
             "noise50": (torch.rand((n, 3, s, s), generator=gen, device=dev) < 0.5).to(torch.uint8)}
    px = n * 3 * s * s

    variants, alg_bytes = {}, {}
    for mname, m in masks.items():
        for op in OPS:
            for kw, kh in SIZES:
                key = f"{op}{kw}x{kh}:{mname}"
                variants[key] = lambda m=m, op=op, k=(kw, kh): prepost.mask_morphology(m, op, k)
                alg_bytes[key] = 2 * px
        variants[f"fill_holes:{mname}"] = lambda m=m: prepost.fill_holes(m)
        alg_bytes[f"fill_holes:{mname}"] = 2 * px
        opened = prepost.mask_morphology(m, "open", (3, 3))
        variants[f"components8:{mname}"] = lambda m=m: prepost.mask_components(m)
        variants[f"components8_after_open3x3:{mname}"] = lambda o=opened: prepost.mask_components(o)
        variants[f"open3x3+components8:{mname}"] = (
            lambda m=m: prepost.mask_components(prepost.mask_morphology(m, "open", (3, 3))))
    for op in OPS:
        key = f"{op}3x3_packed:fixture"
        variants[key] = lambda op=op: prepost.mask_morphology(fwd_bits, op, (3, 3), packed=True)
        alg_bytes[key] = 2 * px // 8
    variants["fill_holes_packed:fixture"] = lambda: prepost.fill_holes(fwd_bits, packed=True)
    alg_bytes["fill_holes_packed:fixture"] = 2 * px // 8
    variants["forward:fixture"] = lambda: eng.run(x, want_logits=False, thresholds=THR, mask_out=fwd_mask)

    names = list(variants)
    for name in names:
        for _ in range(3):
            variants[name]()
    torch.cuda.synchronize()
    times = {k: [] for k in names}
    stream = torch.cuda.current_stream(dev)
    for r in range(args.rounds):
        for name in names[r % len(names):] + names[:r % len(names)]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                variants[name]()
            e1.record(stream)
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)

    counts = {name: component_counts(m, prepost) for name, m in masks.items()}
    trained = "not measured"
    if args.trained_steps > 0:
        from tw_invoice_unet_ocr_llm_b200.synthetic import train_fixture_state
        state, loss = train_fixture_state(str(dev), steps=args.trained_steps)
        teng = Engine(state, dev)
        tmask = torch.empty_like(fwd_mask)
        teng.run(x, want_logits=False, thresholds=THR, mask_out=tmask)
        trained = {"steps": args.trained_steps, "final_loss": float(loss), "components_per_plane":
                   component_counts(tmask, prepost), "set_fraction": float(tmask.float().mean())}

    res = {"gpu": gpu_info(), "torch": torch.__version__, "shape": [n, 3, s, s], "steps_per_sample": args.steps,
           "rounds": args.rounds, "device_ms": {}, "components_per_plane": counts, "trained_checkpoint": trained,
           "workspace_bytes": {op: prepost.nat.lib().unetb200_morph_workspace_bytes(n * 3, s, s, code)
                               for op, code in (("open", prepost.nat.MORPH_OPEN),
                                                ("fill_holes", prepost.nat.MORPH_FILL_HOLES))}}
    for name in names:
        t = times[name]
        med = statistics.median(t)
        row = {"median": med, "min": min(t), "max": max(t), "samples": t}
        if name in alg_bytes:
            row["alg_bytes"] = alg_bytes[name]
            row["alg_GBps"] = alg_bytes[name] / (med * 1e-3) / 1e9
        res["device_ms"][name] = row
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "morph_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"],
                      "device_ms_median": {k: round(v["median"], 4) for k, v in res["device_ms"].items()},
                      "components_per_plane": counts, "trained": trained}))
    print("wrote", path)


if __name__ == "__main__":
    main()
