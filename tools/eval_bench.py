#!/usr/bin/env python
"""Accuracy of the trained stand-in under each clean-up setting, and the cost of scoring (prepost.mask_match), on
one GPU.

    python tools/eval_bench.py --out DIR [--train-steps 300 --n-eval 256 --n 64 --size 512 --steps 10 --rounds 7]

Accuracy: the UNet trained by synthetic.train_fixture_state (seed 0, `--train-steps` steps on marked_invoices seed
300) is scored by inference.evaluate_masks on a held-out marked_invoices(`--n-eval`, 512, seed=303) set, at the
reference's thresholds, for clean=None, [("open", (3, 3))] and the README recipe [("close", (9, 3)), "fill_holes",
("open", (3, 3))], each at connectivity 4 and 8 (min_pixels 1, IoU > 0.5).  Per field: pixel IoU, region
precision / recall / F1, PQ and the raw counts.

Cost: mask_match at `--n` x 3 x `--size`^2 (8-connectivity, IoU 0.5) on three plane sets -- the trained model's
masks against their ground truth, 50 % noise against 50 % noise, and the (x + y) % 2 checkerboard against itself
("checker4": one region per plane at 8-connectivity, so every row merges into one entry) -- each with byte and with
bit-packed inputs; beside them, for scale, the forward with bit-packed masks and two mask_components calls (pred and
gt, byte planes).  Each variant is timed with CUDA events
around `--steps` back-to-back calls, alternated within each of `--rounds` rounds (rotated start) after a warm-up; the
medians are reported.  The host oracle (oracle/mask_match.py) is timed per plane on one core on the trained masks.

Writes DIR/eval_bench.json with the GPU's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.io_formats_bench import gpu_info  # noqa: E402

SETTINGS = {"none": None, "open3x3": [("open", (3, 3))],
            "close9x3_fill_open3x3": [("close", (9, 3)), "fill_holes", ("open", (3, 3))]}
REPORT = ("pixel_iou", "precision", "recall", "f1", "pq")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--train-steps", type=int, default=300)
    ap.add_argument("--n-eval", type=int, default=256)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()

    import numpy as np
    import torch
    from oracle import mask_match as om
    from tw_invoice_unet_ocr_llm_b200 import inference as inf
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import marked_invoices, train_fixture_state
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    t0 = time.perf_counter()
    state, loss = train_fixture_state(dev, steps=args.train_steps, seed=0)
    train_s = time.perf_counter() - t0
    model = UNet(3, 3)
    model.load_state_dict(state)
    model = model.to(dev).eval()
    x_eval, gt_eval = marked_invoices(args.n_eval, 512, seed=303)

    accuracy = {}
    for name, clean in SETTINGS.items():
        for conn in (4, 8):
            r = inf.evaluate_masks(model, x_eval, gt_eval, clean=clean, connectivity=conn)
            accuracy[f"{name}:conn{conn}"] = {f: {k: r[f][k] for k in REPORT + ("iou_sum",) + tuple(prepost.MATCH_COUNTS)}
                                              for f in inf.FIELDS}

    # ---- cost at n x 3 x size^2
    n, s = args.n, args.size
    thr = [inf.THRESHOLDS[f] for f in inf.FIELDS]
    x, gt = marked_invoices(n, s, seed=304)
    x = x.to(dev)
    gt_u8 = (gt != 0).to(torch.uint8).to(dev)
    eng = Engine(state, dev)
    _, fwd = eng.run(x, want_logits=False, thresholds=thr)
    gen = torch.Generator(device=dev).manual_seed(3)
    noise = [(torch.rand((n, 3, s, s), generator=gen, device=dev) < 0.5).to(torch.uint8) for _ in range(2)]
    yy, xx = torch.meshgrid(torch.arange(s, device=dev), torch.arange(s, device=dev), indexing="ij")
    chk = ((xx + yy) % 2 == 0).to(torch.uint8).expand(n, 3, s, s).contiguous()
    sets = {"trained": (fwd, gt_u8), "noise50": tuple(noise), "checker4": (chk, chk)}

    def packed(t):
        return torch.from_numpy(np.packbits(t.cpu().numpy(), axis=-1, bitorder="little")).to(dev)

    variants = {}
    n_regions = {}
    for name, (p, g) in sets.items():
        pb, gb = packed(p), packed(g)
        variants[f"mask_match:{name}:bytes"] = lambda p=p, g=g: prepost.mask_match(p, g)
        variants[f"mask_match:{name}:packed"] = lambda p=pb, g=gb: prepost.mask_match(p, g, pred_packed=True,
                                                                                     gt_packed=True)
        variants[f"2x_mask_components:{name}"] = lambda p=p, g=g: (prepost.mask_components(p),
                                                                   prepost.mask_components(g))
        c, _ = prepost.mask_match(p, g)
        c = c.view(-1, 8).cpu()
        n_regions[name] = {"pred_per_plane": float(c[:, 3].float().mean()), "gt_per_plane": float(c[:, 4].float().mean()),
                           "matched_per_plane": float(c[:, 5].float().mean())}
    variants["forward_bits:trained"] = lambda: eng.run(x, want_logits=False, thresholds=thr, mask_bits=True)
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

    # ---- the host oracle, per plane on one core
    torch.set_num_threads(1)
    fp, gp = fwd.cpu().numpy(), gt_u8.cpu().numpy()
    planes = [(i, c) for i in range(min(n, 8)) for c in range(3)]
    t0 = time.perf_counter()
    for i, c in planes:
        om.match_plane(fp[i, c], gp[i, c])
    oracle_ms = (time.perf_counter() - t0) * 1e3 / len(planes)

    res = {"gpu": gpu_info(), "torch": torch.__version__,
           "trained": {"steps": args.train_steps, "final_loss": float(loss), "train_s": train_s},
           "eval_set": {"n": args.n_eval, "size": 512, "seed": 303, "thresholds": thr},
           "accuracy": accuracy, "timing_shape": [n, 3, s, s], "steps_per_sample": args.steps,
           "rounds": args.rounds, "regions": n_regions, "oracle_ms_per_plane_one_core": oracle_ms,
           "workspace_bytes": prepost.nat.lib().unetb200_match_workspace_bytes(n * 3, s, s), "device_ms": {}}
    for name in names:
        t = times[name]
        res["device_ms"][name] = {"median": statistics.median(t), "min": min(t), "max": max(t), "samples": t}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "eval_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    short = {k: {f: {m: (None if v[f][m] is None else round(v[f][m], 4)) for m in REPORT} for f in inf.FIELDS}
             for k, v in accuracy.items()}
    print(json.dumps({"gpu": res["gpu"], "accuracy": short, "regions": n_regions,
                      "device_ms_median": {k: round(v["median"], 4) for k, v in res["device_ms"].items()},
                      "oracle_ms_per_plane_one_core": round(oracle_ms, 3)}))
    print("wrote", path)


if __name__ == "__main__":
    main()
