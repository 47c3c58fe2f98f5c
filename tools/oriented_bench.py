#!/usr/bin/env python
"""Cost of the oriented boxes (prepost.mask_components_oriented) and of the upright crops (prepost.warp_crops) on one
GPU.

    python tools/oriented_bench.py --out DIR [--n 64 --size 512 --steps 10 --rounds 7 --frames 64 --crops 192]

* Labelling: the fixture checkpoint's forward masks of bench.py's synthetic invoices (64 x 3 x 512^2), 8-connectivity,
  K = 4 and 16: mask_components against mask_components_oriented (scale 1920/512, 1080/512).  The difference is the
  cost of the oriented passes (moments, axis, extents).
* Warp: `--crops` upright crops (300..700 x 30..120 px at angles -60..60 degrees, three per frame) cut from `--frames`
  1080p RGB frames on the device, in one warp_crops call; against cv2.warpAffine per crop on one host core
  (cv2.setNumThreads(1)), the same crops.

Each device variant is timed with CUDA events around `--steps` back-to-back calls, alternated within each of
`--rounds` rounds (rotated start) after a warm-up pass; medians are reported.  Writes DIR/oriented_bench.json with
the GPU's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.io_formats_bench import THR, gpu_info  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--crops", type=int, default=192)
    args = ap.parse_args()

    import cv2
    import numpy as np
    import torch
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import make_fixture_state, synthetic_invoices_u8
    if not torch.cuda.is_available():
        raise SystemExit("oriented_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n, s = args.n, args.size
    eng = Engine(make_fixture_state(), dev)
    x = torch.from_numpy(synthetic_invoices_u8(n, s, s, seed=7)).to(dev)
    mask = torch.empty((n, 3, s, s), dtype=torch.uint8, device=dev)
    eng.run(x, want_logits=False, thresholds=THR, mask_out=mask)
    scale = (1920 / s, 1080 / s)

    # 1080p frames: one synthetic invoice tiled with per-frame noise (generating 64 distinct ones costs minutes)
    base = torch.from_numpy(synthetic_invoices_u8(1, 1080, 1920, seed=5)[0]).to(dev)
    gen = torch.Generator(device=dev).manual_seed(11)
    frames = [(base.to(torch.int16) + torch.randint(-8, 9, base.shape, generator=gen, device=dev, dtype=torch.int16))
              .clamp_(0, 255).to(torch.uint8) for _ in range(args.frames)]
    rng = np.random.default_rng(3)
    mats, sizes, which = [], [], []
    for k in range(args.crops):
        t = math.radians(rng.uniform(-60, 60))
        ow, oh = int(rng.integers(300, 701)), int(rng.integers(30, 121))
        cx, cy = rng.uniform(400, 1520), rng.uniform(200, 880)
        e1, e2 = (math.cos(t), math.sin(t)), (-math.sin(t), math.cos(t))
        ox = cx - 0.5 * (ow - 1) * e1[0] - 0.5 * (oh - 1) * e2[0]
        oy = cy - 0.5 * (ow - 1) * e1[1] - 0.5 * (oh - 1) * e2[1]
        mats.append(np.array([[e1[0], e2[0], ox], [e1[1], e2[1], oy]]))
        sizes.append((ow, oh))
        which.append(k % args.frames)
    crop_frames = [frames[i] for i in which]
    torch.cuda.synchronize()

    variants = {}
    for k in (4, 16):
        variants[f"components8:K{k}"] = lambda k=k: prepost.mask_components(mask, max_components=k)
        variants[f"oriented8:K{k}"] = lambda k=k: prepost.mask_components_oriented(mask, max_components=k,
                                                                                   scale=scale)
    variants["warp_crops"] = lambda: prepost.warp_crops(crop_frames, mats, sizes)

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

    # the same crops with OpenCV on one host core; the device result must match it
    cv2.setNumThreads(1)
    hosts = [f.cpu().numpy() for f in frames]
    crops_dev, _ = prepost.warp_crops(crop_frames, mats, sizes)
    host_ms, mismatched = [], 0
    for rep in range(3):
        t0 = time.perf_counter()
        outs = [cv2.warpAffine(hosts[i], m, sz, flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP,
                               borderMode=cv2.BORDER_REPLICATE) for i, m, sz in zip(which, mats, sizes)]
        host_ms.append((time.perf_counter() - t0) * 1e3)
    for o, c in zip(outs, crops_dev):
        mismatched += int(not np.array_equal(o, c.cpu().numpy()))

    _, cnt = prepost.mask_components(mask)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "cv2": cv2.__version__, "mask_shape": [n, 3, s, s],
           "scale": scale, "frames": args.frames, "crops": args.crops,
           "crop_pixels": int(sum(w * h for w, h in sizes)), "steps_per_sample": args.steps, "rounds": args.rounds,
           "components_per_plane_mean": float(cnt.float().mean()), "device_ms": {},
           "cv2_host_ms_all_crops_median": statistics.median(host_ms), "cv2_mismatched_crops": mismatched}
    for name in names:
        t = times[name]
        res["device_ms"][name] = {"median": statistics.median(t), "min": min(t), "max": max(t), "samples": t}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "oriented_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "device_ms_median": {k: round(v["median"], 4) for k, v in res["device_ms"].items()},
                      "cv2_host_ms": round(res["cv2_host_ms_all_crops_median"], 3), "cv2_mismatched": mismatched}))
    print("wrote", path)


if __name__ == "__main__":
    main()
