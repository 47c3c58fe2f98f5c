#!/usr/bin/env python
"""Cost of connected-component labelling (prepost.mask_components) at batch 64 x 3 x 512 x 512 on one GPU.

    python tools/components_bench.py --out DIR [--n 64 --size 512 --steps 10 --rounds 7 --scipy-planes 24]

Mask sets: the fixture checkpoint's forward masks of bench.py's synthetic invoices, 50 % noise, and the 4-connected
checkerboard (the most components a plane can have: H * W / 2).  Variants, each timed with CUDA events around
`--steps` back-to-back calls, alternated within each of `--rounds` rounds (rotated start) after a warm-up pass:
mask_components (8- and 4-connectivity, K = 8, byte masks; the fixture masks also bit-packed and with labels),
mask_bbox of the same masks for scale, and the forward that produces the fixture masks.  The medians are reported.
The masks (50 MB) stay in L2 between calls; the workspace (14 bytes per pixel) does not.  scipy.ndimage.label +
find_objects + bincount on the host, one plane at a time, gives the CPU figure (host time, one core).

Writes DIR/components_bench.json with the GPU's name, power limit and max SM clock.
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

from tools.io_formats_bench import THR, gpu_info  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--scipy-planes", type=int, default=24)
    args = ap.parse_args()

    import numpy as np
    import torch
    from scipy import ndimage
    from tw_invoice_unet_ocr_llm_b200 import prepost
    from tw_invoice_unet_ocr_llm_b200.engine import Engine
    from tw_invoice_unet_ocr_llm_b200.synthetic import make_fixture_state, synthetic_invoices_u8
    if not torch.cuda.is_available():
        raise SystemExit("components_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n, s = args.n, args.size
    eng = Engine(make_fixture_state(), dev)
    x = torch.from_numpy(synthetic_invoices_u8(n, s, s, seed=7)).to(dev)
    fwd_mask = torch.empty((n, 3, s, s), dtype=torch.uint8, device=dev)
    eng.run(x, want_logits=False, thresholds=THR, mask_out=fwd_mask)
    _, fwd_bits = eng.run(x, want_logits=False, thresholds=THR, mask_bits=True)
    gen = torch.Generator(device=dev).manual_seed(3)
    yy, xx = torch.meshgrid(torch.arange(s, device=dev), torch.arange(s, device=dev), indexing="ij")
    masks = {
        "fixture": fwd_mask,
        "noise50": (torch.rand((n, 3, s, s), generator=gen, device=dev) < 0.5).to(torch.uint8),
        "checker": ((yy + xx) % 2 == 0).to(torch.uint8).expand(n, 3, s, s).contiguous(),
    }
    torch.cuda.synchronize()

    variants = {}
    for name, m in masks.items():
        for conn in (8, 4):
            variants[f"components{conn}:{name}"] = (lambda m=m, c=conn: prepost.mask_components(m, connectivity=c))
        variants[f"bbox:{name}"] = (lambda m=m: prepost.mask_bbox(m))
    variants["components8_packed:fixture"] = lambda: prepost.mask_components(fwd_bits, packed=True)
    variants["components8_labels:fixture"] = lambda: prepost.mask_components(fwd_mask, labels=True)
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

    counts = {}
    for name, m in masks.items():
        for conn in (8, 4):
            _, cnt = prepost.mask_components(m, connectivity=conn)
            c = cnt.cpu().numpy()
            counts[f"{name}/{conn}"] = {"mean": float(c.mean()), "max": int(c.max())}

    host = {}
    for name, m in masks.items():
        planes = m.reshape(-1, s, s)[: args.scipy_planes].cpu().numpy() != 0
        per = []
        for p in planes:
            t0 = time.perf_counter()
            lab, k = ndimage.label(p, np.ones((3, 3), bool))
            ndimage.find_objects(lab)
            np.bincount(lab.ravel(), minlength=k + 1)
            per.append((time.perf_counter() - t0) * 1e3)
        host[name] = {"ms_per_plane_median": statistics.median(per), "planes": len(per)}

    res = {"gpu": gpu_info(), "torch": torch.__version__, "shape": [n, 3, s, s], "steps_per_sample": args.steps,
           "rounds": args.rounds, "cpu_count": os.cpu_count(), "device_ms": {}, "components_per_plane": counts,
           "scipy_host": host,
           "workspace_bytes": prepost.nat.lib().unetb200_components_workspace_bytes(n * 3, s, s)}
    for name in names:
        t = times[name]
        res["device_ms"][name] = {"median": statistics.median(t), "min": min(t), "max": max(t), "samples": t}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "components_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "device_ms_median": {k: round(v["median"], 4) for k, v in res["device_ms"].items()},
                      "scipy_ms_per_plane": {k: round(v["ms_per_plane_median"], 3) for k, v in host.items()},
                      "components_per_plane": counts}))
    print("wrote", path)


if __name__ == "__main__":
    main()
