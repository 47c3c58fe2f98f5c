#!/usr/bin/env python
"""Input formats x logits types at batch 64 x 512 x 512 on one GPU.

    python tools/io_formats_bench.py --out DIR [--n 64 --size 512 --steps 10 --rounds 7]

Every input format (fp32 / fp16 / bf16, NCHW or channels-last, and uint8 NHWC) with every logits type (fp32 /
fp16 / bf16) runs the forward of bench.py's default step (logits + byte masks into preallocated buffers).  A variant
is timed with CUDA events around `--steps` back-to-back forwards; the variants alternate within each of `--rounds`
rounds (rotated start), after one warm-up pass over all of them, and the median per-step time is reported.  The
first conv's time comes from a separate pass with option profile = 1 (Engine.layer_times_ms()[0]; graph replay and
programmatic dependent launch are off while profiling, so those step times are not comparable with the timed ones).
`cl_fp32_copy` is the path a channels-last fp32 input took before the NHWC formats existed: x.contiguous(), then
the fp32 NCHW forward (the copy is inside the timed region).  Masks of every variant must equal the fp32 NCHW ones.

Writes DIR/io_formats_bench.json with the GPU's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

THR = [0.25, 0.40, 0.30]


def gpu_info() -> dict:
    """Name, power limit and max SM clock of GPU 0 (read-only nvidia-smi query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        keys = [k.strip() for k in out[0].split(",")]
        vals = [v.strip() for v in out[1].split(",")]
        return dict(zip(keys, vals))
    except Exception as e:   # the numbers are worthless without this, but keep them
        return {"error": f"nvidia-smi query failed: {e}"}


def bytes_per_step(n, h, w, c, x_elem, logits_elem, ncls=3):
    return {"input_bytes": n * c * h * w * x_elem, "logits_bytes": n * ncls * h * w * logits_elem}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--profile-reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    from tw_invoice_unet_ocr_llm_b200.synthetic import make_fixture_state, synthetic_invoices_u8
    from tw_invoice_unet_ocr_llm_b200.unet_model import UNet
    if not torch.cuda.is_available():
        raise SystemExit("io_formats_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    model = UNet(3, 3)
    model.load_state_dict(make_fixture_state())
    eng = model.to(dev).eval().engine(dev)
    n, h, w = args.n, args.size, args.size

    u8 = torch.from_numpy(synthetic_invoices_u8(n, h, w, seed=7)).to(dev)        # [N,H,W,3]
    x32 = u8.permute(0, 3, 1, 2).float().div_(255.0).contiguous()               # what preprocess makes
    inputs = {"u8_nhwc": u8}
    for name, dt in (("fp32", torch.float32), ("fp16", torch.float16), ("bf16", torch.bfloat16)):
        inputs[f"{name}_nchw"] = x32.to(dt).contiguous()
        inputs[f"{name}_cl"] = x32.to(dt).to(memory_format=torch.channels_last)
    ldt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}
    logits = {k: torch.empty((n, 3, h, w), dtype=t, device=dev) for k, t in ldt.items()}
    masks = {}
    variants = {}
    for xin in inputs:
        for lk in ldt:
            variants[f"{xin}->{lk}"] = (xin, lk, False)
    variants["cl_fp32_copy->fp32"] = ("fp32_cl", "fp32", True)

    def step(name):
        xin, lk, copy = variants[name]
        x = inputs[xin].contiguous() if copy else inputs[xin]
        m = masks.setdefault(name, torch.empty((n, 3, h, w), dtype=torch.uint8, device=dev))
        eng.run(x, want_logits=True, thresholds=THR, logits_out=logits[lk], mask_out=m, logits_dtype=ldt[lk])

    names = list(variants)
    for name in names:                       # warm-up: plans, graphs (second use), clocks
        for _ in range(3):
            step(name)
    torch.cuda.synchronize()

    times = {k: [] for k in names}
    stream = torch.cuda.current_stream(dev)
    for r in range(args.rounds):
        order = names[r % len(names):] + names[:r % len(names)]
        for name in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                step(name)
            e1.record(stream)
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)

    # every variant wrote its own mask buffer, from the same pixel values
    masks_equal = {k: bool(torch.equal(masks[k], masks["fp32_nchw->fp32"])) for k in names}

    # first-conv time (layer 0) with per-launch events
    eng.set_option("profile", 1)
    first = {k: [] for k in names}
    for rep in range(args.profile_reps):
        for name in names:
            step(name)
            first[name].append(eng.layer_times_ms()[0])
    eng.set_option("profile", 0)

    res = {"gpu": gpu_info(), "torch": torch.__version__, "shape": [n, 3, h, w], "steps_per_sample": args.steps,
           "rounds": args.rounds, "thresholds": THR, "variants": {}}
    elem = {"u8": 1, "fp32": 4, "fp16": 2, "bf16": 2}
    for name in names:
        xin, lk, copy = variants[name]
        res["variants"][name] = {
            "input": xin, "logits": lk, "host_copy_to_nchw": copy,
            "step_ms_median": statistics.median(times[name]), "step_ms_min": min(times[name]),
            "step_ms_max": max(times[name]), "step_ms": times[name],
            "first_conv_ms_median": statistics.median(first[name]),
            "images_per_s": n / statistics.median(times[name]) * 1e3,
            "masks_equal_fp32_nchw": masks_equal[name],
            **bytes_per_step(n, h, w, 3, elem[xin.split("_")[0]], elem[lk]),
        }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "io_formats_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "summary": {k: [round(v["step_ms_median"], 4), round(v["first_conv_ms_median"], 4),
                                                          v["masks_equal_fp32_nchw"]]
                                                      for k, v in res["variants"].items()}}))
    print("wrote", path)


if __name__ == "__main__":
    main()
