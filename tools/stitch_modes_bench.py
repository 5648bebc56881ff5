"""Throughput of the three stitch settings of TiledSegmenter on bench.py's workload (BASELINE.json configs[1]:
3000x2000 colour images resident in HBM, the BN-folded inference plan with the fused up-sample + stitch),
measured in ONE process so that the three rows share the card, the clocks and the inputs:

    default           stitch="reference", confidence=False   (bench.py's `value` path)
    reference+conf    stitch="reference", confidence=True    (same labels, + the u8 confidence plane)
    mean+conf         stitch="mean",      confidence=True    (labels from the mean of the covering softmaxes)

Cases alternate round by round; each prints one JSON line with the median Mpx/s over the rounds, the card's name
and its power limit read in the same run.

    python tools/stitch_modes_bench.py [--images 16] [--steps 3] [--rounds 5] [--out stitch_modes.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

CASES = (("default", "reference", False), ("reference+confidence", "reference", True), ("mean+confidence", "mean", True))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=16)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch-tiles", type=int, default=45)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stitch_modes_bench.py needs a CUDA device")
    from pylc_b200 import _lib
    from pylc_b200.pipeline import TiledSegmenter
    cfg = bench.CONFIGS[1]
    bench.W_FULL, bench.H_FULL, bench.CH = cfg["w"], cfg["h"], cfg["ch"]
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    _lib.load()
    torch.backends.cudnn.benchmark = False
    model = bench.build_model(device)
    imgs, masks = bench.make_inputs(list(range(args.images)), model.meta.palette_rgb)
    segs = {}
    fused = None
    for name, stitch, conf in CASES:
        seg = TiledSegmenter(model, batch_tiles=args.batch_tiles, fuse_network=fused is None, stitch=stitch, confidence=conf)
        if fused is None:
            fused = seg.fused
        else:
            seg.fused, seg.s2d, seg.fuse_upsample = fused, segs["default"].s2d, segs["default"].fuse_upsample
        segs[name] = seg
    base = segs["default"]
    resident = [base.stage_device(imgs[i], masks[i], index=i) for i in range(args.images)]
    torch.cuda.synchronize()
    mpx = args.images * cfg["w"] * cfg["h"] / 1e6
    times = {name: [] for name, _, _ in CASES}
    for name, _, _ in CASES:
        for _ in range(args.warmup):
            segs[name].reset()
            segs[name].run_resident(resident)
    for _ in range(args.rounds):
        for name, _, _ in CASES:
            seg = segs[name]
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                seg.reset()
                seg.run_resident(resident)
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)
    confs = {name: segs[name].conf.cpu().numpy() for name, _, _ in CASES}
    gpu, limit = card()
    rows = []
    for name, stitch, conf in CASES:
        ms = float(np.median(times[name]))
        rows.append({"case": name, "stitch": stitch, "confidence": conf, "mpx_per_s": round(mpx / (ms / 1e3), 2),
                     "ms_per_step_median": round(ms, 3), "ms_per_step_all": [round(t, 3) for t in times[name]],
                     "images_per_step": args.images, "steps": args.steps, "rounds": args.rounds,
                     "confusion_equals_default": bool(np.array_equal(confs[name], confs["default"])),
                     "gpu": gpu, "power_limit": limit, "workload": "configs[1] 3000x2000 colour, resident in HBM"})
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
