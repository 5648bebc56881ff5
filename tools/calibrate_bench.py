"""Cost of temperature calibration on the GPU, one JSON line per row, each with the card's name and power limit:

    stitch        the mean stitch at temperature 1.7 against the same call at temperature 1, in the same process
                  and alternating, for both routes (two-kernel: [n, C, T, T] logits; fused: channels-last decoder
                  outputs with the x4 up-sample in the stitch), at 45 and 273 tiles, C = 9, T = 512
    prob_scores   pylc_prob_scores, NLL only and with the Brier score, at 3000x2000 and 6000x4000 (C = 9; the
                  probability map at the fitted size of each, 3072x2048 and 6144x4096)
    fit           `pylc calibrate`'s work on N synthetic 3000x2000 images (bench.py's workload, random-init network):
                  retention (one network pass per image), the search, and the two reports

Kernel rows are the median of --rounds rounds of --reps back-to-back calls between CUDA events.

    python tools/calibrate_bench.py [--images 4] [--rounds 7] [--reps 20] [--out calibrate.jsonl]
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from stitch_modes_bench import card  # noqa: E402


def timed(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def alternate(cases, rounds, reps):
    """{name: median ms} over `rounds` rounds that run every case once each, in turn."""
    for fn in cases.values():
        fn()
    times = {k: [] for k in cases}
    for _ in range(rounds):
        for k, fn in cases.items():
            times[k].append(timed(fn, reps))
    return {k: float(np.median(v)) for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("calibrate_bench.py needs a CUDA device")
    from pylc_b200 import _lib, ops
    _lib.load()
    gpu, limit = card()
    rows = []

    def emit(row):
        row.update(gpu=gpu, power_limit=limit)
        rows.append(row)
        print(json.dumps(row), flush=True)

    C, T, S, tpb = 9, 512, 256, 45
    g = torch.Generator(device="cuda").manual_seed(0)
    for nr, nc in ((5, 9), (13, 21)):
        n = nr * nc
        logits = [(torch.randn(min(tpb, n - i), C, T, T, device="cuda", generator=g) * 3) for i in range(0, n, tpb)]
        dec = [(torch.randn(min(tpb, n - i), C, T // 4, T // 4, device="cuda", generator=g) * 3)
               .contiguous(memory_format=torch.channels_last) for i in range(0, n, tpb)]
        for route, fn, src in (("two-kernel", ops.stitch_probs, logits), ("fused", ops.stitch_upsample_probs, dec)):
            h, w = ops.stitch_dims(nr, nc, T, S)
            out = {"labels": torch.empty((h, w), dtype=torch.uint8, device="cuda"),
                   "confidence": torch.empty((h, w), dtype=torch.uint8, device="cuda")}
            med = alternate({t: (lambda t=t: fn(src, nr, nc, T, S, mode="mean", tiles_per_batch=tpb, out=out,
                                                temperature=t)) for t in (1.0, 1.7)}, args.rounds, args.reps)
            emit({"row": "stitch", "route": route, "tiles": n, "C": C, "ms_t1": round(med[1.0], 4),
                  "ms_t1.7": round(med[1.7], 4), "ratio": round(med[1.7] / med[1.0], 4)})
        del logits, dec

    for (w_full, h_full), (w, h) in (((3000, 2000), (3072, 2048)), ((6000, 4000), (6144, 4096))):
        P = torch.softmax(torch.randn(C, h, w, device="cuda", generator=g), dim=0).contiguous()
        y = torch.randint(0, C, (h_full, w_full), device="cuda", generator=g, dtype=torch.int64).to(torch.uint8)
        ws = torch.empty((_lib.SCORES_WS_DOUBLES,), dtype=torch.float64, device="cuda")
        maps = ops.device_index_maps(w, h, w_full, h_full, "cuda")
        med = alternate({b: (lambda b=b: ops.prob_scores(P, y, w_full, h_full, want_brier=b, maps=maps, workspace=ws))
                         for b in (False, True)}, args.rounds, args.reps)
        for b in (False, True):
            # bytes the kernel must move at least: the truth plane, the index maps, and the gathered f32 values
            need = h_full * w_full * (1 + 4 * (C if b else 1)) + 4 * (w_full + h_full)
            emit({"row": "prob_scores", "brier": b, "full": [w_full, h_full], "fitted": [w, h], "C": C,
                  "ms": round(med[b], 4), "gb_per_s_of_gathered_bytes": round(need / (med[b] * 1e-3) / 1e9, 1)})
        del P, y

    from pylc_b200.pipeline import TiledSegmenter
    from pylc_b200.utils.calibrate import TemperatureFit
    cfg = bench.CONFIGS[1]
    bench.W_FULL, bench.H_FULL, bench.CH = cfg["w"], cfg["h"], cfg["ch"]
    model = bench.build_model(torch.device("cuda", 0))
    imgs, masks = bench.make_inputs(list(range(args.images)), model.meta.palette_rgb)
    seg = TiledSegmenter(model, batch_tiles=32, stitch="mean")
    fit = TemperatureFit(seg, torch.cuda.mem_get_info()[0] / 2)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for img, mask in zip(imgs, masks):
        fit.add(img.numpy(), mask.numpy())
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    res = fit.fit()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    before, after = fit.report(1.0), fit.report(res["temperature"])
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    emit({"row": "fit", "images": args.images, "size": [cfg["w"], cfg["h"]], "route": "eager network (pylc calibrate)",
          "retained_gb": round(fit.bytes / 1e9, 3), "s_retain": round(t1 - t0, 3), "s_search": round(t2 - t1, 3),
          "evaluations": len(res["evals"]), "ms_per_evaluation": round((t2 - t1) * 1e3 / len(res["evals"]), 3),
          "s_reports": round(t3 - t2, 3), "temperature": res["temperature"], "at_bound": res["at_bound"],
          "nll_before": before["nll"], "nll_after": after["nll"], "ln_T": round(math.log(res["temperature"]), 6)})
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
