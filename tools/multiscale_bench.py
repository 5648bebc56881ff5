"""Multi-scale inference on a B200: the combine kernel alone and bench.py's workload end to end, in one process.

    combine   pylc_multiscale_combine at 3000x2000 and 6000x4000 output, K = 1, 2, 3 members (scales (1.0,),
              (0.75, 1.0), (0.75, 1.0, 1.25) of that image, planes of the fitted sizes), C = 9: median of CUDA-event
              times over many launches with L2 flushed between them (tools/kbench.py's Timer), algorithmic bytes
              (every plane read once, labels + confidence written) and their share of the 6553 GB/s copy peak
              measured for this project (profiles/kbench_r2.jsonl)
    e2e       bench.py's workload (BASELINE.json configs[1]: 3000x2000 colour images resident in HBM, the
              random-init network's inference plan) through TiledSegmenter.run_resident with stitch="mean",
              confidence=True and scales (1.0,), (0.75, 1.0), (0.75, 1.0, 1.25), one case after the other; Mpx/s
              of evaluated (full-resolution) pixels, the combine kernel's share of the step (images x its isolated
              time / step time) and whether the (1.0,) run's confusion matrix and labels equal the single-scale
              mean stitch's
    ptxas     registers / spills of every instantiation from `nvcc -Xptxas -v` of csrc/multiscale.cu

Every record carries the card's name and power limit, read in the same run.

    python tools/multiscale_bench.py [--images 64] [--rounds 2] [--out-dir profiles]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402

COPY_PEAK_GBS = 6553.0
SCALE_SETS = ((1.0,), (0.75, 1.0), (0.75, 1.0, 1.25))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def ptxas_report():
    src = os.path.join(ROOT, "pylc_b200", "csrc", "multiscale.cu")
    with tempfile.TemporaryDirectory() as tmp:
        out = subprocess.run(["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                              "-c", src, "-o", os.path.join(tmp, "m.o")], capture_output=True, text=True, check=True).stderr
    rows, name = [], None
    for line in out.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            spill = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            k = re.search(r"ILi(\d+)E", name)
            rows.append((int(k.group(1)) if k else name, int(m.group(1)), spill))
            name = None
    return sorted(rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--batch-tiles", type=int, default=45)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multiscale_bench.py needs a CUDA device")
    from kbench import Timer
    from pylc_b200 import _lib, ops
    from pylc_b200.pipeline import TiledSegmenter, multiscale_geometry
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    _lib.load()
    torch.backends.cudnn.benchmark = False
    gpu, limit = card()
    rows = []

    def emit(r):
        r.update({"gpu": gpu, "power_limit": limit})
        rows.append(r)
        print(json.dumps(r), flush=True)

    # ---- the combine kernel alone -------------------------------------------------------------
    C = 9
    timer = Timer(args.iters)
    combine_ms = {}
    for W, H in ((3000, 2000), (6000, 4000)):
        for scales in SCALE_SETS:
            geo = multiscale_geometry(W, H, 512, scales)
            g = torch.Generator(device=device).manual_seed(W + len(scales))
            planes = [torch.rand((C, g_["fitted"][1], g_["fitted"][0]), generator=g, device=device) for g_ in geo]
            out = {"labels": torch.empty((H, W), dtype=torch.uint8, device=device),
                   "confidence": torch.empty((H, W), dtype=torch.uint8, device=device)}
            med, best = timer.run(lambda: ops.multiscale_combine(planes, W, H, out=out))
            nbytes = sum(p.numel() * 4 for p in planes) + 2 * W * H
            combine_ms[(W, H, scales)] = med
            emit({"what": "combine", "kernel": "multiscale_combine_kernel<%d>" % len(scales), "w_full": W, "h_full": H,
                  "K": len(scales), "C": C, "scales": list(scales), "planes": [list(g_["fitted"]) for g_ in geo],
                  "ms_median": round(med, 4), "ms_min": round(best, 4), "alg_bytes": nbytes,
                  "gbs": round(nbytes / (med / 1e3) / 1e9, 1),
                  "share_of_copy_peak": round(nbytes / (med / 1e3) / 1e9 / COPY_PEAK_GBS, 3),
                  "l2": "flushed between launches", "iters": args.iters})
            del planes, out
    del timer
    torch.cuda.empty_cache()

    # ---- end to end: bench.py's workload --------------------------------------------------------
    cfg = bench.CONFIGS[1]
    bench.W_FULL, bench.H_FULL, bench.CH = cfg["w"], cfg["h"], cfg["ch"]
    W, H = cfg["w"], cfg["h"]
    model = bench.build_model(device)
    imgs, masks = bench.make_inputs(list(range(args.images)), model.meta.palette_rgb)
    base = TiledSegmenter(model, batch_tiles=args.batch_tiles, fuse_network=True, stitch="mean", confidence=True)
    segs = {}
    for scales in SCALE_SETS:
        seg = TiledSegmenter(model, batch_tiles=args.batch_tiles, fuse_network=False, stitch="mean", confidence=True,
                             scales=scales)
        seg.fused, seg.s2d, seg.fuse_upsample = base.fused, base.s2d, base.fuse_upsample
        segs[scales] = seg
    mpx = args.images * W * H / 1e6
    times = {s: [] for s in SCALE_SETS}
    for scales in SCALE_SETS:            # one case's images are resident at a time: K members each
        seg = segs[scales]
        resident = [seg.stage_device(imgs[i], masks[i], index=i) for i in range(args.images)]
        torch.cuda.synchronize()
        seg.reset()
        seg.run_resident(resident)      # warm-up
        for _ in range(args.rounds):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            seg.reset()
            seg.run_resident(resident)
            e1.record()
            e1.synchronize()
            times[scales].append(e0.elapsed_time(e1))
        if scales == (1.0,):
            one = []
            seg.reset()
            seg.run_resident(resident[:4], results=one)
            ref_res = []
            ref_stage = [base.stage_device(imgs[i], masks[i], index=i) for i in range(4)]
            base.reset()
            base.run_resident(ref_stage, results=ref_res)
            maps = [ops.resample_encode_confusion(b["labels"], W, H, n_classes=base.C, want_pred=True)["pred_full"] for b in ref_res]
            confs = [ops.confidence_resample(b["confidence"], W, H)["confidence_full"] for b in ref_res]
            same = bool(torch.equal(seg.conf, base.conf)) and all(
                torch.equal(a["labels"], m) and torch.equal(a["confidence"], q) for a, m, q in zip(one, maps, confs))
            del ref_stage, ref_res, one
        del resident
        torch.cuda.empty_cache()
    for scales in SCALE_SETS:
        ms = float(np.median(times[scales]))
        comb = args.images * combine_ms[(W, H, scales)]
        emit({"what": "e2e", "scales": list(scales), "images_per_step": args.images, "mpx_per_s": round(mpx / (ms / 1e3), 2),
              "ms_per_step_median": round(ms, 1), "ms_per_step_all": [round(t, 1) for t in times[scales]],
              "sum_s2": round(sum(s * s for s in scales), 4),
              "combine_share_of_step": round(comb / ms, 4), "combine_share_basis": "images x isolated kernel median / step",
              "outputs_equal_single_scale_mean": same if scales == (1.0,) else None,
              "workload": "configs[1] %dx%d colour, resident in HBM, stitch=mean, confidence=True" % (W, H)})

    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "multiscale_r4.jsonl"), "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    with open(os.path.join(args.out_dir, "multiscale_r4_ptxas.md"), "w") as f:
        f.write("# pylc_multiscale_combine: registers and spills (`nvcc -Xptxas -v`, sm_100a, -O3)\n\n"
                "| instantiation | registers | spill stores / loads (bytes) |\n|---|---|---|\n")
        for k, regs, spill in ptxas_report():
            f.write("| multiscale_combine_kernel<%s> | %d | %d / %d |\n" % (k, regs, spill[0], spill[1]))


if __name__ == "__main__":
    main()
