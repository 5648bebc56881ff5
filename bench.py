#!/usr/bin/env python
"""
bench.py -- end-to-end tiled inference + evaluation throughput (BASELINE.json metric:
megapixels/s at 1/2/4/8 B200, kernel HBM GB/s as a fraction of the measured peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): a DST.A-shaped colour batch of 64 synthetic 3000x2000
image/mask pairs per GPU, schema_a (9 classes), DeepLabv3+/ResNet-101 random-init, 512x512 tiles
with 50 % overlap (45 tiles per image after the fit-resize to 2560x1536), stitch + argmax,
nearest-neighbour resample to full resolution, confusion matrix -> weighted IoU / F1 / MCC.
One "step" = one pass over the 64 images of a rank.  Weak scaling: every rank owns 64 images; the
only collective is the all-reduce of the [9,9] i64 confusion matrix.

    value   Mpx/s with the fitted images and ground truths already resident in HBM
    e2e     Mpx/s through pylc_b200.pipeline.TiledSegmenter.run_host: decoded images in pinned
            host memory -> pitched H2D on the copy engine -> device fit-resize (bit-exact INTER_AREA)
            -> gather -> network -> stitch -> resample + confusion -> D2H of the confusion matrix;
            every byte of every step's input crosses PCIe inside the timed region
    roofline   the custom kernel with the largest share of the timed step, timed live with CUDA
            events on its stream inside the timed steps; `kernels` lists every custom launch
    cpu_baseline / --impl reference   the reference's CPU path (oracle port: same per-class
            passes, band-merge loops, scikit-learn calls; torch CPU network) on the host cores

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (see dump_outputs); the inputs
and the network's weights are seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_IMAGES, W_FULL, H_FULL, CH, TILES_PER_IMAGE = 64, 3000, 2000, 3, 45
WORKLOAD = "configs[1]: 64 synthetic 3000x2000 colour image/mask pairs per GPU, schema_a, DeepLabv3+ " \
           "ResNet-101 random-init, 512px tiles stride 256, stitch+argmax+resample+confusion/mIoU"
METRIC = "megapixels/sec end-to-end tiled inference"
# BASELINE.json configs this file can run (--config): image set, geometry, channels.  configs[1] is the
# one the metric is quoted on (and what the driver runs); configs[4] is the sharded 6000x4000 gray set.
CONFIGS = {
    1: dict(n=64, w=3000, h=2000, ch=3, tiles=45,
            name="configs[1]: 64 synthetic 3000x2000 colour image/mask pairs {per}, schema_a, DeepLabv3+ "
                 "ResNet-101 random-init, 512px tiles stride 256, stitch+argmax+resample+confusion/mIoU"),
    4: dict(n=16, w=6000, h=4000, ch=1, tiles=273,
            name="configs[4]: 16 synthetic 6000x4000 grayscale image/mask pairs {per}, schema_a, DeepLabv3+ "
                 "ResNet-101 random-init, 512px tiles stride 256 (273 tiles/image), stitch+argmax+resample+confusion"),
}


def peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
        reasons = []
        for k, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
            if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_inputs(global_indices, palette):
    """The rank's decoded image / RGB-mask pairs as tightly packed [H,W(,3)] u8 tensors in PINNED host
    memory -- what cv2.imread hands the reference, page-locked.  Image g is a function of its GLOBAL
    index only, so every partition of the same set over any number of ranks sees the same pixels."""
    from pylc_b200 import synth

    def one(g):
        return (torch.from_numpy(synth.image(g, W_FULL, H_FULL, CH)).pin_memory(),
                torch.from_numpy(synth.mask(g, W_FULL, H_FULL, palette)).pin_memory())
    with cf.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 4)) as ex:
        pairs = list(ex.map(one, global_indices))
    imgs = [p[0] for p in pairs]
    masks = [p[1] for p in pairs]
    return imgs, masks


def build_model(device, seed=0):
    from pylc_b200.config import defaults
    from pylc_b200.models.model import Model
    torch.manual_seed(seed)
    model = Model()
    model.track = False
    model.device = device
    px_mean = list(defaults.px_rgb_mean) if CH == 3 else [defaults.px_grayscale_mean]
    px_std = list(defaults.px_rgb_std) if CH == 3 else [defaults.px_grayscale_std]
    model.update_meta({"ch": CH, "arch": "deeplab", "backbone": "resnet", "pretrained": False,
                       "px_mean": px_mean, "px_std": px_std,
                       "weights": [1.0] * defaults.n_classes, "normalize_default": False})
    model.build()
    model.net.eval()
    return model


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU path on a bounded sample
# ---------------------------------------------------------------------------------------------

def reference_sample():
    """Bounded sample of the workload at image granularity: ONE whole image of the configuration and its
    mask (configs[1]: 3000x2000 -> fitted 2560x1536 -> all 45 tiles), i.e. 1/64 of a step; every phase
    of the path is per image."""
    from pylc_b200 import synth
    from pylc_b200.config import defaults
    img = synth.image(0, W_FULL, H_FULL, CH)
    gt = synth.mask(0, W_FULL, H_FULL, defaults.palette_rgb)
    return img, gt, "image 0 of the set, whole (%dx%d, %s + RGB mask): all its tiles, every phase incl. the CPU network" % (
        W_FULL, H_FULL, "colour" if CH == 3 else "gray")


class ReferenceCPU(object):
    """pylc.py test on the CPU as the reference runs it (test.py:52-115), via the oracle port."""

    def __init__(self):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import pylc_oracle as orc                       # allowed here: cpu_baseline / reference leg
        from pylc_b200.config import defaults
        from pylc_b200.models.deeplab import DeepLab    # stock torch ops; state_dict == reference's
        self.orc, self.meta = orc, defaults
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        torch.manual_seed(0)
        self.net = DeepLab(n_classes=defaults.n_classes).eval()
        if CH == 3:
            self.mean = torch.tensor(defaults.px_rgb_mean)[None, :, None, None]
            self.std = torch.tensor(defaults.px_rgb_std)[None, :, None, None]
        else:                                            # model.py:433-435: one gray mean / std
            self.mean = torch.tensor([defaults.px_grayscale_mean])[None, :, None, None]
            self.std = torch.tensor([defaults.px_grayscale_std])[None, :, None, None]

    def step(self, img, gt):
        import cv2
        orc, meta, T, S = self.orc, self.meta, 512, 256
        ph = {}
        t0 = time.perf_counter()
        w_fit, h_fit = orc.fit_dims(img.shape[1], img.shape[0], T)
        fitted = cv2.resize(img, (w_fit, h_fit), interpolation=cv2.INTER_AREA)      # tools.py:194
        tiles = orc.split_tiles(fitted, T, S)                                       # extract.py:296-310
        ph["fit+split"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        outs = []
        with torch.no_grad():
            for lo in range(0, len(tiles), 8):                                       # test.py:68-83, batch 8
                x = torch.tensor(tiles[lo:lo + 8]).float()
                x = ((x - self.mean) / self.std) / 255                               # model.py:443-445
                if x.shape[1] == 1:
                    x = torch.cat((x, x, x), 1)                                      # model.py:376-377
                outs.append(self.net(x).numpy())
        ph["network_cpu"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        rgb = orc.reconstruct_port(outs, h_fit, w_fit, img.shape[1], img.shape[0], T, S, meta.palette_rgb,
                                   meta.n_classes)                                   # tools.py:209-319
        ph["reconstruct"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        y_pred = orc.class_encode_port(np.moveaxis(rgb.astype(np.uint8), 2, 0)[None], meta.palette_rgb).ravel()
        y_true = orc.class_encode_port(np.moveaxis(gt, 2, 0)[None], meta.palette_rgb).ravel()  # evaluate.py:103-108
        ph["class_encode x2"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        y_true, y_pred = orc.inject_coverage(y_true, y_pred, len(meta.class_codes))  # evaluate.py:172-174
        res = orc.metrics_port(y_true, y_pred, meta.class_codes)                     # metrics.py:45-87
        ph["sklearn_metrics"] = time.perf_counter() - t0
        return res, ph


def run_reference(args, rank):
    if rank != 0:
        return
    img, gt, desc = reference_sample()
    ref = ReferenceCPU()
    mpx = img.shape[0] * img.shape[1] / 1e6
    for _ in range(args.warmup):
        ref.step(img, gt)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, phases = ref.step(img, gt)
    dt = time.perf_counter() - t0
    v = mpx * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mpx/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample_per_step": desc},
            "cpu_baseline": {"value": v, "unit": "Mpx/s", "cores": ref.cores, "kind": "port", "sample": desc,
                             "phases_s": {k: round(x, 3) for k, x in phases.items()}},
            "e2e": {"value": v, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline():
    img, gt, desc = reference_sample()
    ref = ReferenceCPU()
    t0 = time.perf_counter()
    _, phases = ref.step(img, gt)
    dt = time.perf_counter() - t0
    return {"value": img.shape[0] * img.shape[1] / 1e6 / dt, "unit": "Mpx/s", "cores": ref.cores, "kind": "port",
            "sample": desc + "; 1 pass, no warm-up", "phases_s": {k: round(x, 3) for k, x in phases.items()}}


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------

class KernelTimer(object):
    """Wraps the ops.* calls of the pipeline with CUDA events on the launching stream and counts the
    algorithmic bytes of every launch (SURVEY.md 8d: compulsory HBM traffic of the call)."""

    def __init__(self, ops):
        self.ops, self.on, self.rows, self.orig = ops, False, {}, {}
        nb = lambda t: t.numel() * t.element_size()          # noqa: E731

        def stitch_bytes(a, k, out):
            lg = a[0]
            n_logit = sum(t.numel() for t in lg) if isinstance(lg, (list, tuple)) else lg.numel()
            return n_logit * 4 + out[0].numel()               # every logit once + 1 B label per output px
        self.bytes_of = {
            "fit_resize_area": lambda a, k, out: (a[1] * a[2] + a[5] * a[6]) * a[3],         # source once + fitted once
            "tile_gather_norm_s2d": lambda a, k, out: a[1] * a[2] * a[3] + nb(out),          # fitted image once + tiles
            "tile_gather_norm_f32": lambda a, k, out: a[1] * a[2] * a[3] + nb(out),
            "maxpool3x3s2_nhwc": lambda a, k, out: nb(a[0]) + nb(out),
            "upsample_concat_nhwc": lambda a, k, out: nb(a[0]) + nb(a[1]) + nb(out),
            "upsample_nhwc_to_nchw": lambda a, k, out: nb(a[0]) + nb(out),
            "stitch_argmax_colour": stitch_bytes,
            "stitch_upsample_argmax_colour": stitch_bytes,     # decoder output once + 1 B label per output px
            "resample_encode_confusion": lambda a, k, out: a[1] * a[2] * 4,                  # 3 B ground truth + 1 B label per px
        }

    def __enter__(self):
        for name, fn_bytes in self.bytes_of.items():
            orig = getattr(self.ops, name)
            self.orig[name] = orig

            def timed(*a, _orig=orig, _name=name, _fb=fn_bytes, **k):
                if not self.on:
                    return _orig(*a, **k)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = _orig(*a, **k)
                e.record()
                row = self.rows.setdefault(_name, {"pairs": [], "bytes": 0})
                row["pairs"].append((s, e))
                row["bytes"] += _fb(a, k, out)
                return out
            setattr(self.ops, name, timed)
        return self

    def __exit__(self, *a):
        for name, orig in self.orig.items():
            setattr(self.ops, name, orig)

    def result(self, peak, step_ms, steps):
        out = []
        for name, row in self.rows.items():
            ms = [s.elapsed_time(e) for s, e in row["pairs"]]
            if not ms:
                continue
            avg_ms, avg_b = sum(ms) / len(ms), row["bytes"] / len(ms)
            out.append({"op": name, "launches_per_step": len(ms) // steps, "avg_launch_ms": avg_ms,
                        "algorithmic_bytes_per_launch": avg_b, "achieved_gbs": avg_b / (avg_ms * 1e-3) / 1e9,
                        "frac": avg_b / (avg_ms * 1e-3) / 1e9 / peak, "share_of_step": sum(ms) / steps / step_ms})
        return sorted(out, key=lambda r: -r["share_of_step"])


def ncu_traffic(tag, kernel_prefix):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu captures
    (profiles/traffic_r2.json, else traffic_r1.json; written by tools/summarise_profiles.py)."""
    for name in ("traffic_r2.json", "traffic_r1.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                for row in json.load(f).get(tag, []):
                    if row["kernel"].startswith(kernel_prefix):
                        return row["dram_bytes"], "profiles/" + name
        except Exception:
            pass
    return None, None


# op of the pipeline -> (kernel it launches, tag of its ncu capture in profiles/traffic_r*.json, bound)
KERNEL_OF = {
    "stitch_argmax_colour": ("stitch_kernel", "stitch45", "hbm"),
    "stitch_upsample_argmax_colour": ("stitch_up_kernel", "stitchup", "issue (exp + FMA per class; reads 16x fewer bytes than the logits)"),
    "upsample_concat_nhwc": ("upsample_concat_staged_kernel", "netglue", "hbm"),
    "maxpool3x3s2_nhwc": ("maxpool3x3s2_kernel", "netglue", "hbm"),
    "upsample_nhwc_to_nchw": ("upsample_to_nchw_staged_kernel", "netglue", "hbm"),
    "tile_gather_norm_s2d": ("gather_norm_s2d_staged_kernel", "gather_s2d", "hbm"),
    "tile_gather_norm_f32": ("gather_norm_staged_kernel", "gather_norm", "hbm"),
    "fit_resize_area": ("area_resize_x2_kernel", "resize", "issue (OpenCV's float sequence replayed exactly, two elements per FFMA2 / FADD2)"),
    "resample_encode_confusion": ("resample_confusion_tma_kernel", "resample", "hbm in the steady state; set-up and flush of a 15 us launch"),
}


def roofline_of(kernels, peak, peak_kind, images_per_step, step_ms):
    """The `roofline` object of the JSON line: the custom kernel with the largest share of the timed step
    (timed live with CUDA events on its stream; every custom launch is listed under `kernels`)."""
    if not kernels:
        return None
    top = max(kernels, key=lambda r: r["share_of_step"])
    kern, tag, bound = KERNEL_OF.get(top["op"], (top["op"], None, "hbm"))
    traffic, src = ncu_traffic(tag, kern) if tag else (None, None)
    return {"kernel": "%s (pylc op %s)" % (kern, top["op"]), "bound": "hbm", "limited_by": bound,
            "achieved": top["achieved_gbs"], "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": top["frac"],
            "avg_launch_ms": top["avg_launch_ms"], "algorithmic_bytes_per_launch": top["algorithmic_bytes_per_launch"],
            "traffic": traffic, "traffic_source": (src + ": ncu --set full capture of this launch shape, dram read + write") if src else None,
            "share_of_step": top["share_of_step"],
            "why_this_kernel": "the custom kernel with the largest share of the timed step; every custom launch of the step is listed under `kernels` with its own fraction"}


LABEL_SAMPLE = 1 << 22      # label values --dump-outputs writes (16 MB as float32)


def dump_outputs(out_dir, conf, conf_e2e, results, n_images):
    """--dump-outputs: what the last timed step of each timed pass returned, as float arrays.
        confusion.npy      [C,C] confusion matrix of the resident pass (all-reduced; counts are exact in float64)
        confusion_e2e.npy  [C,C] the matrix run_host returned
        labels.npy         [images, k] this rank's fitted-resolution label maps at k fixed positions
        labels_index.npy   [k] those positions, flat indices into one [h,w] map, drawn with seed 0
    The convolution routes and cuDNN engines are fixed per layer shape rather than timed (models/fused.py), so
    repeated runs with the same arguments write the same arrays.
    """
    if len(results) != n_images:
        raise SystemExit("bench.py: the last timed step returned %d per-image results for %d images" % (len(results), n_images))
    maps = torch.stack([r["labels"] for r in results]).flatten(1)
    n, hw = maps.shape
    k = min(hw, max(1, LABEL_SAMPLE // n))
    index = np.sort(np.random.default_rng(0).choice(hw, size=k, replace=False))
    sample = maps[:, torch.from_numpy(index).to(maps.device)].cpu().numpy()
    arrays = {"confusion": conf.astype(np.float64), "confusion_e2e": conf_e2e.astype(np.float64),
              "labels": sample.astype(np.float32), "labels_index": index.astype(np.float64)}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    from pylc_b200 import _lib, ops
    from pylc_b200 import dist as pdist
    from pylc_b200.pipeline import TiledSegmenter

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    _lib.load()
    # cuDNN's heuristic engines, not timed ones: a timed choice can differ between runs, and with it the TF32 sums
    torch.backends.cudnn.benchmark = False
    dtype = {"fp32": None, "bf16": torch.bfloat16, "fp16": torch.float16}[args.backbone_dtype]

    model = build_model(device)
    seg = TiledSegmenter(model, batch_tiles=args.batch_tiles, channels_last=not args.no_channels_last,
                         autocast_dtype=dtype, host_workers=args.host_workers, fuse_network=not args.no_fuse,
                         device_fit=not args.host_fit, fuse_upsample=not args.no_fuse_upsample)
    # weak: every rank owns N_IMAGES images (global index rank * N_IMAGES + i); strong: ONE set of
    # N_IMAGES images dealt round-robin over the ranks (dist.shard_indices, SURVEY.md 8e)
    strong = args.scaling == "strong"
    gidx = pdist.shard_indices(N_IMAGES, rank, world) if strong else [rank * N_IMAGES + i for i in range(N_IMAGES)]
    imgs, masks = make_inputs(gidx, model.meta.palette_rgb)
    n_mine = len(gidx)
    mpx_job = (N_IMAGES if strong else N_IMAGES * world) * W_FULL * H_FULL / 1e6      # whole job, all ranks
    d2h = seg.C * seg.C * 8

    def barrier_sync():
        torch.cuda.synchronize()
        pdist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM -------------------------------------------------------
    stage = seg.stage_device if seg.can_fit_on_device(imgs[0]) else (lambda im, gt, index: seg.stage(im.numpy(), gt.numpy(), index=index))
    resident = [stage(imgs[i], masks[i], index=gidx[i]) for i in range(n_mine)]
    torch.cuda.synchronize()
    h2d = sum(im.numel() + gt.numel() for im, gt in zip(imgs, masks)) if seg.can_fit_on_device(imgs[0]) \
        else sum(f.img.numel() + f.gt.numel() for f in resident)      # bytes run_host copies per step
    clocks = ClockSampler(local_rank)
    last_results = []
    with KernelTimer(ops) as st:
        for _ in range(args.warmup):
            seg.reset()
            seg.run_resident(resident)
        barrier_sync()
        st.on = True
        clocks.start()
        launches0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.profiler.start()     # no-op unless run under `ncu --profile-from-start off` (tools/gpu_profile.sh)
        ev0.record()
        for step in range(args.steps):
            seg.reset()
            seg.run_resident(resident, results=last_results if args.dump_outputs and step == args.steps - 1 else None)
            conf_dev = pdist.all_reduce_(seg.conf.clone()) if world > 1 else seg.conf
        ev1.record()
        barrier_sync()
        torch.cuda.profiler.stop()
        st.on = False
        launches = _lib.launch_count() - launches0
        ms = pdist.max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        kernels = st.result(peak_gbs()[0], ms, args.steps)
    conf_resident = conf_dev.cpu().numpy()
    del resident

    # ---- e2e: host buffers, copies inside the timed region -------------------------------------
    for _ in range(max(1, min(args.warmup, 2))):
        seg.reset()
        seg.run_host(imgs, masks, distributed=world > 1, global_indices=gidx)
    barrier_sync()
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        seg.reset()
        conf_host, _ = seg.run_host(imgs, masks, distributed=world > 1, global_indices=gidx)
    ev1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = pdist.max_over_ranks(max(ev0.elapsed_time(ev1), wall_ms)) / args.steps
    barrier_sync()
    clk = clocks.summary()

    if rank != 0:
        return
    peak, peak_kind = peak_gbs()
    scores = seg.scores(conf_host)
    line = {
        "metric": METRIC, "value": mpx_job / (ms * 1e-3), "unit": "Mpx/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32 hot-path kernels (u8/i64 integer paths); network %s" % (
            "fp32 with cuDNN TF32 (PyTorch default, as the reference would run)" if dtype is None else args.backbone_dtype),
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "images_per_gpu": n_mine, "images_total": N_IMAGES if strong else N_IMAGES * world,
                   "tiles_per_image": TILES_PER_IMAGE, "batch_tiles": args.batch_tiles,
                   "network_plan": "eager nn.Module" if args.no_fuse else "BatchNorm folded, cuDNN fused conv+bias(+add)+ReLU, channels_last, space-to-depth stem, pylc max-pool / up-sample+concat / final up-sample kernels",
                   "l2": "inputs larger than L2 (each step streams > 20 GB of logits per GPU)",
                   "parallelism": "dp%d, images sharded (%s), one [9,9] i64 all-reduce per step" % (
                       world, "one fixed set dealt round-robin" if strong else "a fixed set per rank"),
                   "fit_resize": "host cv2 threads" if args.host_fit else "device (pylc_fit_resize_area_u8, bit-exact INTER_AREA)",
                   "value_region": ("fitted" if args.host_fit else "decoded") + " u8 images + RGB ground truth resident in HBM -> all-reduced confusion matrix",
                   "weighted_iou": scores["iou"], "confusion_sum": int(conf_host.sum()),
                   "resident_equals_e2e": bool(np.array_equal(conf_resident, conf_host))},
        "e2e": {"value": mpx_job / (e2e_ms * 1e-3), "unit": "Mpx/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "api": "pylc_b200.pipeline.TiledSegmenter.run_host"},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": roofline_of(kernels, peak, peak_kind, n_mine, ms),
        "kernels": kernels,
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, conf_resident, conf_host, last_results, n_mine)
    print(json.dumps(line), flush=True)
    if not line["config"]["resident_equals_e2e"]:
        # both paths process the same images with ONE coverage injection (global image 0): the integer
        # matrices must be identical at every GPU count -- anything else is a parity failure
        raise SystemExit("bench.py: confusion matrix of the resident pass differs from the end-to-end pass")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--backbone-dtype", default="fp32", choices=["fp32", "bf16", "fp16"])
    ap.add_argument("--batch-tiles", type=int, default=45)
    ap.add_argument("--host-workers", type=int, default=6)
    ap.add_argument("--no-channels-last", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--host-fit", action="store_true", help="fit-resize on host threads with cv2 (the reference's call) "
                    "instead of the bit-exact device kernel")
    ap.add_argument("--no-fuse", action="store_true", help="run the eager nn.Module instead of the BN-folded cuDNN-fused plan")
    ap.add_argument("--no-fuse-upsample", action="store_true", help="final x4 up-sample and stitch as two kernels instead of "
                    "the fused stitch that reads the decoder output (same results, bit for bit)")
    ap.add_argument("--images", type=int, default=None, help="images per GPU per step (weak) or in total (strong); "
                    "default: the configuration's own count (profiling runs use fewer)")
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS), help="BASELINE.json configs index: 1 = the "
                    "colour 3000x2000 set the metric is quoted on (default, what the driver runs); 4 = gray 6000x4000")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: --images per GPU (default); "
                    "strong: ONE set of --images dealt round-robin over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last "
                    "timed step returned to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = CONFIGS[args.config]
    n_img = cfg["n"] if args.images is None else args.images
    globals().update(N_IMAGES=n_img, W_FULL=cfg["w"], H_FULL=cfg["h"], CH=cfg["ch"], TILES_PER_IMAGE=cfg["tiles"],
                     WORKLOAD=cfg["name"].format(per="per GPU" if args.scaling == "weak" else "in total (strong scaling)")
                     .replace("%d synthetic" % cfg["n"], "%d synthetic" % n_img))
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")))
        return
    from pylc_b200 import dist as pdist
    rank, world, local_rank = pdist.init_from_env()
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus %d needs torchrun (one process per GPU); WORLD_SIZE is 1" % args.gpus)
    run_ours(args, rank, world, local_rank)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
