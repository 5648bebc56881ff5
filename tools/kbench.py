"""Per-kernel micro-benchmark: achieved algorithmic HBM GB/s of every custom kernel at the
BASELINE sizes, against the measured peak in MEASURED_PEAKS.json.  CUDA events around each
launch on the launching stream, L2 flushed between launches.  Writes one JSON line per kernel.

    python tools/kbench.py [--iters 20] [--out gpurun_out/kbench.jsonl] [--only stitch,loss]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from pylc_b200 import ops  # noqa: E402
from pylc_b200.config import Parameters  # noqa: E402


def peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class Timer:
    def __init__(self, iters, warmup=3):
        self.iters, self.warmup = iters, warmup
        self.flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def run(self, fn):
        for _ in range(self.warmup):
            fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(self.iters):
            # evict L2 (126 MB) between timed launches: a 512 MB fill, then a 512 MB read.  Together
            # they also keep the GPU busy (~200 us) while the host enqueues the timed launch, so
            # host-side launch cost (ctypes marshalling) never shows up between the two events
            self.flush.zero_()
            self.sink = self.flush.view(torch.int32).sum()   # read pass: leaves CLEAN lines, so no dirty
            #                                                  write-backs compete with the timed kernel
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            e.synchronize()
            times.append(s.elapsed_time(e))
        return float(np.median(times)), float(np.min(times))

    def run_sweep(self, fns, rounds=6):
        """Back-to-back launches over DISTINCT input sets whose combined footprint exceeds L2 (so every
        launch streams from HBM without a flush in between): the shape of an extraction / evaluation
        sweep over many images.  Returns ms per launch."""
        for fn in fns:
            fn()
        torch.cuda.synchronize()
        self.flush.zero_()
        self.sink = self.flush.view(torch.int32).sum()
        # the launches are captured into one CUDA graph so that host-side enqueue cost (ctypes, Python)
        # cannot throttle the back-to-back stream
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(rounds):
                for fn in fns:
                    fn()
        graph.replay()
        torch.cuda.synchronize()
        self.flush.zero_()
        self.sink = self.flush.view(torch.int32).sum()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        graph.replay()
        e.record()
        e.synchronize()
        return s.elapsed_time(e) / (rounds * len(fns))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    only = set(filter(None, args.only.split(",")))
    import pylc_oracle as orc
    peak, peak_kind = peak_gbs()
    tm = Timer(args.iters)
    meta = Parameters()
    pal, C = meta.palette_rgb, meta.n_classes
    T = 512
    rows = []

    def report(name, alg_bytes, fn, note=""):
        if only and not any(o in name for o in only):
            return
        med, best = tm.run(fn)
        gbs = alg_bytes / (med * 1e-3) / 1e9
        row = {"kernel": name, "ms_median": round(med, 4), "ms_min": round(best, 4), "alg_MB": round(alg_bytes / 1e6, 2),
               "achieved_gbs": round(gbs, 1), "peak_gbs": peak, "peak_kind": peak_kind, "frac": round(gbs / peak, 4),
               "note": note}
        rows.append(row)
        print(json.dumps(row), flush=True)

    def report_sweep(name, alg_bytes, fns, note=""):
        if only and not any(o in name for o in only):
            return
        ms = tm.run_sweep(fns)
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        row = {"kernel": name, "ms_per_launch": round(ms, 4), "launches": 6 * len(fns), "alg_MB": round(alg_bytes / 1e6, 2),
               "achieved_gbs": round(gbs, 1), "peak_gbs": peak, "peak_kind": peak_kind, "frac": round(gbs / peak, 4),
               "timing": "events around %d back-to-back launches over %d distinct input sets (> L2)" % (6 * len(fns), len(fns)),
               "note": note}
        rows.append(row)
        print(json.dumps(row), flush=True)

    # ---- the harness's floor: what this timer reads for a launch that does (almost) nothing -------------
    one = torch.ones((4,), dtype=torch.float32, device="cuda")
    unit = torch.ones((1,), dtype=torch.float32, device="cuda")
    report("launch floor: pylc_scale_unless_one_f32 on 4 floats (reads one scalar, returns)", 16,
           lambda: ops.scale_unless_one_(one, unit),
           "events around ONE launch after an L2 flush: every single-launch row above ~10 us of kernel time contains about this much "
           "launch latency; the `sweep` rows (one CUDA graph of back-to-back launches) do not")

    # ---- extraction ------------------------------------------------------------------------
    W, H = 6000, 4000
    mask = orc.synth_mask(0, W, H, pal, skew=True)
    d_mask, mp = ops.upload_image(mask)
    nH, nW = ops.tile_grid(H, W, T, 512)
    m_out = torch.empty((nH * nW, T, T), dtype=torch.uint8, device="cuda")
    tile_px = nH * nW * T * T
    m_hist = torch.zeros((nH * nW, C), dtype=torch.int64, device="cuda")
    report("mask_gather_encode_hist 6000x4000 S512 C9", tile_px * 4,
           lambda: ops.mask_gather_encode_hist(d_mask, H, W, mp, T, 512, pal, out=m_out, px_dist=m_hist),
           "3 B in + 1 B out per tile px; 50-px label blocks, 0.1 % off-palette pixels")
    if not only or any("mask_gather" in o for o in only):
        rng = np.random.default_rng(3)
        noise = np.asarray(pal, dtype=np.uint8)[rng.integers(0, C, size=(H, W))]
        d_noise, np_ = ops.upload_image(np.ascontiguousarray(noise))
        report("mask_gather_encode_hist 6000x4000 S512 C9, worst case: per-pixel noise labels", tile_px * 4,
               lambda: ops.mask_gather_encode_hist(d_noise, H, W, np_, T, 512, pal, out=m_out, px_dist=m_hist),
               "run length 1: every 4-pixel group is re-encoded pixel by pixel")
        del d_noise, noise
        W2, H2 = 2000, 1500
        d_small, sp = ops.upload_image(orc.synth_mask(1, W2, H2, pal, skew=True))
        nH3, nW3 = ops.tile_grid(H2, W2, T, 512)
        report("mask_gather_encode_hist 2000x1500 S512 C9 (6 tiles)", nH3 * nW3 * T * T * 4,
               lambda: ops.mask_gather_encode_hist(d_small, H2, W2, sp, T, 512, pal, out=m_out[:nH3 * nW3], px_dist=m_hist[:nH3 * nW3]),
               "configs[0] size; launch-bound")
    if not only or any("sweep" in o or "mask_gather" in o for o in only):
        sets = []
        for i in range(4):
            dm, dp = ops.upload_image(orc.synth_mask(i, W, H, pal, skew=True))
            sets.append((dm, dp, torch.empty_like(m_out)))
        report_sweep("mask_gather_encode_hist 6000x4000 S512 C9, sweep", tile_px * 4,
                     [lambda d=d, q=q, o=o: ops.mask_gather_encode_hist(d, H, W, q, T, 512, pal, out=o, px_dist=m_hist) for d, q, o in sets],
                     "3 B in + 1 B out per tile px")
        del sets
    if not only or any("stack" in o for o in only):
        # configs[3] geometry: 24 gray image + schema_b mask pairs of 2000x1500 as one stack per kernel
        pal_b = Parameters({"schema": "./schemas/schema_b.json"}).palette_rgb
        Ws, Hs, K = 2000, 1500, 24
        d_ms, mps, _ = ops.upload_stack([orc.synth_mask(100 + i, Ws, Hs, pal_b, skew=True) for i in range(K)])
        d_is, ips, _ = ops.upload_stack([orc.synth_image(100 + i, Ws, Hs, 1) for i in range(K)])
        nHs, nWs = ops.tile_grid(Hs, Ws, T, 512)
        n_t = nHs * nWs * K
        s_m = torch.empty((n_t, T, T), dtype=torch.uint8, device="cuda")
        s_i = torch.empty((n_t, 1, T, T), dtype=torch.uint8, device="cuda")
        s_h = torch.zeros((n_t, len(pal_b)), dtype=torch.int64, device="cuda")
        s_st = torch.zeros((n_t, 1, 2), dtype=torch.int64, device="cuda")
        report("mask_gather_encode_hist stack of 24 x 2000x1500 S512 C11 (one launch)", n_t * T * T * 4,
               lambda: ops.mask_gather_encode_hist_stack(d_ms, Hs, Ws, mps, T, 512, pal_b, out=s_m, px_dist=s_h),
               "3 B in + 1 B out per tile px; pylc_mask_gather_encode_hist_stack")
        report("tile_gather_u8 gray + moments stack of 24 x 2000x1500 S512 (one launch)", n_t * T * T * 2,
               lambda: ops.tile_gather_u8_stack(d_is, Hs, Ws, 1, ips, T, 512, stats=True, out=s_i, stat_out=s_st),
               "1 B in + 1 B out per tile px; pylc_tile_gather_u8_stack (the moments buffer is zeroed by a memset inside the timed region)")
        if not only or any("sweep" in o or "stack" in o for o in only):
            sets = []
            for j in range(4):
                dj, _, _ = ops.upload_stack([orc.synth_image(200 + 24 * j + i, Ws, Hs, 1) for i in range(K)])
                sets.append((dj, torch.empty_like(s_i)))
            lib = ops._lib.load()

            def gray_stack(d, o):       # the C entry point directly: no memset of the moments between launches
                ops.check(lib.pylc_tile_gather_u8_stack(ops._p(d), K, Hs * ips, Hs, Ws, 1, ips, T, 512, ops._p(o), ops._p(s_st),
                                                        ops._stream()), "pylc_tile_gather_u8_stack")
            report_sweep("tile_gather_u8 gray + moments stack of 24 x 2000x1500 S512, sweep", n_t * T * T * 2,
                         [lambda d=d, o=o: gray_stack(d, o) for d, o in sets], "1 B in + 1 B out per tile px")
            del sets
        del d_ms, d_is, s_m, s_i, s_h, s_st
    enc_out = torch.empty((1, H, W), dtype=torch.uint8, device="cuda")
    palc0, _ = ops._lib.palette_array(pal)
    enc_hist = torch.zeros((C,), dtype=torch.int64, device="cuda")

    def encode_full():
        ops._lib.check(ops._lib.load().pylc_class_encode(ops._p(d_mask), 1, H, W, mp, 0, palc0, C, ops._p(enc_out),
                                                         ops._p(enc_hist), ops._stream()), "pylc_class_encode")
    report("class_encode + hist 6000x4000 interleaved C9", H * W * 4, encode_full, "3 B in + 1 B out per px")
    del enc_out
    Wf, Hf = 5632, 3584
    img1 = orc.synth_image(0, Wf, Hf, 1)
    d_img1, ip1 = ops.upload_image(img1)
    nH2, nW2 = ops.tile_grid(Hf, Wf, T, 256)
    g_out = torch.empty((nH2 * nW2, 1, T, T), dtype=torch.uint8, device="cuda")
    report("tile_gather_u8 gray 5632x3584 S256", nH2 * nW2 * T * T * 1.25,
           lambda: ops.tile_gather_u8(d_img1, Hf, Wf, 1, ip1, T, 256, out=g_out), "1.25 B per tile px")
    img3 = orc.synth_image(1, Wf, Hf, 3)
    d_img3, ip3 = ops.upload_image(img3)
    g3_out = torch.empty((nH2 * nW2, 3, T, T), dtype=torch.uint8, device="cuda")
    report("tile_gather_u8 rgb 5632x3584 S256", nH2 * nW2 * T * T * 3.75,
           lambda: ops.tile_gather_u8(d_img3, Hf, Wf, 3, ip3, T, 256, out=g3_out), "3.75 B per tile px")
    n_out = torch.empty((nH2 * nW2, 3, T, T), dtype=torch.float32, device="cuda")
    report("tile_gather_norm_f32 rgb 5632x3584 S256", nH2 * nW2 * T * T * (0.75 + 12),
           lambda: ops.tile_gather_norm_f32(d_img3, Hf, Wf, 3, ip3, T, 256, [128.0] * 3, [60.0] * 3, out=n_out),
           "0.75 B in + 12 B out per tile px")
    report("profile_tiles hist 273 tiles", m_out.numel() * 1.0,
           lambda: ops.profile_tiles(None, m_out, C), "1 B per px")
    # an existing tile database is profiled in ONE launch (utils/profile.py sweeps the whole DB); the
    # reference's DST.A historic set holds 3574 tiles (pylc_gpu.ipynb cell 9)
    db_masks = m_out[torch.arange(3574, device="cuda") % m_out.shape[0]].contiguous()
    report("profile_tiles hist 3574 tiles (DST.A-sized DB)", db_masks.numel() * 1.0,
           lambda: ops.profile_tiles(None, db_masks, C), "1 B per px")
    del db_masks
    report("profile_tiles moments 273x3 planes", g3_out.numel() * 1.0,
           lambda: ops.profile_tiles(g3_out, None, C), "1 B per px")
    del g3_out, n_out, g_out

    # ---- network glue (bench.py batch: 45 tiles of 512 x 512) ------------------------------------------
    if not only or any(o in "glue upsample_concat maxpool upsample_nhwc_to_nchw gather_norm_s2d" for o in only):
        Bt, cl = 45, torch.channels_last
        xa = torch.randn((Bt, 256, 32, 32), device="cuda").contiguous(memory_format=cl)
        lo = torch.randn((Bt, 48, 128, 128), device="cuda").contiguous(memory_format=cl)
        report("upsample_concat_nhwc 45x(256@32^2 -> 128^2 + 48)", (xa.numel() + lo.numel() + Bt * 304 * 128 * 128) * 4,
               lambda: ops.upsample_concat_nhwc(xa, lo), "x + low read once, [B,304,128,128] written once")
        st_ = torch.randn((Bt, 64, 256, 256), device="cuda").contiguous(memory_format=cl)
        report("maxpool3x3s2_nhwc 45x64@256^2", (st_.numel() + st_.numel() // 4) * 4, lambda: ops.maxpool3x3s2_nhwc(st_),
               "input read once, output written once")
        de = torch.randn((Bt, 9, 128, 128), device="cuda").contiguous(memory_format=cl)
        report("upsample_nhwc_to_nchw 45x9@128^2 -> 512^2", (de.numel() + Bt * 9 * 512 * 512) * 4,
               lambda: ops.upsample_nhwc_to_nchw(de, (512, 512)), "decoder output read once, planar logits written once")
        del xa, lo, st_, de
        fit3 = torch.from_numpy(orc.synth_image(3, 2560, 1536, 3)).cuda()
        report("tile_gather_norm_s2d rgb 2560x1536 S256 (45 tiles)", 2560 * 1536 * 3 + 45 * 259 * 259 * 64,
               lambda: ops.tile_gather_norm_s2d(fit3, 1536, 2560, 3, 2560 * 3, T, 256, [128.0] * 3, [60.0] * 3),
               "source read once + 64 B per space-to-depth pixel written")
        del fit3

    # ---- test-time fit resize -----------------------------------------------------------------
    for (Wr, Hr, chr_) in ((3000, 2000, 3), (6000, 4000, 1)):
        wr, hr = orc.fit_dims(Wr, Hr, T)
        raw, rp = ops.upload_image(orc.synth_image(2, Wr, Hr, chr_))      # 16-byte pitched rows, as TiledSegmenter uploads them
        fitted = torch.empty((hr, ops.pitch_for(wr * chr_)), dtype=torch.uint8, device="cuda")
        ops.fit_resize_area(raw, Hr, Wr, chr_, rp, hr, wr, out=fitted)      # builds + caches the tables
        report("fit_resize_area %dx%d ch%d -> %dx%d" % (Wr, Hr, chr_, wr, hr), (Wr * Hr + wr * hr) * chr_,
               lambda raw=raw, rp=rp, fitted=fitted, Wr=Wr, Hr=Hr, chr_=chr_, wr=wr, hr=hr:
               ops.fit_resize_area(raw, Hr, Wr, chr_, rp, hr, wr, out=fitted),
               "source read once + fitted image written once; 16-byte pitched source rows")
        del raw, fitted

    # ---- stitch ------------------------------------------------------------------------------
    nr, nc = Hf // 256 - 1, Wf // 256 - 1
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn((nr * nc, C, T, T), generator=g, device="cuda") * 3
    lut = pal
    hw = Hf * Wf
    report("stitch_argmax_colour 273 tiles C9 labels", logits.numel() * 4 + hw,
           lambda: ops.stitch_argmax_colour(logits, nr, nc, T, 256), "every logit once + 1 B label")
    report("stitch_argmax_colour 273 tiles C9 labels+rgb", logits.numel() * 4 + hw * 4,
           lambda: ops.stitch_argmax_colour(logits, nr, nc, T, 256, lut_rgb=lut, want_rgb=True))
    labels, _, _ = ops.stitch_argmax_colour(logits, nr, nc, T, 256)
    # the bench.py geometry: one fitted 2560x1536 image = 45 tiles (5 x 9)
    report("stitch_argmax_colour 45 tiles C9 labels (bench.py image)", 45 * C * T * T * 4 + 2560 * 1536,
           lambda: ops.stitch_argmax_colour(logits[:45], 5, 9, T, 256), "every logit once + 1 B label")
    # per-pixel probabilities: labels + the u8 confidence plane, reference labels or the argmax of the mean
    c_out = {"labels": torch.empty((Hf, Wf), dtype=torch.uint8, device="cuda"),
             "confidence": torch.empty((Hf, Wf), dtype=torch.uint8, device="cuda")}
    for mode in ("reference", "mean"):
        report("stitch_probs 273 tiles C9 %s+confidence" % mode, logits.numel() * 4 + hw * 2,
               lambda mode=mode: ops.stitch_probs(logits, nr, nc, T, 256, mode=mode, out=c_out),
               "every logit once + 1 B label + 1 B confidence")
        report("stitch_probs 45 tiles C9 %s+confidence (bench.py image)" % mode, 45 * C * T * T * 4 + 2560 * 1536 * 2,
               lambda mode=mode: ops.stitch_probs(logits[:45], 5, 9, T, 256, mode=mode), "every logit once + 2 B per px")
    del logits, c_out
    # §8f-1: the same image stitched straight from the decoder's [45, 9, 128, 128] channels-last output, the
    # final x4 bilinear up-sample evaluated in the kernel (no 424 MB logits round trip)
    dec = (torch.randn((45, C, T // 4, T // 4), generator=g, device="cuda") * 3).contiguous(memory_format=torch.channels_last)
    report("stitch_upsample_argmax_colour 45 tiles C9 labels (bench.py image)", dec.numel() * 4 + 2560 * 1536,
           lambda: ops.stitch_upsample_argmax_colour(dec, 5, 9, T, 256),
           "decoder output once + 1 B label; replaces upsample_nhwc_to_nchw + stitch_argmax_colour (2 x 424.7 MB + 26.5 MB of traffic); "
           "exp- and blend-bound, not HBM-bound: compare its time with the sum of those two rows")
    for mode in ("mean", "reference"):
        report("stitch_upsample_probs 45 tiles C9 %s+confidence (bench.py image)" % mode, dec.numel() * 4 + 2560 * 1536 * 2,
               lambda mode=mode: ops.stitch_upsample_probs(dec, 5, 9, T, 256, mode=mode),
               "decoder output once + 2 B per px; mean mode skips the interior's second softmax (36 instead of 54 "
               "exponentials per interior pixel at C = 9), compare with the row above")
    del dec

    # ---- evaluation --------------------------------------------------------------------------
    maps = (torch.from_numpy(ops.nn_index_map(Wf, W)).cuda(), torch.from_numpy(ops.nn_index_map(Hf, H)).cuda())
    conf = torch.zeros((C, C), dtype=torch.int64, device="cuda")
    # a predicted label map is spatially coherent (the network's logits are a x4 bilinear up-sample);
    # the argmax of i.i.d. random logits above is salt-and-pepper noise, kept as the worst case
    coherent = torch.from_numpy(orc.synth_labels(3, Wf, Hf, C, skew=True, block=37)).cuda()
    report("resample_encode_confusion 6000x4000 C9", H * W * 4,
           lambda: ops.resample_encode_confusion(coherent, W, H, gt_rgb=d_mask, gt_pitch=mp, palette=pal, n_inject=C,
                                                 conf=conf, maps=maps), "3 B GT + 1 B label per full-res px; 37-px label blocks")
    report("resample_encode_confusion 6000x4000 C9 worst-case noise labels", H * W * 4,
           lambda: ops.resample_encode_confusion(labels, W, H, gt_rgb=d_mask, gt_pitch=mp, palette=pal, n_inject=C,
                                                 conf=conf, maps=maps), "labels = argmax of i.i.d. random logits (run length ~1)")
    if not only or any("sweep" in o or "resample" in o for o in only):
        sets = []
        for i in range(4):
            dm, dp = ops.upload_image(orc.synth_mask(10 + i, W, H, pal, skew=True))
            sets.append((dm, dp, torch.from_numpy(orc.synth_labels(20 + i, Wf, Hf, C, skew=True, block=37)).cuda()))
        report_sweep("resample_encode_confusion 6000x4000 C9, sweep", H * W * 4,
                     [lambda d=d, q=q, l=l: ops.resample_encode_confusion(l, W, H, gt_rgb=d, gt_pitch=q, palette=pal, n_inject=C,
                                                                         conf=conf, maps=maps) for d, q, l in sets],
                     "3 B GT + 1 B label per full-res px")
        del sets
    # the bench.py geometry: a 2560x1536 label map against a 3000x2000 ground truth
    Wb, Hb, wb, hb = 3000, 2000, 2560, 1536
    dmb, dpb = ops.upload_image(orc.synth_mask(30, Wb, Hb, pal, skew=True))
    lab_b = torch.from_numpy(orc.synth_labels(31, wb, hb, C, skew=True, block=37)).cuda()
    maps_b = (torch.from_numpy(ops.nn_index_map(wb, Wb)).cuda(), torch.from_numpy(ops.nn_index_map(hb, Hb)).cuda())
    report("resample_encode_confusion 3000x2000 C9 (bench.py image)", Hb * Wb * 4,
           lambda: ops.resample_encode_confusion(lab_b, Wb, Hb, gt_rgb=dmb, gt_pitch=dpb, palette=pal, n_inject=C,
                                                 conf=conf, maps=maps_b), "3 B GT + 1 B label per full-res px")
    if not only or any("sweep" in o or "resample" in o for o in only):
        sets_b = []
        for i in range(12):                      # 12 x (18 MB + 3.9 MB) of distinct inputs > L2
            dm, dp = ops.upload_image(orc.synth_mask(40 + i, Wb, Hb, pal, skew=True))
            sets_b.append((dm, dp, torch.from_numpy(orc.synth_labels(60 + i, wb, hb, C, skew=True, block=37)).cuda()))
        report_sweep("resample_encode_confusion 3000x2000 C9 (bench.py image), sweep", Hb * Wb * 4,
                     [lambda d=d, q=q, l=l: ops.resample_encode_confusion(l, Wb, Hb, gt_rgb=d, gt_pitch=q, palette=pal, n_inject=C,
                                                                         conf=conf, maps=maps_b) for d, q, l in sets_b],
                     "3 B GT + 1 B label per full-res px; back-to-back launches as inside an evaluation sweep")
        del sets_b
    pred_full = torch.empty((H, W), dtype=torch.uint8, device="cuda")
    gt_full = torch.empty((H, W), dtype=torch.uint8, device="cuda")

    def with_outputs():
        ops._lib.check(ops._lib.load().pylc_resample_encode_confusion(
            ops._p(coherent), Hf, Wf, ops._p(maps[0]), ops._p(maps[1]), H, W, ops._p(d_mask), mp, palc, None, C, C,
            ops._p(conf), ops._p(pred_full), None, ops._p(gt_full), ops._stream()), "resample")
    palc, _ = ops._lib.palette_array(pal)
    report("resample_encode_confusion 6000x4000 C9 + label outputs", H * W * 6, with_outputs,
           "3 B GT + 1 B label in, 2 x 1 B label maps out")

    # confidence plane to full resolution + reliability table (fitted u8 plane, full-res predicted / true classes)
    for (Wc, Hc) in ((3000, 2000), (6000, 4000)):
        wc, hc = orc.fit_dims(Wc, Hc, T)
        c_fit = torch.from_numpy(orc.synth_labels(5, wc, hc, 256, block=37)).cuda()
        c_pred = torch.from_numpy(orc.synth_labels(6, Wc, Hc, C, skew=True, block=37)).cuda()
        c_true = torch.from_numpy(orc.synth_labels(7, Wc, Hc, C, skew=True, block=37)).cuda()
        c_maps = ops.device_index_maps(wc, hc, Wc, Hc, c_fit.device)
        rel = torch.zeros((C, 256, 2), dtype=torch.int64, device="cuda")
        c_full = torch.empty((Hc, Wc), dtype=torch.uint8, device="cuda")

        def conf_resample(c_fit=c_fit, c_pred=c_pred, c_true=c_true, c_maps=c_maps, rel=rel, c_full=c_full, Wc=Wc, Hc=Hc, wc=wc, hc=hc):
            ops._lib.check(ops._lib.load().pylc_confidence_resample(
                ops._p(c_fit), hc, wc, ops._p(c_maps[0]), ops._p(c_maps[1]), Hc, Wc, ops._p(c_pred), ops._p(c_true), C,
                ops._p(c_full), ops._p(rel), ops._stream()), "pylc_confidence_resample")
        report("confidence_resample %dx%d C9 + reliability" % (Wc, Hc), Hc * Wc * 3, conf_resample,
               "1 B pred + 1 B truth in, 1 B confidence out per full-res px; 37-px blocks")
        del c_fit, c_pred, c_true, c_full

    # ---- multi-loss --------------------------------------------------------------------------
    B = 64
    z = torch.randn((B, C, T, T), generator=g, device="cuda") * 3
    t64 = torch.randint(0, C, (B, T, T), generator=g, device="cuda")
    t8 = t64.to(torch.uint8)
    cfg = ops.loss_cfg()
    npx = B * T * T
    part = torch.zeros((2 * C + 3,), dtype=torch.float64, device="cuda")
    report("multiloss_reduce B64 C9 i64 target", npx * (4 * C + 8),
           lambda: ops.multiloss_reduce(z, t64, cfg, partials=part), "fwd only: 4C + 8 B/px")
    report("multiloss_reduce B64 C9 u8 target", npx * (4 * C + 1),
           lambda: ops.multiloss_reduce(z, t8, cfg, partials=part), "fwd only: 4C + 1 B/px")
    part = ops.multiloss_reduce(z, t64, cfg)
    grad = torch.empty_like(z)
    report("multiloss_grad B64 C9 i64 target", npx * (8 * C + 8),
           lambda: ops.multiloss_grad(z, t64, cfg, part, npx, out=grad), "8C + 8 B/px physically moved")

    def fwd_bwd():
        p = torch.zeros((2 * C + 3,), dtype=torch.float64, device="cuda")
        ops.multiloss_reduce(z, t64, cfg, partials=p)
        ops.multiloss_grad(z, t64, cfg, p, npx, out=grad)
    report("multiloss fwd+bwd B64 C9 (algorithmic 8C+8)", npx * (8 * C + 8), fwd_bwd,
           "two passes physically move 12C + 16 B/px")

    def fused():
        p = torch.zeros((2 * C + 3,), dtype=torch.float64, device="cuda")
        ops.multiloss_fwd_bwd(z, t64, cfg, out=grad, partials=p)
    report("multiloss fwd+bwd B64 C9, one cooperative launch (algorithmic 8C+8)", npx * (8 * C + 8), fused,
           "reduce + grid barrier + gradient back to front; physically moves <= 12C + 16 B/px")

    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
