"""TEST INFRASTRUCTURE ONLY -- live comparison of the oracle with the unmodified reference.

Runs in its own process (the harness changes the working directory and puts the reference's flat module
names -- config, utils, db, models -- at the front of sys.path): imports the reference checkout named by
PYLC_REFERENCE_ROOT through oracle/ref_harness.py and checks every restatement in oracle/pylc_oracle.py against
the reference function it cites, on seeded inputs that are NOT the ones frozen in tests/golden/ (other seeds,
other sizes).

    PYLC_REFERENCE_ROOT=<PyLC checkout> python oracle/live_check.py [--seed N]
                                                exit code 0 = all equal, 1 = mismatch, 77 = reference absent

tests/test_oracle_vs_reference.py runs it.
"""
import argparse
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import pylc_oracle as orc      # noqa: E402
import ref_harness             # noqa: E402
from gen_golden import palettes, rand_mask_rgb   # noqa: E402

FAIL = []


def check(name, ok):
    print("%-46s %s" % (name, "ok" if ok else "MISMATCH"))
    if not ok:
        FAIL.append(name)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=4242)
    args = ap.parse_args()
    if not ref_harness.available():
        print("reference not available")
        return 77
    ref = ref_harness.load()
    rng = np.random.default_rng(args.seed)
    pa, pb = palettes(ref)

    # Extractor.__split (utils/extract.py:279-310)
    for shape, T, S in [((90, 131), 32, 32), ((97, 70, 3), 32, 16), ((64, 64), 64, 32)]:
        img = rng.integers(0, 256, size=shape, dtype=np.uint8)
        ex = ref.extract.Extractor({"tile_size": T, "stride": S, "ch": 3 if len(shape) == 3 else 1})
        tiles, _ = ex._Extractor__split(img)
        check("split %s T%d S%d" % (shape, T, S), np.array_equal(tiles.numpy(), orc.split_tiles(img, T, S)))

    # tools.class_encode (utils/tools.py:412-449), both shipped palettes, off-palette pixels
    for name, pal in (("schema_a", pa), ("schema_b", pb)):
        rgb = np.stack([rand_mask_rgb(rng, 48, 40, pal, block=3, off=0.05) for _ in range(2)])
        tiles = np.moveaxis(rgb, 3, 1).copy()
        want = ref.tools.class_encode(torch.tensor(tiles), pal).numpy()
        check("class_encode %s (port)" % name, np.array_equal(orc.class_encode_port(tiles, pal), want))
        check("class_encode %s (closed form)" % name, np.array_equal(orc.class_encode(tiles, pal), want))
        check("class_encode_hwc %s" % name, np.array_equal(orc.class_encode_hwc(rgb[0], pal), want[0]))

    # tools.colourize (utils/tools.py:322-358)
    for name, pal in (("schema_a", pa), ("schema_b", pb)):
        lab = rng.integers(0, len(pal), size=(1, 31, 17)).astype(np.int64)
        want = ref.tools.colourize(lab, len(pal), palette=pal)
        check("colourize %s" % name, np.array_equal(orc.colourize(lab, len(pal), pal), want)
              and np.array_equal(orc.colourize_port(lab, len(pal), pal), want))

    # tools.adjust_to_tile (utils/tools.py:151-206): fitted size and the INTER_AREA pixels
    for (W, H, ch) in [(301, 203, 1), (257, 190, 3)]:
        img = rng.integers(0, 256, size=(H, W) if ch == 1 else (H, W, 3), dtype=np.uint8)
        fitted, w, h, off = ref.tools.adjust_to_tile(img, 64, 32, ch)
        check("adjust_to_tile dims %dx%d ch%d" % (W, H, ch), orc.fit_dims(W, H, 64) == (w, h) and off == 0)
        check("adjust_to_tile pixels %dx%d ch%d" % (W, H, ch), np.array_equal(orc.resize_area(img, w, h), fitted))

    # tools.reconstruct (utils/tools.py:209-319): stitched map through the argmax spy, RGB result
    captured = {}
    real_argmax = np.argmax

    def spy(a, *aa, **kw):
        captured["map"] = np.array(a, copy=True)
        return real_argmax(a, *aa, **kw)

    for pal, nr, nc, T, S, (w_full, h_full) in [(pa, 2, 4, 32, 16, (91, 50)), (pb, 3, 2, 32, 16, (50, 77))]:
        C = len(pal)
        h, w = (nr + 1) * S, (nc + 1) * S
        tiles = (rng.standard_normal((nr * nc, C, T, T)) * 3).astype(np.float32)
        meta = ref.config.Parameters({"tile_size": T, "stride": S})
        meta.palette_rgb, meta.n_classes = pal, C
        meta.extract = {"w_fitted": w, "h_fitted": h, "w_scaled": w_full, "h_scaled": h_full, "offset": 0}
        np.argmax = spy
        try:
            with ref_harness.quiet():
                rgb = ref.tools.reconstruct([torch.tensor(tiles[i:i + 3]) for i in range(0, len(tiles), 3)], meta)
        finally:
            np.argmax = real_argmax
        check("reconstruct map %dx%d C%d (port, bit-equal)" % (nr, nc, C), np.array_equal(orc.stitch_map_port(tiles, h, w, T, S), captured["map"][0]))
        check("reconstruct map %dx%d C%d (closed form, 1e-6)" % (nr, nc, C),
              np.allclose(orc.stitch_map(tiles, nr, nc, T, S), captured["map"][0], rtol=1e-6, atol=1e-7))
        got = orc.reconstruct_port([tiles[i:i + 3] for i in range(0, len(tiles), 3)], h, w, w_full, h_full, T, S, pal, C)
        check("reconstruct rgb %dx%d C%d" % (nr, nc, C), np.array_equal(np.asarray(got), np.asarray(rgb)))

    # MultiLoss forward + autograd backward (models/modules/loss.py:23-215)
    ref.config.defaults.device = "cpu"
    for C, weighted in ((9, False), (11, True)):
        B, H, W = 2, 12, 18
        z = (rng.standard_normal((B, C, H, W)) * 3).astype(np.float32)
        t = rng.integers(0, C, size=(B, H, W)).astype(np.int64)
        wts = (rng.random(C) * 0.9 + 0.1).astype(np.float32)
        with ref_harness.quiet():
            crit = ref.loss.MultiLoss(loss_weights={"weighted": weighted, "weights": wts.tolist(), "ce": 0.5, "dice": 0.5, "focal": 0.5},
                                      schema={"n_classes": C, "class_codes": ["c%d" % i for i in range(C)],
                                              "class_labels": ["l%d" % i for i in range(C)]})
        zt = torch.tensor(z, requires_grad=True)
        loss = crit.forward(zt, torch.tensor(t))
        loss.backward()
        want = np.array([loss.item(), crit.ce.item(), crit.dsc.item(), crit.fl.item()])
        got = orc.multiloss(z, t, C, weights=wts, weighted=weighted)
        check("MultiLoss values C%d weighted=%s" % (C, weighted), np.allclose(got[:4], want, rtol=1e-5))
        check("MultiLoss gradient C%d weighted=%s" % (C, weighted), np.allclose(got[4], zt.grad.numpy(), rtol=2e-4, atol=1e-9))
        port = orc.multiloss_port(z, t, C, weights=wts, weighted=weighted)
        check("MultiLoss port C%d weighted=%s" % (C, weighted), np.allclose(np.asarray(port[:4], dtype=np.float64), want, rtol=1e-6))

    # Metrics (utils/metrics.py:45-87, scikit-learn) from one confusion matrix
    C = len(pa)
    yt = rng.integers(0, C, size=5000).astype(np.uint8)
    yp = np.where(rng.random(5000) < 0.7, yt, rng.integers(0, C, size=5000)).astype(np.uint8)
    yt, yp = orc.inject_coverage(yt, yp, C)
    with ref_harness.in_workdir(), ref_harness.quiet():
        m = ref.metrics.Metrics()
        m.f1_score(yt, yp)
        m.jaccard(yt, yp)
        m.mcc(yt, yp)
        m.confusion_matrix(yt, yp, labels=ref.config.defaults.class_codes)
    mine = orc.metrics_from_confusion(orc.confusion_counts(yt, yp, C))
    check("metrics f1 / iou / mcc from the matrix", mine["f1"] == m.results["f1"] and mine["iou"] == m.results["iou"] and mine["mcc"] == m.results["mcc"])
    check("row-normalised confusion matrix", np.array_equal(mine["cmatrix"], np.asarray(m.cmatrix)))

    print("%d mismatches" % len(FAIL))
    return 1 if FAIL else 0


if __name__ == "__main__":
    sys.exit(main())
