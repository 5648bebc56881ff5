"""
TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by executing the UNMODIFIED PyLC
reference on small seeded inputs.  The reference is not part of this repository, so the vectors
are committed; regenerate them with

    PYLC_REFERENCE_ROOT=<PyLC checkout> python oracle/gen_golden.py

Tile size 32 / stride 16 keep the fixtures small; the reference code paths exercised are
size-independent.  Every fixture file stays under 1 MB.
"""
import hashlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import ref_harness  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def palettes(ref):
    # Parameters only reads `schema` from an attribute-style namespace (config.py:107)
    pa = ref.config.Parameters(types.SimpleNamespace(schema="./schemas/schema_a.json")).palette_rgb
    pb = ref.config.Parameters(types.SimpleNamespace(schema="./schemas/schema_b.json")).palette_rgb
    assert len(pa) == 9 and len(pb) == 11
    return pa, pb


def rand_mask_rgb(rng, h, w, palette, block=5, off=0.02):
    lab = rng.integers(0, len(palette), size=((h + block - 1) // block, (w + block - 1) // block))
    lab = np.kron(lab, np.ones((block, block), dtype=np.int64))[:h, :w]
    rgb = np.asarray(palette, dtype=np.uint8)[lab]
    n_off = int(h * w * off)
    rgb[rng.integers(0, h, n_off), rng.integers(0, w, n_off)] = rng.integers(0, 256, (n_off, 3), dtype=np.uint8)
    return rgb


def gen_split(ref, out):
    rng = np.random.default_rng(11)
    for name, shape, T, S in [("gray_s32", (75, 101), 32, 32), ("gray_s16", (80, 96), 32, 16),
                              ("rgb_s32", (70, 97, 3), 32, 32), ("rgb_s16", (64, 80, 3), 32, 16)]:
        img = rng.integers(0, 256, size=shape, dtype=np.uint8)
        ex = ref.extract.Extractor({"tile_size": T, "stride": S, "ch": 3 if len(shape) == 3 else 1})
        tiles, n = ex._Extractor__split(img)
        out["split_%s_img" % name] = img
        out["split_%s_tiles" % name] = tiles.numpy()
        out["split_%s_TS" % name] = np.array([T, S])


def gen_encode(ref, out):
    rng = np.random.default_rng(12)
    pa, pb = palettes(ref)
    for name, pal in (("a", pa), ("b", pb)):
        rgb = np.stack([rand_mask_rgb(rng, 32, 32, pal) for _ in range(3)])
        tiles = np.moveaxis(rgb, 3, 1).copy()
        enc = ref.tools.class_encode(torch.tensor(tiles), pal)
        out["encode_%s_in" % name] = tiles
        out["encode_%s_out" % name] = enc.numpy()
        out["palette_%s" % name] = np.asarray(pal, dtype=np.uint8)
    # duplicate palette entries: later entry wins (utils/tools.py:441-444)
    dup = [[0, 0, 0], [10, 20, 30], [10, 20, 30], [1, 2, 3]]
    rgb = rand_mask_rgb(rng, 32, 32, dup)[None]
    tiles = np.moveaxis(rgb, 3, 1).copy()
    out["encode_dup_in"] = tiles
    out["encode_dup_out"] = ref.tools.class_encode(torch.tensor(tiles), dup).numpy()
    out["palette_dup"] = np.asarray(dup, dtype=np.uint8)


def gen_colourize(ref, out):
    rng = np.random.default_rng(13)
    pa, pb = palettes(ref)
    for name, pal in (("a", pa), ("b", pb)):
        lab = rng.integers(0, len(pal), size=(2, 20, 24)).astype(np.int64)
        out["colourize_%s_in" % name] = lab
        out["colourize_%s_out" % name] = ref.tools.colourize(lab, len(pal), palette=pal)


def gen_extract_profile(ref, out):
    import cv2
    rng = np.random.default_rng(14)
    pa, pb = palettes(ref)
    for name, ch, pal, schema in (("gray_a", 1, pa, "schema_a"), ("rgb_b", 3, pb, "schema_b")):
        with ref_harness.in_workdir() as wd:
            idir = os.path.join(wd, "in_%s" % name, "img")
            mdir = os.path.join(wd, "in_%s" % name, "mask")
            os.makedirs(idir)
            os.makedirs(mdir)
            imgs, masks = [], []
            for k, (h, w) in enumerate([(70, 100), (64, 64), (97, 66)]):
                if ch == 1:
                    img = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
                    cv2.imwrite(os.path.join(idir, "f%d.tif" % k), img)
                else:
                    img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
                    cv2.imwrite(os.path.join(idir, "f%d.tif" % k), cv2.cvtColor(img, cv2.COLOR_RGB2BGR))
                m = rand_mask_rgb(rng, h, w, pal)
                cv2.imwrite(os.path.join(mdir, "f%d.png" % k), cv2.cvtColor(m, cv2.COLOR_RGB2BGR))
                imgs.append(img)
                masks.append(m)
            params = types.SimpleNamespace(schema="./schemas/%s.json" % schema, ch=ch, tile_size=32,
                                           stride=32, tile_px_count=32 * 32)
            with ref_harness.quiet():
                ex = ref.extract.Extractor(params).load(idir, mdir).extract()
                tiles_img = ex.imgs.copy()
                tiles_mask = ex.masks.copy()
                ex.profile()
            meta = ex.get_meta()
            files = ref.tools.collate(idir, mdir)
            order = [int(os.path.basename(f["img"])[1]) for f in files]
        out["exprof_%s_order" % name] = np.array(order)
        for k in range(3):
            out["exprof_%s_img%d" % (name, k)] = imgs[k]
            out["exprof_%s_mask%d" % (name, k)] = masks[k]
        out["exprof_%s_tiles_img" % name] = tiles_img
        out["exprof_%s_tiles_mask" % name] = tiles_mask
        out["exprof_%s_px_dist" % name] = np.asarray(meta.px_dist, dtype=np.int64)
        out["exprof_%s_dset_px_dist" % name] = np.asarray(meta.dset_px_dist, dtype=np.int64)
        out["exprof_%s_dset_px_count" % name] = np.array(meta.dset_px_count)
        out["exprof_%s_probs" % name] = np.asarray(meta.probs)
        out["exprof_%s_weights" % name] = np.asarray(meta.weights)
        out["exprof_%s_m2jsd" % name] = np.array([meta.m2, meta.jsd])
        out["exprof_%s_px_mean" % name] = np.asarray(meta.px_mean, dtype=np.float32)
        out["exprof_%s_px_std" % name] = np.asarray(meta.px_std, dtype=np.float32)


def gen_fit(ref, out):
    import cv2
    rows = []
    for (W, H) in [(2000, 1500), (3000, 2000), (6000, 4000), (3453, 4940), (4940, 3453), (1024, 1024),
                   (1100, 2300), (5999, 3999), (513, 1027)]:
        img = np.zeros((H, W), dtype=np.uint8)
        _, w_fit, h_fit, off = ref.tools.adjust_to_tile(img, 512, 256, 1)
        rows.append([W, H, w_fit, h_fit, off])
    out["fit_dims"] = np.array(rows)
    # the fitted pixels themselves: the reference's adjust_to_tile (cv2 INTER_AREA) on small seeded images
    rng = np.random.default_rng(77)
    for name, (W, H, T, ch) in {"g": (150, 110, 32, 1), "c": (100, 75, 32, 3), "n": (97, 161, 32, 3)}.items():
        img = rng.integers(0, 256, size=(H, W) if ch == 1 else (H, W, ch), dtype=np.uint8)
        fitted, w_fit, h_fit, off = ref.tools.adjust_to_tile(img, T, T // 2, ch)
        assert fitted.shape[:2] == (h_fit, w_fit) and off == 0
        out["fitimg_%s_in" % name] = img
        out["fitimg_%s_out" % name] = fitted
    # OpenCV nearest-neighbour index maps (cv2.resize of a ramp), several size pairs
    pairs = [(1536, 2000), (1024, 1500), (2560, 3000), (5632, 6000), (3584, 4000), (64, 75), (48, 50),
             (3072, 3453), (4608, 4940), (512, 513)]
    out["nn_pairs"] = np.array(pairs)
    for (src, dst) in pairs:
        ramp = np.arange(src, dtype=np.float32)[None, :]
        out["nn_map_%d_%d" % (src, dst)] = cv2.resize(ramp, (dst, 1), interpolation=cv2.INTER_NEAREST)[0].astype(np.int32)


def gen_reconstruct(ref, out):
    rng = np.random.default_rng(15)
    pa, pb = palettes(ref)
    captured = {}
    real_argmax = np.argmax

    def spy(a, *args, **kw):
        captured["map"] = np.array(a, copy=True)
        return real_argmax(a, *args, **kw)

    cases = [("a_2x3", pa, 2, 3, 32, 16, (75, 50)), ("a_3x2", pa, 3, 2, 32, 16, (50, 70)),
             ("a_3x3", pa, 3, 3, 32, 16, (64, 64)), ("a_2x1", pa, 2, 1, 32, 16, (33, 50)),
             ("b_4x5", pb, 4, 5, 32, 16, (101, 83)), ("a_s32_2x3", pa, 2, 3, 32, 32, (100, 70))]
    names = []
    for name, pal, nr, nc, T, S, (w_full, h_full) in cases:
        C = len(pal)
        if S < T:
            h, w = (nr + 1) * S, (nc + 1) * S
        else:
            h, w = nr * S, nc * S
        tiles = (rng.standard_normal((nr * nc, C, T, T)) * 3).astype(np.float32)
        meta = ref.config.Parameters({"tile_size": T, "stride": S})
        meta.palette_rgb = pal
        meta.n_classes = C
        meta.extract = {"w_fitted": w, "h_fitted": h, "w_scaled": w_full, "h_scaled": h_full, "offset": 0}
        # split into batches of <= 4 tiles like the data loader does
        batches = [torch.tensor(tiles[i:i + 4]) for i in range(0, len(tiles), 4)]
        np.argmax = spy
        try:
            rgb = ref.tools.reconstruct(batches, meta)
        finally:
            np.argmax = real_argmax
        out["recon_%s_tiles_sha256" % name] = np.array(hashlib.sha256(tiles.tobytes()).hexdigest())   # see orc.reconstruct_fixture_tiles
        out["recon_%s_geom" % name] = np.array([nr, nc, T, S, h, w, w_full, h_full, C])
        out["recon_%s_map" % name] = captured["map"][0]
        out["recon_%s_rgb" % name] = rgb
        names.append(name)
    out["recon_cases"] = np.array(names)


def gen_evaluate(ref, out):
    import cv2
    rng = np.random.default_rng(16)
    pa, _ = palettes(ref)
    C = len(pa)
    h, w = 60, 90
    gt = rand_mask_rgb(rng, h, w, pa, block=7, off=0.01)
    lab_pred = rng.integers(0, C, size=((h + 5) // 6, (w + 5) // 6))
    lab_pred = np.kron(lab_pred, np.ones((6, 6), dtype=np.int64))[:h, :w]
    # make prediction correlated with GT
    gt_lab = ref.tools.class_encode(torch.tensor(np.moveaxis(gt, 2, 0)[None].copy()), pa).numpy()[0]
    keep = rng.random((h, w)) < 0.6
    lab_pred = np.where(keep, gt_lab, lab_pred)
    pred_rgb = np.asarray(pa, dtype=np.uint8)[lab_pred].astype(np.float32)
    with ref_harness.in_workdir() as wd:
        gpath = os.path.join(wd, "gt_eval.png")
        cv2.imwrite(gpath, cv2.cvtColor(gt, cv2.COLOR_RGB2BGR))
        meta = ref.config.Parameters({"id": "golden_eval"})
        meta.extract = {"fid": "golden", "w_scaled": w, "h_scaled": h}
        with ref_harness.quiet():
            ev = ref.evaluate.Evaluator(meta)
            ev.load(pred_rgb, meta, mask_true_path=gpath, scale=None)
            y_true_raw = ev.y_true.numpy().copy()
            y_pred_raw = ev.y_pred.numpy().copy()
            ev.evaluate()
    out["eval_gt_rgb"] = gt
    out["eval_pred_rgb"] = pred_rgb
    out["eval_y_true_raw"] = y_true_raw
    out["eval_y_pred_raw"] = y_pred_raw
    out["eval_y_true"] = ev.y_true.numpy()
    out["eval_y_pred"] = ev.y_pred.numpy()
    out["eval_scalars"] = np.array([ev.metrics.results["f1"], ev.metrics.results["iou"], ev.metrics.results["mcc"]])
    out["eval_cmatrix"] = np.asarray(ev.metrics.cmatrix)
    out["eval_report_json"] = np.array(json.dumps(ev.metrics.results["report"]))
    out["eval_labels"] = np.array(ev.labels)


def gen_loss(ref, out):
    rng = np.random.default_rng(17)
    pa, pb = palettes(ref)
    ref.config.defaults.device = "cpu"
    for name, C, weighted in (("a_unw", 9, False), ("a_w", 9, True), ("b_w", 11, True)):
        B, H, W = 3, 16, 20
        z = (rng.standard_normal((B, C, H, W)) * 3).astype(np.float32)
        t = rng.integers(0, C, size=(B, H, W)).astype(np.int64)
        if name == "a_unw":
            t[t == 5] = 0  # a class absent from the batch
        wts = (rng.random(C) * 0.9 + 0.1).astype(np.float32)
        crit = ref.loss.MultiLoss(
            loss_weights={"weighted": weighted, "weights": wts.tolist(), "ce": 0.5, "dice": 0.5, "focal": 0.5},
            schema={"n_classes": C, "class_codes": ["c%d" % i for i in range(C)],
                    "class_labels": ["l%d" % i for i in range(C)]})
        zt = torch.tensor(z, requires_grad=True)
        loss = crit.forward(zt, torch.tensor(t))
        loss.backward()
        out["loss_%s_z" % name] = z
        out["loss_%s_t" % name] = t
        out["loss_%s_w" % name] = wts
        out["loss_%s_vals" % name] = np.array([loss.item(), crit.ce.item(), crit.dsc.item(), crit.fl.item()],
                                              dtype=np.float64)
        out["loss_%s_grad" % name] = zt.grad.numpy()


def gen_augment(ref, out):
    """Augmentor.optimize (utils/augment.py:92-187) run by the reference itself on seeded profile metadata."""
    import types
    import utils.augment as ref_augment
    rng = np.random.default_rng(41)
    for name, (N, C, T) in {"a": (300, 9, 64), "b": (500, 11, 32)}.items():
        # skewed per-tile class histograms that sum to T*T, like get_profile's px_dist
        conc = np.concatenate([[8.0, 0.05, 3.0, 1.0], np.full(C - 4, 0.3)])
        p = rng.dirichlet(conc, size=N)
        px = np.floor(p * T * T).astype(np.int64)
        px[:, 0] += T * T - px.sum(axis=1)
        probs = px.sum(axis=0) / px.sum()
        aug = ref_augment.Augmentor()
        aug.input_meta = types.SimpleNamespace(px_dist=px, tile_px_count=T * T, probs=probs, n_classes=C)
        aug.input_size = N
        aug.optimize()
        om = aug.optim_meta
        out["aug_%s_px_dist" % name] = px
        out["aug_%s_probs" % name] = probs
        out["aug_%s_meta" % name] = np.array([N, C, T * T])
        out["aug_%s_rates" % name] = np.asarray(om['rates'])
        out["aug_%s_optim" % name] = np.array([om['threshold'], om['rate_coef'], om['jsd'], om['m2'], om['n_samples'],
                                                  om['aug_n_samples']], dtype=np.float64)
        out["aug_%s_optim_probs" % name] = np.asarray(om['probs'])


def gen_warp(ref, out):
    """tools.augment_transform (utils/tools.py:452-594) on a formula-generated tile, with the dtypes the
    reference's loader hands it (float32 image, int64 mask; db/dataset.py:62-63) and the RandomState(j) seeds
    Augmentor.oversample uses (utils/augment.py:213-215)."""
    import pylc_oracle as orc
    for ch in (1, 3):
        img, mask = orc.augment_fixture_tile(ch)
        for seed in (0, 1, 3):
            a, b = ref.tools.augment_transform(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
            out["warp_ch%d_s%d_img" % (ch, seed)] = np.asarray(a).astype(np.uint8)
            assert np.array_equal(np.asarray(b), np.asarray(b).astype(np.uint8))
            out["warp_ch%d_s%d_mask" % (ch, seed)] = np.asarray(b).astype(np.uint8)


def gen_model(ref, out):
    """Model-file boundary: the reference's DeepLabv3+/ResNet-101 state-dict keys and shapes, its output
    on a seeded input with deterministic weights (oracle.fill_state_dict), and a model file whose `meta` is
    the reference's own pickled config.Parameters (models/modules/checkpoint.py:53-66) with an empty
    state dict -- what Model.load has to unpickle (models/model.py:78-121)."""
    import pylc_oracle as orc
    mm = ref_harness.load_model_modules()
    with ref_harness.in_workdir(), ref_harness.quiet():
        model = mm.model.Model()
        model.meta.update(types.SimpleNamespace(ch=3, arch='deeplab', backbone='resnet', pretrained=False))
        model.meta.px_mean, model.meta.px_std = [130.0, 140.0, 150.0], [25.0, 22.0, 19.0]
        model.meta.weights = [1.0] * model.meta.n_classes
        model.build()
        net = model.net.cpu().eval()
        sd = net.state_dict()
        out["keys"] = np.array(list(sd.keys()))
        out["shapes"] = np.array(json.dumps([list(v.shape) for v in sd.values()]))
        out["dtypes"] = np.array([str(v.dtype) for v in sd.values()])
        net.load_state_dict(orc.fill_state_dict(sd))
        x = torch.randn(2, 3, 96, 80, generator=torch.Generator().manual_seed(123))
        with torch.no_grad():
            y = net(x)
        out["x"] = x.numpy()
        out["y"] = y.numpy()
        torch.save({"model": {}, "optim": None, "meta": model.meta}, os.path.join(OUT, "ref_meta_model.pth"))
        out["meta_id"] = np.array(str(model.meta.id))
        out["meta_n_classes"] = np.array(model.meta.n_classes)


def main():
    ref = ref_harness.load()
    # get_image() upscales anything whose short side is below defaults.tile_size
    # (utils/tools.py:139-146), so the global default follows the small fixture tile size.
    ref.config.defaults.tile_size = 32
    os.makedirs(OUT, exist_ok=True)
    for fname, fn in (("split", gen_split), ("encode", gen_encode), ("colourize", gen_colourize),
                      ("extract_profile", gen_extract_profile), ("fit", gen_fit),
                      ("reconstruct", gen_reconstruct), ("evaluate", gen_evaluate), ("loss", gen_loss),
                      ("augment", gen_augment), ("model", gen_model), ("warp", gen_warp)):
        out = {}
        fn(ref, out)
        path = os.path.join(OUT, fname + ".npz")
        np.savez_compressed(path, **out)
        print("%-18s %7.1f KB  %d arrays" % (fname, os.path.getsize(path) / 1024, len(out)))


if __name__ == "__main__":
    main()
