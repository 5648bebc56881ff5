"""The CPU oracle (oracle/pylc_oracle.py) against vectors produced by the unmodified reference
(oracle/gen_golden.py).  This is what pins the oracle: the reference ships no tests of its own."""
import json
import os

import numpy as np
import pytest

import pylc_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("name", ["gray_s32", "gray_s16", "rgb_s32", "rgb_s16"])
def test_split(golden, name):
    g = golden("split")
    T, S = g["split_%s_TS" % name]
    assert np.array_equal(orc.split_tiles(g["split_%s_img" % name], int(T), int(S)), g["split_%s_tiles" % name])


@pytest.mark.parametrize("name", ["a", "b", "dup"])
def test_class_encode(golden, name):
    g = golden("encode")
    pal = g["palette_%s" % name].tolist()
    assert np.array_equal(orc.class_encode_port(g["encode_%s_in" % name], pal), g["encode_%s_out" % name])
    assert np.array_equal(orc.class_encode(g["encode_%s_in" % name], pal), g["encode_%s_out" % name])
    # off-palette pixels exist in the fixture and land in class 1
    assert (g["encode_%s_out" % name] == 1).any()


@pytest.mark.parametrize("name", ["a", "b"])
def test_colourize(golden, palettes, name):
    g = golden("colourize")
    pal = palettes[name]
    lab = g["colourize_%s_in" % name]
    assert np.array_equal(orc.colourize_port(lab, len(pal), pal), g["colourize_%s_out" % name])
    assert np.array_equal(orc.colourize(lab, len(pal), pal), g["colourize_%s_out" % name])


def test_colourize_grey_chain():
    # a palette whose class-0 colour is the grey [2,2,2] is re-mapped by the later pass i=2
    pal = [[2, 2, 2], [9, 9, 9], [50, 60, 70]]
    lab = np.array([[[0, 1, 2]]])
    assert np.array_equal(orc.colourize_port(lab, 3, pal), orc.colourize(lab, 3, pal))
    assert orc.colourize(lab, 3, pal)[0, 0, 0].tolist() == [50, 60, 70]


@pytest.mark.parametrize("name,ch,pk", [("gray_a", 1, "a"), ("rgb_b", 3, "b")])
def test_extract_profile(golden, palettes, name, ch, pk):
    g = golden("extract_profile")
    pal = palettes[pk]
    C = len(pal)
    imgs, masks = [], []
    for k in g["exprof_%s_order" % name]:
        imgs.append(orc.split_tiles(g["exprof_%s_img%d" % (name, k)], 32, 32))
        mt = orc.split_tiles(g["exprof_%s_mask%d" % (name, k)], 32, 32)
        masks.append(orc.class_encode(mt, pal))
    imgs = np.concatenate(imgs)
    masks = np.concatenate(masks)
    assert np.array_equal(imgs, g["exprof_%s_tiles_img" % name])
    assert np.array_equal(masks, g["exprof_%s_tiles_mask" % name])
    for prof in (orc.profile_port(imgs, masks, C, 32), orc.profile(imgs, masks, C, 32)):
        assert np.array_equal(prof["px_dist"], g["exprof_%s_px_dist" % name])
        assert np.array_equal(prof["dset_px_dist"], g["exprof_%s_dset_px_dist" % name])
        assert prof["dset_px_count"] == int(g["exprof_%s_dset_px_count" % name])
        np.testing.assert_allclose(prof["probs"], g["exprof_%s_probs" % name], rtol=0, atol=0)
        np.testing.assert_allclose(prof["weights"], g["exprof_%s_weights" % name], rtol=1e-15)
        np.testing.assert_allclose([prof["m2"], prof["jsd"]], g["exprof_%s_m2jsd" % name], rtol=1e-14)
        np.testing.assert_allclose(prof["px_mean"], g["exprof_%s_px_mean" % name], rtol=1e-5)
        np.testing.assert_allclose(prof["px_std"], g["exprof_%s_px_std" % name], rtol=1e-5)


def test_fit_dims(golden):
    for W, H, w_fit, h_fit, off in golden("fit")["fit_dims"]:
        assert orc.fit_dims(int(W), int(H), 512) == (w_fit, h_fit)
        assert off == 0


@pytest.mark.parametrize("W,H,T,ch", [(2000, 1500, 512, 1), (3000, 2000, 512, 3), (1300, 900, 256, 3), (1500, 1100, 512, 1),
                                      (700, 650, 128, 3)])
def test_resize_area_equals_cv2(W, H, T, ch):
    """The INTER_AREA restatement (oracle for the device fit-resize) against the installed OpenCV,
    the library the reference itself calls at utils/tools.py:194: every byte equal."""
    import cv2
    w, h = orc.fit_dims(W, H, T)
    img = orc.synth_image(3, W, H, ch)
    ref = cv2.resize(img, (w, h), interpolation=cv2.INTER_AREA)
    assert np.array_equal(orc.resize_area(img, w, h), ref)
    noise = np.random.default_rng(W).integers(0, 256, size=img.shape, dtype=np.uint8)
    assert np.array_equal(orc.resize_area(noise, w, h), cv2.resize(noise, (w, h), interpolation=cv2.INTER_AREA))


def test_resize_area_golden_fit(golden):
    """... and against the reference's own adjust_to_tile output (tests/golden/fit.npz)."""
    g = golden("fit")
    keys = [k for k in g.files if k.startswith("fitimg_") and k.endswith("_in")]
    assert len(keys) == 3
    for k in keys:
        src, ref = g[k], g[k.replace("_in", "_out")]
        assert np.array_equal(orc.resize_area(src, ref.shape[1], ref.shape[0]), ref)


def test_nn_index_map(golden):
    g = golden("fit")
    for src, dst in g["nn_pairs"]:
        assert np.array_equal(orc.nn_index_map(int(src), int(dst)), g["nn_map_%d_%d" % (src, dst)]), (src, dst)


def _recon_cases(golden):
    return [str(c) for c in golden("reconstruct")["recon_cases"]]


@pytest.mark.parametrize("case", ["a_2x3", "a_3x2", "a_3x3", "a_2x1", "b_4x5", "a_s32_2x3"])
def test_reconstruct(golden, palettes, case):
    g = golden("reconstruct")
    nr, nc, T, S, h, w, w_full, h_full, C = [int(v) for v in g["recon_%s_geom" % case]]
    pal = palettes["b" if case.startswith("b") else "a"]
    tiles = orc.reconstruct_fixture_tiles(g, case)
    ref_map = g["recon_%s_map" % case]
    assert orc.stitch_grid(h, w, T, S) == (nr, nc)
    # the step-by-step port is bit-equal to the reference
    port = orc.stitch_map_port(tiles, h, w, T, S)
    assert np.array_equal(port, ref_map)
    # and so is the closed form (SURVEY.md A.3)
    closed = orc.stitch_map(tiles, nr, nc, T, S)
    assert np.array_equal(closed, ref_map)
    # labels -> NN resample -> colourise == reference RGB output
    labels = orc.stitch_labels(closed)
    full = orc.resample_labels(labels, w_full, h_full)
    rgb = orc.colourize(full[None], C, pal)[0].astype(np.float32)
    assert np.array_equal(rgb, g["recon_%s_rgb" % case])
    batches = [tiles[i:i + 4] for i in range(0, len(tiles), 4)]
    assert np.array_equal(orc.reconstruct_port(batches, h, w, w_full, h_full, T, S, pal, C), g["recon_%s_rgb" % case])


def test_evaluate(golden, palettes):
    g = golden("evaluate")
    pal = palettes["a"]
    C = len(pal)
    y_pred = orc.class_encode_hwc(g["eval_pred_rgb"].astype(np.uint8), pal).ravel()
    y_true = orc.class_encode_hwc(g["eval_gt_rgb"], pal).ravel()
    assert np.array_equal(y_pred, g["eval_y_pred_raw"])
    assert np.array_equal(y_true, g["eval_y_true_raw"])
    yt, yp = orc.inject_coverage(y_true, y_pred, C)
    assert np.array_equal(yt, g["eval_y_true"]) and np.array_equal(yp, g["eval_y_pred"])
    labels = [str(s) for s in g["eval_labels"]]
    M = orc.confusion_counts(yt, yp, C)
    assert M.sum() == yt.size
    ref_report = json.loads(str(g["eval_report_json"]))
    for res in (orc.metrics_from_confusion(M, labels), orc.metrics_port(yt, yp, labels)):
        np.testing.assert_allclose([res["f1"], res["iou"], res["mcc"]], g["eval_scalars"], rtol=1e-12)
        np.testing.assert_allclose(res["cmatrix"], g["eval_cmatrix"], rtol=1e-15)
        for key, val in ref_report.items():
            if isinstance(val, dict):
                for k2, v2 in val.items():
                    assert res["report"][key][k2] == pytest.approx(v2, rel=1e-12), (key, k2)
            else:
                assert res["report"][key] == pytest.approx(val, rel=1e-12)


@pytest.mark.parametrize("name,C,weighted", [("a_unw", 9, False), ("a_w", 9, True), ("b_w", 11, True)])
def test_multiloss(golden, name, C, weighted):
    g = golden("loss")
    z, t, w = g["loss_%s_z" % name], g["loss_%s_t" % name], g["loss_%s_w" % name]
    ref_vals, ref_grad = g["loss_%s_vals" % name], g["loss_%s_grad" % name]
    port = orc.multiloss_port(z, t, C, weights=w, weighted=weighted)
    np.testing.assert_allclose(port[:4], ref_vals, rtol=1e-6)
    np.testing.assert_allclose(port[4], ref_grad, rtol=1e-5, atol=1e-9)
    loss, ce, dice, focal, grad, partials = orc.multiloss(z, t, C, weights=w, weighted=weighted)
    # north_star tolerance: loss values within 1e-4 relative
    np.testing.assert_allclose([loss, ce, dice, focal], ref_vals, rtol=1e-5)
    np.testing.assert_allclose(grad, ref_grad, rtol=2e-4, atol=2e-9)
    assert partials.shape == (2 * C + 3,)


@pytest.mark.parametrize("name", ["a", "b"])
def test_augment_optimize(golden, name):
    """Augmentor.optimize restatement against the reference's own run (tests/golden/augment.npz)."""
    g = golden("augment")
    N, C, px_count = (int(v) for v in g["aug_%s_meta" % name])
    best, data = orc.augment_optimize_port(g["aug_%s_px_dist" % name], px_count, g["aug_%s_probs" % name], C, N)
    assert np.array_equal(best["rates"], g["aug_%s_rates" % name])
    ref = g["aug_%s_optim" % name]
    assert [best["threshold"], best["rate_coef"], best["jsd"], best["m2"], best["n_samples"], best["aug_n_samples"]] == list(ref)
    assert np.array_equal(best["probs"], g["aug_%s_optim_probs" % name])


# ---------------------------------------------------------------------------------------------
# model-file boundary (models/modules/checkpoint.py:53-66, models/model.py:78-121)
# ---------------------------------------------------------------------------------------------

def test_deeplab_state_dict_manifest_equals_reference(golden):
    """pylc_b200's DeepLabv3+/ResNet-101 has the reference network's state-dict keys, order, shapes and
    dtypes (so a reference model file loads with strict keys, and ours loads in the reference)."""
    import json
    import torch
    from pylc_b200.models.deeplab import DeepLab
    g = golden("model")
    sd = DeepLab(n_classes=int(g["meta_n_classes"])).state_dict()
    assert list(sd.keys()) == [str(k) for k in g["keys"]]
    assert [list(v.shape) for v in sd.values()] == json.loads(str(g["shapes"]))
    assert [str(v.dtype) for v in sd.values()] == [str(d) for d in g["dtypes"]]


def test_deeplab_forward_equals_reference_network(golden):
    """Same weights (oracle.fill_state_dict, a deterministic fill), same input -> the reference network's
    own output, recorded by gen_golden.py from the unmodified reference: the two networks are the same
    function, not just the same parameter names."""
    import torch
    from pylc_b200.models.deeplab import DeepLab
    g = golden("model")
    net = DeepLab(n_classes=int(g["meta_n_classes"])).eval()
    net.load_state_dict(orc.fill_state_dict(net.state_dict()))
    with torch.no_grad():
        y = net(torch.from_numpy(g["x"])).numpy()
    want = g["y"]
    assert y.shape == want.shape
    assert np.abs(want).max() > 1e-3                         # a live output, not zeros
    assert np.abs(y - want).max() <= 1e-5 * np.abs(want).max()


def test_model_load_reads_reference_pickled_meta(tmp_path, monkeypatch):
    """A model file written by the reference pickles `meta` as config.Parameters of ITS module tree
    (checkpoint.py:53-66); Model.load resolves it to pylc_b200.config.Parameters and builds from it."""
    import torch
    from pylc_b200.config import Parameters
    from pylc_b200.models.model import _load_model_file
    path = os.path.join(GOLDEN, "ref_meta_model.pth")
    data = _load_model_file(path, torch.device("cpu"))
    assert set(data) >= {"model", "meta"}
    meta = data["meta"]
    assert isinstance(meta, Parameters)
    assert meta.arch == "deeplab" and meta.backbone == "resnet" and meta.ch == 3 and meta.n_classes == 9
    assert meta.px_mean == [130.0, 140.0, 150.0] and len(meta.palette_rgb) == 9
    fresh = Parameters()
    fresh.update(vars(meta))                                  # Model.load: self.meta.update(model_data["meta"])
    assert fresh.class_codes == meta.class_codes


# ---------------------------------------------------------------------------------------------
# augmentation warps (utils/tools.py:452-594) -- host OpenCV calls in the reference and here
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("seed", [0, 1, 3])
def test_augment_transform_equals_reference(golden, ch, seed):
    """pylc_b200.utils.tools.augment_transform gives the bytes the reference's own function gave for the same
    tile, dtypes and RandomState seed (perspective jitter, reflect border, crop + resize, brightness shift)."""
    from pylc_b200.utils import tools
    g = golden("warp")
    img, mask = orc.augment_fixture_tile(ch)
    a, b = tools.augment_transform(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
    want_img, want_mask = g["warp_ch%d_s%d_img" % (ch, seed)], g["warp_ch%d_s%d_mask" % (ch, seed)]
    assert np.asarray(a).dtype == np.uint8 and np.array_equal(np.asarray(a), want_img)
    assert np.array_equal(np.asarray(b).astype(np.uint8), want_mask)
    assert not np.array_equal(want_img.reshape(img.shape[1:] if ch == 3 else img.shape[2:]), img[0] if ch == 3 else img[0, 0])


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("seed", [0, 1, 3])
def test_augment_transform_port_equals_reference_golden(golden, ch, seed):
    """The OpenCV-free restatement (oracle.augment_transform_port: fixed-point warp coordinates, float bilinear
    table, reflect-101, the enlarging INTER_AREA taps without FMA, int16 brightness shift) reproduces the
    reference's bytes."""
    g = golden("warp")
    img, mask = orc.augment_fixture_tile(ch)
    a, b = orc.augment_transform_port(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
    assert a.dtype == np.uint8 and np.array_equal(a, g["warp_ch%d_s%d_img" % (ch, seed)])
    assert np.array_equal(b.astype(np.uint8), g["warp_ch%d_s%d_mask" % (ch, seed)])


@pytest.mark.parametrize("ch,seed", [(1, 4), (1, 7), (3, 5), (3, 11)])
def test_augment_transform_port_equals_opencv_chain(ch, seed):
    """Same restatement against the OpenCV call chain itself (tools.augment_transform = the reference's calls,
    pinned above) on noise tiles and other seeds: every rounding decision of cv2.warpPerspective and cv2.resize."""
    from pylc_b200.utils import tools
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(1, ch, 512, 512), dtype=np.uint8)
    mask = rng.integers(0, 11, size=(1, 512, 512))
    a, b = tools.augment_transform(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
    c, d = orc.augment_transform_port(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
    assert np.array_equal(np.asarray(a), c) and np.array_equal(np.asarray(b), d)
    # the pieces on their own
    import cv2
    m_inv, _ = orc.augment_params(np.random.RandomState(seed), 512)
    m = cv2.invert(m_inv)[1]
    hwc = np.moveaxis(img[0], 0, -1).astype(np.float32)
    hwc = hwc[..., 0] if ch == 1 else hwc
    want = cv2.warpPerspective(hwc, m, (512, 512), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REFLECT_101)
    got = orc.warp_perspective_linear_f32(hwc, cv2.invert(m)[1])
    assert np.array_equal(want, got)
    crop = np.ascontiguousarray(want[30:482, 30:482])
    assert np.array_equal(cv2.resize(crop, (512, 512), interpolation=cv2.INTER_AREA), orc.resize_area_upscale_f32(crop, 512))
