"""Per-pixel probabilities, confidence and calibration on the GPU (pylc_stitch_probs, pylc_stitch_upsample_probs,
pylc_confidence_resample) against the CPU oracle in tests/confidence_oracle.py, and through the pipeline,
the evaluator and the CLI."""
import glob
import json
import os

import cv2
import numpy as np
import pytest
import torch

import confidence_oracle as co
import pylc_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MARGIN = 1e-6


@pytest.fixture(scope="module")
def ops():
    from pylc_b200 import ops as _ops
    _ops._lib.load()
    return _ops


def _tiles(C, nr, nc, T, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(nr * nc, C, T, T, generator=g) * 3).numpy()


def _src(tiles, tpb):
    if tpb:
        return [torch.from_numpy(tiles[i:i + tpb]).cuda() for i in range(0, len(tiles), tpb)]
    return torch.from_numpy(tiles).cuda()


def _offset_u8(shape, dev, off):
    """A u8 tensor of `shape` whose data starts `off` bytes into its allocation (odd / misaligned outputs)."""
    n = int(np.prod(shape))
    return torch.empty(n + off, dtype=torch.uint8, device=dev)[off:].view(shape)


def _check_probs_vs_oracle(res_ref, res_mean, tiles, nr, nc, T, S, lut):
    P = co.stitch_probs(tiles, nr, nc, T, S)
    M = orc.stitch_map(tiles, nr, nc, T, S)
    probs = res_mean["probs"].cpu().numpy()
    assert np.all(np.abs(probs - P) <= 1e-5 * np.abs(P) + 1e-7)
    # mean-mode labels: argmax of P wherever it is decided
    lab_mean = res_mean["labels"].cpu().numpy()
    assert np.array_equal(lab_mean, np.argmax(probs, axis=0))
    bad = (lab_mean != np.argmax(P, axis=0)) & (orc.top2_margin(P) > MARGIN)
    assert not bad.any()
    # edge blocks: mean-mode P is bit-for-bit the reference-mode stitched map
    kinds = co.block_kinds(nr, nc, T, S)
    edge = kinds == 2
    m_ref = res_ref["probs"].cpu().numpy()
    assert np.array_equal(probs[:, edge], m_ref[:, edge])
    # confidence: the u8 of P at the label, within 1 of the oracle and exact away from rounding boundaries,
    # compared where the reference's labels are decided
    lab_ref = res_ref["labels"].cpu().numpy()
    decided = orc.top2_margin(M) > MARGIN
    for res, lab in ((res_ref, lab_ref), (res_mean, lab_mean)):
        q = res["confidence"].cpu().numpy().astype(np.int64)
        want = co.confidence_u8(P, lab).astype(np.int64)
        p_at = np.take_along_axis(P, lab[None].astype(np.int64), axis=0)[0] * 255.0
        safe = np.abs(p_at - np.floor(p_at) - 0.5) > 1e-3
        assert np.abs(q - want)[decided].max() <= 1
        assert np.array_equal(q[decided & safe], want[decided & safe])
    # reference-mode confidence == u8 of mean-mode probs at the reference label, bit for bit
    p_ref = torch.gather(res_mean["probs"], 0, res_ref["labels"].long()[None])[0]
    q_ref = torch.clamp(torch.round(p_ref * 255.0), max=255).to(torch.uint8)
    assert torch.equal(res_ref["confidence"], q_ref)
    if lut is not None:
        assert np.array_equal(res_mean["rgb"].cpu().numpy(), np.asarray(lut, dtype=np.uint8)[lab_mean])


GEOMS = [(4, 2, 3, 64, 32), (9, 3, 4, 64, 32), (11, 2, 3, 64, 32), (12, 2, 2, 64, 32), (20, 2, 3, 64, 32),
         (9, 2, 3, 64, 64), (11, 2, 2, 32, 32), (9, 3, 3, 62, 31)]


@pytest.mark.parametrize("C,nr,nc,T,S", GEOMS)
@pytest.mark.parametrize("tpb", [None, 2])
def test_stitch_probs_vs_reference_route_and_oracle(ops, palettes, C, nr, nc, T, S, tpb):
    tiles = _tiles(C, nr, nc, T, C * 1000 + nr * 10 + nc)
    lut = (palettes["a"] + palettes["b"] + palettes["a"])[:C]
    src = _src(tiles, tpb)
    lab0, rgb0, map0 = ops.stitch_argmax_colour(src, nr, nc, T, S, lut_rgb=lut, want_rgb=True, want_stitched=True,
                                                tiles_per_batch=tpb)
    kw = dict(lut_rgb=lut, want_rgb=True, want_probs=True, tiles_per_batch=tpb)
    ref = ops.stitch_probs(src, nr, nc, T, S, mode="reference", **kw)
    mean = ops.stitch_probs(src, nr, nc, T, S, mode="mean", **kw)
    # reference mode: today's outputs, bit for bit
    assert torch.equal(ref["labels"], lab0) and torch.equal(ref["rgb"], rgb0) and torch.equal(ref["probs"], map0)
    _check_probs_vs_oracle(ref, mean, tiles, nr, nc, T, S, lut)
    # odd / misaligned output pointers (the one-pixel path) give the same bytes
    h, w = ops.stitch_dims(nr, nc, T, S)
    for mode, want in (("reference", ref), ("mean", mean)):
        out = {"labels": _offset_u8((h, w), lab0.device, 1), "confidence": _offset_u8((h, w), lab0.device, 3)}
        got = ops.stitch_probs(src, nr, nc, T, S, mode=mode, tiles_per_batch=tpb, out=out)
        assert torch.equal(got["labels"], want["labels"]) and torch.equal(got["confidence"], want["confidence"])
        # labels only, no confidence: the same labels
        lab_only = ops.stitch_probs(src, nr, nc, T, S, mode=mode, want_confidence=False, tiles_per_batch=tpb)
        assert torch.equal(lab_only["labels"], want["labels"]) and lab_only["confidence"] is None


def test_stitch_probs_argument_errors(ops):
    from pylc_b200._lib import PylcError
    tiles = torch.zeros((4, 9, 32, 32), device="cuda")
    with pytest.raises(PylcError):
        ops.stitch_probs(tiles, 2, 2, 32, 16, mode="max")
    lib = ops._lib.load()
    lab = torch.empty((48, 48), dtype=torch.uint8, device="cuda")
    rc = lib.pylc_stitch_probs(ops._p(tiles), None, 4, 2, 2, 9, 32, 16, 2, None, ops._p(lab), None, None, None, None)
    assert rc == -1                                           # PYLC_ERR_ARG: unknown mode


@pytest.mark.parametrize("C,nr,nc,T,S,tpb", [(9, 3, 5, 512, 256, 8), (11, 2, 2, 512, 256, 4), (5, 2, 3, 512, 512, 6),
                                             (12, 1, 2, 512, 256, 2), (9, 2, 2, 256, 128, 3), (4, 2, 3, 128, 64, 4)])
def test_stitch_upsample_probs_equals_two_kernel_route(ops, palettes, C, nr, nc, T, S, tpb):
    n, hs = nr * nc, T // 4
    g = torch.Generator().manual_seed(C * 100 + n + 7)
    dec_all = (torch.randn(n, C, hs, hs, generator=g) * 3).cuda().contiguous(memory_format=torch.channels_last)
    batches = [dec_all[i:i + tpb].contiguous(memory_format=torch.channels_last) for i in range(0, n, tpb)]
    lut = (palettes["a"] + palettes["b"])[:C]
    logits = [ops.upsample_nhwc_to_nchw(b, (T, T)) for b in batches]
    src = logits if len(logits) > 1 else logits[0]
    kw = dict(lut_rgb=lut, want_rgb=True, want_probs=True, tiles_per_batch=tpb)
    for mode in ("reference", "mean"):
        two = ops.stitch_probs(src, nr, nc, T, S, mode=mode, **kw)
        one = ops.stitch_upsample_probs(batches, nr, nc, T, S, mode=mode, **kw)
        for k in ("labels", "rgb", "confidence", "probs"):
            assert torch.equal(one[k], two[k]), (mode, k)
    lab0, _, map0 = ops.stitch_upsample_argmax_colour(batches, nr, nc, T, S, want_stitched=True, tiles_per_batch=tpb)
    ref = ops.stitch_upsample_probs(batches, nr, nc, T, S, mode="reference", want_probs=True, tiles_per_batch=tpb)
    assert torch.equal(ref["labels"], lab0) and torch.equal(ref["probs"], map0)
    if n * T * T <= 4 * 512 * 512:
        mean = ops.stitch_upsample_probs(batches, nr, nc, T, S, mode="mean", want_probs=True, tiles_per_batch=tpb)
        _check_probs_vs_oracle(ref, mean, torch.cat(logits).cpu().numpy(), nr, nc, T, S, None)


def test_stitch_upsample_probs_misaligned_confidence_is_an_error(ops):
    from pylc_b200._lib import PylcError
    dec = torch.zeros((4, 9, 32, 32), device="cuda").contiguous(memory_format=torch.channels_last)
    h, w = ops.stitch_dims(2, 2, 128, 64)
    with pytest.raises(PylcError, match="align"):
        ops.stitch_upsample_probs([dec], 2, 2, 128, 64, out={"confidence": _offset_u8((h, w), dec.device, 1)})


@pytest.mark.parametrize("w_full,h_full,w,h", [(3000, 2000, 2560, 1536), (6000, 4000, 5632, 3584), (3001, 1999, 2560, 1536),
                                               (777, 555, 512, 512)])
def test_confidence_resample_and_reliability(ops, w_full, h_full, w, h):
    C = 9
    rng = np.random.default_rng(w_full + h_full)
    conf = rng.integers(0, 256, (h, w)).astype(np.uint8)
    conf[:, : w // 3] = 200                                       # a uniform region: contention on one counter
    pred = rng.integers(0, C, (h_full, w_full)).astype(np.uint8)
    pred[: h_full // 2] = 3
    true = np.where(rng.random((h_full, w_full)) < 0.7, pred, rng.integers(0, C, (h_full, w_full))).astype(np.uint8)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    res = ops.confidence_resample(d(conf), w_full, h_full, y_pred_full=d(pred), y_true_full=d(true), n_classes=C)
    want_full = conf[ops.nn_index_map(h, h_full)[:, None], ops.nn_index_map(w, w_full)[None, :]]
    assert np.array_equal(res["confidence_full"].cpu().numpy(), want_full)
    assert np.array_equal(res["reliability"].cpu().numpy(), co.reliability_table(want_full, pred, true, C))
    # added into; table only; plane only
    ops.confidence_resample(d(conf), w_full, h_full, y_pred_full=d(pred), y_true_full=d(true), n_classes=C,
                            reliability=res["reliability"], want_full=False)
    assert np.array_equal(res["reliability"].cpu().numpy(), 2 * co.reliability_table(want_full, pred, true, C))
    only = ops.confidence_resample(d(conf), w_full, h_full)
    assert only["reliability"] is None and torch.equal(only["confidence_full"], res["confidence_full"])


def test_confidence_resample_uniform_image_and_errors(ops):
    C = 11
    conf = torch.full((1536, 2560), 255, dtype=torch.uint8, device="cuda")
    pred = torch.full((2000, 3000), 7, dtype=torch.uint8, device="cuda")
    res = ops.confidence_resample(conf, 3000, 2000, y_pred_full=pred, y_true_full=pred, n_classes=C)
    table = res["reliability"].cpu().numpy()
    assert table[7, 255, 1] == 3000 * 2000 and table.sum() == 3000 * 2000
    lib = ops._lib.load()
    maps = ops.device_index_maps(2560, 1536, 3000, 2000, conf.device)
    rel = torch.zeros((C, 256, 2), dtype=torch.int64, device="cuda")
    rc = lib.pylc_confidence_resample(ops._p(conf), 1536, 2560, ops._p(maps[0]), ops._p(maps[1]), 2000, 3000, ops._p(pred),
                                      None, C, None, ops._p(rel), None)
    assert rc == -1                                           # reliability needs both label planes


def _tiny_model():
    from test_gpu_host import _tiny_model as tiny
    return tiny(3)


@pytest.mark.parametrize("fuse", [False, True])
def test_pipeline_confidence_and_mean_mode(ops, palettes, fuse):
    from pylc_b200.pipeline import TiledSegmenter
    model = _tiny_model()
    pal = palettes["a"]
    W, H = 1600, 1200
    img = orc.synth_image(41, W, H, 3)
    gt = orc.synth_mask(41, W, H, pal, skew=True)
    kw = dict(batch_tiles=8, keep_masks=True, fuse_network=fuse, channels_last=fuse)
    base = TiledSegmenter(model, **kw)
    conf0, res0 = base.run_host([img], [gt])
    withc = TiledSegmenter(model, confidence=True, **kw)
    withc.fused = base.fused
    conf1, res1 = withc.run_host([img], [gt])
    assert np.array_equal(conf0, conf1)
    assert torch.equal(res0[0]["labels"], res1[0]["labels"]) and torch.equal(res0[0]["pred_full"], res1[0]["pred_full"])
    assert "confidence" not in res0[0]
    c_fit, c_full = res1[0]["confidence"], res1[0]["confidence_full"]
    assert tuple(c_full.shape) == (H, W)
    x, y = ops.nn_index_map(c_fit.shape[1], W), ops.nn_index_map(c_fit.shape[0], H)
    assert np.array_equal(c_full.cpu().numpy(), c_fit.cpu().numpy()[y[:, None], x[None, :]])
    # mean mode: run_host and run_resident agree
    mean = TiledSegmenter(model, stitch="mean", confidence=True, **kw)
    mean.fused = base.fused
    conf_h, res_h = mean.run_host([img], [gt])
    mean.reset()
    out = []
    mean.run_resident([mean.stage(img, gt, index=0)], results=out)
    assert np.array_equal(mean.conf.cpu().numpy(), conf_h)
    assert torch.equal(out[0]["labels"], res_h[0]["labels"]) and torch.equal(out[0]["confidence"], res_h[0]["confidence"])


def _cli(cwd, *argv):
    import subprocess
    import sys
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-m", "pylc_b200.pylc"] + list(argv), cwd=str(cwd), env=env,
                         capture_output=True, text=True, timeout=900, stdin=subprocess.DEVNULL)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    return out.stdout


def _tree(root):
    out = {}
    for p in sorted(glob.glob(os.path.join(root, "**", "*"), recursive=True)):
        if os.path.isfile(p) and not p.endswith(".pdf"):
            with open(p, "rb") as f:
                out[os.path.relpath(p, root)] = f.read()
    return out


def test_cli_stitch_mean_save_confidence(tmp_path, palettes):
    from pylc_b200.config import Parameters
    from pylc_b200.models.deeplab import DeepLab
    pal = palettes["a"]
    C = len(pal)
    W, H = 1300, 1000
    os.makedirs(tmp_path / "imgs")
    os.makedirs(tmp_path / "masks")
    for k in range(2):
        assert cv2.imwrite(str(tmp_path / "imgs" / ("s%d.tif" % k)), orc.synth_image(50 + k, W, H, 1))
        assert cv2.imwrite(str(tmp_path / "masks" / ("s%d.png" % k)),
                           np.ascontiguousarray(orc.synth_mask(50 + k, W, H, pal)[..., ::-1]))
    torch.manual_seed(0)
    net = DeepLab(n_classes=C, in_channels=1)
    m = Parameters()
    m.update({"ch": 1, "arch": "deeplab", "backbone": "resnet", "pretrained": False, "px_mean": [120.0], "px_std": [40.0],
              "weights": [1.0] * C, "normalize_default": False, "id": "conf_model"})
    model_file = str(tmp_path / "conf_model.pth")
    torch.save({"model": net.state_dict(), "optim": None, "meta": m}, model_file)
    runs = {}
    for name, extra in (("default", []), ("mean", ["--stitch", "mean", "--save_confidence"]),
                        ("ref_conf", ["--save_confidence"]), ("agg", ["--stitch", "mean", "--save_confidence", "--aggregate_metrics"])):
        cwd = tmp_path / name
        os.makedirs(cwd)
        _cli(cwd, "test", "--model", model_file, "--img", str(tmp_path / "imgs"), "--mask", str(tmp_path / "masks"), *extra)
        roots = glob.glob(str(cwd / "data" / "outputs" / "*"))
        assert len(roots) == 1
        runs[name] = roots[0]
    # a default run writes no confidence directory and no calibration
    assert not os.path.exists(os.path.join(runs["default"], "confidence"))
    for p in glob.glob(os.path.join(runs["default"], "metrics", "*_eval.json")):
        assert "calibration" not in json.load(open(p))
    # --save_confidence without --stitch mean: labels, masks and scores are the default run's
    d, r = _tree(runs["default"]), _tree(runs["ref_conf"])
    for k, v in d.items():
        if k.endswith("_eval.json"):
            got = json.load(open(os.path.join(runs["ref_conf"], k)))
            assert got.pop("calibration")["n_pixels"] == W * H
            assert got == json.loads(v)
        else:
            assert r[k] == v, k
    for name in ("mean", "ref_conf", "agg"):
        pngs = sorted(glob.glob(os.path.join(runs[name], "confidence", "*.png")))
        assert len(pngs) == 2
        for p in pngs:
            q = cv2.imread(p, cv2.IMREAD_UNCHANGED)
            assert q.dtype == np.uint8 and q.shape == (H, W) and q.max() > 0
    for p in glob.glob(os.path.join(runs["mean"], "metrics", "*_eval.json")):
        cal = json.load(open(p))["calibration"]
        assert 0.0 <= cal["ece"] <= cal["mce"] <= 1.0 and cal["n_pixels"] == W * H
    agg = glob.glob(os.path.join(runs["agg"], "metrics", "aggregate_metrics_eval.json"))
    assert len(agg) == 1
    assert json.load(open(agg[0]))["calibration"]["n_pixels"] == 2 * W * H
