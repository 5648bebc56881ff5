"""Multi-scale inference on the GPU: pylc_multiscale_combine against the CPU oracle in tests/multiscale_oracle.py,
the one-scale anchors against the single-scale mean stitch, the per-scale orchestration of TiledSegmenter and the
CLI."""
import glob
import json
import os

import cv2
import numpy as np
import pytest
import torch

import confidence_oracle as co
import multiscale_oracle as mo
import pylc_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MARGIN = 1e-6


@pytest.fixture(scope="module")
def ops():
    from pylc_b200 import ops as _ops
    _ops._lib.load()
    return _ops


def _planes(seed, C, sizes):
    rng = np.random.default_rng(seed)
    return [co.softmax64(rng.standard_normal((C, h, w)) * 3).astype(np.float32) for w, h in sizes]


def _offset_u8(shape, dev, off):
    """A u8 tensor of `shape` whose data starts `off` bytes into its allocation (odd / misaligned outputs)."""
    n = int(np.prod(shape))
    return torch.empty(n + off, dtype=torch.uint8, device=dev)[off:].view(shape)


def _check_vs_oracle(got, probs, w_full, h_full, lut):
    m32, lab32, q32 = mo.combine_f32(probs, w_full, h_full)
    assert np.array_equal(got["labels"].cpu().numpy(), lab32)
    assert np.array_equal(got["confidence"].cpu().numpy(), q32)
    m64, lab64, q64 = mo.combine_f64(probs, w_full, h_full)
    decided = orc.top2_margin(m64) > MARGIN if m64.shape[0] > 1 else np.ones(lab64.shape, dtype=bool)
    assert np.array_equal(lab32[decided], lab64[decided])
    assert np.abs(q32.astype(np.int64) - q64).max() <= 1
    if lut is not None:
        assert np.array_equal(got["rgb"].cpu().numpy(), np.asarray(lut, dtype=np.uint8)[lab32])


CASES = [   # K, C, member sizes (w, h), output (w, h)
    (1, 9, [(1536, 1024)], (1301, 997)),
    (1, 1, [(64, 48)], (128, 96)),
    (2, 2, [(512, 512), (1024, 512)], (1301, 997)),
    (2, 9, [(1024, 512), (1536, 1024)], (1800, 1300)),
    (3, 9, [(1024, 512), (1536, 1024), (2048, 1536)], (1600, 1200)),
    (3, 11, [(257, 129), (300, 200), (511, 383)], (301, 199)),
    (8, 20, [(64 + 16 * k, 48 + 8 * k) for k in range(8)], (131, 97)),
    (3, 32, [(128, 64), (256, 128), (384, 256)], (333, 222)),
]


@pytest.mark.parametrize("K,C,sizes,out", CASES)
def test_combine_equals_restatement_and_definition(ops, K, C, sizes, out):
    assert len(sizes) == K
    w_full, h_full = out
    probs = _planes(K * 100 + C, C, sizes)
    lut = [list(v) for v in np.random.default_rng(C).integers(0, 256, (C, 3))]
    d = [torch.from_numpy(p).cuda() for p in probs]
    got = ops.multiscale_combine(d, w_full, h_full, lut_rgb=lut, want_rgb=True)
    _check_vs_oracle(got, probs, w_full, h_full, lut)
    # misaligned outputs take the byte path and give the same bytes; each output alone as well
    dev = d[0].device
    odd = {"labels": _offset_u8((h_full, w_full), dev, 1), "rgb": _offset_u8((h_full, w_full, 3), dev, 2),
           "confidence": _offset_u8((h_full, w_full), dev, 3)}
    mis = ops.multiscale_combine(d, w_full, h_full, lut_rgb=lut, want_rgb=True, out=odd)
    for k in ("labels", "rgb", "confidence"):
        assert torch.equal(mis[k], got[k]), k
    lab = ops.multiscale_combine(d, w_full, h_full, want_confidence=False)
    conf = ops.multiscale_combine(d, w_full, h_full, want_labels=False)
    assert lab["confidence"] is None and torch.equal(lab["labels"], got["labels"])
    assert conf["labels"] is None and torch.equal(conf["confidence"], got["confidence"])


def test_combine_argument_errors(ops):
    import ctypes
    from pylc_b200._lib import PylcError
    lib = ops._lib.load()
    p = torch.rand((9, 32, 48), device="cuda")
    xo, yo = ops.device_index_maps(48, 32, 64, 40, p.device)
    lab = torch.empty((40, 64), dtype=torch.uint8, device="cuda")

    def call(K, C, planes=None):
        n = max(K, 1)
        planes = planes if planes is not None else [p.data_ptr()] * n
        arr = lambda v: (ctypes.c_void_p * n)(*v)           # noqa: E731
        ints = lambda v: (ctypes.c_int * n)(*([v] * n))      # noqa: E731
        return lib.pylc_multiscale_combine(arr(planes), arr([xo.data_ptr()] * n), arr([yo.data_ptr()] * n), ints(32),
                                           ints(48), K, C, 40, 64, None, ops._p(lab), None, None, None)
    assert call(2, 9) == 0
    assert call(0, 9) == -1 and call(9, 9) == -1                       # PYLC_ERR_ARG: K outside [1, 8]
    assert call(2, 9, planes=[p.data_ptr(), None]) == -1               # a null plane
    assert call(1, 0) == -2 and call(1, 33) == -2                      # PYLC_ERR_CLASSES
    torch.cuda.synchronize()
    with pytest.raises(PylcError):
        ops.multiscale_combine([p] * 9, 64, 40)
    with pytest.raises(PylcError):
        ops.multiscale_combine([p, torch.rand((8, 32, 48), device="cuda")], 64, 40)


def _tiles(C, nr, nc, T, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(nr * nc, C, T, T, generator=g) * 3


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("w_full,h_full", [(1800, 1300), (1301, 997)])
def test_one_scale_anchor_equals_mean_stitch_resampled(ops, fused, w_full, h_full):
    C, nr, nc, T, S, tpb = 9, 3, 5, 512, 256, 4
    if fused:
        dec = _tiles(C, nr, nc, T // 4, 11).cuda().contiguous(memory_format=torch.channels_last)
        src = [dec[i:i + tpb].contiguous(memory_format=torch.channels_last) for i in range(0, nr * nc, tpb)]
        st = ops.stitch_upsample_probs(src, nr, nc, T, S, mode="mean", want_probs=True, tiles_per_batch=tpb)
    else:
        src = _tiles(C, nr, nc, T, 12).cuda()
        st = ops.stitch_probs(src, nr, nc, T, S, mode="mean", want_probs=True)
    got = ops.multiscale_combine([st["probs"]], w_full, h_full)
    pred = ops.resample_encode_confusion(st["labels"], w_full, h_full, n_classes=C, want_pred=True)["pred_full"]
    conf = ops.confidence_resample(st["confidence"], w_full, h_full)["confidence_full"]
    assert torch.equal(got["labels"], pred)
    assert torch.equal(got["confidence"], conf)


def _tiny_model():
    from test_gpu_host import _tiny_model as tiny
    return tiny(3)


def _reliability(ops, res, gt_full, C):
    return ops.confidence_resample(res["confidence"], gt_full.shape[1], gt_full.shape[0], y_pred_full=res["pred_full"],
                                   y_true_full=gt_full, n_classes=C, want_full=False)["reliability"]


@pytest.mark.parametrize("fuse", [False, True])
def test_pipeline_one_scale_equals_mean_stitch(ops, palettes, fuse):
    from pylc_b200.pipeline import TiledSegmenter
    model = _tiny_model()
    pal = palettes["a"]
    W, H = 1600, 1200
    img = orc.synth_image(61, W, H, 3)
    gt = orc.synth_mask(61, W, H, pal, skew=True)
    gt_full = torch.from_numpy(orc.class_encode_hwc(gt, pal)).cuda()
    kw = dict(batch_tiles=8, keep_masks=True, fuse_network=fuse, channels_last=fuse, stitch="mean", confidence=True)
    base = TiledSegmenter(model, **kw)
    one = TiledSegmenter(model, scales=(1.0,), **kw)
    one.fused = base.fused
    for runner in ("host", "resident"):
        outs = []
        for seg in (base, one):
            seg.reset()
            if runner == "host":
                conf, res = seg.run_host([img], [gt])
            else:
                res = []
                seg.run_resident([seg.stage(img, gt, index=0)], results=res)
                conf = seg.conf.cpu().numpy()
            outs.append((conf, res[0]))
        (c0, r0), (c1, r1) = outs
        assert np.array_equal(c0, c1), runner
        for k in ("pred_full", "pred_rgb", "confidence_full"):
            assert torch.equal(r0[k], r1[k]), (runner, k)
        assert torch.equal(_reliability(ops, r0, gt_full, 9), _reliability(ops, r1, gt_full, 9)), runner


def test_pipeline_refuses_scales_without_mean_stitch():
    from pylc_b200.pipeline import TiledSegmenter
    model = _tiny_model()
    with pytest.raises(ValueError, match="mean"):
        TiledSegmenter(model, scales=(1.0,))
    with pytest.raises(ValueError):
        TiledSegmenter(model, stitch="mean", scales=(1.0, 1.0))


def test_pipeline_multiscale_orchestration(ops, palettes):
    from pylc_b200.pipeline import TiledSegmenter, multiscale_geometry
    from pylc_b200.utils import tools
    model = _tiny_model()
    pal = palettes["a"]
    W, H, T, scales = 2400, 1800, 512, (0.75, 1.0, 1.25)
    img = orc.synth_image(71, W, H, 3)
    gt = orc.synth_mask(71, W, H, pal, skew=True)
    kw = dict(batch_tiles=8, keep_masks=True, stitch="mean", confidence=True, scales=scales)
    dev_seg = TiledSegmenter(model, **kw)
    host_seg = TiledSegmenter(model, device_fit=False, **kw)
    geo = multiscale_geometry(W, H, T, scales)
    assert [g["device"] for g in geo] == [True, True, False]
    # each member's P is a single-scale mean stitch of the test's own cv2 resize + fit
    f = dev_seg.stage_device(img, gt, index=0)
    torch.cuda.current_stream().wait_event(f.ready)
    planes = dev_seg.member_probs(f)
    fh = host_seg.stage(img, gt, index=0)
    torch.cuda.current_stream().wait_event(fh.ready)
    assert all(m[1] is not None for m in fh.members)
    planes_host = host_seg.member_probs(fh)
    for g, P, Ph in zip(geo, planes, planes_host):
        x = img if g["scale"] == 1.0 else cv2.resize(img, g["resized"], interpolation=cv2.INTER_AREA)
        fitted, w, h, _ = tools.adjust_to_tile(x, T, T // 2, 3)
        assert (w, h) == g["fitted"]
        d, pitch = ops.upload_image(fitted)
        ref = dev_seg._stitch_probs(dev_seg._tiles(d, pitch, h, w), h // 256 - 1, w // 256 - 1, want_labels=False,
                                    want_confidence=False, want_probs=True)["probs"]
        assert torch.equal(P, ref), g["scale"]
        assert torch.equal(Ph, ref), g["scale"]             # made on the host: the same member
    want = ops.multiscale_combine(planes, W, H)
    # the pipeline: labels and confidence are the combine of those planes; run_host == run_resident == host route
    conf_h, res_h = dev_seg.run_host([img], [gt])
    assert torch.equal(res_h[0]["labels"], want["labels"]) and torch.equal(res_h[0]["confidence"], want["confidence"])
    assert torch.equal(res_h[0]["confidence_full"], want["confidence"])
    assert torch.equal(res_h[0]["pred_full"], want["labels"])
    dev_seg.reset()
    out = []
    dev_seg.run_resident([dev_seg.stage_device(img, gt, index=0)], results=out)
    assert np.array_equal(dev_seg.conf.cpu().numpy(), conf_h)
    assert torch.equal(out[0]["labels"], want["labels"]) and torch.equal(out[0]["confidence"], want["confidence"])
    conf_x, res_x = host_seg.run_host([img], [gt])
    assert np.array_equal(conf_x, conf_h) and torch.equal(res_x[0]["labels"], want["labels"])
    # the confusion matrix: a CPU count of the full-resolution labels against the encoded truth, with the injection
    yt, yp = orc.inject_coverage(orc.class_encode_hwc(gt, pal), want["labels"].cpu().numpy(), 9)
    assert np.array_equal(conf_h, orc.confusion_counts(yt, yp, 9))


def test_combine_full_size_equals_restatement(ops):
    from pylc_b200.pipeline import multiscale_geometry
    geo = multiscale_geometry(6000, 4000, 512, (0.75, 1.0, 1.25))
    probs = _planes(6, 9, [g["fitted"] for g in geo])
    got = ops.multiscale_combine([torch.from_numpy(p).cuda() for p in probs], 6000, 4000)
    _, lab, q = mo.combine_f32(probs, 6000, 4000)
    assert np.array_equal(got["labels"].cpu().numpy(), lab)
    assert np.array_equal(got["confidence"].cpu().numpy(), q)


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


def _cli_inputs(tmp, name, W, H, pal, seed):
    for sub in ("imgs", "masks"):
        os.makedirs(tmp / name / sub)
    for k in range(2):
        assert cv2.imwrite(str(tmp / name / "imgs" / ("s%d.tif" % k)), orc.synth_image(seed + k, W, H, 1))
        assert cv2.imwrite(str(tmp / name / "masks" / ("s%d.png" % k)),
                           np.ascontiguousarray(orc.synth_mask(seed + k, W, H, pal)[..., ::-1]))
    return tmp / name / "imgs", tmp / name / "masks"


def test_cli_multiscale(tmp_path, palettes):
    from pylc_b200.config import Parameters
    from pylc_b200.models.deeplab import DeepLab
    pal = palettes["a"]
    C = len(pal)
    torch.manual_seed(0)
    net = DeepLab(n_classes=C, in_channels=1)
    m = Parameters()
    m.update({"ch": 1, "arch": "deeplab", "backbone": "resnet", "pretrained": False, "px_mean": [120.0], "px_std": [40.0],
              "weights": [1.0] * C, "normalize_default": False, "id": "ms_model"})
    model_file = str(tmp_path / "ms_model.pth")
    torch.save({"model": net.state_dict(), "optim": None, "meta": m}, model_file)
    small = _cli_inputs(tmp_path, "small", 1600, 1200, pal, 80)
    large = _cli_inputs(tmp_path, "large", 2600, 2000, pal, 90)
    runs = {}
    for name, (imgs, masks), extra in (
            ("mean", small, ["--stitch", "mean", "--save_confidence"]),
            ("one", small, ["--stitch", "mean", "--multiscale", "1.0", "--save_confidence"]),
            ("two", large, ["--stitch", "mean", "--multiscale", "1.0", "0.8", "--save_confidence", "--aggregate_metrics"])):
        cwd = tmp_path / name
        os.makedirs(cwd)
        _cli(cwd, "test", "--model", model_file, "--img", str(imgs), "--mask", str(masks), *extra)
        roots = glob.glob(str(cwd / "data" / "outputs" / "*"))
        assert len(roots) == 1
        runs[name] = roots[0]
    # --multiscale 1.0: the files of the single-scale mean run; the scores carry the scales
    a, b = _tree(runs["mean"]), _tree(runs["one"])
    assert set(a) == set(b) and any(k.endswith(".png") and k.startswith("confidence") for k in a)
    for k, v in a.items():
        if k.endswith("_eval.json"):
            got = json.loads(b[k])
            assert got.pop("multiscale") == [1.0]
            assert got == json.loads(v)
        else:
            assert b[k] == v, k
    # two scales with aggregate metrics: masks, confidence and a calibration over every pixel
    assert len(glob.glob(os.path.join(runs["two"], "masks", "*.png"))) == 2
    for p in sorted(glob.glob(os.path.join(runs["two"], "confidence", "*.png"))):
        q = cv2.imread(p, cv2.IMREAD_UNCHANGED)
        assert q.dtype == np.uint8 and q.shape == (2000, 2600) and q.max() > 0
    agg = json.load(open(os.path.join(runs["two"], "metrics", "aggregate_metrics_eval.json")))
    assert agg["multiscale"] == [0.8, 1.0] and agg["calibration"]["n_pixels"] == 2 * 2600 * 2000
