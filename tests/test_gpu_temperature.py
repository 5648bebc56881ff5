"""Temperature scaling of the mean stitch on the GPU (pylc_stitch_probs_t, pylc_stitch_upsample_probs_t,
pylc_prob_scores, utils/calibrate.py) against the f64 oracle in tests/temperature_oracle.py, through the pipeline and
the command line."""
import glob
import json
import math
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest
import torch

import confidence_oracle as co
import pylc_oracle as orc
import temperature_oracle as to

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MARGIN = 1e-6
GEOMS = [(4, 2, 3, 64, 32), (9, 3, 4, 64, 32), (11, 2, 3, 64, 32), (12, 2, 2, 64, 32), (20, 2, 3, 64, 32),
         (9, 2, 3, 64, 64), (11, 2, 2, 32, 32), (9, 3, 3, 62, 31)]        # those of test_gpu_confidence.py


@pytest.fixture(scope="module")
def ops():
    from pylc_b200 import ops as _ops
    _ops._lib.load()
    return _ops


def _tiles(C, nr, nc, T, seed, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(nr * nc, C, T, T, generator=g) * scale).numpy()


def _outputs(ops, C, h, w):
    return {"labels": torch.empty((h, w), dtype=torch.uint8, device="cuda"),
            "confidence": torch.empty((h, w), dtype=torch.uint8, device="cuda"),
            "probs": torch.empty((C, h, w), dtype=torch.float32, device="cuda")}


def _raw_stitch(ops, src, nr, nc, T, S, mode, temperature=None):
    """One call of pylc_stitch_probs (temperature None) or pylc_stitch_probs_t, outputs allocated here."""
    lib = ops._lib.load()
    lp, bp, tpb, C, _, table = ops._tile_source(src, nr, nc, None)
    h, w = ops.stitch_dims(nr, nc, T, S)
    out = _outputs(ops, C, h, w)
    args = [lp, bp, tpb, nr, nc, C, T, S, mode, None, ops._p(out["labels"]), None, ops._p(out["confidence"]),
            ops._p(out["probs"])]
    rc = lib.pylc_stitch_probs(*args, None) if temperature is None else lib.pylc_stitch_probs_t(*args, temperature, None)
    torch.cuda.synchronize()
    return rc, out


def _raw_stitch_up(ops, dec, nr, nc, T, S, mode, temperature=None):
    lib = ops._lib.load()
    table, tpb, C, hs, ws, _ = ops._decoder_source(dec, nr, nc, None)
    h, w = ops.stitch_dims(nr, nc, T, S)
    out = _outputs(ops, C, h, w)
    args = [ops._p(table), tpb, nr, nc, C, T, S, hs, ws, mode, None, ops._p(out["labels"]), None,
            ops._p(out["confidence"]), ops._p(out["probs"])]
    rc = lib.pylc_stitch_upsample_probs(*args, None) if temperature is None \
        else lib.pylc_stitch_upsample_probs_t(*args, temperature, None)
    torch.cuda.synchronize()
    return rc, out


def _same(a, b):
    return all(torch.equal(a[k], b[k]) for k in ("labels", "confidence", "probs"))


def _decoder(C, nr, nc, T, seed):
    g = torch.Generator().manual_seed(seed)
    d = (torch.randn(nr * nc, C, T // 4, T // 4, generator=g) * 3).cuda()
    return [d.contiguous(memory_format=torch.channels_last)]


# ---- 1. T = 1 anchors ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("C,nr,nc,T,S", GEOMS)
def test_tempered_entry_points_at_one_equal_the_untempered_ones(ops, C, nr, nc, T, S):
    src = torch.from_numpy(_tiles(C, nr, nc, T, C * 100 + nr * 10 + nc)).cuda()
    for mode in (0, 1):
        rc0, a = _raw_stitch(ops, src, nr, nc, T, S, mode)
        rc1, b = _raw_stitch(ops, src, nr, nc, T, S, mode, 1.0)
        assert rc0 == rc1 == 0 and _same(a, b), mode


@pytest.mark.parametrize("C,S", [(4, 32), (9, 32), (11, 32), (12, 32), (9, 64)])
def test_fused_tempered_entry_point_at_one_equals_the_untempered_one(ops, C, S):
    nr, nc, T = 2, 3, 64
    dec = _decoder(C, nr, nc, T, C + S)
    for mode in (0, 1):
        rc0, a = _raw_stitch_up(ops, dec, nr, nc, T, S, mode)
        rc1, b = _raw_stitch_up(ops, dec, nr, nc, T, S, mode, 1.0)
        assert rc0 == rc1 == 0 and _same(a, b), mode


def test_temperature_argument_errors(ops):
    from pylc_b200._lib import PylcError
    src = torch.from_numpy(_tiles(9, 2, 2, 32, 1)).cuda()
    dec = _decoder(9, 2, 2, 64, 2)
    for bad in (2.0, 0.5):                                    # reference mode takes T = 1 only
        assert _raw_stitch(ops, src, 2, 2, 32, 16, 0, bad)[0] == -1
        assert _raw_stitch_up(ops, dec, 2, 2, 64, 32, 0, bad)[0] == -1
        with pytest.raises(PylcError):
            ops.stitch_probs(src, 2, 2, 32, 16, mode="reference", temperature=bad)
    for bad in (0.0, -1.0, float("nan"), float("inf"), -float("inf")):
        assert _raw_stitch(ops, src, 2, 2, 32, 16, 1, bad)[0] == -1
        assert _raw_stitch_up(ops, dec, 2, 2, 64, 32, 1, bad)[0] == -1
        with pytest.raises(PylcError):
            ops.stitch_probs(src, 2, 2, 32, 16, mode="mean", temperature=bad)


# ---- 2. against the oracle ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("temperature", [0.25, 0.5, 2.0, 7.5])
@pytest.mark.parametrize("C,nr,nc,T,S", [(4, 2, 3, 64, 32), (9, 3, 4, 64, 32), (11, 2, 3, 64, 32), (12, 2, 2, 64, 32),
                                         (20, 2, 3, 64, 32), (9, 2, 3, 64, 64), (11, 2, 2, 32, 32)])
def test_tempered_stitch_vs_oracle(ops, C, nr, nc, T, S, temperature):
    tiles = _tiles(C, nr, nc, T, C * 1000 + nr * 10 + nc)
    res = ops.stitch_probs(torch.from_numpy(tiles).cuda(), nr, nc, T, S, mode="mean", want_probs=True,
                           temperature=temperature)
    P = to.stitch_probs_t(tiles, nr, nc, T, S, temperature)
    probs = res["probs"].cpu().numpy()
    assert np.all(np.abs(probs - P) <= 1e-5 * np.abs(P) + 1e-7)
    lab = res["labels"].cpu().numpy()
    assert np.array_equal(lab, np.argmax(probs, axis=0))
    assert not ((lab != np.argmax(P, axis=0)) & (orc.top2_margin(P) > MARGIN)).any()
    decided = orc.top2_margin(P) > MARGIN
    q = res["confidence"].cpu().numpy().astype(np.int64)
    want = co.confidence_u8(P, lab).astype(np.int64)
    p_at = np.take_along_axis(P, lab[None].astype(np.int64), axis=0)[0] * 255.0
    safe = np.abs(p_at - np.floor(p_at) - 0.5) > 1e-3
    assert np.abs(q - want)[decided].max() <= 1
    assert np.array_equal(q[decided & safe], want[decided & safe])


# ---- 3. fused route ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("temperature", [0.5, 3.0])
@pytest.mark.parametrize("C,nr,nc,T,S,tpb", [(9, 3, 5, 512, 256, 4), (11, 2, 2, 512, 256, 4), (5, 2, 3, 512, 512, 6)])
def test_fused_route_equals_two_kernel_route_tempered(ops, C, nr, nc, T, S, tpb, temperature):
    g = torch.Generator().manual_seed(C * 7 + nr)
    dec = (torch.randn(nr * nc, C, T // 4, T // 4, generator=g) * 3).cuda().contiguous(memory_format=torch.channels_last)
    batches = [dec[i:i + tpb].contiguous(memory_format=torch.channels_last) for i in range(0, nr * nc, tpb)]
    logits = [ops.upsample_nhwc_to_nchw(b, (T, T)) for b in batches]
    kw = dict(mode="mean", want_probs=True, tiles_per_batch=tpb, temperature=temperature)
    a = ops.stitch_upsample_probs(batches, nr, nc, T, S, **kw)
    b = ops.stitch_probs(logits, nr, nc, T, S, **kw)
    assert _same(a, b)
    one = ops.stitch_probs(logits, nr, nc, T, S, mode="mean", want_probs=True, tiles_per_batch=tpb)
    assert not torch.equal(a["probs"], one["probs"])      # the temperature did reach the kernels


# ---- 4. pylc_prob_scores -------------------------------------------------------------------------------------------

def _probs(C, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.softmax(torch.randn(C, h, w, generator=g) * 3, dim=0).contiguous()


def _offset_u8(arr, off):
    t = torch.empty(arr.size + off, dtype=torch.uint8, device="cuda")[off:]
    t.copy_(torch.from_numpy(arr.ravel()))
    return t.view(arr.shape)


@pytest.mark.parametrize("C,h,w,h_full,w_full,off", [(9, 37, 53, 101, 203, 1), (11, 64, 96, 61, 97, 3),
                                                     (32, 40, 48, 123, 157, 0), (9, 256, 384, 513, 767, 2)])
def test_prob_scores_vs_oracle(ops, C, h, w, h_full, w_full, off):
    P = _probs(C, h, w, C + h)
    rng = np.random.default_rng(h_full)
    y = rng.integers(0, C, size=(h_full, w_full)).astype(np.uint8)
    y_d = _offset_u8(y, off)
    x_ofs, y_ofs = ops.nn_index_map(w, w_full), ops.nn_index_map(h, h_full)
    nll, brier = to.prob_scores(P.numpy(), y, x_ofs, y_ofs)
    got = ops.prob_scores(P.cuda(), y_d, w_full, h_full).cpu().numpy()
    assert got[0] == pytest.approx(nll, rel=1e-6) and got[1] == pytest.approx(brier, rel=1e-6)
    # NLL only: the same NLL sum bit for bit, no Brier
    nll_only = ops.prob_scores(P.cuda(), y_d, w_full, h_full, want_brier=False).cpu().numpy()
    assert nll_only[0] == got[0] and nll_only[1] == 0.0


def test_prob_scores_full_size_deterministic(ops):
    C, h, w, h_full, w_full = 9, 2048, 3072, 4000, 6000
    P = _probs(C, h, w, 5)
    rng = np.random.default_rng(6)
    y = rng.integers(0, C, size=(h_full, w_full)).astype(np.uint8)
    y_d = torch.from_numpy(y).cuda()
    Pd = P.cuda()
    a = ops.prob_scores(Pd, y_d, w_full, h_full)
    b = ops.prob_scores(Pd, y_d, w_full, h_full)
    assert torch.equal(a, b)                                   # the same bits on every call
    nll, brier = to.prob_scores(P.numpy(), y, ops.nn_index_map(w, w_full), ops.nn_index_map(h, h_full))
    got = a.cpu().numpy()
    assert got[0] == pytest.approx(nll, rel=1e-6) and got[1] == pytest.approx(brier, rel=1e-6)


def test_prob_scores_floor_at_exact_zeros(ops):
    C, h, w = 4, 8, 16
    P = torch.zeros(C, h, w)
    P[1] = 1.0                                                 # class 0 has probability exactly 0
    y = np.zeros((h, w), dtype=np.uint8)
    y[:, ::2] = 1
    got = ops.prob_scores(P.cuda(), torch.from_numpy(y).cuda(), w, h).cpu().numpy()
    n0 = int((y == 0).sum())
    assert got[0] == pytest.approx(n0 * -math.log(float(np.float32(1e-12))), rel=1e-6)
    assert got[1] == pytest.approx(2.0 * n0, rel=1e-12)


def test_prob_scores_argument_errors(ops):
    from pylc_b200._lib import PylcError
    with pytest.raises(PylcError):
        ops.prob_scores(torch.zeros((3, 4, 4), device="cuda"), torch.zeros((5, 5), dtype=torch.uint8, device="cuda"), 4, 4)
    lib = ops._lib.load()
    ws = torch.empty(ops._lib.SCORES_WS_DOUBLES, dtype=torch.float64, device="cuda")
    assert lib.pylc_prob_scores(None, 3, 4, 4, None, None, 4, 4, None, 1, ops._p(ws), ops._p(ws), None) == -1
    p = torch.zeros((33, 1, 1), device="cuda")
    m = torch.zeros(1, dtype=torch.int32, device="cuda")
    y = torch.zeros(1, dtype=torch.uint8, device="cuda")
    assert lib.pylc_prob_scores(ops._p(p), 33, 1, 1, ops._p(m), ops._p(m), 1, 1, ops._p(y), 1, ops._p(ws), ops._p(ws),
                                None) == -2


# ---- 5. fit --------------------------------------------------------------------------------------------------------

def _gpu_objective(ops, tiles, y, geom):
    C, nr, nc, T, S = geom
    src = torch.from_numpy(tiles).cuda()
    y_d = torch.from_numpy(y).cuda()
    h, w = y.shape
    maps = ops.device_index_maps(w, h, w, h, "cuda")

    def f(u):
        P = ops.stitch_probs(src, nr, nc, T, S, mode="mean", want_labels=False, want_confidence=False, want_probs=True,
                             temperature=math.exp(u))["probs"]
        return float(ops.prob_scores(P, y_d, w, h, want_brier=False, maps=maps)[0].item()) / y.size
    return f


@pytest.mark.parametrize("T0", [0.5, 2.0])
def test_fit_agrees_with_oracle_and_recovers_planted_temperature(ops, T0):
    from pylc_b200.utils.calibrate import fit_temperature
    tiles, y, geom = to.planted_case(T0)
    r = fit_temperature(_gpu_objective(ops, tiles, y, geom))
    T, f, at_bound, _ = to.fit_temperature(lambda u: to.mean_nll(tiles, y, geom, math.exp(u)))
    assert abs(math.log(r["temperature"]) - math.log(T)) <= 5e-3
    assert r["f"] == pytest.approx(f, rel=1e-6)
    assert not r["at_bound"] and not at_bound
    assert abs(r["temperature"] / T0 - 1) < 0.03


# ---- 6. pipeline ---------------------------------------------------------------------------------------------------

def _tiny_model():
    from test_gpu_host import _tiny_model as tiny
    return tiny(3)


def _direct(ops, seg, img, temperature):
    """The ops composition the pipeline runs for one image: host fit, tiles, network, tempered stitch, resample."""
    from pylc_b200.utils import tools
    fitted, w, h, _ = tools.adjust_to_tile(img, seg.T, seg.S, 3)
    d, pitch = ops.upload_image(fitted)
    src = seg.network_output(seg._tiles(d, pitch, h, w))
    return src, seg.stitch_output(src, h // seg.S - 1, w // seg.S - 1, temperature=temperature, want_probs=True)


@pytest.mark.parametrize("fuse", [False, True])
def test_pipeline_temperature_equals_ops_composition(ops, palettes, fuse):
    from pylc_b200.pipeline import TiledSegmenter
    model = _tiny_model()
    pal = palettes["a"]
    W, H = 1600, 1200
    img = orc.synth_image(41, W, H, 3)
    gt = orc.synth_mask(41, W, H, pal, skew=True)
    kw = dict(batch_tiles=8, keep_masks=True, fuse_network=fuse, channels_last=fuse, stitch="mean", confidence=True)
    plain = TiledSegmenter(model, **kw)
    one = TiledSegmenter(model, temperature=1.0, **kw)
    hot = TiledSegmenter(model, temperature=2.5, **kw)
    one.fused = hot.fused = plain.fused
    _, want = _direct(ops, hot, img, 2.5)
    _, want1 = _direct(ops, plain, img, 1.0)
    for runner in ("host", "resident"):
        got = {}
        for name, seg in (("plain", plain), ("one", one), ("hot", hot)):
            seg.reset()
            if runner == "host":
                conf, res = seg.run_host([img], [gt])
            else:
                res = []
                seg.run_resident([seg.stage(img, gt, index=0)], results=res)
                conf = seg.conf.cpu().numpy()
            got[name] = (conf, res[0])
        assert torch.equal(got["hot"][1]["labels"], want["labels"]), runner
        assert torch.equal(got["hot"][1]["confidence"], want["confidence"]), runner
        assert torch.equal(got["plain"][1]["labels"], want1["labels"]), runner
        assert np.array_equal(got["plain"][0], got["one"][0]), runner
        for k in ("labels", "confidence", "pred_full", "pred_rgb", "confidence_full"):
            assert torch.equal(got["plain"][1][k], got["one"][1][k]), (runner, k)


def test_multiscale_members_are_tempered(ops, palettes):
    from pylc_b200.pipeline import TiledSegmenter
    model = _tiny_model()
    W, H = 2400, 1800
    img = orc.synth_image(43, W, H, 3)
    gt = orc.synth_mask(43, W, H, palettes["a"], skew=True)
    seg = TiledSegmenter(model, batch_tiles=8, keep_masks=True, stitch="mean", confidence=True, scales=(0.75, 1.0),
                         temperature=0.7)
    f = seg.stage_device(img, gt, index=0)
    torch.cuda.current_stream().wait_event(f.ready)
    planes = seg.member_probs(f)
    _, direct = _direct(ops, seg, img, 0.7)
    assert torch.equal(planes[1], direct["probs"])           # the 1.0 member is the tempered single-scale stitch
    want = ops.multiscale_combine(planes, W, H)
    _, res = seg.run_host([img], [gt])
    assert torch.equal(res[0]["labels"], want["labels"]) and torch.equal(res[0]["confidence"], want["confidence"])


def test_pipeline_refuses_temperature_without_mean_stitch():
    from pylc_b200.pipeline import TiledSegmenter
    model = _tiny_model()
    with pytest.raises(ValueError, match="mean"):
        TiledSegmenter(model, temperature=2.0)
    with pytest.raises(ValueError):
        TiledSegmenter(model, stitch="mean", temperature=0.0)
    TiledSegmenter(model, temperature=1.0)                    # T = 1 is today's reference stitch


# ---- 7. command line -----------------------------------------------------------------------------------------------

def _run(cwd, *argv):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    return subprocess.run([sys.executable, "-m", "pylc_b200.pylc"] + list(argv), cwd=str(cwd), env=env,
                          capture_output=True, text=True, timeout=900, stdin=subprocess.DEVNULL)


def _cli(cwd, *argv):
    out = _run(cwd, *argv)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    return out.stdout


def _tree(root, sub):
    out = {}
    for p in sorted(glob.glob(os.path.join(root, sub, "*"))):
        with open(p, "rb") as f:
            out[os.path.basename(p)] = f.read()
    return out


def test_cli_calibrate_and_test(tmp_path, palettes, monkeypatch):
    from pylc_b200.config import Parameters
    from pylc_b200.models.deeplab import DeepLab
    pal = palettes["a"]
    C = len(pal)
    torch.manual_seed(0)
    net = DeepLab(n_classes=C, in_channels=1)
    m = Parameters()
    m.update({"ch": 1, "arch": "deeplab", "backbone": "resnet", "pretrained": False, "px_mean": [120.0], "px_std": [40.0],
              "weights": [1.0] * C, "normalize_default": False, "id": "cal_model"})
    model_file = str(tmp_path / "cal_model.pth")
    torch.save({"model": net.state_dict(), "optim": None, "meta": m}, model_file)
    for sub in ("imgs", "masks"):
        os.makedirs(tmp_path / sub)
    W, H = 1600, 1200
    for k in range(2):
        assert cv2.imwrite(str(tmp_path / "imgs" / ("s%d.tif" % k)), orc.synth_image(20 + k, W, H, 1))
        assert cv2.imwrite(str(tmp_path / "masks" / ("s%d.png" % k)),
                           np.ascontiguousarray(orc.synth_mask(20 + k, W, H, pal)[..., ::-1]))
    # a budget below one image: exit 2 with the count, nothing written
    os.makedirs(tmp_path / "tiny")
    out = _run(tmp_path / "tiny", "calibrate", "-l", model_file, "-i", str(tmp_path / "imgs"), "-m",
               str(tmp_path / "masks"), "-o", str(tmp_path / "never.pth"), "--max_resident_gb", "0.001")
    assert out.returncode == 2 and "0 image(s) fit" in out.stderr
    assert not os.path.exists(tmp_path / "never.pth")
    assert not glob.glob(str(tmp_path / "tiny" / "data" / "outputs" / "*" / "metrics" / "*"))
    # the fit: a calibrated copy next to the model and the fit report
    os.makedirs(tmp_path / "cal")
    _cli(tmp_path / "cal", "calibrate", "-l", model_file, "-i", str(tmp_path / "imgs"), "-m", str(tmp_path / "masks"))
    copy = str(tmp_path / "cal_model_calibrated.pth")
    assert os.path.isfile(copy)
    rep = json.load(open(glob.glob(str(tmp_path / "cal" / "data" / "outputs" / "*" / "metrics" /
                                       "calibration_fit.json"))[0]))
    T = rep["temperature"]
    assert 0.05 <= T <= 20 and rep["before"]["nll"] >= rep["after"]["nll"]
    assert len(rep["evaluations"]) > 25 and rep["evaluations"][12][0] == 1.0
    for blk in ("before", "after"):
        assert set(rep[blk]) >= {"nll", "brier", "accuracy", "ece", "mce"}
    from pylc_b200.models.model import _load_model_file
    cal = _load_model_file(copy, "cpu")["calibration"]
    assert cal["temperature"] == T and cal["n_images"] == 2 and cal["n_px"] == 2 * W * H
    assert cal["nll_before"] == rep["before"]["nll"] and cal["nll_after"] == rep["after"]["nll"]
    # pylc test with the copy: the stored temperature applies to the mean stitch and is recorded
    runs = {}
    for name, model, extra in (("plain", model_file, []), ("copy", copy, []), ("copy_t1", copy, ["--temperature", "1"])):
        os.makedirs(tmp_path / name)
        _cli(tmp_path / name, "test", "--model", model, "--img", str(tmp_path / "imgs"), "--mask", str(tmp_path / "masks"),
             "--stitch", "mean", "--save_confidence", *extra)
        runs[name] = glob.glob(str(tmp_path / name / "data" / "outputs" / "*"))[0]
    evs = sorted(glob.glob(os.path.join(runs["copy"], "metrics", "*_eval.json")))
    assert evs and all(json.load(open(p))["temperature"] == T for p in evs)
    assert all("temperature" not in json.load(open(p))
               for p in glob.glob(os.path.join(runs["copy_t1"], "metrics", "*_eval.json")))
    # --temperature 1 turns it off: masks and confidence byte for byte those of the uncalibrated model
    for sub in ("masks", "confidence"):
        a, b = _tree(runs["plain"], sub), _tree(runs["copy_t1"], sub)
        assert a and a == b, sub
    # the calibrated run's masks are a TiledSegmenter(temperature=T*) run of the same images
    from pylc_b200.models.model import Model
    from pylc_b200.pipeline import TiledSegmenter
    from pylc_b200.utils import tools
    monkeypatch.chdir(tmp_path / "copy")
    model = Model().load(copy)
    model.net.eval()
    assert model.calibration["temperature"] == T
    seg = TiledSegmenter(model, batch_tiles=32, keep_masks=True, stitch="mean", temperature=T)
    for k in range(2):
        img = tools.get_image(str(tmp_path / "imgs" / ("s%d.tif" % k)), 1)[0]
        _, res = seg.run_host([img])
        png = glob.glob(os.path.join(runs["copy"], "masks", "s%d*.png" % k))[0]
        rgb = cv2.cvtColor(cv2.imread(png, cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
        assert np.array_equal(rgb, res[0]["pred_rgb"].cpu().numpy()), k
    # a calibrated model with the reference stitch says the temperature is not applied
    os.makedirs(tmp_path / "ref")
    out = _cli(tmp_path / "ref", "test", "--model", copy, "--img", str(tmp_path / "imgs" / "s0.tif"))
    assert "not applied" in out
