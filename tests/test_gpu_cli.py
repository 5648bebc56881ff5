"""CLI-level run of BASELINE.json configs[0] on the GPU: `pylc extract` -> `pylc profile --db` -> `pylc test
--mask` on one synthetic 2000x1500 grayscale image / RGB mask written to disk, schema_a, random-init
DeepLabv3+/ResNet-101 model file (reference pylc.py:19-40, preprocess.py:21-51, test.py:23-115).
Every sub-command runs as its own process, exactly as a user would start it; what they write (tile
database + metadata, predicted mask PNG, *_eval.json, *_cmap.npy) is compared with the oracle's port
of the reference's functions."""
import glob
import json
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest
import torch

import pylc_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T = 512


def _cli(cwd, *argv):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-m", "pylc_b200.pylc"] + list(argv), cwd=str(cwd), env=env,
                         capture_output=True, text=True, timeout=900, stdin=subprocess.DEVNULL)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    return out.stdout


def test_cli_extract_profile_test_on_files(tmp_path, palettes, monkeypatch):
    pal = palettes["a"]
    C = len(pal)
    W, H = 2000, 1500
    img = orc.synth_image(0, W, H, 1)
    mask = orc.synth_mask(0, W, H, pal)
    os.makedirs(tmp_path / "imgs")
    os.makedirs(tmp_path / "masks")
    os.makedirs(tmp_path / "db")
    assert cv2.imwrite(str(tmp_path / "imgs" / "scene.tif"), img)
    assert cv2.imwrite(str(tmp_path / "masks" / "scene.png"), np.ascontiguousarray(mask[..., ::-1]))

    # ---- pylc extract: decode (get_image) -> tiles + encoded masks + profile -> database file --------
    _cli(tmp_path, "extract", "--ch", "1", "--img", "imgs", "--mask", "masks", "--output", "db")
    dbs = glob.glob(str(tmp_path / "db" / "*.npz")) + glob.glob(str(tmp_path / "db" / "*.h5"))
    assert len(dbs) == 1
    from pylc_b200.db.dataset import DB
    data = DB._read(dbs[0])
    want_img = orc.split_tiles(img, T, T)                       # extract.py:279-310, stride = tile size
    want_mask = orc.class_encode(orc.split_tiles(mask, T, T), pal)
    got_img, got_mask = np.asarray(data["img"]), np.asarray(data["mask"])
    assert got_img.shape == want_img.shape and got_mask.shape == want_mask.shape
    # coshuffle (tools.py:361-385) applies ONE unseeded permutation to both arrays: compare as pairs
    key = lambda a, b: (a.tobytes(), b.tobytes())               # noqa: E731
    assert sorted(key(a, b) for a, b in zip(got_img, got_mask)) == sorted(key(a, b) for a, b in zip(want_img, want_mask))
    meta = data["meta"]
    ref = orc.profile_port(want_img, want_mask, C, T)
    assert meta.n_samples == 6 and meta.ch == 1 and meta.n_classes == C
    assert meta.dset_px_dist == [int(v) for v in ref["dset_px_dist"]]
    assert sorted(map(tuple, meta.px_dist)) == sorted(map(tuple, np.asarray(ref["px_dist"]).tolist()))
    assert np.allclose(meta.probs, ref["probs"], rtol=0, atol=0) and np.allclose(meta.weights, ref["weights"], rtol=0, atol=0)
    assert np.allclose(meta.px_mean, ref["px_mean"], rtol=1e-5) and np.allclose(meta.px_std, ref["px_std"], rtol=1e-5)
    assert meta.m2 == ref["m2"] and meta.jsd == ref["jsd"]

    # ---- pylc profile --db: re-profiles the stored tiles (what README.md:161-167 documents) ----------
    out = _cli(tmp_path, "profile", "--db", dbs[0])
    assert "Profile Metadata" in out and "{:30s} {}".format("Samples", 6) in out
    assert "{:30s} {}".format("Dataset pixel count", 6 * T * T) in out

    # ---- a random-init model file in the reference's format (checkpoint.py:53-66) -------------------
    from pylc_b200.config import Parameters
    from pylc_b200.models.deeplab import DeepLab
    torch.manual_seed(0)
    net = DeepLab(n_classes=C, in_channels=1)
    m = Parameters()
    m.update({"ch": 1, "arch": "deeplab", "backbone": "resnet", "pretrained": False, "px_mean": meta.px_mean,
              "px_std": meta.px_std, "weights": meta.weights, "normalize_default": False, "id": "cli_model"})
    os.makedirs(tmp_path / "models")
    model_file = str(tmp_path / "models" / "cli_model.pth")
    torch.save({"model": net.state_dict(), "optim": None, "meta": m}, model_file)

    # ---- pylc test --mask: fit -> tiles -> network -> stitch -> resample -> metrics, files written ------
    _cli(tmp_path, "test", "--model", model_file, "--img", "imgs/scene.tif", "--mask", "masks/scene.png", "--save_logits")
    out_root = glob.glob(str(tmp_path / "data" / "outputs" / "*"))
    assert len(out_root) == 1
    png = glob.glob(os.path.join(out_root[0], "masks", "*.png"))
    ev = glob.glob(os.path.join(out_root[0], "metrics", "*_eval.json"))
    cm = glob.glob(os.path.join(out_root[0], "metrics", "*_cmap.npy"))
    lg = glob.glob(os.path.join(out_root[0], "logits", "*_output.pth"))
    assert len(png) == len(ev) == len(cm) == len(lg) == 1
    # the label map the run stitched (fitted resolution 1536x1024), then the reference's tail in the oracle:
    labels = torch.load(lg[0], weights_only=False)["results"][0].numpy()
    w_fit, h_fit = orc.fit_dims(W, H, T)
    assert labels.shape == (h_fit, w_fit) and labels.max() < C
    pred_full = orc.resample_labels(labels, W, H)                      # tools.py:316-317
    rgb = cv2.cvtColor(cv2.imread(png[0], cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
    assert np.array_equal(rgb, np.asarray(pal, dtype=np.uint8)[pred_full])   # tools.py:312-313 colourize
    decoded_mask = cv2.cvtColor(cv2.imread(str(tmp_path / "masks" / "scene.png"), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
    yt, yp = orc.inject_coverage(orc.class_encode_hwc(decoded_mask, pal), pred_full, C)   # evaluate.py:103-108,172-174
    want = orc.metrics_port(yt, yp, Parameters().class_codes)          # metrics.py:45-87 (scikit-learn)
    with open(ev[0]) as f:
        got = json.load(f)
    assert got["f1"] == want["f1"] and got["iou"] == want["iou"] and got["mcc"] == want["mcc"]
    assert np.array_equal(np.load(cm[0]), want["cmatrix"])
    # and the label map itself is the reference's reconstruct of THIS network's logits (near-ties aside)
    from pylc_b200.models.model import Model
    monkeypatch.chdir(tmp_path)                                        # Model creates ./data/save/<id>, as the CLI did
    model = Model().load(model_file)
    model.net.eval()                                                   # test.py:41
    fitted = cv2.resize(img, (w_fit, h_fit), interpolation=cv2.INTER_AREA)
    tiles = torch.from_numpy(orc.split_tiles(fitted, T, T // 2))
    logits = torch.cat([model.test(tiles[i:i + 8])[0] for i in range(0, len(tiles), 8)]).cpu().numpy()
    ref_map = orc.stitch_map(logits, h_fit // 256 - 1, w_fit // 256 - 1, T, 256)
    ref_lab = orc.stitch_labels(ref_map)
    # the CLI ran the network in its own process with another batch size: TF32 convolution noise (~1e-3 of
    # the logit scale) moves near-ties, so compare outside a margin of that size
    clear = orc.top2_margin(ref_map) > 2e-2
    assert clear.mean() > 0.5
    assert (labels[clear] == ref_lab[clear]).mean() > 0.999


def test_cli_augment_on_database(tmp_path, palettes):
    """`pylc augment --db` (reference preprocess.py:54-74, utils/argparse.py:91-106): sample-rate search, over-sampling
    and re-profiling of a tile database written by the extractor; the `_aug<id>` database it writes holds the input
    tiles plus the warped copies Augmentor.oversample produces in-process for the same rates."""
    from pylc_b200.config import Parameters
    from pylc_b200.db.dataset import DB
    from pylc_b200.utils.augment import Augmentor
    from pylc_b200.utils.extract import Extractor
    pal = palettes["a"]
    meta = Parameters()
    meta.update({"ch": 1})
    os.makedirs(tmp_path / "db")
    meta.output_dir = str(tmp_path / "db")
    imgs = [orc.synth_image(30 + i, 1100, 1100, 1) for i in range(4)]
    masks = [orc.synth_mask(30 + i, 1100, 1100, pal, skew=True) for i in range(4)]
    ex = Extractor(meta)
    ex.verbose = False
    db_path = ex.load_arrays(imgs, masks).extract().profile().get_data().save()
    n_in = 16

    out = _cli(tmp_path, "augment", "--db", db_path)
    assert "Augmentation Results" in out and "Augmentation done" in out
    aug_files = [p for p in glob.glob(str(tmp_path / "db" / "_aug*")) if p != db_path]
    assert len(aug_files) == 1
    got = DB._read(aug_files[0])

    want = Augmentor().load(db_path)
    want.optimize().oversample(shuffle=False)
    n_out = n_in + int(np.sum(want.rates))
    assert got["img"].shape == (n_out, 1, T, T) and got["mask"].shape == (n_out, T, T)
    key = lambda a, b: (a.tobytes(), b.tobytes())               # noqa: E731  (the CLI shuffles: compare as pairs)
    assert sorted(key(a, b) for a, b in zip(got["img"], got["mask"])) == \
        sorted(key(a, b) for a, b in zip(want.output_imgs, want.output_masks))
    m = got["meta"]
    assert m.n_samples == n_out and m.id == "_aug" + str(want.input_meta.id)
    assert m.dset_px_dist == np.bincount(np.asarray(got["mask"]).ravel(), minlength=len(pal)).tolist()
