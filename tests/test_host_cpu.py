"""CPU-side tests of the host logic: metrics from one confusion matrix vs scikit-learn, the tile
dataset, geometry helpers, config/schema handling and the data-parallel plumbing (gloo, 2 ranks).
No CUDA kernel is executed here."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import pylc_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- metrics --------------------------------------------------------------------------------

@pytest.mark.parametrize("C,seed,missing", [(9, 0, None), (11, 1, None), (9, 2, 4), (3, 3, None)])
def test_scores_from_confusion_equal_sklearn(C, seed, missing):
    from pylc_b200.utils.metrics import scores_from_confusion
    rng = np.random.default_rng(seed)
    yt = rng.integers(0, C, 50000).astype(np.uint8)
    yp = np.where(rng.random(50000) < 0.7, yt, rng.integers(0, C, 50000)).astype(np.uint8)
    if missing is not None:                       # a class present in neither vector is dropped (unique_labels)
        yt[yt == missing] = 0
        yp[yp == missing] = 0
    labels = ["c%d" % i for i in range(C)]
    present = sorted(set(yt.tolist()) | set(yp.tolist()))
    want = orc.metrics_port(yt, yp, [labels[i] for i in present])
    got = scores_from_confusion(orc.confusion_counts(yt, yp, C), labels)
    assert got["f1"] == want["f1"] and got["iou"] == want["iou"] and got["mcc"] == want["mcc"]
    assert np.array_equal(got["cmatrix"], want["cmatrix"])
    assert got["report"] == want["report"]


def test_metrics_object_from_counts():
    from pylc_b200.utils.metrics import Metrics, format_report
    M = np.array([[5, 1, 0], [2, 7, 1], [0, 0, 4]])
    m = Metrics().set_counts(M, ["a", "b", "c"])
    m.f1_score(None, None)
    m.jaccard(None, None)
    m.mcc(None, None)
    m.confusion_matrix(None, None, labels=["a", "b", "c"])
    m.report(None, None, labels=["a", "b", "c"])
    assert set(m.results) == {"f1", "iou", "mcc", "report"}
    assert np.allclose(m.cmatrix.sum(axis=1), 1.0)
    assert "weighted avg" in format_report(m.results["report"])
    json.dumps(m.results)                          # what save_metrics writes


def test_jsd_m2_match_oracle():
    from pylc_b200.utils.metrics import jsd, m2
    p = np.array([0.55, 0.0, 0.22, 0.08, 0.1, 0.001, 0.001, 0.035, 0.013])
    q = np.full(9, 1 / 9)
    assert jsd(p, q) == orc.jsd(p, q) and m2(p, 9) == orc.m2(p, 9)
    with pytest.raises(AssertionError):
        m2(p, 1)


# ---- geometry / host tools -------------------------------------------------------------------

def test_fit_dims_and_nn_maps_match_reference_golden(golden):
    """tests/golden/fit.npz was produced by the reference's adjust_to_tile / cv2.resize."""
    from pylc_b200.ops import nn_index_map
    from pylc_b200.utils import tools
    g = golden("fit")
    for W, H, w_fit, h_fit, off in g["fit_dims"]:
        assert tools.fit_dims(int(W), int(H), 512) == (w_fit, h_fit) and off == 0
    for n_src, n_dst in g["nn_pairs"]:
        assert np.array_equal(nn_index_map(int(n_src), int(n_dst)), g["nn_map_%d_%d" % (n_src, n_dst)])
    img = orc.synth_image(0, 1300, 900, 3)
    out, w, h, off = tools.adjust_to_tile(img, 512, 256, 3)
    assert (w, h, off) == (1024, 512, 0) and out.shape == (512, 1024, 3)
    with pytest.raises(AssertionError):
        tools.adjust_to_tile(np.zeros((600, 600), np.uint8), 512, 300, 1)


def test_colourize_lut_follows_sequential_passes(palettes):
    from pylc_b200.utils.tools import colourize_lut
    for pal in palettes.values():
        assert colourize_lut(len(pal), pal) == [list(c) for c in pal]
    chain = [[2, 2, 2], [9, 9, 9], [7, 7, 7]]       # label 0 -> grey 2 -> re-mapped by pass 2
    assert colourize_lut(3, chain) == orc.colourize_lut(3, chain).tolist() == [[7, 7, 7], [9, 9, 9], [7, 7, 7]]


def test_nn_index_map_equals_opencv():
    import cv2
    from pylc_b200.ops import nn_index_map
    for n_src, n_dst in [(2560, 3000), (1536, 2000), (5632, 6000), (1024, 1500), (512, 512), (1536, 1100)]:
        ramp = np.arange(n_src, dtype=np.float32)[None, :]
        want = cv2.resize(ramp, (n_dst, 1), interpolation=cv2.INTER_NEAREST)[0].astype(np.int32)
        assert np.array_equal(nn_index_map(n_src, n_dst), want)


def test_collate_pairs_by_basename(tmp_path):
    from pylc_b200.utils import tools
    (tmp_path / "img").mkdir()
    (tmp_path / "mask").mkdir()
    for n in ("b", "a"):
        (tmp_path / "img" / (n + ".tif")).write_bytes(b"x")
        (tmp_path / "mask" / (n + ".png")).write_bytes(b"x")
    files = tools.collate(str(tmp_path / "img"), str(tmp_path / "mask"))
    assert [os.path.basename(f["img"]) for f in files] == ["a.tif", "b.tif"]
    assert all(os.path.basename(f["mask"])[0] == os.path.basename(f["img"])[0] for f in files)
    (tmp_path / "mask" / "c.png").write_bytes(b"x")
    with pytest.raises(SystemExit):
        tools.collate(str(tmp_path / "img"), str(tmp_path / "mask"))


# ---- config / dataset ------------------------------------------------------------------------

def test_get_image_decodes_files_like_the_reference(tmp_path, palettes):
    """tools.get_image (reference tools.py:77-148) on real files: gray .tif, colour .png mask; channel order,
    the grayscale check of colour requests, and the scale rule (INTER_AREA image / INTER_NEAREST mask)."""
    import cv2
    from pylc_b200.utils import tools
    gray = orc.synth_image(3, 700, 600, 1)
    mask = orc.synth_mask(3, 700, 600, palettes["a"])
    cv2.imwrite(str(tmp_path / "g.tif"), gray)
    cv2.imwrite(str(tmp_path / "m.png"), cv2.cvtColor(mask, cv2.COLOR_RGB2BGR))
    img, w, h, ws, hs = tools.get_image(str(tmp_path / "g.tif"), 1)
    assert (w, h, ws, hs) == (700, 600, 700, 600) and np.array_equal(img, gray)
    m, w, h, ws, hs = tools.get_image(str(tmp_path / "m.png"), 3, interpolate=cv2.INTER_NEAREST)
    assert np.array_equal(m, mask)                                   # RGB order restored
    with pytest.raises(SystemExit):                                   # a gray file asked for as colour stops
        tools.get_image(str(tmp_path / "g.tif"), 3)
    img2, w, h, ws, hs = tools.get_image(str(tmp_path / "g.tif"), 1, scale=0.5)
    assert np.array_equal(img2, cv2.resize(gray, (ws, hs), interpolation=cv2.INTER_AREA)) and (w, h) == (700, 600)


def test_ordered_prefetch_keeps_order_and_surfaces_errors(tmp_path):
    """The decode look-ahead of the file loops (Extractor.extract, pylc test): results in item order whatever
    the completion order, bounded look-ahead, worker exceptions / exit(1) raised at the item's position."""
    import threading
    import time
    import cv2
    from pylc_b200.utils import tools
    started = []
    lock = threading.Lock()

    def slow(i):
        with lock:
            started.append(i)
        time.sleep(0.02 * ((7 - i) % 4))                              # later items finish first
        return i * i

    for workers in (0, 1, 4):
        assert list(tools.ordered_prefetch(slow, range(12), workers=workers)) == [i * i for i in range(12)]
    assert list(tools.ordered_prefetch(slow, [], workers=4)) == []
    # bounded look-ahead: after taking the first result at most depth + 1 items have been started
    del started[:]
    gen = tools.ordered_prefetch(slow, range(40), workers=2, depth=3)
    assert next(gen) == 0
    with lock:
        assert len(started) <= 5
    gen.close()

    def boom(i):
        if i == 3:
            exit(1)                                                   # the reference's error convention
        if i == 5:
            raise ValueError("bad file")
        return i

    got = []
    with pytest.raises(SystemExit):
        for v in tools.ordered_prefetch(boom, range(8), workers=4):
            got.append(v)
    assert got == [0, 1, 2]
    # real files decode identically through the look-ahead
    imgs = [orc.synth_image(10 + i, 320, 240, 1) for i in range(6)]
    for i, im in enumerate(imgs):
        cv2.imwrite(str(tmp_path / ("f%d.png" % i)), im)
    out = list(tools.ordered_prefetch(lambda i: tools.get_image(str(tmp_path / ("f%d.png" % i)), 1)[0], range(6), workers=3))
    assert all(np.array_equal(a, b) for a, b in zip(out, imgs))


def test_extractor_stack_grouping_host_logic(monkeypatch, palettes):
    """Host logic of Extractor.extract without a GPU: the device entry points are replaced by oracle stand-ins that
    record their calls, so what is checked is the grouping of consecutive equally sized files into stacks
    (STACK_MAX, size changes, images without masks), the file order of the tiles and the `meta.extract` record
    (reference utils/extract.py:132-222)."""
    from pylc_b200 import ops
    from pylc_b200.config import Parameters
    from pylc_b200.utils import extract as ex_mod
    from pylc_b200.utils import tools
    calls = []

    def upload_stack(images, device=None, staging=None):
        a = np.stack([np.asarray(im).reshape(im.shape[0], -1) for im in images])
        return torch.from_numpy(a), a.shape[2], None

    def tile_gather_u8_stack(src, H, W, ch, pitch, T, S, stats=False, out=None, stat_out=None):
        calls.append(("img", src.shape[0], H, W))
        tiles = np.concatenate([orc.split_tiles(im.numpy().reshape((H, W) if ch == 1 else (H, W, ch)), T, S) for im in src])
        x = tiles.astype(np.int64).reshape(tiles.shape[0], ch, -1)
        stat = torch.from_numpy(np.stack([x.sum(-1), (x * x).sum(-1)], axis=-1))
        return (torch.from_numpy(tiles), stat) if stats else torch.from_numpy(tiles)

    def mask_gather_encode_hist_stack(src, H, W, pitch, T, S, palette, hist=True, out=None, px_dist=None):
        calls.append(("mask", src.shape[0], H, W))
        enc = np.concatenate([orc.class_encode(orc.split_tiles(m.numpy().reshape(H, W, 3), T, S), palette) for m in src])
        return torch.from_numpy(enc), torch.from_numpy(orc.tile_histograms(enc, len(palette)))

    monkeypatch.setattr(ops, "upload_stack", upload_stack)
    monkeypatch.setattr(ops, "tile_gather_u8_stack", tile_gather_u8_stack)
    monkeypatch.setattr(ops, "mask_gather_encode_hist_stack", mask_gather_encode_hist_stack)
    monkeypatch.setattr(ops, "tile_grid", lambda H, W, T, S: ((H - T) // S + 1 if H >= T else 0, (W - T) // S + 1 if W >= T else 0))
    monkeypatch.setattr(tools, "_device", lambda: torch.device("cpu"))
    monkeypatch.setenv("PYLC_DECODE_THREADS", "3")

    pal = palettes["a"]
    meta = Parameters()
    meta.update({"ch": 1})
    T = meta.tile_size
    sizes = [(1100, 1050)] * 5 + [(1050, 1100)] + [(1100, 1050)] * 2
    imgs = [orc.synth_image(70 + i, w, h, 1) for i, (w, h) in enumerate(sizes)]
    masks = [orc.synth_mask(70 + i, w, h, pal) for i, (w, h) in enumerate(sizes)]
    ex = ex_mod.Extractor(meta)
    ex.verbose = False
    ex.STACK_MAX = 3
    ex.load_arrays(imgs, masks).extract()
    # runs: 5 equal (3 + 2 by STACK_MAX) | 1 odd | 2 equal ; one image and one mask call per stack
    assert [c[1] for c in calls if c[0] == "img"] == [3, 2, 1, 2]
    assert [c[1] for c in calls if c[0] == "mask"] == [3, 2, 1, 2]
    ref_i = np.concatenate([orc.split_tiles(im, T, T) for im in imgs])
    ref_m = np.concatenate([orc.class_encode(orc.split_tiles(m, T, T), pal) for m in masks])
    got_i, got_m = ex.host()
    assert np.array_equal(got_i, ref_i) and np.array_equal(got_m, ref_m)          # file order kept across stacks
    e = ex.get_meta().extract
    assert (e["n"], e["w_full"], e["h_full"], e["w_fitted"], e["h_fitted"], e["offset"]) == (4, 1100, 1050, 1100, 1050, 0)
    assert ex.get_meta().n_tiles == len(ref_i) == 32 and ex.mask_idx == 32
    ex.profile()                                                                  # from the kernels' by-products
    want = orc.profile_port(ref_i, ref_m, len(pal), T)
    assert np.array_equal(np.array(ex.get_meta().px_dist), want["px_dist"])
    np.testing.assert_allclose(ex.get_meta().px_mean, want["px_mean"], rtol=1e-5)
    np.testing.assert_allclose(ex.get_meta().px_std, want["px_std"], rtol=1e-5)
    # images only: no mask calls, a zero mask buffer of matching length (extract.py:96-102)
    del calls[:]
    ex.load_arrays(imgs[:4]).extract()
    assert [c[0] for c in calls] == ["img", "img"] and [c[1] for c in calls] == [3, 1]
    assert ex.masks.shape[0] == ex.imgs.shape[0] == 16 and int(ex.masks.sum()) == 0


def test_cli_parser_accepts_reference_command_lines():
    """The sub-commands and flags of the reference parser (utils/argparse.py:40-335) for the path: every form a PyLC
    user types parses here to the same destinations."""
    from pylc_b200.pylc import get_parser
    p = get_parser()
    a = p.parse_args("extract --ch 3 --img ./imgs --mask ./masks".split())
    assert (a.action, a.ch, a.img, a.mask) == ("extract", 3, "./imgs", "./masks")
    a = p.parse_args("extract --ch 1 -i ./imgs".split())                  # masks are optional (argparse.py:60-66)
    assert a.mask is None and a.ch == 1
    a = p.parse_args("augment --db data/db/x.h5".split())
    assert a.action == "augment" and a.db == "data/db/x.h5"
    a = p.parse_args("profile --db data/db/x.h5".split())
    assert a.action == "profile"
    a = p.parse_args(("train --db x.h5 --arch deeplab --backbone resnet --weighted --pretrained --resume --normalize batch "
                      "--activation relu --up_mode upsample --optim adam --sched step_lr --lr 0.001 --batch_size 8 --n_epochs 2 "
                      "--n_workers 0 --report 10 --clip 0.5 --ce_weight 0.5 --dice_weight 0.3 --focal_weight 0.2").split())
    assert a.weighted is True and a.pretrained is True and a.resume is True and a.clip == 0.5
    a = p.parse_args("train --db x.h5 --weighted True --pretrained ./w.pth".split())   # value forms
    assert a.weighted == "True" and a.pretrained == "./w.pth"
    a = p.parse_args("train --db x.h5".split())
    assert a.weighted is None and a.pretrained is None and not a.resume
    a = p.parse_args("test -l m.pth -i img.tif -m mask.png --scale 0.5 --save_logits --aggregate_metrics".split())
    assert (a.model, a.img, a.mask, a.scale, a.save_logits, a.aggregate_metrics) == ("m.pth", "img.tif", "mask.png", 0.5, True, True)
    with pytest.raises(SystemExit):
        p.parse_args("extract --ch 2 --img x".split())                    # ch in {1, 3}


def _live_golden():
    """What the *_live tests compare, recorded by oracle/gen_live_golden.py."""
    with open(os.path.join(ROOT, "tests", "golden", "host_live.json")) as f:
        return json.load(f)


def test_cli_parser_covers_reference_options_live():
    """Every option of the reference's extract / augment / train / test sub-parsers exists here with the same destination
    and choices: against tests/golden/host_live.json, and against the reference's parser when it is present (merge /
    grayscale are stubs in the reference and are not provided)."""
    import argparse
    import importlib
    import ref_harness
    import host_record as hr
    from pylc_b200.pylc import get_parser as our_parser
    stored, ours_rec = _live_golden()["parser"], hr.record_parser(our_parser())      # tests/golden/host_live.json
    assert set(stored["commands"]) <= set(ours_rec["commands"])
    for cmd in ("extract", "augment", "train", "test"):
        for opts, want in stored[cmd].items():
            assert ours_rec[cmd].get(opts) == want, (cmd, opts)
    if not ref_harness.available():
        return
    ref_harness.load()
    sys.path.insert(0, ref_harness.REF_ROOT)
    try:
        ref_parser = importlib.import_module("utils.argparse").get_parser()
    finally:
        sys.path.remove(ref_harness.REF_ROOT)
    from pylc_b200.pylc import get_parser

    def subs(parser):
        for act in parser._actions:
            if isinstance(act, argparse._SubParsersAction):
                return {name: {tuple(x.option_strings): x for x in sp._actions if x.option_strings and x.dest != "help"}
                        for name, sp in act.choices.items()}
        return {}
    ref, ours = subs(ref_parser), subs(get_parser())
    assert set(ref) - set(ours) == {"merge", "grayscale"}
    for cmd in ("extract", "augment", "train", "test"):
        for opts, act in ref[cmd].items():
            assert opts in ours[cmd], (cmd, opts)
            mine = ours[cmd][opts]
            assert mine.dest == act.dest and mine.choices == act.choices, (cmd, opts)
            if act.default is not None and act.type is not None:          # typed defaults are the reference's
                assert mine.default == act.default, (cmd, opts, mine.default, act.default)


def test_python_surface_covers_reference_live():
    """SURVEY.md section 8b, against tests/golden/host_live.json and, when present, the reference: every public method of the reference's path classes and every
    function of its path modules exists here under the same module path and name, with the reference's leading
    parameters (extra trailing parameters with defaults are extensions).  Omissions are listed, with the reason."""
    import importlib
    import inspect
    import ref_harness
    import host_record as hr
    stored, ours_rec = _live_golden()["surface"], hr.record_surface(hr.package_modules())   # tests/golden/host_live.json
    for owner, members in stored.items():
        for n, params in members.items():
            assert n in ours_rec[owner] and ours_rec[owner][n][:len(params)] == params, (owner, n)
    if not ref_harness.available():
        return
    ref_harness.load()
    omitted = {
        ("Evaluator", "save_tex"): "LaTeX table helper (analysis, SURVEY.md section 2: out of scope)",
        ("Augmentor", "grayscale"): "bare stub in the reference (augment.py)",
        ("Augmentor", "merge_dbs"): "body commented out in the reference (augment.py:241-300)",
    }
    classes = [("utils.extract", "Extractor"), ("utils.evaluate", "Evaluator"), ("models.modules.loss", "MultiLoss"),
               ("models.modules.loss", "RunningLoss"), ("models.modules.checkpoint", "Checkpoint"), ("models.model", "Model"),
               ("db.dataset", "MLPDataset"), ("utils.metrics", "Metrics"), ("utils.augment", "Augmentor"), ("config", "Parameters")]
    modules = ["utils.tools", "utils.profile", "utils.metrics"]

    def names(fn):
        return [p.name for p in inspect.signature(fn).parameters.values()]

    def ref_import(name):
        sys.path.insert(0, ref_harness.REF_ROOT)
        try:
            return importlib.import_module(name)
        finally:
            sys.path.remove(ref_harness.REF_ROOT)
    problems = []
    for mod, cls in classes:
        R = getattr(ref_import(mod), cls)
        O = getattr(importlib.import_module("pylc_b200." + mod), cls)
        mine = dict(inspect.getmembers(O, inspect.isfunction))
        for n, f in inspect.getmembers(R, inspect.isfunction):
            if (n.startswith("_") and n != "__init__") or (cls, n) in omitted:
                continue
            if n not in mine:
                problems.append("%s.%s missing" % (cls, n))
            elif names(mine[n])[:len(names(f))] != names(f):
                problems.append("%s.%s%s != reference %s" % (cls, n, names(mine[n]), names(f)))
    for mod in modules:
        R, O = ref_import(mod), importlib.import_module("pylc_b200." + mod)
        for n, f in inspect.getmembers(R, inspect.isfunction):
            if f.__module__ != R.__name__:
                continue
            if not hasattr(O, n):
                problems.append("%s.%s missing" % (mod, n))
            elif names(getattr(O, n))[:len(names(f))] != names(f):
                problems.append("%s.%s%s != reference %s" % (mod, n, names(getattr(O, n)), names(f)))
    assert not problems, problems


@pytest.mark.parametrize("schema", ["schema_a", "schema_b"])
def test_parameters_table_equals_reference_live(schema):
    """`json.dumps(vars(Parameters))` is the metadata record of database and model files (reference database.py:216-235,
    checkpoint.py:53-66): attribute names and default values must be the reference's, key for key."""
    import importlib
    import ref_harness
    import host_record as hr
    from pylc_b200.config import Parameters as OurParameters
    assert hr.record_parameters(OurParameters, schema) == _live_golden()["parameters"][schema]   # tests/golden/host_live.json
    if not ref_harness.available():
        return
    ref_harness.load()
    sys.path.insert(0, ref_harness.REF_ROOT)
    try:
        ref_cfg = importlib.import_module("config")
    finally:
        sys.path.remove(ref_harness.REF_ROOT)
    from pylc_b200.config import Parameters
    import argparse
    # a Namespace, as the CLI passes it: the reference ignores a dict's "schema" key at construction (config.py:108 tests
    # hasattr), which this package accepts as an extension
    args = argparse.Namespace(schema="./schemas/%s.json" % schema)
    want, got = vars(ref_cfg.Parameters(args)), vars(Parameters(args))
    assert set(want) == set(got)
    for k in want:
        if k != "seed":                     # np.random seed of the process, different by construction
            assert want[k] == got[k], k


def _oracle_host_lib():
    """oracle/_build/libpylc_oracle_host.so: the augmentation kernel's per-pixel function compiled for the host."""
    import ctypes
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = os.path.join(root, "oracle", "_build", "libpylc_oracle_host.so")
    if not os.path.isfile(path):
        subprocess.run(["make", "-C", os.path.join(root, "oracle")], check=True, stdout=subprocess.DEVNULL)
    lib = ctypes.CDLL(path)
    fn = lib.pylc_oracle_augment_tiles_host
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 3 + [ctypes.c_int] + [ctypes.c_void_p] * 2
    return fn


def _augment_tiles_host(src_imgs, src_masks, job_src, job_minv, job_shift):
    fn = _oracle_host_lib()
    imgs = np.ascontiguousarray(np.asarray(src_imgs), dtype=np.uint8)
    masks = np.ascontiguousarray(np.asarray(src_masks), dtype=np.uint8)
    src = np.ascontiguousarray(job_src, dtype=np.int32)
    minv = np.ascontiguousarray(np.asarray(job_minv, dtype=np.float64).reshape(-1, 9))
    shift = np.ascontiguousarray(job_shift, dtype=np.int32)
    n, ch, T = imgs.shape[0], imgs.shape[1], imgs.shape[2]
    out_i, out_m = np.zeros((len(src), ch, T, T), np.uint8), np.zeros((len(src), T, T), np.uint8)
    assert fn(imgs.ctypes.data, masks.ctypes.data, n, ch, T, src.ctypes.data, minv.ctypes.data, shift.ctypes.data, len(src),
              out_i.ctypes.data, out_m.ctypes.data) == 0
    return out_i, out_m


@pytest.mark.parametrize("ch", [1, 3])
def test_augment_kernel_arithmetic_on_host_equals_reference_golden(golden, ch):
    """csrc/augment_math.cuh -- the per-pixel function of pylc_augment_tiles_u8 -- compiled for the host: the bytes
    the reference's augment_transform produced (golden warp vectors) and, on noise tiles, the OpenCV chain itself."""
    from pylc_b200.utils import tools
    g = golden("warp")
    img, mask = orc.augment_fixture_tile(ch)
    seeds = [0, 1, 3]
    params = [tools.augment_params(np.random.RandomState(s), 512) for s in seeds]
    out_i, out_m = _augment_tiles_host(img, mask, [0] * 3, np.stack([p[0] for p in params]), [p[1] for p in params])
    for j, s in enumerate(seeds):
        assert np.array_equal(out_i[j].reshape(g["warp_ch%d_s%d_img" % (ch, s)].shape), g["warp_ch%d_s%d_img" % (ch, s)])
        assert np.array_equal(out_m[j], g["warp_ch%d_s%d_mask" % (ch, s)])
    rng = np.random.default_rng(ch)
    img = rng.integers(0, 256, size=(2, ch, 512, 512), dtype=np.uint8)
    mask = rng.integers(0, 11, size=(2, 512, 512)).astype(np.uint8)
    seeds = [2, 5, 8]
    params = [tools.augment_params(np.random.RandomState(s), 512) for s in seeds]
    out_i, out_m = _augment_tiles_host(img, mask, [1, 0, 1], np.stack([p[0] for p in params]), [p[1] for p in params])
    for j, (s, src) in enumerate(zip(seeds, [1, 0, 1])):
        a, b = tools.augment_transform(img[src:src + 1].astype(np.float32), mask[src:src + 1].astype(np.int64), np.random.RandomState(s))
        assert np.array_equal(np.asarray(a).reshape(out_i[j].shape), out_i[j]) and np.array_equal(np.asarray(b), out_m[j])


@pytest.mark.parametrize("T,ch,seed", [(62, 1, 0), (128, 3, 7), (384, 1, 7), (1024, 1, 7)])
def test_augment_kernel_arithmetic_other_tile_sizes(T, ch, seed):
    """The same host-compiled kernel function and the NumPy restatement against the OpenCV chain at other tile sizes.
    The control points are fixed for 512-pixel tiles (tools.py:576), so at 1024 the jitter is a strong perspective whose
    denominator crosses zero inside the tile: coordinates saturate to 16 bits, as OpenCV's remap receives them, and the
    reflect-101 border is applied many times over."""
    from pylc_b200.utils import tools
    rng = np.random.default_rng(T + ch)
    img = rng.integers(0, 256, size=(1, ch, T, T), dtype=np.uint8)
    mask = rng.integers(0, 9, size=(1, T, T)).astype(np.uint8)
    m_inv, shift = tools.augment_params(np.random.RandomState(seed), T)
    out_i, out_m = _augment_tiles_host(img, mask, [0], m_inv[None], [shift])
    a, b = tools.augment_transform(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
    assert np.array_equal(np.asarray(a).reshape(out_i[0].shape), out_i[0]) and np.array_equal(np.asarray(b), out_m[0])
    c, d = orc.augment_transform_port(img.astype(np.float32), mask.astype(np.int64), np.random.RandomState(seed))
    assert np.array_equal(np.asarray(a), c) and np.array_equal(np.asarray(b), d)


def test_oversample_device_plumbing_equals_host_path(monkeypatch):
    """Augmentor.oversample(device=True): job table (RandomState(j) draws per copy), slot order (each original followed
    by its copies) and dtypes -- with the device entry point replaced by its host twin, the result equals the default
    path through the reference's OpenCV calls, array for array (reference utils/augment.py:184-239)."""
    from pylc_b200 import ops
    from pylc_b200.config import Parameters
    from pylc_b200.db.dataset import MLPDataset
    from pylc_b200.utils import profile, tools
    from pylc_b200.utils.augment import Augmentor

    def fake(src_imgs, src_masks, job_src, job_minv, job_shift, out_imgs=None, out_masks=None):
        a, b = _augment_tiles_host(src_imgs.numpy(), src_masks.numpy(), job_src, job_minv, job_shift)
        return torch.from_numpy(a), torch.from_numpy(b)
    monkeypatch.setattr(ops, "augment_tiles", fake)
    monkeypatch.setattr(tools, "_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(profile, "get_profile", lambda dset: dset.get_meta())
    rng = np.random.default_rng(0)
    imgs = rng.integers(0, 256, size=(4, 1, 512, 512), dtype=np.uint8)
    masks = rng.integers(0, 9, size=(4, 512, 512)).astype(np.uint8)
    meta = Parameters()
    meta.update({"ch": 1})
    outs = []
    for device in (False, True):
        aug = Augmentor().load(MLPDataset(input_data={"img": imgs, "mask": masks, "meta": meta}))
        aug.rates = np.array([2, 0, 1, 3])
        aug.oversample(shuffle=False, device=device)
        outs.append((aug.output_imgs, aug.output_masks))
        assert aug.output_imgs.shape == (10, 1, 512, 512) and aug.output_meta.id.startswith("_aug")
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    assert np.array_equal(outs[1][0][[0, 3, 4, 6]], imgs)           # originals at the head of their groups


def test_parameters_schema_b_and_update():
    from pylc_b200.config import Parameters
    p = Parameters({"schema": "./schemas/schema_b.json", "ch": 1})
    assert p.n_classes == 11 and len(p.palette_rgb) == 11 and p.ch_label == "grayscale"
    p.update({"px_mean": np.array([1.0, 2.0]), "not_a_field": 3})
    assert p.px_mean == [1.0, 2.0] and not hasattr(p, "not_a_field")
    assert p.tiles_per_image == 700
    json.dumps({k: v for k, v in vars(p).items()})   # the HDF5 `meta` attribute must stay JSON-serialisable


def test_dataset_partition_iteration_and_npz_roundtrip(tmp_path):
    from pylc_b200.config import Parameters
    from pylc_b200.db.dataset import MLPDataset
    rng = np.random.default_rng(0)
    imgs = rng.integers(0, 256, (10, 1, 16, 16), dtype=np.uint8)
    masks = rng.integers(0, 9, (10, 16, 16), dtype=np.uint8)
    meta = Parameters({"ch": 1})
    meta.id, meta.output_dir = "unit_db", str(tmp_path)
    full = MLPDataset(input_data={"img": imgs, "mask": masks, "meta": meta})
    train = MLPDataset(input_data={"img": imgs, "mask": masks, "meta": meta}, partition=(0, 0.8))
    valid = MLPDataset(input_data={"img": imgs, "mask": masks, "meta": meta}, partition=(0.8, 1.0))
    assert (full.size, train.size, valid.size) == (10, 8, 2)
    items = list(valid)
    assert items[0][0].dtype == torch.float32 and items[0][1].dtype == torch.int64
    assert torch.equal(items[1][1], torch.from_numpy(masks[9]).long())
    loader, n_batches = train.loader(batch_size=4, drop_last=True)
    assert n_batches == 2 and [b[0].shape[0] for b in loader] == [4, 4]
    path = full.save()
    assert path.endswith(".npz") or path.endswith(".h5")
    back = MLPDataset(db_path=path)
    assert np.array_equal(back.get_data("img"), imgs) and np.array_equal(back.get_data("mask"), masks)
    assert back.get_meta().id == "unit_db" and back.get_meta().n_classes == 9


# ---- data-parallel plumbing (gloo, world_size 2) ----------------------------------------------

_WORKER = r"""
import os, sys, json
import numpy as np, torch
sys.path.insert(0, %r)
from pylc_b200 import dist as pdist
rank, world, _ = pdist.init_from_env(backend="gloo")
mine = pdist.shard_indices(7)
rng = np.random.default_rng(0)
conf_all = rng.integers(0, 1000, (7, 9, 9))
local = conf_all[mine].sum(axis=0)
total = pdist.all_reduce_i64(local)
part = torch.tensor([0.5 * (rank + 1), 2.0], dtype=torch.float64)
pdist.all_reduce_(part)
t = pdist.max_over_ranks(1.0 + rank)
ex = pdist.loss_exchange()          # collective; gloo has no peer-addressable memory: every rank agrees on None
pdist.barrier()
if rank == 0:
    print(json.dumps({"world": world, "mine": mine, "ok": bool(np.array_equal(total, conf_all.sum(axis=0))),
                      "part": part.tolist(), "t": t, "exchange": ex is not None}))
torch.distributed.destroy_process_group()
"""


def test_dist_gloo_two_ranks(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % ROOT)
    port = 29000 + os.getpid() % 2000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(script)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    assert res == {"world": 2, "mine": [0, 2, 4, 6], "ok": True, "part": [1.5, 4.0], "t": 2.0, "exchange": False}


def test_rank_steps_equal_on_every_rank():
    """Data-parallel training: every step issues collectives, so every rank must take the same number of
    steps whatever the batch count (pylc.py train / _validate)."""
    from pylc_b200.pylc import rank_steps
    for world in (1, 2, 3, 4, 8):
        for n_batches in range(0, 40):
            steps = rank_steps(n_batches, world)
            taken = [sum(1 for i in range(n_batches) if i < steps * world and i % world == r) for r in range(world)]
            assert taken == [steps] * world
            assert n_batches - steps * world < world          # at most world-1 trailing batches dropped


def test_checkpoint_of_ddp_wrapped_net_has_bare_keys(tmp_path):
    """Model files written from a DistributedDataParallel-wrapped network carry the bare network's keys
    (reference checkpoint.py:53-66 format), and a 'module.'-prefixed dict still loads."""
    import types
    from pylc_b200.models.model import Checkpoint, strip_module_prefix
    net = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 1), torch.nn.BatchNorm2d(4))
    wrapper = torch.nn.Module()
    wrapper.module = net                                   # what DDP / DataParallel look like from outside
    optim = torch.optim.SGD(net.parameters(), lr=0.1)
    model = types.SimpleNamespace(net=wrapper, optim=optim, meta={"id": "x"}, epoch=1, iter=2)
    ck = Checkpoint("ddp_case", save_dir=str(tmp_path))
    ck.save(model, is_best=True)
    for f in (ck.checkpoint_file, ck.model_file):
        keys = list(torch.load(f, weights_only=False)["model"].keys())
        assert keys == list(net.state_dict().keys())
    prefixed = {"module." + k: v for k, v in net.state_dict().items()}
    assert list(strip_module_prefix(prefixed).keys()) == list(net.state_dict().keys())
    assert strip_module_prefix(net.state_dict()) is not None and list(strip_module_prefix(net.state_dict())) == list(net.state_dict())


def test_shard_indices_cover_everything_once():
    from pylc_b200.dist import shard_indices
    for world in (1, 2, 4, 8):
        got = sorted(i for r in range(world) for i in shard_indices(64, r, world))
        assert got == list(range(64))


# ---- bench.py reference arm contract ----------------------------------------------------------

def test_bench_cli_contract_flags():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl"):
        assert flag in out.stdout


# ---- inference plan (BN folding) ---------------------------------------------------------------

def test_fused_deeplab_matches_eval_network_on_cpu():
    from pylc_b200.models.deeplab import DeepLab
    from pylc_b200.models.fused import FusedDeepLab
    torch.manual_seed(0)
    net = DeepLab(n_classes=9).eval()
    g = torch.Generator().manual_seed(1)
    for m in net.modules():                      # non-trivial running statistics and affine terms
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)
    x = torch.randn(1, 3, 128, 128, generator=g)
    with torch.no_grad():
        want = net(x)
    got = FusedDeepLab(net, channels_last=False)(x)
    assert got.shape == want.shape and got.is_contiguous()
    scale = want.abs().max().item()
    assert (got - want).abs().max().item() <= 2e-4 * scale


@pytest.mark.parametrize("ssize,dsize", [(3000, 2560), (2000, 1536), (4000, 3584), (1100, 512), (513, 512), (512, 512)])
def test_area_table_host_equals_oracle(ssize, dsize):
    """pylc_area_table (host code of the CUDA library, no GPU needed) == the oracle's restatement of
    OpenCV's computeResizeAreaTab, weight for weight."""
    from pylc_b200 import ops
    start, count, weights = ops.area_table_host(ssize, dsize)
    tab = orc.area_table(ssize, dsize)
    k = 0
    for d in range(dsize):
        for j in range(count[d]):
            dd, si, a = tab[k]
            assert (dd, si) == (d, start[d] + j) and weights[d, j] == a
            k += 1
    assert k == len(tab)
