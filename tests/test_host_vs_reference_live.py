"""The host-side helpers of the path (decode, file collation, fit, shuffles, C-vector statistics) on the same files and
arrays as the unmodified reference: against the record in tests/golden/host_live.json (oracle/gen_live_golden.py), and
side by side with the reference itself when PYLC_REFERENCE_ROOT names a PyLC checkout."""
import importlib
import json
import os
import sys

import cv2
import numpy as np
import pytest

import host_record as hr
import ref_harness

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_live.json")))
PACKAGE = hr.package_modules()


@pytest.fixture(scope="module")
def ref():
    if not ref_harness.available():
        return None
    ref_harness.load()
    sys.path.insert(0, ref_harness.REF_ROOT)
    try:
        mods = {n: importlib.import_module(m) for n, m in (("tools", "utils.tools"), ("profile", "utils.profile"),
                                                            ("metrics", "utils.metrics"), ("config", "config"))}
    finally:
        sys.path.remove(ref_harness.REF_ROOT)
    return type("Ref", (), mods)


@pytest.fixture(scope="module")
def files(tmp_path_factory, palettes):
    d = tmp_path_factory.mktemp("live")
    hr.make_files(str(d), palettes["a"])
    return d


def test_collate_and_load_files(ref, files):
    from pylc_b200.utils import tools
    d = str(files)
    assert hr.record_file_lists(PACKAGE, d) == GOLDEN["files"]
    if ref is None:
        return
    run = hr.run
    for args in ((d + "/img", d + "/mask"), (d + "/img",), (d + "/img/a.tif", d + "/mask/a.png"),
                 (d + "/img", d + "/odd"), (d + "/missing",)):
        want, got = run(ref.tools.collate, *args), run(tools.collate, *args)
        assert want[:2] == got[:2], args
    assert run(ref.tools.load_files, d + "/img", [".tif", ".png"])[:2] == run(tools.load_files, d + "/img", [".tif", ".png"])[:2]
    for p in ("/x/y/abc.def.tif", "rel/name.png", "noext"):
        assert ref.tools.get_fname(p) == tools.get_fname(p)


@pytest.mark.parametrize("name,ch,scale,interp", hr.GET_IMAGE_CASES)
def test_get_image(ref, files, name, ch, scale, interp, monkeypatch):
    from pylc_b200.utils import tools
    case = (name, ch, scale, interp)
    assert hr.record_get_image(PACKAGE, str(files), case) == GOLDEN["get_image"][hr.get_image_key(case)]
    if ref is None:
        return
    monkeypatch.setattr("builtins.input", lambda *a: "y")
    path = str(files / name)
    want = hr.run(ref.tools.get_image, path, ch, scale=scale, interpolate=getattr(cv2, interp))
    got = hr.run(tools.get_image, path, ch, scale=scale, interpolate=getattr(cv2, interp))
    assert want[0] == got[0]
    if want[0] == "ok":
        assert np.array_equal(want[1][0], got[1][0]) and tuple(want[1][1:]) == tuple(got[1][1:])


def test_adjust_to_tile_coshuffle_and_statistics(ref):
    from pylc_b200.utils import metrics, tools
    assert hr.record_helpers(PACKAGE) == GOLDEN["helpers"]
    if ref is None:
        return
    import pylc_oracle as orc
    for seed, (w, h, ch) in enumerate([(700, 500, 1), (650, 430, 3), (512, 512, 1)]):
        img = orc.synth_image(seed, w, h, ch)
        want, got = ref.tools.adjust_to_tile(img, 128, 64, ch), tools.adjust_to_tile(img, 128, 64, ch)
        assert np.array_equal(want[0], got[0]) and tuple(want[1:]) == tuple(got[1:])
    a, b = np.arange(40).reshape(10, 4), np.arange(10)
    np.random.seed(5)
    want = ref.tools.coshuffle(a.copy(), b.copy())
    np.random.seed(5)
    got = tools.coshuffle(a.copy(), b.copy())
    assert all(np.array_equal(x, y) for x, y in zip(want, got))
    rng = np.random.default_rng(0)
    for C in (2, 9, 11):
        p = rng.random(C)
        p /= p.sum()
        q = np.full(C, 1.0 / C)
        assert ref.metrics.jsd(p, q) == metrics.jsd(p, q) and ref.metrics.m2(p, C) == metrics.m2(p, C)
    for c in ([0, 0, 0], [255, 128, 7]):
        assert ref.tools.rgb2hex(c) == tools.rgb2hex(c)
