"""TEST INFRASTRUCTURE ONLY -- what the host-side live tests compare, in a form that can be stored.

Each record_* function runs one group of host helpers on fixed inputs and returns a JSON-serialisable record:
outcomes of the reference's error convention (print + exit), values, and arrays as shape / dtype / SHA-256.
`src` is a namespace with the modules the tests compare -- the PyLC reference's (ref_harness.load()) or this
package's (package_modules()) -- so one function produces the stored golden record and the record under test.
oracle/gen_live_golden.py writes tests/golden/host_live.json; tests/test_host_vs_reference_live.py and the *_live
tests of tests/test_host_cpu.py compare this package with it (and with the reference itself when it is present).
"""
import argparse
import contextlib
import hashlib
import importlib
import inspect
import io
import json
import os

import numpy as np

import pylc_oracle as orc

# the file cases of test_get_image: (file, ch, scale, interpolation name)
GET_IMAGE_CASES = [
    ("img/a.tif", 3, None, "INTER_AREA"), ("img/b.png", 3, 0.5, "INTER_AREA"), ("img/c.jpg", 3, None, "INTER_AREA"),
    ("mask/a.png", 3, 0.4, "INTER_NEAREST"), ("gray.tif", 1, None, "INTER_AREA"), ("gray.tif", 1, 0.7, "INTER_AREA"),
    ("gray.tif", 3, None, "INTER_AREA"),        # a gray file asked for as colour: print + exit(1)
    ("img/a.tif", 1, None, "INTER_AREA"),       # a colour file asked for as gray (the reference prompts; answered "y")
]

# reference class / module paths of the Python surface, and what is deliberately not provided
SURFACE_CLASSES = [("utils.extract", "Extractor"), ("utils.evaluate", "Evaluator"), ("models.modules.loss", "MultiLoss"),
                   ("models.modules.loss", "RunningLoss"), ("models.modules.checkpoint", "Checkpoint"),
                   ("models.model", "Model"), ("db.dataset", "MLPDataset"), ("utils.metrics", "Metrics"),
                   ("utils.augment", "Augmentor"), ("config", "Parameters")]
SURFACE_MODULES = ["utils.tools", "utils.profile", "utils.metrics"]
SURFACE_OMITTED = {
    ("Evaluator", "save_tex"): "LaTeX table helper (analysis, SURVEY.md section 2: out of scope)",
    ("Augmentor", "grayscale"): "bare stub in the reference (augment.py)",
    ("Augmentor", "merge_dbs"): "body commented out in the reference (augment.py:241-300)",
}
# Parameters attributes that are not part of the table: the process's random seed and the machine's device
PARAMETERS_VOLATILE = ("seed", "device")


def package_modules():
    """This package's modules under the reference's module paths."""
    return lambda path: importlib.import_module("pylc_b200." + path)


def make_files(d, palette):
    """The decoded-file fixture: three image / mask pairs (.tif / .png / .jpg), a stray text file, an image without
    a mask and a gray .tif, written with OpenCV from seeded synthetic pixels."""
    import cv2
    for sub in ("img", "mask", "odd"):
        os.makedirs(os.path.join(d, sub))
    for i, (name, ext) in enumerate([("a", ".tif"), ("b", ".png"), ("c", ".jpg")]):
        assert cv2.imwrite(os.path.join(d, "img", name + ext), orc.synth_image(i, 300, 200, 3)[..., ::-1])
        assert cv2.imwrite(os.path.join(d, "mask", name + ".png"), np.ascontiguousarray(orc.synth_mask(i, 300, 200, palette)[..., ::-1]))
    with open(os.path.join(d, "img", "notes.txt"), "w") as f:
        f.write("not an image")
    assert cv2.imwrite(os.path.join(d, "odd", "only.png"), orc.synth_image(5, 64, 64, 3))
    assert cv2.imwrite(os.path.join(d, "gray.tif"), orc.synth_image(9, 300, 200, 1))


def run(fn, *a, **k):
    """(outcome, value, printed text): the reference signals errors with print + exit(1)."""
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            val = fn(*a, **k)
        return "ok", val, buf.getvalue()
    except SystemExit as e:
        return "exit", e.code, buf.getvalue()
    except AssertionError:
        return "assert", None, buf.getvalue()


def plain(v, d=None):
    """JSON form of a value: arrays by shape / dtype / SHA-256, paths below `d` relative to it."""
    if isinstance(v, np.ndarray) or type(v).__module__ == "torch":
        a = np.ascontiguousarray(np.asarray(v))
        return {"shape": list(a.shape), "dtype": a.dtype.str, "sha256": hashlib.sha256(a.tobytes()).hexdigest()}
    if isinstance(v, np.generic):
        return v.item()
    if isinstance(v, dict):
        return {str(k): plain(x, d) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [plain(x, d) for x in v]
    if isinstance(v, str) and d is not None:
        return v.replace(d, "<dir>")
    return v


def outcome(fn, *a, d=None, **k):
    """(outcome, value) of one call in JSON form."""
    res = run(fn, *a, **k)
    return plain(list(res[:2]), d)


def record_file_lists(src, d):
    tools = src("utils.tools")
    rec = {}
    for args in ((d + "/img", d + "/mask"), (d + "/img",), (d + "/img/a.tif", d + "/mask/a.png"), (d + "/img", d + "/odd"),
                 (d + "/missing",)):
        rec["collate " + " ".join(plain(list(args), d))] = outcome(tools.collate, *args, d=d)
    rec["load_files <dir>/img .tif .png"] = outcome(tools.load_files, d + "/img", [".tif", ".png"], d=d)
    for p in ("/x/y/abc.def.tif", "rel/name.png", "noext"):
        rec["get_fname " + p] = tools.get_fname(p)
    return rec


def get_image_key(case):
    return "%s ch%d scale %s %s" % case


def record_get_image(src, d, case):
    """get_image on one file case; a colour file asked for as gray makes the reference prompt, answered "y"."""
    import builtins
    import cv2
    name, ch, scale, interp = case
    prompt = builtins.input
    builtins.input = lambda *a: "y"
    try:
        return outcome(src("utils.tools").get_image, os.path.join(d, name), ch, scale=scale,
                       interpolate=getattr(cv2, interp), d=d)
    finally:
        builtins.input = prompt


def record_helpers(src):
    tools, metrics = src("utils.tools"), src("utils.metrics")
    rec = {}
    for seed, (w, h, ch) in enumerate([(700, 500, 1), (650, 430, 3), (512, 512, 1)]):
        rec["adjust_to_tile %dx%d ch%d" % (w, h, ch)] = plain(list(tools.adjust_to_tile(orc.synth_image(seed, w, h, ch), 128, 64, ch)))
    a, b = np.arange(40).reshape(10, 4), np.arange(10)
    np.random.seed(5)
    rec["coshuffle seed 5"] = [np.asarray(x).tolist() for x in tools.coshuffle(a.copy(), b.copy())]
    rng = np.random.default_rng(0)
    for C in (2, 9, 11):
        p = rng.random(C)
        p /= p.sum()
        q = np.full(C, 1.0 / C)
        rec["jsd m2 C%d" % C] = [float(metrics.jsd(p, q)), float(metrics.m2(p, C))]
    for c in ([0, 0, 0], [255, 128, 7]):
        rec["rgb2hex %s" % c] = tools.rgb2hex(c)
    return rec


def record_parser(parser):
    """extract / augment / train / test options: option strings -> destination, choices, typed default."""
    for act in parser._actions:
        if isinstance(act, argparse._SubParsersAction):
            out = {"commands": sorted(act.choices)}
            for name in ("extract", "augment", "train", "test"):
                opts = {}
                for x in act.choices[name]._actions:
                    if x.option_strings and x.dest != "help":
                        opts[" ".join(x.option_strings)] = {
                            "dest": x.dest, "choices": list(x.choices) if x.choices is not None else None,
                            "default": x.default if x.default is not None and x.type is not None else None}
                out[name] = opts
            return out
    return {}


def record_surface(src):
    """Public methods of the path classes and functions of the path modules with their parameter names."""
    def names(fn):
        return [p.name for p in inspect.signature(fn).parameters.values()]
    out = {}
    for mod, cls in SURFACE_CLASSES:
        C = getattr(src(mod), cls)
        out[cls] = {n: names(f) for n, f in inspect.getmembers(C, inspect.isfunction)      # not torch.nn.Module's own
                    if not (n.startswith("_") and n != "__init__") and (cls, n) not in SURFACE_OMITTED
                    and not f.__module__.startswith("torch")}
    for mod in SURFACE_MODULES:
        M = src(mod)
        out[mod] = {n: names(f) for n, f in inspect.getmembers(M, inspect.isfunction) if f.__module__ == M.__name__}
    return out


def record_parameters(Parameters, schema):
    """vars(Parameters) as the CLI builds it (a Namespace with `schema`), without the volatile attributes."""
    table = vars(Parameters(argparse.Namespace(schema="./schemas/%s.json" % schema)))
    return json.loads(json.dumps({k: plain(v) for k, v in table.items() if k not in PARAMETERS_VOLATILE}))
