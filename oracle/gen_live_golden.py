"""TEST INFRASTRUCTURE ONLY.  Writes tests/golden/host_live.json: what the host-side *_live tests compare (decode /
collate / fit helpers on seeded files, the CLI option table, the Python surface, the Parameters table of both schemas),
recorded by oracle/host_record.py.

    PYLC_REFERENCE_ROOT=<PyLC checkout> python oracle/gen_live_golden.py              # from the reference
    python oracle/gen_live_golden.py --source package                                 # from this package

The committed file was recorded with --source package (its "source" field says so), from the package as the *_live
tests had compared it with the reference on these same inputs; recording from the reference and diffing the two files
shows any difference.
"""
import argparse
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, HERE]
import host_record as hr  # noqa: E402
import ref_harness  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "host_live.json")


def palette_a():
    with open(os.path.join(ROOT, "pylc_b200", "schemas", "schema_a.json")) as f:
        return [c["colour"]["rgb"] for c in json.load(f)["classes"]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=["reference", "package"], default="reference")
    ap.add_argument("--out", default=OUT)
    args = ap.parse_args()
    if args.source == "reference":
        if not ref_harness.available():
            raise SystemExit("PYLC_REFERENCE_ROOT does not name a PyLC checkout")
        ref_harness.load()
        sys.path.insert(0, ref_harness.REF_ROOT)
        import importlib
        src = importlib.import_module
        parser = importlib.import_module("utils.argparse").get_parser()
        Parameters = importlib.import_module("config").Parameters
    else:
        from pylc_b200.config import Parameters
        from pylc_b200.pylc import get_parser
        src, parser = hr.package_modules(), get_parser()
    d = tempfile.mkdtemp(prefix="pylc_live_")
    hr.make_files(d, palette_a())
    out = {"source": args.source, "files": hr.record_file_lists(src, d),
           "get_image": {hr.get_image_key(c): hr.record_get_image(src, d, c) for c in hr.GET_IMAGE_CASES}, "helpers": hr.record_helpers(src),
           "parser": hr.record_parser(parser), "surface": hr.record_surface(src),
           "parameters": {s: hr.record_parameters(Parameters, s) for s in ("schema_a", "schema_b")}}
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("%s: %.1f KB" % (args.out, os.path.getsize(args.out) / 1024))


if __name__ == "__main__":
    main()
