"""Temperature scaling of the mean stitch without a GPU: the f64 oracle (tests/temperature_oracle.py), the search of
pylc_b200/utils/calibrate.py against analytic objectives and against the oracle's planted temperatures, the
calibrated model-file copy and the command-line checks."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import confidence_oracle as co
import temperature_oracle as to

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_k_t_is_log2e_at_one_and_one_f32_division():
    assert to.k_t(1.0) == to.KLOG2E
    for T in (0.05, 0.25, 0.5, 2.0, 7.5, 20.0):
        assert to.k_t(T) == np.float32(np.float32(1.4426950408889634) / np.float32(T))


def test_oracle_at_one_equals_the_mean_stitch_oracle():
    rng = np.random.default_rng(3)
    for C, nr, nc, T, S in ((4, 2, 3, 32, 16), (9, 3, 3, 32, 16), (11, 2, 2, 16, 16)):
        tiles = (rng.standard_normal((nr * nc, C, T, T)) * 3).astype(np.float32)
        # k_T * ln 2 is 1 up to the f32 rounding of log2(e)
        assert np.allclose(to.stitch_probs_t(tiles, nr, nc, T, S, 1.0), co.stitch_probs(tiles, nr, nc, T, S),
                           rtol=1e-6, atol=1e-9)


def test_oracle_scores_by_hand():
    P = np.array([[[0.5, 0.0]], [[0.5, 1.0]]])          # C = 2, h = 1, w = 2
    y = np.array([[0, 0]], dtype=np.uint8)
    nll, brier = to.prob_scores(P, y, [0, 1], [0])
    assert nll == pytest.approx(-math.log(0.5) - math.log(1e-12))
    assert brier == pytest.approx(0.25 + 0.25 + 1.0 + 1.0)


@pytest.mark.parametrize("fit", ["package", "oracle"])
@pytest.mark.parametrize("u0", [-1.3, 0.0, 0.37, 2.2])
def test_search_finds_the_minimum_of_a_parabola(fit, u0):
    obj = lambda u: (u - u0) ** 2 + 1.0                     # noqa: E731
    if fit == "package":
        from pylc_b200.utils.calibrate import fit_temperature
        r = fit_temperature(obj)
        T, at_bound, n = r["temperature"], r["at_bound"], len(r["evals"])
        assert r["evals"][12][0] == 1.0                      # T = 1 exactly at the grid's centre
    else:
        T, _, at_bound, ev = to.fit_temperature(obj)
        n = len(ev)
    assert abs(math.log(T) - u0) < 1e-4 and not at_bound and n > 25


@pytest.mark.parametrize("slope,bound", [(1.0, 0.05), (-1.0, 20.0)])
def test_search_flags_a_minimum_at_the_grid_bound(slope, bound):
    from pylc_b200.utils.calibrate import fit_temperature
    r = fit_temperature(lambda u: slope * u)
    assert r["at_bound"] and r["temperature"] == pytest.approx(bound, rel=1e-12)
    T, _, at_bound, _ = to.fit_temperature(lambda u: slope * u)
    assert at_bound and T == pytest.approx(bound, rel=1e-12)


def test_search_resolves_ties_to_the_first_evaluation():
    from pylc_b200.utils.calibrate import fit_temperature
    r = fit_temperature(lambda u: 0.0)                       # every point ties: the first grid point wins
    assert r["temperature"] == pytest.approx(0.05, rel=1e-12) and r["at_bound"]
    # a flat valley around the centre: grid points 11..13 tie, the first of them (i = 11) is T*
    valley = lambda u: 0.0 if abs(u) <= math.log(20.0) / 12 + 1e-12 else 1.0     # noqa: E731
    r = fit_temperature(valley)
    assert r["temperature"] == pytest.approx(math.exp(-math.log(20.0) / 12), rel=1e-12)
    assert to.fit_temperature(valley)[0] == pytest.approx(r["temperature"], rel=1e-12)


def test_package_search_matches_the_oracle_search_step_for_step():
    from pylc_b200.utils.calibrate import fit_temperature
    obj = lambda u: math.cosh(u - 0.3) + 0.1 * u          # noqa: E731
    r = fit_temperature(obj)
    T, f, at_bound, ev = to.fit_temperature(obj)
    assert [math.log(t) for t, _ in r["evals"]] == pytest.approx([u for u, _ in ev], abs=1e-12)
    assert r["temperature"] == pytest.approx(T, rel=1e-12) and r["f"] == f and r["at_bound"] == at_bound


@pytest.mark.parametrize("T0", [0.5, 2.0])
def test_oracle_fit_recovers_a_planted_temperature(T0):
    tiles, y, geom = to.planted_case(T0)
    T, _, at_bound, _ = to.fit_temperature(lambda u: to.mean_nll(tiles, y, geom, math.exp(u)))
    assert not at_bound and abs(T / T0 - 1) < 0.03


def test_calibrated_copy_round_trips_and_plain_files_have_none(tmp_path):
    """In a child process: Model.load configures the process-wide defaults."""
    code = r"""
import json, os, sys, torch
from pylc_b200.config import Parameters
from pylc_b200.models.deeplab import DeepLab
from pylc_b200.models.model import Model, _load_model_file
from pylc_b200.utils.calibrate import write_calibrated_copy
torch.manual_seed(0)
m = Parameters()
m.update({"ch": 1, "n_classes": 4, "arch": "deeplab", "backbone": "resnet", "pretrained": False, "id": "cal_model"})
torch.save({"model": DeepLab(n_classes=4, in_channels=1).state_dict(), "optim": None, "meta": m}, "plain.pth")
cal = {"temperature": 1.75, "n_images": 2, "n_px": 123, "nll_before": 1.5, "nll_after": 1.25}
write_calibrated_copy("plain.pth", "plain_calibrated.pth", cal)
a, b = _load_model_file("plain.pth", "cpu"), _load_model_file("plain_calibrated.pth", "cpu")
assert set(b) == set(a) | {"calibration"} and all(torch.equal(a["model"][k], b["model"][k]) for k in a["model"])
print(json.dumps([Model().load("plain.pth").calibration, Model().load("plain_calibrated.pth").calibration]))
"""
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    plain, calibrated = json.loads(out.stdout.strip().splitlines()[-1])
    assert plain is None
    assert calibrated == {"temperature": 1.75, "n_images": 2, "n_px": 123, "nll_before": 1.5, "nll_after": 1.25}


def test_cli_parses_calibrate_and_temperature():
    from pylc_b200.config import Parameters
    from pylc_b200.pylc import get_parser
    p = get_parser()
    a = p.parse_args("calibrate -l m.pth -i imgs -m masks --max_resident_gb 4 -o out.pth".split())
    assert a.func.__name__ == "calibrate" and a.max_resident_gb == 4.0 and a.output == "out.pth"
    assert a.scale == Parameters().scale and a.batch_tiles == 32
    with pytest.raises(SystemExit):
        p.parse_args("calibrate -l m.pth -i imgs".split())           # masks are required
    assert p.parse_args("test -l m.pth --stitch mean --temperature 1.5".split()).temperature == 1.5
    assert p.parse_args("test -l m.pth".split()).temperature is None
    assert set(vars(Parameters(a))) == set(vars(Parameters()))


@pytest.mark.parametrize("argv", ["--temperature 2 --stitch reference", "--temperature 2", "--stitch mean --temperature 0",
                                  "--stitch mean --temperature -1", "--stitch mean --temperature nan",
                                  "--stitch mean --temperature inf"])
def test_cli_refuses_bad_temperatures(argv, capsys):
    from pylc_b200 import pylc
    args = pylc.get_parser().parse_args(("test -l m.pth -i img.tif " + argv).split())
    with pytest.raises(SystemExit) as exc:
        pylc.test(args)
    assert exc.value.code == 2
    err = capsys.readouterr().err
    assert "--temperature" in err and len(err.strip().splitlines()) == 1


def test_calibrate_refuses_multi_rank_and_overwriting_the_model(monkeypatch, capsys):
    from pylc_b200 import pylc
    p = pylc.get_parser()
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit) as exc:
        pylc.calibrate(p.parse_args("calibrate -l m.pth -i imgs -m masks".split()))
    assert exc.value.code == 2 and "one GPU" in capsys.readouterr().err
    monkeypatch.setenv("WORLD_SIZE", "1")
    with pytest.raises(SystemExit) as exc:
        pylc.calibrate(p.parse_args("calibrate -l m.pth -i imgs -m masks -o ./m.pth".split()))
    assert exc.value.code == 2 and "copy" in capsys.readouterr().err
