"""Multi-scale inference on the CPU: the oracle's two statements against each other, OpenCV's nearest-neighbour
sampling against the package's index maps, the per-scale geometry and the CLI flag."""
import cv2
import numpy as np
import pytest

import confidence_oracle as co
import multiscale_oracle as mo
import pylc_oracle as orc


def _planes(seed, C, sizes):
    rng = np.random.default_rng(seed)
    return [co.softmax64(rng.standard_normal((C, h, w)) * 3).astype(np.float32) for w, h in sizes]


@pytest.mark.parametrize("C,sizes,w_full,h_full", [
    (9, [(96, 64), (128, 96), (160, 112)], 131, 97),
    (2, [(40, 30), (61, 47)], 80, 60),
    (11, [(33, 21)] * 8, 50, 31),
    (20, [(64, 48)], 64, 48),
])
def test_f64_definition_and_f32_restatement_agree(C, sizes, w_full, h_full):
    probs = _planes(C + len(sizes), C, sizes)
    m64, lab64, q64 = mo.combine_f64(probs, w_full, h_full)
    m32, lab32, q32 = mo.combine_f32(probs, w_full, h_full)
    assert m32.dtype == np.float32 and lab32.shape == (h_full, w_full)
    assert np.abs(m32.astype(np.float64) - m64).max() <= 1e-6
    decided = orc.top2_margin(m64) > 1e-6
    assert np.array_equal(lab32[decided], lab64[decided])
    assert np.abs(q32.astype(np.int64) - q64).max() <= 1
    p = np.take_along_axis(m64, lab64[None].astype(np.int64), axis=0)[0] * 255.0
    safe = decided & (np.abs(p - np.floor(p) - 0.5) > 1e-3)
    assert np.array_equal(q32[safe], q64[safe])


@pytest.mark.parametrize("w,h,w_full,h_full", [(1536, 1024, 3000, 2000), (2560, 1536, 2000, 1300), (511, 257, 1301, 997),
                                               (1301, 997, 511, 257), (7, 5, 7, 5)])
def test_opencv_nearest_equals_the_index_maps(w, h, w_full, h_full):
    from pylc_b200 import ops
    plane = np.random.default_rng(w + h).random((2, h, w)).astype(np.float32)
    got = mo.sample_nearest(plane, w_full, h_full)
    x, y = ops.nn_index_map(w, w_full), ops.nn_index_map(h, h_full)
    assert np.array_equal(got, plane[:, y[:, None], x[None, :]])


def test_one_scale_is_the_argmax_and_confidence_of_its_map():
    (P,) = _planes(5, 9, [(70, 40)])
    m, lab, q = mo.combine_f32([P], 70, 40)
    assert np.array_equal(m, P)
    assert np.array_equal(lab, np.argmax(P, axis=0))
    assert np.array_equal(q, co.confidence_u8(P, lab))


def test_geometry_routes_members_to_device_or_host():
    from pylc_b200.pipeline import multiscale_geometry
    geo = multiscale_geometry(4000, 3000, 512, (1.25, 0.5, 0.75, 1.0))
    assert [g["scale"] for g in geo] == [0.5, 0.75, 1.0, 1.25]
    by = {g["scale"]: g for g in geo}
    assert by[0.5]["resized"] == (2000, 1500) and not by[0.5]["device"]        # integer factor: OpenCV's fast path
    assert by[0.75]["resized"] == (3000, 2250) and by[0.75]["fitted"] == (2560, 1536) and by[0.75]["device"]
    assert by[1.0]["resized"] == (4000, 3000) and by[1.0]["fitted"] == (3584, 2560) and by[1.0]["device"]
    assert by[1.25]["resized"] == (5000, 3750) and not by[1.25]["device"]      # enlarging
    for g in geo:
        w, h = g["fitted"]
        assert w % 512 == 0 and h % 512 == 0 and w <= g["resized"][0]


def test_geometry_refuses_a_scale_that_fits_to_one_tile_row():
    from pylc_b200.pipeline import multiscale_geometry
    assert [g["fitted"] for g in multiscale_geometry(1600, 1200, 512, (1.0,))] == [(1536, 1024)]
    with pytest.raises(ValueError, match=r"scale 0\.75.*1024x512"):
        multiscale_geometry(1600, 1200, 512, (0.75, 1.0))
    with pytest.raises(ValueError, match=r"scale 0\.25.*400x300"):
        multiscale_geometry(1600, 1200, 512, (0.25, 1.0))


@pytest.mark.parametrize("scales", [(), (1.0, 1.0), (0.0, 1.0), (-0.5, 1.0), tuple(0.5 + 0.1 * i for i in range(9))])
def test_scale_lists_refused(scales):
    from pylc_b200.pipeline import check_scales
    with pytest.raises(ValueError):
        check_scales(scales)


def test_scale_lists_are_sorted():
    from pylc_b200.pipeline import check_scales
    assert check_scales([1.25, 0.75, 1]) == (0.75, 1.0, 1.25)


def test_cli_accepts_multiscale_and_parameters_are_unchanged():
    from pylc_b200.config import Parameters
    from pylc_b200.pylc import get_parser
    p = get_parser()
    a = p.parse_args("test -l m.pth -i img.tif --stitch mean --multiscale 0.75 1.0 1.25 --save_confidence".split())
    assert a.multiscale == [0.75, 1.0, 1.25] and a.stitch == "mean"
    assert p.parse_args("test -l m.pth -i img.tif".split()).multiscale is None
    assert set(vars(Parameters(a))) == set(vars(Parameters())) and not hasattr(Parameters(a), "multiscale")


@pytest.mark.parametrize("argv", ["--multiscale 1.0", "--stitch reference --multiscale 0.75 1.0",
                                  "--stitch mean --multiscale 1.0 1.0"])
def test_cli_refuses_multiscale_without_mean_stitch_or_with_bad_scales(argv, capsys):
    from pylc_b200 import pylc
    args = pylc.get_parser().parse_args(("test -l m.pth -i img.tif " + argv).split())
    with pytest.raises(SystemExit) as exc:
        pylc.test(args)
    assert exc.value.code != 0
    assert "--multiscale" in capsys.readouterr().err


def test_cv2_resize_at_identical_size_is_a_copy():
    """The 1.0 member skips the first resize: OpenCV would return the same bytes."""
    img = orc.synth_image(3, 701, 503, 3)
    assert np.array_equal(cv2.resize(img, (701, 503), interpolation=cv2.INTER_AREA), img)

