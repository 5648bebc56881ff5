"""Probability / confidence / calibration extension on the CPU: the oracle's mean-of-softmaxes map against
the reference's golden stitched maps, the calibration figures of a reliability table, and the CLI flags."""
import numpy as np
import pytest

import confidence_oracle as co
import pylc_oracle as orc

CASES = ["a_2x3", "a_3x2", "a_3x3", "a_2x1", "b_4x5"]


def _case(golden, case):
    g = golden("reconstruct")
    nr, nc, T, S, h, w, w_full, h_full, C = [int(v) for v in g["recon_%s_geom" % case]]
    return g, orc.reconstruct_fixture_tiles(g, case), g["recon_%s_map" % case], nr, nc, T, S


@pytest.mark.parametrize("case", CASES)
def test_stitch_probs_is_the_reference_map_on_edges_and_its_softmax_on_corners(golden, case):
    g, tiles, M, nr, nc, T, S = _case(golden, case)
    P = co.stitch_probs(tiles, nr, nc, T, S)
    kinds = co.block_kinds(nr, nc, T, S)
    assert P.shape == M.shape
    edge, corner = kinds == 2, kinds == 1
    assert edge.any() and corner.sum() == 4 * S * S
    # edge blocks: the reference's single softmax-average IS the mean of the two covering softmaxes
    np.testing.assert_allclose(P[:, edge], M[:, edge], rtol=1e-6, atol=0)
    # corner blocks: the reference keeps the raw logits, P is their softmax
    np.testing.assert_allclose(P[:, corner], co.softmax64(M[:, corner]), rtol=1e-6, atol=0)
    # and P is a probability vector everywhere, interior included
    np.testing.assert_allclose(P.sum(axis=0), 1.0, rtol=1e-12)


def test_stitch_probs_without_overlap_is_the_softmax_of_the_scattered_logits(golden):
    g, tiles, M, nr, nc, T, S = _case(golden, "a_s32_2x3")
    assert S == T
    P = co.stitch_probs(tiles, nr, nc, T, S)
    np.testing.assert_allclose(P, co.softmax64(M), rtol=1e-6, atol=0)
    np.testing.assert_allclose(P, co.softmax64(orc.stitch_map(tiles, nr, nc, T, S)), rtol=1e-6, atol=0)


def test_confidence_u8_is_the_probability_at_the_label():
    P = co.softmax64(np.random.default_rng(0).standard_normal((9, 20, 30)) * 3)
    lab = np.argmax(P, axis=0)
    q = co.confidence_u8(P, lab)
    assert q.dtype == np.uint8
    assert np.array_equal(q, np.rint(P.max(axis=0) * 255).astype(np.uint8))
    assert int(co.confidence_u8(np.ones((1, 2, 2)), np.zeros((2, 2), np.uint8)).min()) == 255


def _pixels(seed, n, C):
    rng = np.random.default_rng(seed)
    pred = rng.integers(0, C, n).astype(np.uint8)
    conf = rng.integers(0, 256, n).astype(np.uint8)
    # right more often at high confidence, so the bins differ
    right = rng.random(n) < conf / 255.0 * 0.8
    true = np.where(right, pred, (pred + 1 + rng.integers(0, C - 1, n)) % C).astype(np.uint8)
    return conf, pred, true


def test_calibration_from_reliability_equals_per_pixel_figures():
    from pylc_b200.utils.metrics import calibration_from_reliability
    C = 9
    conf, pred, true = _pixels(1, 200_000, C)
    table = co.reliability_table(conf, pred, true, C)
    assert table.sum() == conf.size
    cal = calibration_from_reliability(table, [str(i) for i in range(C)])
    ece, mce = co.calibration_direct(conf, pred, true)
    assert cal["ece"] == pytest.approx(ece, rel=1e-12, abs=1e-15)
    assert cal["mce"] == pytest.approx(mce, rel=1e-12, abs=1e-15)
    assert sum(cal["bins"]["count"]) == conf.size == cal["n_pixels"]
    for c in range(C):
        sel = pred == c
        k = cal["classes"][str(c)]
        assert k["count"] == int(sel.sum())
        assert k["confidence"] == pytest.approx(conf[sel].mean() / 255.0, rel=1e-12)
        assert k["accuracy"] == pytest.approx((true[sel] == c).mean(), rel=1e-12)


def test_calibration_of_tables_summed_over_ranks_is_exact():
    from pylc_b200.utils.metrics import calibration_from_reliability
    C = 11
    conf, pred, true = _pixels(2, 100_001, C)
    whole = co.reliability_table(conf, pred, true, C)
    half = 37_123
    split = co.reliability_table(conf[:half], pred[:half], true[:half], C) + \
        co.reliability_table(conf[half:], pred[half:], true[half:], C)
    assert np.array_equal(whole, split)
    assert calibration_from_reliability(split) == calibration_from_reliability(whole)


def test_calibration_of_perfectly_calibrated_and_empty_tables():
    from pylc_b200.utils.metrics import calibration_from_reliability
    t = np.zeros((2, 256, 2), dtype=np.int64)
    assert calibration_from_reliability(t)["ece"] == 0.0
    t[0, 255, 1] = 10          # confidence 1.0, always right
    cal = calibration_from_reliability(t)
    assert cal["ece"] == 0.0 and cal["mce"] == 0.0 and cal["classes"]["1"]["count"] == 0
    with pytest.raises(ValueError):
        calibration_from_reliability(np.zeros((2, 255, 2)))


def test_cli_accepts_stitch_and_confidence_flags():
    from pylc_b200.pylc import get_parser
    p = get_parser()
    a = p.parse_args("test -l m.pth -i img.tif -m mask.png --stitch mean --save_confidence".split())
    assert (a.stitch, a.save_confidence, a.save_logits) == ("mean", True, False)
    a = p.parse_args("test -l m.pth -i img.tif".split())
    assert (a.stitch, a.save_confidence) == ("reference", False)
    assert (a.model, a.img, a.mask, a.save_logits, a.aggregate_metrics, a.batch_tiles) == ("m.pth", "img.tif", None, False, False, 32)
    with pytest.raises(SystemExit):
        p.parse_args("test -l m.pth --stitch max".split())


def test_stitch_mode_names():
    from pylc_b200 import ops
    from pylc_b200._lib import PylcError
    assert ops.STITCH_MODES == {"reference": 0, "mean": 1}
    with pytest.raises(PylcError):
        ops._stitch_mode("max")
