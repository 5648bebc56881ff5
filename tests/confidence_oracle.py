"""CPU oracle of the probability / confidence / calibration extension (pylc_stitch_probs,
pylc_confidence_resample, metrics.calibration_from_reliability).

It is written from the definition, independently of the kernels' block decomposition: every tile's
float64 softmax is added into a [C, h, w] sum together with a coverage count, and the mean is the sum
over the count.  The reference has no such map, so there is nothing of it to port here; the golden
reference maps pin it on edge and corner blocks (tests/test_confidence_cpu.py)."""
import numpy as np


def softmax64(x, axis=0):
    x = np.asarray(x, dtype=np.float64)
    e = np.exp(x - x.max(axis=axis, keepdims=True))
    return e / e.sum(axis=axis, keepdims=True)


def stitch_dims(nr, nc, T, S):
    return ((nr + 1) * S, (nc + 1) * S) if S < T else (nr * T, nc * T)


def stitch_probs(tiles, nr, nc, T, S):
    """P [C, h, w] f64: the mean, over the tiles covering each pixel, of softmax_c of the tile's logits.
    Tile (i, j) of the row-major [nr*nc, C, T, T] stack covers rows i*S .. i*S+T-1 and columns
    j*S .. j*S+T-1 of the fitted map."""
    tiles = np.asarray(tiles)
    C = tiles.shape[1]
    h, w = stitch_dims(nr, nc, T, S)
    acc = np.zeros((C, h, w), dtype=np.float64)
    cnt = np.zeros((h, w), dtype=np.float64)
    for i in range(nr):
        for j in range(nc):
            y0, x0 = i * S, j * S
            acc[:, y0:y0 + T, x0:x0 + T] += softmax64(tiles[i * nc + j])
            cnt[y0:y0 + T, x0:x0 + T] += 1
    assert cnt.min() >= 1
    return acc / cnt


def block_kinds(nr, nc, T, S):
    """[h, w] i8: how many tiles cover each pixel (1 corner / 2 edge / 4 interior; 1 everywhere when S == T)."""
    h, w = stitch_dims(nr, nc, T, S)
    cnt = np.zeros((h, w), dtype=np.int8)
    for i in range(nr):
        for j in range(nc):
            cnt[i * S:i * S + T, j * S:j * S + T] += 1
    return cnt


def confidence_u8(P, labels):
    """q = min(255, round-half-even(P[label] * 255)) per pixel, u8."""
    P = np.asarray(P)
    p = np.take_along_axis(P, np.asarray(labels, dtype=np.int64)[None], axis=0)[0]
    return np.minimum(255, np.rint(p * 255.0)).astype(np.uint8)


def reliability_table(conf_full, pred, true, C):
    """[C, 256, 2] i64 pixel counts by (predicted class, confidence level, prediction correct); pixels whose
    predicted or true class is >= C are not counted."""
    q = np.asarray(conf_full, dtype=np.int64).ravel()
    p = np.asarray(pred, dtype=np.int64).ravel()
    t = np.asarray(true, dtype=np.int64).ravel()
    ok = (p < C) & (t < C)
    key = (p[ok] * 256 + q[ok]) * 2 + (p[ok] == t[ok])
    return np.bincount(key, minlength=C * 512).astype(np.int64).reshape(C, 256, 2)


def calibration_direct(conf_full, pred, true, n_bins=15):
    """ECE / MCE straight from per-pixel arrays (float64), for checking the table-based figures."""
    c = np.asarray(conf_full, dtype=np.float64).ravel() / 255.0
    ok = (np.asarray(pred).ravel() == np.asarray(true).ravel()).astype(np.float64)
    b = np.minimum((c * n_bins).astype(np.int64), n_bins - 1)
    ece, mce = 0.0, 0.0
    for k in range(n_bins):
        sel = b == k
        if sel.any():
            gap = abs(ok[sel].mean() - c[sel].mean())
            ece += sel.sum() / c.size * gap
            mce = max(mce, gap)
    return ece, mce
