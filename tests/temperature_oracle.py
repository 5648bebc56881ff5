"""CPU oracle (float64) of temperature scaling for the mean stitch: pylc_stitch_probs_t, pylc_prob_scores and the
temperature search of pylc_b200/utils/calibrate.py, each written from its definition."""
import math

import numpy as np

import confidence_oracle as co

KLOG2E = np.float32(1.4426950408889634)


def k_t(temperature):
    """The kernels' softmax scale: f32(log2(e) / f32(T)), one f32 division."""
    return np.float32(KLOG2E / np.float32(temperature))


def stitch_probs_t(tiles, nr, nc, T, S, temperature):
    """P_T [C, h, w] f64: the mean over the covering tiles of softmax64(L * k_T * ln 2), k_T the f32 constant the
    kernels use (k_T * ln 2 = 1 / T up to f32 rounding)."""
    tiles = np.asarray(tiles)
    scale = float(k_t(temperature)) * math.log(2.0)
    C = tiles.shape[1]
    h, w = co.stitch_dims(nr, nc, T, S)
    acc = np.zeros((C, h, w), dtype=np.float64)
    cnt = np.zeros((h, w), dtype=np.float64)
    for i in range(nr):
        for j in range(nc):
            y0, x0 = i * S, j * S
            acc[:, y0:y0 + T, x0:x0 + T] += co.softmax64(tiles[i * nc + j].astype(np.float64) * scale)
            cnt[y0:y0 + T, x0:x0 + T] += 1
    return acc / cnt


def prob_scores(P, y_true, x_ofs, y_ofs):
    """(sum of -log(max(q, 1e-12)), sum of sum_c (P[c] - [c == g])^2) in float64 over the full-resolution pixels,
    q = P[g][y_ofs[y]][x_ofs[x]], g = y_true[y, x]; a class >= C counts as probability 0."""
    P = np.asarray(P, dtype=np.float64)
    y_true = np.asarray(y_true, dtype=np.int64)
    C = P.shape[0]
    x_ofs = np.asarray(x_ofs, dtype=np.int64)
    nll = brier = 0.0
    for y in range(y_true.shape[0]):
        row = P[:, int(y_ofs[y]), :][:, x_ofs]              # [C, w_full]
        g = y_true[y]
        inside = g < C
        q = np.where(inside, row[np.minimum(g, C - 1), np.arange(g.size)], 0.0)
        nll += float(-np.log(np.maximum(q, 1e-12)).sum())
        onehot = (np.arange(C)[:, None] == g[None, :]).astype(np.float64)
        brier += float(((row - onehot) ** 2).sum())
    return nll, brier


def fit_temperature(objective):
    """The search of the definition over objective(u), u = ln T.  Returns (T*, f(T*), at_bound, [(u, f), ...])."""
    evaluated = []

    def f(u):
        evaluated.append((u, float(objective(u))))
        return evaluated[-1][1]
    grid = [(i - 12) * math.log(20.0) / 12 for i in range(25)]
    values = [f(u) for u in grid]
    i_star = 0
    for i in range(1, 25):
        if values[i] < values[i_star]:
            i_star = i
    a, b = grid[max(i_star - 1, 0)], grid[min(i_star + 1, 24)]
    invphi = (math.sqrt(5.0) - 1.0) / 2.0
    c = b - invphi * (b - a)
    d = a + invphi * (b - a)
    fc, fd = f(c), f(d)
    while not b - a < 1e-4:
        if fc <= fd:                      # keep [a, d]; the old c becomes the new d
            b, d, fd = d, c, fc
            c = b - invphi * (b - a)
            fc = f(c)
        else:                             # keep [c, b]; the old d becomes the new c
            a, c, fc = c, d, fd
            d = a + invphi * (b - a)
            fd = f(d)
    best = 0
    for k in range(1, len(evaluated)):
        if evaluated[k][1] < evaluated[best][1]:
            best = k
    return math.exp(evaluated[best][0]), evaluated[best][1], i_star in (0, 24), evaluated


def planted_case(T0, seed=7, C=9, nr=6, nc=6, T=64, S=32, scale=3.0):
    """Seeded logits and a ground truth sampled per pixel from the oracle's P_T0 (the geometry the planted-temperature
    tests use on the CPU and the GPU).  Returns (tiles f32, y_true u8 [h, w], (C, nr, nc, T, S))."""
    rng = np.random.default_rng(seed)
    tiles = (rng.standard_normal((nr * nc, C, T, T)) * scale).astype(np.float32)
    P = stitch_probs_t(tiles, nr, nc, T, S, T0)
    cum = np.cumsum(P, axis=0)
    u = rng.random(P.shape[1:]) * cum[-1]
    y = np.minimum((u[None] >= cum).sum(axis=0), C - 1).astype(np.uint8)
    return tiles, y, (C, nr, nc, T, S)


def mean_nll(tiles, y, geom, temperature):
    C, nr, nc, T, S = geom
    P = stitch_probs_t(tiles, nr, nc, T, S, temperature)
    h, w = y.shape
    return prob_scores(P, y, np.arange(w), np.arange(h))[0] / y.size
