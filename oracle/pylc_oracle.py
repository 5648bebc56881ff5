"""
TEST INFRASTRUCTURE ONLY -- CPU oracle for the PyLC tiled-segmentation hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product (pylc_b200/) never does: it fails loudly when the CUDA
library is missing.

Every function restates, in NumPy / Torch-CPU, what one reference function computes and cites
the reference file:line it follows (paths relative to the PyLC reference root).  Two flavours
exist for the expensive ones:

  *_port  : same algorithmic steps / same library calls as the reference (per-class passes,
            per-band softmax loops, scikit-learn metrics ...), so its CPU time is representative
            of the reference.  This is what bench.py times as `cpu_baseline` (kind "port").
  (plain) : closed-form vectorised restatement used as the fast checker in tests.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md section 4).  The oracle
is pinned instead against outputs of the unmodified reference executed in the build container
(oracle/gen_golden.py -> tests/golden/*.npz; tests/test_oracle_golden.py) and, when
PYLC_REFERENCE_ROOT names a reference checkout, live (tests/test_oracle_vs_reference.py).
"""
import hashlib
import math

import numpy as np
import torch

# ----------------------------------------------------------------------------------------------
# Tiling geometry  (utils/extract.py:279-310, utils/tools.py:151-206)
# ----------------------------------------------------------------------------------------------


def tile_grid(H, W, T, S):
    """Tensor.unfold(0,T,S).unfold(1,T,S) tile counts (utils/extract.py:302-305)."""
    if H < T or W < T:
        return 0, 0
    return (H - T) // S + 1, (W - T) // S + 1


def split_tiles(img, T, S):
    """utils/extract.py:279-310  Extractor.__split: [H,W] or [H,W,3] u8 -> [nH*nW, ch, T, T] u8,
    row-major tile order, trailing remainder dropped, HWC -> CHW for colour."""
    img = np.asarray(img, dtype=np.uint8)
    ch = 3 if img.ndim == 3 else 1
    nH, nW = tile_grid(img.shape[0], img.shape[1], T, S)
    out = np.empty((nH * nW, ch, T, T), dtype=np.uint8)
    for r in range(nH):
        for c in range(nW):
            blk = img[r * S:r * S + T, c * S:c * S + T]
            out[r * nW + c] = blk[None] if ch == 1 else np.moveaxis(blk, 2, 0)
    return out


def fit_dims(W, H, T):
    """utils/tools.py:178-192  adjust_to_tile target size: w'=(W//T)*T, h'=(ceil(w'/(W/H))//T)*T."""
    aspect = W / H
    w_fit = (W // T) * T
    h_fit = (math.ceil(w_fit / aspect) // T) * T
    return w_fit, h_fit


def area_table(ssize, dsize):
    """One axis of OpenCV's computeResizeAreaTab (imgproc/resize.cpp; cv2 is a third-party dependency
    of the reference -- requirements.txt:8 -- whose INTER_AREA call sits at utils/tools.py:194).
    Returns a list of (dst index, src index, float32 weight) in OpenCV's order.  Pinned by
    tests/test_oracle_golden.py against the installed cv2 itself."""
    inv_scale = float(dsize) / float(ssize)
    scale = 1.0 / inv_scale
    tab = []
    for dx in range(dsize):
        fsx1 = dx * scale
        fsx2 = fsx1 + scale
        cell = min(scale, ssize - fsx1)
        sx1, sx2 = math.ceil(fsx1), math.floor(fsx2)
        sx2 = min(sx2, ssize - 1)
        sx1 = min(sx1, sx2)
        if sx1 - fsx1 > 1e-3:
            tab.append((dx, sx1 - 1, np.float32((sx1 - fsx1) / cell)))
        for sx in range(sx1, sx2):
            tab.append((dx, sx, np.float32(1.0 / cell)))
        if fsx2 - sx2 > 1e-3:
            tab.append((dx, sx2, np.float32(min(min(fsx2 - sx2, 1.0), cell) / cell)))
    return tab


def resize_area(img, w, h):
    """cv2.resize(img, (w, h), interpolation=cv2.INTER_AREA) for u8 images and non-integer down-scales,
    restated from OpenCV's resizeArea_<uchar, float>: per source row a float buffer
    buf[dx] = sum_k S[sx_k]*alpha_k (sequential, multiply and add rounded separately), rows combined
    as sum = beta_0*buf, sum += beta_j*buf, output cvRound(sum) saturated.  Bit-exact with cv2 4.13."""
    img = np.asarray(img)
    sh, sw = img.shape[:2]
    cn = 1 if img.ndim == 2 else img.shape[2]
    src = img.reshape(sh, sw, cn)
    xt, yt = area_table(sw, w), area_table(sh, h)
    K = max(np.bincount([t[0] for t in xt]))
    xi = np.zeros((w, K), np.int64)
    xa = np.zeros((w, K), np.float32)
    xn = np.zeros(w, np.int64)
    for d, si, a in xt:
        xi[d, xn[d]], xa[d, xn[d]] = si, a
        xn[d] += 1
    out = np.zeros((h, w, cn), np.uint8)
    acc, prev_dy = None, -1
    for dy, sy, beta in yt:
        row = src[sy].astype(np.float32)
        buf = np.zeros((w, cn), np.float32)
        for k in range(K):
            term = (row[xi[:, k]] * xa[:, k][:, None]).astype(np.float32)
            buf = np.where((xn > k)[:, None], (buf + term).astype(np.float32), buf)
        scaled = (np.float32(beta) * buf).astype(np.float32)
        if dy != prev_dy:
            if prev_dy >= 0:
                out[prev_dy] = np.clip(np.rint(acc), 0, 255).astype(np.uint8)
            acc, prev_dy = scaled, dy
        else:
            acc = (acc + scaled).astype(np.float32)
    out[prev_dy] = np.clip(np.rint(acc), 0, 255).astype(np.uint8)
    return out.reshape(h, w) if img.ndim == 2 else out


def augment_optimize_port(px_dist, px_count, dset_probs, n_classes, input_size, rate_coef_range=(1, 21),
                          threshold_range=(0, 3.), rate_range=(0, 4), n_samples_ratio=0.36):
    """utils/augment.py:92-187 as written (grid search over rate coefficient x threshold, JSD argmin).
    Returns (optim dict with 'rates', list of per-grid-point dicts)."""
    eps = 1e-8
    px_dist = np.array(px_dist, dtype='long')
    dset_probs = np.array(dset_probs, dtype='float32') + eps
    oversample_filter = np.clip(1 / n_classes - dset_probs, a_min=0, a_max=1.)
    probs = px_dist / px_count
    probs_weighted = np.multiply(np.multiply(probs, 1 / dset_probs), oversample_filter)
    scores = np.sqrt(np.sum(probs_weighted, axis=1))
    rate_coefs = np.arange(min(rate_coef_range), max(rate_coef_range), 1.)
    thresholds = np.arange(min(threshold_range), max(threshold_range), 0.05)
    balanced = np.empty(n_classes)
    balanced.fill(1 / n_classes)
    data, jsds = [], []
    for rate_coef in rate_coefs:
        for threshold in thresholds:
            over_sample = scores > threshold
            rates = np.multiply(over_sample, rate_coef * scores).astype(int)
            rates = np.clip(rates, rate_range[0], rate_range[1])
            if np.sum(rates) < int(n_samples_ratio * input_size):
                full_px_dist = px_dist + np.multiply(np.expand_dims(rates, axis=1), px_dist)
                full_px_probs = np.sum(full_px_dist, axis=0) / np.sum(full_px_dist)
                m2_s, jsd_s = m2(full_px_probs, n_classes), jsd(full_px_probs, balanced)
                jsds.append(jsd_s)
                data.append({'probs': full_px_probs, 'threshold': threshold, 'rate_coef': rate_coef, 'rates': rates,
                             'n_samples': int(np.sum(full_px_dist) / px_count), 'aug_n_samples': np.sum(rates),
                             'jsd': jsd_s, 'm2': m2_s})
    assert len(jsds) > 0, 'No augmentation optimization found.'
    return data[int(np.argmin(np.asarray(jsds)))], data


# ----------------------------------------------------------------------------------------------
# class_encode / colourize  (utils/tools.py:412-449, 322-358)
# ----------------------------------------------------------------------------------------------


def class_encode_port(tiles, palette):
    """utils/tools.py:412-449 as written: C full passes with boolean temporaries over
    [N*H*W, 3]; f64 scratch initialised to ONE (437) so unmatched colours become class 1;
    later palette entries overwrite earlier ones."""
    tiles = np.asarray(tiles)
    assert tiles.shape[1] == 3
    n, ch, h, w = tiles.shape
    flat = np.moveaxis(tiles, 1, -1).reshape(n * h * w, ch)
    enc = np.ones(n * h * w)
    for idx, colour in enumerate(palette):
        hit = np.all(flat == np.array(colour), axis=1)
        enc[hit] = idx
    return enc.reshape(n, h, w).astype(np.uint8)


def class_encode(tiles, palette):
    """Same result as class_encode_port via one 24-bit key compare (fast checker)."""
    tiles = np.asarray(tiles, dtype=np.uint8)
    assert tiles.shape[1] == 3
    key = (tiles[:, 0].astype(np.uint32) << 16) | (tiles[:, 1].astype(np.uint32) << 8) | tiles[:, 2]
    out = np.ones(key.shape, dtype=np.uint8)
    for idx, c in enumerate(palette):
        out[key == ((int(c[0]) << 16) | (int(c[1]) << 8) | int(c[2]))] = idx
    return out


def class_encode_hwc(rgb, palette):
    """class_encode on an [H,W,3] image (what Evaluator.load does to pred and GT,
    utils/evaluate.py:103-108) -> [H,W] u8."""
    rgb = np.asarray(rgb, dtype=np.uint8)
    return class_encode(np.moveaxis(rgb, 2, 0)[None], palette)[0]


def colourize_port(labels, n_classes, palette):
    """utils/tools.py:322-358 as written: stack label x3, then for i in range(C) rows equal to
    [i,i,i] <- palette[i], sequentially and in place (so a palette colour [k,k,k] with
    i < k < C would be re-mapped by a later pass)."""
    labels = np.asarray(labels)
    n, a, b = labels.shape
    data = np.moveaxis(np.stack((labels,) * 3, axis=1), 1, -1).reshape(n * a * b, 3)
    for i in range(n_classes):
        hit = np.all(data == np.array([i, i, i]), axis=1)
        data[hit] = palette[i]
    return data.reshape(n, a, b, 3)


def colourize_lut(n_classes, palette):
    """Closed form of the sequential in-place passes of colourize (utils/tools.py:352-356):
    the colour label i finally lands on after passes i+1..C-1 (chains through grey colours)."""
    lut = np.zeros((n_classes, 3), dtype=np.int64)
    for i in range(n_classes):
        cur = [int(v) for v in palette[i]]
        for j in range(i + 1, n_classes):
            if cur == [j, j, j]:
                cur = [int(v) for v in palette[j]]
        lut[i] = cur
    return lut


def colourize(labels, n_classes, palette):
    return colourize_lut(n_classes, palette)[np.asarray(labels)]


# ----------------------------------------------------------------------------------------------
# Profiling  (utils/profile.py:21-150, utils/metrics.py:90-132)
# ----------------------------------------------------------------------------------------------


def jsd(p, q):
    """utils/metrics.py:107-111."""
    eps = 1e-8
    m = 0.5 * (p + q + eps)
    return 0.5 * np.sum(p * np.log(p / m + eps)) + 0.5 * np.sum(q * np.log(q / m + eps))


def m2(p, n_classes):
    """utils/metrics.py:131-132."""
    assert n_classes > 1
    return (n_classes / (n_classes - 1)) * (1 - np.sum(p ** 2))


def tile_histograms(masks, n_classes):
    """utils/profile.py:109-111: px_dist[n, c] = #pixels of class c in tile n (i64)."""
    masks = np.asarray(masks)
    out = np.zeros((masks.shape[0], n_classes), dtype=np.int64)
    for i in range(masks.shape[0]):
        out[i] = np.bincount(masks[i].ravel(), minlength=n_classes)[:n_classes]
    return out


def profile_port(imgs, masks, n_classes, tile_size):
    """utils/profile.py:85-147 as written: batch-1 loop, torch.mean/std (unbiased) per tile in
    f32, one_hot + np.sum histogram, then the C-vector maths in f64."""
    imgs = np.asarray(imgs)
    masks = np.asarray(masks)
    n = imgs.shape[0]
    ch = imgs.shape[1]
    px_mean = torch.zeros(ch)
    px_std = torch.zeros(ch)
    px_dist = []
    for i in range(n):
        img = torch.tensor(imgs[i:i + 1]).float()
        mask = torch.tensor(masks[i:i + 1]).long()
        if ch == 3:
            px_mean += torch.mean(img, (0, 2, 3))
            px_std += torch.std(img, (0, 2, 3))
        else:
            px_mean += torch.mean(img)
            px_std += torch.std(img)
        onehot = torch.nn.functional.one_hot(mask, num_classes=n_classes).permute(0, 3, 1, 2)
        px_dist.append(np.sum(onehot.numpy(), axis=(2, 3)))
    px_mean /= n
    px_std /= n
    px_dist = np.concatenate(px_dist)
    return _profile_tail(px_dist, px_mean.tolist(), px_std.tolist(), n, n_classes, tile_size)


def _profile_tail(px_dist, px_mean, px_std, n, n_classes, tile_size):
    dset_px_dist = np.sum(px_dist, axis=0)
    dset_px_count = np.sum(dset_px_dist)
    probs = dset_px_dist / dset_px_count
    assert dset_px_count / (tile_size * tile_size) == n  # utils/profile.py:125-126
    weights = 1 / (np.log(1.02 + probs))  # utils/profile.py:129-130
    weights = weights / np.max(weights)
    balanced = np.full(n_classes, 1 / n_classes)
    return {
        "px_mean": list(px_mean), "px_std": list(px_std), "px_dist": px_dist,
        "dset_px_dist": dset_px_dist, "dset_px_count": int(dset_px_count),
        "probs": probs, "weights": weights,
        "m2": float(m2(probs, n_classes)), "jsd": float(jsd(probs, balanced)),
    }


def profile(imgs, masks, n_classes, tile_size):
    """Fast checker: per-tile moments from exact integer sums (f64), histograms by bincount."""
    imgs = np.asarray(imgs)
    n, ch = imgs.shape[0], imgs.shape[1]
    x = imgs.reshape(n, ch, -1).astype(np.float64)
    if ch == 3:
        cnt = x.shape[2]
        s1 = x.sum(axis=2)
        s2 = (x * x).sum(axis=2)
    else:
        cnt = x.shape[1] * x.shape[2]
        s1 = x.sum(axis=(1, 2))[:, None]
        s2 = (x * x).sum(axis=(1, 2))[:, None]
    mean = s1 / cnt
    var = (s2 - s1 * s1 / cnt) / (cnt - 1)
    px_mean = mean.mean(axis=0).astype(np.float32)
    px_std = np.sqrt(var).mean(axis=0).astype(np.float32)
    return _profile_tail(tile_histograms(masks, n_classes), px_mean.tolist(), px_std.tolist(),
                         n, n_classes, tile_size)


# ----------------------------------------------------------------------------------------------
# Stitching  (utils/tools.py:209-319)
# ----------------------------------------------------------------------------------------------


def _softmax0(a):
    """torch CPU softmax over axis 0, the call the reference makes (utils/tools.py:267-268)."""
    return torch.nn.functional.softmax(torch.from_numpy(np.ascontiguousarray(a)), dim=0).numpy()


def stitch_grid(h, w, T, S):
    """utils/tools.py:235-236: tiles per row / column that reconstruct() consumes."""
    if S < T:
        return h // S - 1, w // S - 1
    return h // S, w // S


def stitch_map_port(tiles, h, w, T, S):
    """utils/tools.py:239-309 as written (offset == 0): horizontal merge of each tile row with
    softmax-averaged overlap bands, then vertical merge of the row strips, in place on a copy.
    Returns the [C,h,w] f32 map that feeds np.argmax (utils/tools.py:313)."""
    tiles = np.array(tiles, dtype=np.float32, copy=True)
    n_classes = tiles.shape[1]
    n_rows, n_cols = stitch_grid(h, w, T, S)
    olap = T - S
    full = np.empty((n_classes, h, w), dtype=np.float32)
    prev_bottom = None
    row_idx = 0
    for i in range(n_rows):
        cur = tiles[i * n_cols]
        strip = np.empty((n_classes, T, w), dtype=np.float32)
        col = 0
        for j in range(n_cols):
            cw = cur.shape[2]
            if j < n_cols - 1:
                nxt = tiles[i * n_cols + j + 1]
                a = _softmax0(cur[:, :, cw - olap:cw])
                b = _softmax0(nxt[:, :, 0:olap])
                cur[:, :, cw - olap:cw] = (a + b) / 2
                strip[:, :, col:col + cw] = cur
                col += cw
                cur = nxt[:, :, olap:]
            else:
                strip[:, :, col:col + cw] = cur
        sh = strip.shape[1]
        bottom = strip[:, sh - olap:sh, :]
        if i > 0:
            merged = (_softmax0(strip[:, 0:olap, :]) + _softmax0(prev_bottom)) / 2
            strip[:, 0:olap, :] = merged
        if i == 0 or 0 < i < n_rows - 1:
            strip = strip[:, 0:sh - olap, :]
        full[:, row_idx:row_idx + strip.shape[1], :] = strip
        row_idx += strip.shape[1]
        prev_bottom = bottom
    return full


def stitch_map(tiles, nr, nc, T, S):
    """Closed form of stitch_map_port (SURVEY.md A.3).  nr x nc tiles of [C,T,T];
    S == T/2: output (nr+1)S x (nc+1)S; S == T: pure scatter.  Every logit is consumed by
    exactly one S x S output block."""
    tiles = np.asarray(tiles, dtype=np.float32)
    C = tiles.shape[1]
    L = tiles.reshape(nr, nc, C, T, T)
    if S == T:
        return np.ascontiguousarray(L.transpose(2, 0, 3, 1, 4).reshape(C, nr * T, nc * T))
    assert 2 * S == T
    h, w = (nr + 1) * S, (nc + 1) * S

    def hrow(i):
        # merged strip of tile row i: [C, T, w]
        strip = np.empty((C, T, w), dtype=np.float32)
        for kx in range(nc + 1):
            xs = slice(kx * S, (kx + 1) * S)
            if kx == 0:
                strip[:, :, xs] = L[i, 0][:, :, 0:S]
            elif kx == nc:
                strip[:, :, xs] = L[i, nc - 1][:, :, S:T]
            else:
                strip[:, :, xs] = (_softmax0(L[i, kx - 1][:, :, S:T]) + _softmax0(L[i, kx][:, :, 0:S])) / 2
        return strip

    strips = [hrow(i) for i in range(nr)]
    out = np.empty((C, h, w), dtype=np.float32)
    for ky in range(nr + 1):
        ys = slice(ky * S, (ky + 1) * S)
        if ky == 0:
            out[:, ys] = strips[0][:, 0:S]
        elif ky == nr:
            out[:, ys] = strips[nr - 1][:, S:T]
        else:
            out[:, ys] = (_softmax0(strips[ky - 1][:, S:T]) + _softmax0(strips[ky][:, 0:S])) / 2
    return out


def stitch_labels(stitched):
    """utils/tools.py:313: np.argmax over the class axis (first maximum wins)."""
    return np.argmax(stitched, axis=0).astype(np.uint8)


def top2_margin(stitched):
    """Gap between the largest and second-largest class value per pixel (for bucketing
    argmax mismatches by margin, SURVEY.md 7.2)."""
    part = np.partition(stitched, stitched.shape[0] - 2, axis=0)
    return part[-1] - part[-2]


def nn_index_map(n_src, n_dst):
    """OpenCV INTER_NEAREST source index for each destination index
    (cv2.resize in utils/tools.py:316-317): min(floor(x * (1/(n_dst/n_src))), n_src-1),
    evaluated in double precision like resizeNN's x_ofs table."""
    inv_scale = n_dst / n_src
    scale = 1.0 / inv_scale
    idx = np.floor(np.arange(n_dst, dtype=np.float64) * scale).astype(np.int64)
    return np.minimum(idx, n_src - 1).astype(np.int32)


def resample_labels(labels, w_full, h_full):
    """Label-space equivalent of colourize -> cv2.resize(INTER_NEAREST) -> class_encode
    (utils/tools.py:312-317, utils/evaluate.py:104-107; SURVEY.md A.4)."""
    h, w = labels.shape
    return labels[nn_index_map(h, h_full)[:, None], nn_index_map(w, w_full)[None, :]]


def reconstruct_port(tile_batches, h, w, w_full, h_full, T, S, palette, n_classes):
    """utils/tools.py:209-319 end to end: concatenate the per-batch logits, stitch, argmax,
    colourize, cv2.resize(INTER_NEAREST) to (w_full, h_full).  Returns f32 RGB [h_full,w_full,3]."""
    import cv2
    tiles = np.concatenate([np.asarray(t) for t in tile_batches], axis=0)
    full = stitch_map_port(tiles, h, w, T, S)
    rgb = colourize_port(np.argmax(full[None], axis=1), n_classes, palette)
    return cv2.resize(rgb[0].astype("float32"), (w_full, h_full), interpolation=cv2.INTER_NEAREST)


# ----------------------------------------------------------------------------------------------
# Evaluation  (utils/evaluate.py:150-176, utils/metrics.py:45-87)
# ----------------------------------------------------------------------------------------------


def inject_coverage(y_true, y_pred, n_labels):
    """utils/evaluate.py:172-174: y_true[i] = y_pred[i] = i for i < len(labels), in place on
    the flattened vectors."""
    y_true = np.array(y_true, copy=True).ravel()
    y_pred = np.array(y_pred, copy=True).ravel()
    for i in range(min(n_labels, y_true.size)):
        y_true[i] = i
        y_pred[i] = i
    return y_true, y_pred


def confusion_counts(y_true, y_pred, n_classes):
    """i64 confusion matrix M[t, p]."""
    idx = np.asarray(y_true).ravel().astype(np.int64) * n_classes + np.asarray(y_pred).ravel().astype(np.int64)
    return np.bincount(idx, minlength=n_classes * n_classes).reshape(n_classes, n_classes).astype(np.int64)


def metrics_port(y_true, y_pred, labels):
    """utils/metrics.py:45-87 as written: five independent scikit-learn calls."""
    from sklearn.metrics import (classification_report, confusion_matrix, f1_score,
                                 jaccard_score, matthews_corrcoef)
    return {
        "f1": f1_score(y_true, y_pred, average="weighted", zero_division=0),
        "iou": jaccard_score(y_true, y_pred, average="weighted"),
        "mcc": matthews_corrcoef(y_true, y_pred),
        "cmatrix": confusion_matrix(y_true, y_pred, normalize="true"),
        "report": classification_report(y_true, y_pred, target_names=labels, output_dict=True,
                                        zero_division=0),
    }


def metrics_from_confusion(M, labels=None):
    """Everything utils/metrics.py reports, derived from one i64 matrix M[t,p]
    (SURVEY.md A.6; equal to scikit-learn 1.9.0 on the present classes)."""
    M = np.asarray(M, dtype=np.int64)
    C = M.shape[0]
    tp = np.diag(M).astype(np.float64)
    sup = M.sum(axis=1).astype(np.float64)
    pred = M.sum(axis=0).astype(np.float64)
    total = float(M.sum())
    with np.errstate(divide="ignore", invalid="ignore"):
        prec = np.where(pred > 0, tp / pred, 0.0)
        rec = np.where(sup > 0, tp / sup, 0.0)
        den = 2 * tp + (pred - tp) + (sup - tp)
        f1 = np.where(den > 0, 2 * tp / den, 0.0)
        union = pred + sup - tp
        iou = np.where(union > 0, tp / union, 0.0)
        cm = np.where(sup[:, None] > 0, M / sup[:, None], 0.0)
    wf1 = float((f1 * sup).sum() / total)
    wiou = float((iou * sup).sum() / total)
    c = tp.sum()
    cov_ytyp = c * total - (sup * pred).sum()
    cov_ypyp = total * total - (pred * pred).sum()
    cov_ytyt = total * total - (sup * sup).sum()
    mcc = 0.0 if cov_ypyp * cov_ytyt == 0 else float(cov_ytyp / math.sqrt(cov_ytyt * cov_ypyp))
    out = {"f1": wf1, "iou": wiou, "mcc": mcc, "cmatrix": cm}
    if labels is not None:
        rep = {}
        for i in range(C):
            rep[labels[i]] = {"precision": float(prec[i]), "recall": float(rec[i]),
                              "f1-score": float(f1[i]), "support": float(sup[i])}
        rep["accuracy"] = float(c / total)
        rep["macro avg"] = {"precision": float(prec.mean()), "recall": float(rec.mean()),
                            "f1-score": float(f1.mean()), "support": total}
        rep["weighted avg"] = {"precision": float((prec * sup).sum() / total),
                               "recall": float((rec * sup).sum() / total),
                               "f1-score": wf1, "support": total}
        out["report"] = rep
    return out


# ----------------------------------------------------------------------------------------------
# Multi-loss  (models/modules/loss.py:71-194)
# ----------------------------------------------------------------------------------------------

LOSS_DEFAULTS = dict(ce=0.5, dice=0.5, focal=0.5, smooth=1.0, gamma=2.0, alpha=0.25, eps=1e-8)


def multiloss_port(pred, target, n_classes, weights=None, weighted=False, need_grad=True, **kw):
    """models/modules/loss.py:107-112,137-146,174-194 as written, on torch CPU with autograd:
    CrossEntropyLoss (+class weights if `weighted`), softmax/one_hot Dice, softmax/one_hot Focal.
    Returns (loss, ce, dice, focal, grad-or-None) as numpy."""
    k = dict(LOSS_DEFAULTS)
    k.update(kw)
    z = torch.tensor(np.asarray(pred, dtype=np.float32), requires_grad=need_grad)
    t = torch.tensor(np.asarray(target)).long()
    if weighted:
        ce_fn = torch.nn.CrossEntropyLoss(torch.tensor(np.asarray(weights)).float())
    else:
        ce_fn = torch.nn.CrossEntropyLoss()
    ce = ce_fn(z, t)
    onehot = torch.nn.functional.one_hot(t, num_classes=n_classes).permute(0, 3, 1, 2)
    probs = torch.nn.functional.softmax(z, dim=1)
    inter = torch.sum(probs * onehot, dim=(0, 2, 3))
    card = torch.sum(probs + onehot, dim=(0, 2, 3))
    dice = (1 - (2.0 * inter + k["smooth"]) / (card + k["smooth"])).mean()
    soft = torch.nn.functional.softmax(z, dim=1) + k["eps"]
    focal_px = torch.sum(onehot * (-k["alpha"] * torch.pow(-soft + 1.0, k["gamma"]) * torch.log(soft)), dim=1)
    focal = torch.mean(focal_px)
    loss = k["ce"] * ce + k["dice"] * dice + k["focal"] * focal
    grad = None
    if need_grad:
        loss.backward()
        grad = z.grad.numpy()
    return (loss.item(), ce.item(), dice.item(), focal.item(), grad)


def multiloss(pred, target, n_classes, weights=None, weighted=False, **kw):
    """Closed form (SURVEY.md A.5) in f64: returns (loss, ce, dice, focal, grad[B,C,H,W] f64,
    partials[2C+3] = [I_c..., K_c..., ce_num, ce_den, focal_sum])."""
    k = dict(LOSS_DEFAULTS)
    k.update(kw)
    z = np.asarray(pred, dtype=np.float32).astype(np.float64)
    t = np.asarray(target).astype(np.int64)
    B, C, H, W = z.shape
    N = B * H * W
    zmax = z.max(axis=1, keepdims=True)
    e = np.exp(z - zmax)
    ssum = e.sum(axis=1, keepdims=True)
    p = e / ssum
    lse = (zmax + np.log(ssum))[:, 0]
    onehot = np.moveaxis(np.eye(C)[t], 3, 1)
    wv = np.asarray(weights, dtype=np.float32).astype(np.float64) if weighted else np.ones(C)
    wt = wv[t]
    zt = np.take_along_axis(z, t[:, None], axis=1)[:, 0]
    pt = np.take_along_axis(p, t[:, None], axis=1)[:, 0]
    ce_num = float((wt * (lse - zt)).sum())
    ce_den = float(wt.sum())
    ce = ce_num / ce_den
    I = (p * onehot).sum(axis=(0, 2, 3))
    K = (p + onehot).sum(axis=(0, 2, 3))
    s = k["smooth"]
    dice = float(np.mean(1 - (2 * I + s) / (K + s)))
    q = pt + k["eps"]
    focal_sum = float((-k["alpha"] * (1 - q) ** k["gamma"] * np.log(q)).sum())
    focal = focal_sum / N
    loss = k["ce"] * ce + k["dice"] * dice + k["focal"] * focal
    # gradient
    g_ce = (wt / ce_den)[:, None] * (p - onehot)
    a = -2.0 / ((K + s) * C)
    b = (2 * I + s) / ((K + s) ** 2 * C)
    g = a[None, :, None, None] * onehot + b[None, :, None, None]
    g_dice = p * (g - (g * p).sum(axis=1, keepdims=True))
    dq = (k["alpha"] / N) * (k["gamma"] * (1 - q) ** (k["gamma"] - 1) * np.log(q) - (1 - q) ** k["gamma"] / q)
    g_focal = (dq * pt)[:, None] * (onehot - p)
    grad = k["ce"] * g_ce + k["dice"] * g_dice + k["focal"] * g_focal
    partials = np.concatenate([I, K, [ce_num, ce_den, focal_sum]])
    return loss, ce, dice, focal, grad, partials


# ----------------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md 8d) -- shared by tests and bench so both sides see the same bytes
# ----------------------------------------------------------------------------------------------

MLP_SKEW = [0.5495, 0.0, 0.2215, 0.0804, 0.1015, 0.0007, 0.0010, 0.0321, 0.0132]


def synth_image(index, W, H, ch):
    """u8 image: 64-px blocky uniform noise + per-pixel noise (three different fields for
    colour so the image is not grey)."""
    rng = np.random.default_rng(1000 + index)
    planes = []
    for _ in range(ch):
        coarse = rng.integers(40, 216, size=((H + 63) // 64, (W + 63) // 64), dtype=np.int32)
        field = np.kron(coarse, np.ones((64, 64), dtype=np.int32))[:H, :W]
        field = field + rng.integers(-32, 33, size=(H, W), dtype=np.int32)
        planes.append(np.clip(field, 0, 255).astype(np.uint8))
    return planes[0] if ch == 1 else np.stack(planes, axis=2)


def synth_labels(index, W, H, n_classes, skew=False, block=50):
    rng = np.random.default_rng(5000 + index)
    if skew:
        p = np.zeros(n_classes)
        p[:len(MLP_SKEW)] = MLP_SKEW[:n_classes]
        p = p / p.sum()
    else:
        p = np.full(n_classes, 1.0 / n_classes)
    coarse = rng.choice(n_classes, size=((H + block - 1) // block, (W + block - 1) // block), p=p)
    return np.kron(coarse, np.ones((block, block), dtype=np.int64))[:H, :W].astype(np.uint8)


def synth_mask(index, W, H, palette, skew=False, off_palette=0.001):
    """RGB u8 mask from the schema palette over 50-px label blocks, plus a fraction of
    off-palette pixels (exercises the 'unmatched -> class 1' rule)."""
    labels = synth_labels(index, W, H, len(palette), skew=skew)
    rgb = np.asarray(palette, dtype=np.uint8)[labels]
    if off_palette > 0:
        rng = np.random.default_rng(9000 + index)
        n_off = int(W * H * off_palette)
        ys = rng.integers(0, H, n_off)
        xs = rng.integers(0, W, n_off)
        rgb[ys, xs] = rng.integers(0, 256, size=(n_off, 3), dtype=np.uint8)
    return rgb


# ---------------------------------------------------------------------------------------------
# model-file boundary (models/modules/checkpoint.py:53-66, models/model.py:78-121)
# ---------------------------------------------------------------------------------------------

def fill_state_dict(state_dict):
    """Deterministic, name-independent fill of a network state dict (tensor i of the ordered dict is drawn
    from generator seed i), used to give the reference DeepLab and ours THE SAME weights without shipping a
    240 MB file: gen_golden.py runs the reference network with these weights and stores the output."""
    out = type(state_dict)()
    for i, (k, v) in enumerate(state_dict.items()):
        g = torch.Generator().manual_seed(i)
        if v.dtype in (torch.int64, torch.int32):
            out[k] = torch.zeros_like(v)
        elif k.endswith("running_var"):
            out[k] = torch.rand(v.shape, generator=g) * 0.5 + 0.75
        elif k.endswith("running_mean"):
            out[k] = torch.randn(v.shape, generator=g) * 0.05
        elif v.dim() <= 1:                       # BatchNorm affine terms, biases
            out[k] = 1.0 + torch.randn(v.shape, generator=g) * 0.05 if k.endswith("weight") else torch.randn(v.shape, generator=g) * 0.05
        else:                                    # convolution kernels: keep activations O(1) through 100 layers
            fan_in = v[0].numel()
            out[k] = torch.randn(v.shape, generator=g) * (1.6 / fan_in) ** 0.5
    return out


def augment_fixture_tile(ch, T=512):
    """Formula-generated tile + label mask for the augment_transform golden vectors (smooth enough to compress)."""
    yy, xx = np.mgrid[0:T, 0:T]
    img = np.stack([(xx // 7 * 5 + yy // 11 * 3 + 40 * c) % 256 for c in range(ch)]).astype(np.uint8)[None]
    mask = ((xx // 60 + yy // 45) % 9).astype(np.uint8)[None]
    return img, mask


def reconstruct_fixture_tiles(fixture, case):
    """Logit tiles of one case of tests/golden/reconstruct.npz.  gen_golden.py draws them case after case from one
    generator (seed 15); random floats do not compress, so the file keeps only the SHA-256 of each case's tiles and
    the draw is repeated here and checked against it."""
    rng = np.random.default_rng(15)
    for name in (str(c) for c in fixture["recon_cases"]):
        nr, nc, T, S, h, w, w_full, h_full, C = (int(v) for v in fixture["recon_%s_geom" % name])
        tiles = (rng.standard_normal((nr * nc, C, T, T)) * 3).astype(np.float32)
        if name == case:
            digest = hashlib.sha256(tiles.tobytes()).hexdigest()
            assert digest == str(fixture["recon_%s_tiles_sha256" % name]), "regenerated tiles differ from the fixture's"
            return tiles
    raise KeyError(case)


# ---------------------------------------------------------------------------------------------
# Augmentation warps: tools.augment_transform (reference utils/tools.py:452-594) restated without
# OpenCV's image functions.  The reference calls cv2.warpPerspective / cv2.resize (OpenCV is not
# vendored; requirements.txt:8 pins cv2 >= 3.4); their published algorithms are restated here and
# pinned three ways: the golden vectors the reference produced (tests/golden/warp.npz), the
# reference's own function on other seeds (tests/test_oracle_golden.py, build container) and the
# installed cv2 run on the same inputs.  Only cv2.getPerspectiveTransform / cv2.invert (an 8x8 and
# a 3x3 solve on the host) are still OpenCV calls, as in the product.
# ---------------------------------------------------------------------------------------------

def _reflect101(p, n):
    """cv2.BORDER_REFLECT_101 (borderInterpolate): ... 2 1 | 0 1 2 ... n-2 n-1 | n-2 n-3 ..., reflected until inside
    (closed form: the pattern has period 2(n-1))."""
    p = np.asarray(p)
    if n == 1:
        return np.zeros_like(p)
    q = np.mod(p, 2 * (n - 1))
    return np.where(q < n, q, 2 * (n - 1) - q)


def _sat_short(v):
    """saturate_cast<short>: warpPerspective hands remap its integer coordinates as 16-bit values."""
    return np.clip(v, -32768, 32767)


def warp_fixed_coords(m_inv, w, h, tab):
    """Source coordinates of cv2.warpPerspective for every destination pixel, as OpenCV computes them
    (imgproc/imgwarp.cpp WarpPerspectiveInvoker): double precision, per block of bw0 columns the
    numerators / denominator at the block's first column plus M * x1 inside it, scaled by tab / W
    (tab = 32 sub-pixel steps for INTER_LINEAR, 1 for INTER_NEAREST), rounded half-to-even."""
    bh0 = min(16, h)
    bw0 = min(1024 // bh0, w)
    xb = (np.arange(w) // bw0 * bw0).astype(np.float64)[None, :]
    x1 = (np.arange(w) % bw0).astype(np.float64)[None, :]
    y = np.arange(h, dtype=np.float64)[:, None]
    M = np.asarray(m_inv, dtype=np.float64)
    X0 = M[0, 0] * xb + M[0, 1] * y + M[0, 2]
    Y0 = M[1, 0] * xb + M[1, 1] * y + M[1, 2]
    W0 = M[2, 0] * xb + M[2, 1] * y + M[2, 2]
    W = W0 + M[2, 0] * x1
    W = np.where(W != 0, tab / np.where(W != 0, W, 1.0), 0.0)
    fX = np.clip((X0 + M[0, 0] * x1) * W, -2.0 ** 31, 2.0 ** 31 - 1)
    fY = np.clip((Y0 + M[1, 0] * x1) * W, -2.0 ** 31, 2.0 ** 31 - 1)
    return np.rint(fX).astype(np.int64), np.rint(fY).astype(np.int64)


def warp_perspective_linear_f32(img, m_inv):
    """cv2.warpPerspective(img f32, M, (w, h), INTER_LINEAR, BORDER_REFLECT_101) given inv(M) (what the
    reference's flags=INTER_AREA resolves to): 1/32-pixel coordinates, float bilinear table
    (1-fy)(1-fx), (1-fy)fx, fy(1-fx), fy*fx.  For 8-bit valued inputs every product and sum is exact."""
    h, w = img.shape[:2]
    X, Y = warp_fixed_coords(m_inv, w, h, 32.0)
    sx, sy = _sat_short(X >> 5), _sat_short(Y >> 5)
    one = np.float32(1)
    fx, fy = ((X & 31) / 32.0).astype(np.float32), ((Y & 31) / 32.0).astype(np.float32)
    wts = [(one - fy) * (one - fx), (one - fy) * fx, fy * (one - fx), fy * fx]
    if img.ndim == 3:
        wts = [t[..., None] for t in wts]
    x0, x1, y0, y1 = _reflect101(sx, w), _reflect101(sx + 1, w), _reflect101(sy, h), _reflect101(sy + 1, h)
    im = img.astype(np.float32)
    return im[y0, x0] * wts[0] + im[y0, x1] * wts[1] + im[y1, x0] * wts[2] + im[y1, x1] * wts[3]


def warp_perspective_nearest(mask, m_inv):
    """cv2.warpPerspective(mask, M, (w, h), INTER_NEAREST, BORDER_REFLECT_101) given inv(M)."""
    h, w = mask.shape[:2]
    X, Y = warp_fixed_coords(m_inv, w, h, 1.0)
    return mask[_reflect101(_sat_short(Y), h), _reflect101(_sat_short(X), w)]


def area_upscale_tab(ssize, dsize):
    """Tap table of cv2.resize(f32, INTER_AREA) when ENLARGING (imgproc/resize.cpp, area_mode with the linear
    kernel): first tap sx = floor(dx * ssize/dsize), second-tap weight fx = frac((dx+1) - (sx+1) * dsize/ssize)
    as f32 (0 when not positive), taps clamped to the last source sample."""
    scale, inv = ssize / dsize, dsize / ssize
    sx, fx = np.zeros(dsize, np.int64), np.zeros(dsize, np.float32)
    for dx in range(dsize):
        s = int(np.floor(dx * scale))
        f = np.float32((dx + 1) - (s + 1) * inv)
        f = np.float32(0) if f <= 0 else np.float32(f - np.floor(f))
        if s >= ssize - 1:
            f, s = np.float32(0), ssize - 1
        sx[dx], fx[dx] = s, f
    return sx, fx


def resize_area_upscale_f32(src, dsize):
    """cv2.resize(src f32 [S,S(,C)], (dsize, dsize), INTER_AREA) for dsize > S: rows first, then columns, every
    product and sum rounded to f32 separately (no fused multiply-add), as the installed OpenCV does."""
    S = src.shape[0]
    sx, fx = area_upscale_tab(S, dsize)
    one = np.float32(1)
    a0, a1 = one - fx, fx
    if src.ndim == 3:
        a0, a1 = a0[None, :, None], a1[None, :, None]
    rows = src[:, sx] * a0 + src[:, np.minimum(sx + 1, S - 1)] * a1
    b0 = (one - fx).reshape((-1,) + (1,) * (src.ndim - 1))
    b1 = fx.reshape(b0.shape)
    return (rows[sx] * b0 + rows[np.minimum(sx + 1, S - 1)] * b1).astype(np.float32)


def augment_params(random_state, w):
    """The random draws of perspective_shift + channel_shift in the reference's order (tools.py:577-580, 550):
    returns (inverse perspective matrix 3x3 f64, brightness shift int)."""
    import cv2
    pts1 = np.float32([[56, 65], [368, 52], [28, 387], [389, 390]])
    pts2 = pts1 + random_state.uniform(-0.06 * w, 0.06 * w, size=pts1.shape).astype(np.float32)
    m_inv = cv2.invert(cv2.getPerspectiveTransform(pts1, pts2))[1]
    return m_inv, int(random_state.uniform(10, 20))


def augment_transform_port(img, mask, random_state):
    """tools.augment_transform (reference utils/tools.py:452-594): img [1,ch,T,T], mask [1,T,T] ->
    (img u8 [ch,T,T] or [T,T], mask f32 [T,T]).  Perspective jitter (bilinear image / nearest mask, reflect-101),
    30-px crop, resize back to T (INTER_AREA image / INTER_NEAREST mask), brightness shift through int16."""
    nch = img.shape[1]
    im = np.squeeze(np.moveaxis(np.asarray(img, dtype=np.float32), 1, -1), axis=0)
    if nch == 1:
        im = im[..., 0]
    mk = np.squeeze(np.asarray(mask), axis=0)
    w = mk.shape[0]
    m_inv, shift = augment_params(random_state, w)
    wim = np.ascontiguousarray(warp_perspective_linear_f32(im, m_inv)[30:w - 30, 30:w - 30])
    wmk = warp_perspective_nearest(mk, m_inv)[30:w - 30, 30:w - 30]
    rim = resize_area_upscale_f32(wim, w)
    idx = np.minimum(np.floor(np.arange(w) * ((w - 60) / w)).astype(np.int64), w - 61)   # cv2 INTER_NEAREST
    rmk = wmk[idx][:, idx].astype(np.float32)
    out = np.uint8(np.clip(np.int16(rim) + shift, 0, 255))                              # channel_shift, tools.py:550-555
    if nch == 3:
        out = np.moveaxis(out, -1, 0)
    return out, rmk
