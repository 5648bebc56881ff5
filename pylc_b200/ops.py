"""
Torch-tensor front end of the C ABI: allocates outputs with the PyTorch caching allocator,
passes raw device pointers + the current CUDA stream to libpylc_b200.so, never synchronises.

PyTorch is plumbing here (device memory, streams); every per-pixel operation is a hand-written
sm_100a kernel behind include/pylc_b200.h.  No function in this module has a CPU path.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import LossCfg, PylcError, check


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise PylcError("pylc_b200 ops take CUDA tensors (there is no CPU fallback)")


def pitch_for(width_bytes):
    """Row pitch (bytes) that keeps every row 16-byte aligned for the vectorised kernels."""
    return (width_bytes + 15) // 16 * 16


def tile_grid(H, W, T, S):
    nH, nW = ctypes.c_int(0), ctypes.c_int(0)
    check(_lib.load().pylc_tile_grid(H, W, T, S, ctypes.byref(nH), ctypes.byref(nW)), "pylc_tile_grid")
    return nH.value, nW.value


def pinned_pitched(img):
    """Host staging: copy an [H,W] / [H,W,3] u8 array into pinned memory with 16-byte-aligned
    rows.  Returns (tensor [H, pitch] u8 pinned, pitch)."""
    img = np.asarray(img)
    H = img.shape[0]
    row = img.shape[1] * (img.shape[2] if img.ndim == 3 else 1)
    pitch = pitch_for(row)
    buf = torch.empty((H, pitch), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    buf.numpy()[:, :row] = img.reshape(H, row)
    return buf, pitch


def upload_image(img, device=None):
    """u8 image -> device tensor [H, pitch] with aligned rows (one async H2D copy)."""
    buf, pitch = pinned_pitched(img)
    return buf.to(device or torch.device("cuda"), non_blocking=True), pitch


def upload_pitched(host, out=None, device=None):
    """pylc_upload_pitched: H2D of a tightly packed (ideally pinned) [H,W] / [H,W,3] u8 host tensor
    or array into a 16-byte-pitched device buffer on the copy engine -- no host-side repack.
    Returns (tensor [H, pitch] u8, pitch)."""
    t = host if torch.is_tensor(host) else torch.from_numpy(np.ascontiguousarray(host))
    if t.is_cuda or t.dtype != torch.uint8 or not t.is_contiguous():
        raise PylcError("upload_pitched takes a contiguous u8 host tensor")
    H = t.shape[0]
    row = t.numel() // H
    pitch = pitch_for(row)
    if out is None:
        out = torch.empty((H, pitch), dtype=torch.uint8, device=device or torch.device("cuda"))
    check(_lib.load().pylc_upload_pitched(_p(out), pitch, ctypes.c_void_p(t.data_ptr()), row, row, H, _stream()),
          "pylc_upload_pitched")
    return out, pitch


# ---- test-time fit resize -------------------------------------------------------------------------

_AREA_TABLES = {}


def area_supported(W, H, w, h):
    """True when cv2.resize((W,H)->(w,h), INTER_AREA) is the general area filter the device kernel
    reproduces bit-exactly (pylc_area_supported)."""
    return bool(_lib.load().pylc_area_supported(int(W), int(H), int(w), int(h)))


def area_table_host(ssize, dsize):
    """pylc_area_table: (start i32 [dsize], count i32 [dsize], weights f32 [dsize, AREA_TAPS]) on the host."""
    start = np.empty(dsize, dtype=np.int32)
    count = np.empty(dsize, dtype=np.int32)
    weights = np.empty((dsize, _lib.AREA_TAPS), dtype=np.float32)
    check(_lib.load().pylc_area_table(int(ssize), int(dsize), start.ctypes.data, count.ctypes.data, weights.ctypes.data),
          "pylc_area_table")
    return start, count, weights


def area_tables(W, H, w, h, device):
    """Device copies of the x and y area tables, cached per geometry."""
    key = (W, H, w, h, str(device))
    hit = _AREA_TABLES.get(key)
    if hit is None:
        if len(_AREA_TABLES) > 64:
            _AREA_TABLES.clear()
        hit = _AREA_TABLES[key] = tuple(torch.from_numpy(a).to(device) for a in area_table_host(W, w) + area_table_host(H, h))
    return hit


def fit_resize_area(src, H, W, ch, pitch, h, w, out=None):
    """pylc_fit_resize_area_u8: cv2.resize(INTER_AREA) of a device-resident u8 image, bit-exact.
    Returns (fitted [h, pitch_out] u8, pitch_out)."""
    _need_cuda(src)
    if not area_supported(W, H, w, h):
        raise PylcError("fit_resize_area: (%d,%d)->(%d,%d) is not OpenCV's general area filter; use the host cv2 path"
                        % (W, H, w, h))
    tabs = area_tables(W, H, w, h, src.device)
    pitch_out = pitch_for(w * ch)
    if out is None:
        out = torch.empty((h, pitch_out), dtype=torch.uint8, device=src.device)
    check(_lib.load().pylc_fit_resize_area_u8(_p(src), H, W, ch, pitch, _p(out), h, w, pitch_out, *[_p(t) for t in tabs],
                                              _stream()), "pylc_fit_resize_area_u8")
    return out, pitch_out


# ---- extraction ---------------------------------------------------------------------------------


def tile_gather_u8(src, H, W, ch, pitch, T, S, stats=False, out=None):
    """pylc_tile_gather_u8: returns tiles [n,ch,T,T] u8 (and stat [n,ch,2] i64 = sum x, sum x^2)."""
    _need_cuda(src)
    nH, nW = tile_grid(H, W, T, S)
    n = nH * nW
    tiles = out if out is not None else torch.empty((n, ch, T, T), dtype=torch.uint8, device=src.device)
    stat = torch.zeros((n, ch, 2), dtype=torch.int64, device=src.device) if stats else None
    check(_lib.load().pylc_tile_gather_u8(_p(src), H, W, ch, pitch, T, S, _p(tiles), _p(stat), _stream()),
          "pylc_tile_gather_u8")
    return (tiles, stat) if stats else tiles


def mask_gather_encode_hist(src, H, W, pitch, T, S, palette, hist=True, out=None, px_dist=None):
    """pylc_mask_gather_encode_hist: returns (tiles [n,T,T] u8, px_dist [n,C] i64 or None).
    `px_dist`: an existing [n,C] i64 tensor to ADD the histograms into (the C ABI accumulates)."""
    _need_cuda(src)
    pal, C = _lib.palette_array(palette)
    nH, nW = tile_grid(H, W, T, S)
    n = nH * nW
    tiles = out if out is not None else torch.empty((n, T, T), dtype=torch.uint8, device=src.device)
    if px_dist is None:
        px_dist = torch.zeros((n, C), dtype=torch.int64, device=src.device) if hist else None
    check(_lib.load().pylc_mask_gather_encode_hist(_p(src), H, W, pitch, T, S, pal, C, _p(tiles), _p(px_dist),
                                                   _stream()), "pylc_mask_gather_encode_hist")
    return tiles, px_dist


def upload_stack(images, device=None, staging=None):
    """Equally sized u8 images [H,W] / [H,W,3] -> ONE device tensor [n, H, pitch] with 16-byte aligned rows
    (the `src` of the *_stack entry points; image stride = H * pitch).  `staging`: a pinned [>= n, H, pitch] u8
    tensor to reuse between calls.  Returns (stack, pitch, staging)."""
    first = np.asarray(images[0])
    H = first.shape[0]
    row = first.shape[1] * (first.shape[2] if first.ndim == 3 else 1)
    pitch = pitch_for(row)
    n = len(images)
    if staging is None or staging.shape[0] < n or tuple(staging.shape[1:]) != (H, pitch):
        staging = torch.empty((n, H, pitch), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    elif torch.cuda.is_available():
        torch.cuda.current_stream().synchronize()      # the previous upload may still be reading the buffer
    view = staging.numpy()
    for i, im in enumerate(images):
        im = np.asarray(im)
        if im.shape != first.shape or im.dtype != np.uint8:
            raise PylcError("upload_stack takes equally sized u8 images")
        view[i, :, :row] = im.reshape(H, row)
    return staging[:n].to(device or torch.device("cuda"), non_blocking=True), pitch, staging


def tile_gather_u8_stack(src, H, W, ch, pitch, T, S, stats=False, out=None, stat_out=None):
    """pylc_tile_gather_u8_stack: `src` [n_img, H, pitch] u8 (equally sized images) -> tiles
    [n_img*n, ch, T, T] u8 in image order (and stat [n_img*n, ch, 2] i64), one launch."""
    _need_cuda(src)
    if src.dim() != 3 or not src.is_contiguous():
        raise PylcError("tile_gather_u8_stack takes a contiguous [n_img, H, pitch] u8 stack")
    n_img, stride = src.shape[0], src.shape[1] * src.shape[2]
    nH, nW = tile_grid(H, W, T, S)
    n = nH * nW * n_img
    tiles = out if out is not None else torch.empty((n, ch, T, T), dtype=torch.uint8, device=src.device)
    stat = None
    if stats:
        stat = stat_out.zero_() if stat_out is not None else torch.zeros((n, ch, 2), dtype=torch.int64, device=src.device)
    check(_lib.load().pylc_tile_gather_u8_stack(_p(src), n_img, stride, H, W, ch, pitch, T, S, _p(tiles), _p(stat), _stream()),
          "pylc_tile_gather_u8_stack")
    return (tiles, stat) if stats else tiles


def mask_gather_encode_hist_stack(src, H, W, pitch, T, S, palette, hist=True, out=None, px_dist=None):
    """pylc_mask_gather_encode_hist_stack: `src` [n_img, H, pitch] u8 RGB masks -> (tiles [n_img*n, T, T] u8,
    px_dist [n_img*n, C] i64 or None) in image order, one launch.  `px_dist` given: added into."""
    _need_cuda(src)
    if src.dim() != 3 or not src.is_contiguous():
        raise PylcError("mask_gather_encode_hist_stack takes a contiguous [n_img, H, pitch] u8 stack")
    n_img, stride = src.shape[0], src.shape[1] * src.shape[2]
    pal, C = _lib.palette_array(palette)
    nH, nW = tile_grid(H, W, T, S)
    n = nH * nW * n_img
    tiles = out if out is not None else torch.empty((n, T, T), dtype=torch.uint8, device=src.device)
    if px_dist is None:
        px_dist = torch.zeros((n, C), dtype=torch.int64, device=src.device) if hist else None
    check(_lib.load().pylc_mask_gather_encode_hist_stack(_p(src), n_img, stride, H, W, pitch, T, S, pal, C, _p(tiles),
                                                         _p(px_dist), _stream()), "pylc_mask_gather_encode_hist_stack")
    return tiles, px_dist


def tile_gather_norm_f32(src, H, W, ch, pitch, T, S, mean, std, post_div=255.0, out_ch=3, out=None):
    """pylc_tile_gather_norm_f32: network-ready f32 tiles [n,out_ch,T,T]."""
    _need_cuda(src)
    nH, nW = tile_grid(H, W, T, S)
    n = nH * nW
    tiles = out if out is not None else torch.empty((n, out_ch, T, T), dtype=torch.float32, device=src.device)
    check(_lib.load().pylc_tile_gather_norm_f32(_p(src), H, W, ch, pitch, T, S, _lib.float3(mean), _lib.float3(std),
                                                float(post_div), out_ch, _p(tiles), _stream()),
          "pylc_tile_gather_norm_f32")
    return tiles


def tile_gather_norm_s2d(src, H, W, ch, pitch, T, S, mean, std, post_div=255.0):
    """pylc_tile_gather_norm_s2d_f32: network-ready tiles in the stem's space-to-depth layout, returned
    as a channels-last tensor of logical shape [n, 16, T/2+3, T/2+3]."""
    _need_cuda(src)
    nH, nW = tile_grid(H, W, T, S)
    n, Hs = nH * nW, T // 2 + 3
    tiles = torch.empty((n, 16, Hs, Hs), dtype=torch.float32, device=src.device, memory_format=torch.channels_last)
    check(_lib.load().pylc_tile_gather_norm_s2d_f32(_p(src), H, W, ch, pitch, T, S, _lib.float3(mean), _lib.float3(std),
                                                    float(post_div), _p(tiles), _stream()),
          "pylc_tile_gather_norm_s2d_f32")
    return tiles


def class_encode_nchw(rgb, palette, hist=False):
    """tools.class_encode on a CUDA [N,3,H,W] u8 tensor -> [N,H,W] u8 (+ [C] i64 histogram)."""
    _need_cuda(rgb)
    if rgb.dim() != 4 or rgb.shape[1] != 3:
        raise PylcError("Input data must be 3 channel (RGB)")
    rgb = rgb.contiguous()
    pal, C = _lib.palette_array(palette)
    n, _, h, w = rgb.shape
    out = torch.empty((n, h, w), dtype=torch.uint8, device=rgb.device)
    hs = torch.zeros((C,), dtype=torch.int64, device=rgb.device) if hist else None
    check(_lib.load().pylc_class_encode(_p(rgb), n, h, w, 0, 1, pal, C, _p(out), _p(hs), _stream()),
          "pylc_class_encode")
    return (out, hs) if hist else out


def class_encode_hwc(rgb, rows, cols, pitch, palette, n_img=1, hist=False):
    """class_encode on interleaved RGB rows (pitch bytes per row) -> [n_img, rows, cols] u8."""
    _need_cuda(rgb)
    pal, C = _lib.palette_array(palette)
    out = torch.empty((n_img, rows, cols), dtype=torch.uint8, device=rgb.device)
    hs = torch.zeros((C,), dtype=torch.int64, device=rgb.device) if hist else None
    check(_lib.load().pylc_class_encode(_p(rgb), n_img, rows, cols, pitch, 0, pal, C, _p(out), _p(hs), _stream()),
          "pylc_class_encode")
    return (out, hs) if hist else out


def profile_tiles(imgs, masks, n_classes):
    """pylc_profile_tiles: (stat [n,ch,2] i64 or None, px_dist [n,C] i64 or None)."""
    _need_cuda(imgs, masks)
    stat = px_dist = None
    n = (imgs if imgs is not None else masks).shape[0]
    ch = 1
    tile_px = 0
    if imgs is not None:
        imgs = imgs.contiguous()
        ch = imgs.shape[1]
        tile_px = imgs.shape[2] * imgs.shape[3]
        stat = torch.zeros((n, ch, 2), dtype=torch.int64, device=imgs.device)
    if masks is not None:
        masks = masks.contiguous()
        tile_px = masks.shape[1] * masks.shape[2]
        px_dist = torch.zeros((n, n_classes), dtype=torch.int64, device=masks.device)
    check(_lib.load().pylc_profile_tiles(_p(imgs), ch, _p(masks), n, tile_px, n_classes, _p(stat), _p(px_dist),
                                         _stream()), "pylc_profile_tiles")
    return stat, px_dist


# ---- stitching ----------------------------------------------------------------------------------


def stitch_dims(nr, nc, T, S):
    return ((nr + 1) * S, (nc + 1) * S) if S < T else (nr * S, nc * S)


def _tile_source(logits, nr, nc, tiles_per_batch):
    """(logits pointer, batch-table pointer, tiles per batch, C, device, batch table | None) of the stitch
    kernels' input: one contiguous [nr*nc,C,T,T] f32 tensor or a list of per-batch tensors."""
    if isinstance(logits, (list, tuple)):
        _need_cuda(*logits)
        C = logits[0].shape[1]
        dev = logits[0].device
        tpb = tiles_per_batch or logits[0].shape[0]
        for i, t in enumerate(logits):
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise PylcError("tile batches must be contiguous float32")
            if i < len(logits) - 1 and t.shape[0] != tpb:
                raise PylcError("all tile batches but the last must hold tiles_per_batch tiles")
        if sum(t.shape[0] for t in logits) != nr * nc:
            raise PylcError("expected %d tiles, got %d" % (nr * nc, sum(t.shape[0] for t in logits)))
        ptrs = torch.tensor([t.data_ptr() for t in logits], dtype=torch.int64)
        batch_table = ptrs.to(dev, non_blocking=True)
        return ctypes.c_void_p(0), _p(batch_table), tpb, C, dev, batch_table
    _need_cuda(logits)
    if logits.dtype != torch.float32 or not logits.is_contiguous():
        raise PylcError("logits must be contiguous float32")
    if logits.shape[0] != nr * nc:
        raise PylcError("expected %d tiles, got %d" % (nr * nc, logits.shape[0]))
    return _p(logits), ctypes.c_void_p(0), nr * nc, logits.shape[1], logits.device, None


def _decoder_source(decoder_batches, nr, nc, tiles_per_batch):
    """(batch table, tiles per batch, C, hs, ws, device) of the fused stitch's channels-last decoder outputs."""
    if torch.is_tensor(decoder_batches):
        decoder_batches = [decoder_batches]
    decoder_batches = list(decoder_batches)
    _need_cuda(*decoder_batches)
    dev = decoder_batches[0].device
    C, hs, ws = decoder_batches[0].shape[1:]
    tpb = tiles_per_batch or decoder_batches[0].shape[0]
    for i, t in enumerate(decoder_batches):
        if not _is_nhwc(t) or tuple(t.shape[1:]) != (C, hs, ws):
            raise PylcError("decoder batches must be channels-last float32 CUDA tensors of one shape")
        if i < len(decoder_batches) - 1 and t.shape[0] != tpb:
            raise PylcError("all tile batches but the last must hold tiles_per_batch tiles")
    if sum(t.shape[0] for t in decoder_batches) != nr * nc:
        raise PylcError("expected %d tiles, got %d" % (nr * nc, sum(t.shape[0] for t in decoder_batches)))
    batch_table = torch.tensor([t.data_ptr() for t in decoder_batches], dtype=torch.int64).to(dev, non_blocking=True)
    return batch_table, tpb, C, hs, ws, dev


def _lut_for(lut_rgb, C, what):
    if lut_rgb is None:
        return None
    pal, c2 = _lib.palette_array(lut_rgb)
    if c2 != C:
        raise PylcError("lut_rgb has %d colours, %s %d classes" % (c2, what, C))
    return pal


def stitch_argmax_colour(logits, nr, nc, T, S, lut_rgb=None, want_labels=True, want_rgb=False,
                         want_stitched=False, tiles_per_batch=None):
    """pylc_stitch_argmax_colour.  `logits` is one contiguous CUDA [nr*nc,C,T,T] f32 tensor, or a list
    of per-batch tensors [<=b,C,T,T] (the reference's `model_outputs` list).
    Returns (labels [h,w] u8 | None, rgb [h,w,3] u8 | None, stitched [C,h,w] f32 | None)."""
    lib = _lib.load()
    lp, bp, tpb, C, dev, batch_table = _tile_source(logits, nr, nc, tiles_per_batch)
    h, w = stitch_dims(nr, nc, T, S)
    labels = torch.empty((h, w), dtype=torch.uint8, device=dev) if want_labels else None
    rgb = torch.empty((h, w, 3), dtype=torch.uint8, device=dev) if want_rgb else None
    stitched = torch.empty((C, h, w), dtype=torch.float32, device=dev) if want_stitched else None
    pal = _lut_for(lut_rgb, C, "logits have")
    check(lib.pylc_stitch_argmax_colour(lp, bp, tpb, nr, nc, C, T, S, pal, _p(labels), _p(rgb), _p(stitched),
                                        _stream()), "pylc_stitch_argmax_colour")
    if batch_table is not None:
        batch_table.record_stream(torch.cuda.current_stream())
    return labels, rgb, stitched


def stitch_upsample_argmax_colour(decoder_batches, nr, nc, T, S, lut_rgb=None, want_labels=True, want_rgb=False,
                                  want_stitched=False, tiles_per_batch=None):
    """pylc_stitch_upsample_argmax_colour: stitch straight from the decoder's channels-last outputs
    [b, C, T/4, T/4] (one tensor per network batch), the final x4 bilinear up-sample evaluated in the kernel.
    Returns (labels [h,w] u8, rgb [h,w,3] u8 or None, stitched [C,h,w] f32 or None), bit-identical to
    stitch_argmax_colour(upsample_nhwc_to_nchw(batch) ...)."""
    lib = _lib.load()
    batch_table, tpb, C, hs, ws, dev = _decoder_source(decoder_batches, nr, nc, tiles_per_batch)
    h, w = stitch_dims(nr, nc, T, S)
    labels = torch.empty((h, w), dtype=torch.uint8, device=dev) if want_labels else None
    rgb = torch.empty((h, w, 3), dtype=torch.uint8, device=dev) if want_rgb else None
    stitched = torch.empty((C, h, w), dtype=torch.float32, device=dev) if want_stitched else None
    pal = _lut_for(lut_rgb, C, "the decoder output has")
    check(lib.pylc_stitch_upsample_argmax_colour(_p(batch_table), tpb, nr, nc, C, T, S, hs, ws, pal, _p(labels), _p(rgb),
                                                 _p(stitched), _stream()), "pylc_stitch_upsample_argmax_colour")
    batch_table.record_stream(torch.cuda.current_stream())
    return labels, rgb, stitched


STITCH_MODES = {"reference": 0, "mean": 1}     # PYLC_STITCH_REFERENCE, PYLC_STITCH_MEAN


def _stitch_mode(mode):
    if mode not in STITCH_MODES:
        raise PylcError("stitch mode must be one of %s, got %r" % (sorted(STITCH_MODES), mode))
    return STITCH_MODES[mode]


def _prob_outputs(C, h, w, dev, want_labels, want_rgb, want_confidence, want_probs, out):
    out = dict(out or {})

    def get(key, shape, dtype, want):
        if out.get(key) is not None:
            return out[key]
        return torch.empty(shape, dtype=dtype, device=dev) if want else None
    return {"labels": get("labels", (h, w), torch.uint8, want_labels),
            "rgb": get("rgb", (h, w, 3), torch.uint8, want_rgb),
            "confidence": get("confidence", (h, w), torch.uint8, want_confidence),
            "probs": get("probs", (C, h, w), torch.float32, want_probs)}


def stitch_probs(logits, nr, nc, T, S, mode="reference", lut_rgb=None, want_labels=True, want_rgb=False,
                 want_confidence=True, want_probs=False, tiles_per_batch=None, out=None, temperature=1.0):
    """pylc_stitch_probs_t: the stitch of stitch_argmax_colour with per-pixel probabilities.
    P = the mean over the covering tiles of their softmaxes.  mode "reference": labels / rgb are those of
    stitch_argmax_colour and `probs` is the reference's merged map M; mode "mean": labels = argmax P and
    `probs` = P.  `confidence` is the u8 plane round(P[label] * 255) in both modes.
    `temperature` (mean mode only; PylcError otherwise unless 1): every tile softmax is softmax(L / temperature);
    1 gives the untempered outputs bit for bit.
    `out`: optional dict of preallocated outputs (any of labels / rgb / confidence / probs).
    Returns dict(labels, rgb, confidence, probs), entries None where not wanted."""
    lib = _lib.load()
    m = _stitch_mode(mode)
    lp, bp, tpb, C, dev, batch_table = _tile_source(logits, nr, nc, tiles_per_batch)
    h, w = stitch_dims(nr, nc, T, S)
    res = _prob_outputs(C, h, w, dev, want_labels, want_rgb, want_confidence, want_probs, out)
    pal = _lut_for(lut_rgb, C, "logits have")
    check(lib.pylc_stitch_probs_t(lp, bp, tpb, nr, nc, C, T, S, m, pal, _p(res["labels"]), _p(res["rgb"]),
                                  _p(res["confidence"]), _p(res["probs"]), float(temperature), _stream()),
          "pylc_stitch_probs_t")
    if batch_table is not None:
        batch_table.record_stream(torch.cuda.current_stream())
    return res


def stitch_upsample_probs(decoder_batches, nr, nc, T, S, mode="reference", lut_rgb=None, want_labels=True,
                          want_rgb=False, want_confidence=True, want_probs=False, tiles_per_batch=None, out=None,
                          temperature=1.0):
    """pylc_stitch_upsample_probs_t: stitch_probs straight from the decoder's channels-last outputs (the fused
    x4 up-sample of stitch_upsample_argmax_colour), bit-identical to
    stitch_probs(upsample_nhwc_to_nchw(batch) ..., temperature=...).  Returns dict(labels, rgb, confidence, probs)."""
    lib = _lib.load()
    m = _stitch_mode(mode)
    batch_table, tpb, C, hs, ws, dev = _decoder_source(decoder_batches, nr, nc, tiles_per_batch)
    h, w = stitch_dims(nr, nc, T, S)
    res = _prob_outputs(C, h, w, dev, want_labels, want_rgb, want_confidence, want_probs, out)
    pal = _lut_for(lut_rgb, C, "the decoder output has")
    check(lib.pylc_stitch_upsample_probs_t(_p(batch_table), tpb, nr, nc, C, T, S, hs, ws, m, pal, _p(res["labels"]),
                                           _p(res["rgb"]), _p(res["confidence"]), _p(res["probs"]), float(temperature),
                                           _stream()), "pylc_stitch_upsample_probs_t")
    batch_table.record_stream(torch.cuda.current_stream())
    return res


def stitch_upsample_supported(C, T, S, hs, ws):
    """Geometry the fused stitch covers (else callers keep up-sample + stitch as two launches)."""
    return C <= 12 and hs * 4 == T and ws * 4 == T and (S == T or 2 * S == T) and S % 8 == 0 and S // 2 <= 256 \
        and 256 % (S // 2) == 0 and (S & (S - 1)) == 0


def colourise_u8(labels, lut_rgb):
    _need_cuda(labels)
    labels = labels.contiguous()
    pal, C = _lib.palette_array(lut_rgb)
    rgb = torch.empty(tuple(labels.shape) + (3,), dtype=torch.uint8, device=labels.device)
    check(_lib.load().pylc_colourise_u8(_p(labels), labels.numel(), pal, C, _p(rgb), _stream()), "pylc_colourise_u8")
    return rgb


# ---- evaluation ---------------------------------------------------------------------------------


def nn_index_map(n_src, n_dst):
    """OpenCV INTER_NEAREST source index per destination index (resizeNN's x_ofs table):
    min(floor(x * (1 / (n_dst / n_src))), n_src - 1) in double precision."""
    scale = 1.0 / (n_dst / n_src)
    idx = np.floor(np.arange(n_dst, dtype=np.float64) * scale).astype(np.int64)
    return np.minimum(idx, n_src - 1).astype(np.int32)


_MAP_CACHE = {}


def device_index_maps(w, h, w_full, h_full, device):
    """(x_ofs [w_full] i32, y_ofs [h_full] i32) on `device`, cached per geometry."""
    key = (w, h, w_full, h_full, str(device))
    maps = _MAP_CACHE.get(key)
    if maps is None:
        if len(_MAP_CACHE) > 64:
            _MAP_CACHE.clear()
        maps = (torch.from_numpy(nn_index_map(w, w_full)).to(device), torch.from_numpy(nn_index_map(h, h_full)).to(device))
        _MAP_CACHE[key] = maps
    return maps


def resample_encode_confusion(labels, w_full, h_full, gt_rgb=None, gt_pitch=0, palette=None, lut_rgb=None,
                              n_classes=None, n_inject=0, conf=None, want_pred=False, want_rgb=False,
                              want_gt=False, maps=None):
    """pylc_resample_encode_confusion.  Returns dict(conf, pred_full, pred_rgb, gt_full)."""
    _need_cuda(labels, gt_rgb)
    h, w = labels.shape
    dev = labels.device
    if maps is None:
        maps = device_index_maps(w, h, w_full, h_full, dev)
    x_ofs, y_ofs = maps
    pal = lut = None
    C = n_classes
    if palette is not None:
        pal, C = _lib.palette_array(palette)
    if lut_rgb is not None:
        lut, C = _lib.palette_array(lut_rgb)
    if gt_rgb is not None and conf is None:
        conf = torch.zeros((C, C), dtype=torch.int64, device=dev)
    pred_full = torch.empty((h_full, w_full), dtype=torch.uint8, device=dev) if want_pred else None
    pred_rgb = torch.empty((h_full, w_full, 3), dtype=torch.uint8, device=dev) if want_rgb else None
    gt_full = torch.empty((h_full, w_full), dtype=torch.uint8, device=dev) if want_gt else None
    check(_lib.load().pylc_resample_encode_confusion(
        _p(labels), h, w, _p(x_ofs), _p(y_ofs), h_full, w_full, _p(gt_rgb), gt_pitch, pal, lut, C, n_inject,
        _p(conf if gt_rgb is not None else None), _p(pred_full), _p(pred_rgb), _p(gt_full), _stream()),
        "pylc_resample_encode_confusion")
    return {"conf": conf, "pred_full": pred_full, "pred_rgb": pred_rgb, "gt_full": gt_full}


def confusion_u8(y_true, y_pred, n_classes, n_inject=0, conf=None):
    _need_cuda(y_true, y_pred)
    y_true = y_true.contiguous().view(-1)
    y_pred = y_pred.contiguous().view(-1)
    if y_true.numel() != y_pred.numel():
        raise PylcError("Input dimensions %s not same as target %s." % (tuple(y_pred.shape), tuple(y_true.shape)))
    if conf is None:
        conf = torch.zeros((n_classes, n_classes), dtype=torch.int64, device=y_true.device)
    check(_lib.load().pylc_confusion_u8(_p(y_true), _p(y_pred), y_true.numel(), n_classes, n_inject, _p(conf),
                                        _stream()), "pylc_confusion_u8")
    return conf


def confidence_resample(confidence, w_full, h_full, y_pred_full=None, y_true_full=None, n_classes=None,
                        reliability=None, want_full=True, maps=None):
    """pylc_confidence_resample: the fitted u8 confidence [h,w] to full resolution with the label map's
    INTER_NEAREST index maps, and, given the full-resolution predicted and true classes, the reliability table
    [C,256,2] i64 (pred, confidence level, correct) ADDED INTO `reliability` (allocated zeroed when None).
    Returns dict(confidence_full, reliability)."""
    _need_cuda(confidence, y_pred_full, y_true_full)
    confidence = confidence.contiguous()
    h, w = confidence.shape
    dev = confidence.device
    if maps is None:
        maps = device_index_maps(w, h, w_full, h_full, dev)
    x_ofs, y_ofs = maps
    counting = y_pred_full is not None or y_true_full is not None
    if counting:
        if y_pred_full is None or y_true_full is None or n_classes is None:
            raise PylcError("confidence_resample: the reliability table needs y_pred_full, y_true_full and n_classes")
        y_pred_full, y_true_full = y_pred_full.contiguous(), y_true_full.contiguous()
        if y_pred_full.numel() != h_full * w_full or y_true_full.numel() != h_full * w_full:
            raise PylcError("confidence_resample: label planes must hold h_full * w_full pixels")
        if reliability is None:
            reliability = torch.zeros((n_classes, 256, 2), dtype=torch.int64, device=dev)
    else:
        reliability = None
    full = torch.empty((h_full, w_full), dtype=torch.uint8, device=dev) if want_full else None
    check(_lib.load().pylc_confidence_resample(_p(confidence), h, w, _p(x_ofs), _p(y_ofs), h_full, w_full, _p(y_pred_full),
                                               _p(y_true_full), int(n_classes or 0), _p(full), _p(reliability), _stream()),
          "pylc_confidence_resample")
    return {"confidence_full": full, "reliability": reliability}


_CHECKED_MAPS = set()


def _checked_index_maps(w, h, w_full, h_full, device):
    """device_index_maps, with every index checked to lie inside the (w, h) plane once per geometry (the C ABI
    takes that as a precondition)."""
    key = (w, h, w_full, h_full)
    if key not in _CHECKED_MAPS:
        for src, dst in ((w, w_full), (h, h_full)):
            m = nn_index_map(src, dst)
            if m.min() < 0 or m.max() >= src:
                raise PylcError("index map %d -> %d leaves its plane" % (src, dst))
        _CHECKED_MAPS.add(key)
    return device_index_maps(w, h, w_full, h_full, device)


def prob_scores(probs, y_true_full, w_full, h_full, want_brier=True, maps=None, workspace=None):
    """pylc_prob_scores: [2] f64 CUDA tensor {sum of -log(max(P[g], 1e-12)), sum of the Brier score} over the
    h_full x w_full pixels of `y_true_full` (u8 encoded classes), P = the mean-mode `probs` [C, h, w] sampled with
    the label map's INTER_NEAREST index maps (`maps`, default device_index_maps).  The Brier entry is 0 without
    `want_brier`.  Deterministic: the same inputs give the same bits.  `workspace`: optional f64 scratch of
    _lib.SCORES_WS_DOUBLES entries, reused across calls on one stream."""
    _need_cuda(probs, y_true_full)
    if probs.dtype != torch.float32 or probs.dim() != 3 or not probs.is_contiguous():
        raise PylcError("prob_scores takes a contiguous [C, h, w] float32 map")
    if y_true_full.dtype != torch.uint8 or y_true_full.numel() != h_full * w_full or not y_true_full.is_contiguous():
        raise PylcError("prob_scores: y_true_full must be a contiguous u8 plane of h_full * w_full pixels")
    C, h, w = probs.shape
    dev = probs.device
    x_ofs, y_ofs = _checked_index_maps(w, h, w_full, h_full, dev) if maps is None else maps
    if x_ofs.numel() != w_full or y_ofs.numel() != h_full:
        raise PylcError("prob_scores: index maps must hold w_full / h_full entries")
    if workspace is None:
        workspace = torch.empty((_lib.SCORES_WS_DOUBLES,), dtype=torch.float64, device=dev)
    sums = torch.empty((2,), dtype=torch.float64, device=dev)
    check(_lib.load().pylc_prob_scores(_p(probs), C, h, w, _p(x_ofs), _p(y_ofs), int(h_full), int(w_full), _p(y_true_full),
                                       1 if want_brier else 0, _p(workspace), _p(sums), _stream()), "pylc_prob_scores")
    return sums


def multiscale_combine(probs, w_full, h_full, lut_rgb=None, want_labels=True, want_rgb=False, want_confidence=True,
                       out=None):
    """pylc_multiscale_combine: the probability maps of K <= 8 image scales, a list of [C, h_k, w_k] f32 CUDA tensors
    (mean-mode `probs` of stitch_probs / stitch_upsample_probs), sampled onto the [h_full, w_full] grid with the label
    map's INTER_NEAREST index maps and averaged in scale order: labels = first argmax of the mean, confidence =
    min(255, round(mean[label] * 255)).  `out`: optional dict of preallocated outputs (labels / rgb / confidence).
    Returns dict(labels, rgb, confidence), entries None where not wanted."""
    probs = list(probs)
    if not 1 <= len(probs) <= _lib.MAX_SCALES:
        raise PylcError("multiscale_combine takes 1 to %d probability maps, got %d" % (_lib.MAX_SCALES, len(probs)))
    _need_cuda(*probs)
    C, dev = probs[0].shape[0], probs[0].device
    for p in probs:
        if p.dtype != torch.float32 or p.dim() != 3 or not p.is_contiguous() or p.shape[0] != C or p.device != dev:
            raise PylcError("multiscale_combine takes contiguous [C, h, w] float32 maps of one class count and device")
    K = len(probs)
    maps = [_checked_index_maps(p.shape[2], p.shape[1], w_full, h_full, dev) for p in probs]
    res = _prob_outputs(C, h_full, w_full, dev, want_labels, want_rgb, want_confidence, False, out)
    res.pop("probs")
    pal = _lut_for(lut_rgb, C, "the probability maps have")
    ptrs = lambda ts: (ctypes.c_void_p * K)(*[t.data_ptr() for t in ts])     # noqa: E731
    ints = lambda vals: (ctypes.c_int * K)(*vals)                             # noqa: E731
    check(_lib.load().pylc_multiscale_combine(ptrs(probs), ptrs([m[0] for m in maps]), ptrs([m[1] for m in maps]),
                                              ints([p.shape[1] for p in probs]), ints([p.shape[2] for p in probs]), K, C,
                                              int(h_full), int(w_full), pal, _p(res["labels"]), _p(res["rgb"]),
                                              _p(res["confidence"]), _stream()), "pylc_multiscale_combine")
    return res


# ---- multi-loss ---------------------------------------------------------------------------------


def loss_cfg(ce=0.5, dice=0.5, focal=0.5, smooth=1.0, gamma=2.0, alpha=0.25, eps=1e-8):
    return LossCfg(ce, dice, focal, smooth, gamma, alpha, eps)


def _loss_inputs(logits, target):
    _need_cuda(logits, target)
    if logits.dtype != torch.float32:
        raise PylcError("logits must be float32")
    logits = logits.contiguous()
    target = target.contiguous()
    if target.dtype == torch.int64:
        is_i64 = 1
    elif target.dtype == torch.uint8:
        is_i64 = 0
    else:
        raise PylcError("target must be int64 or uint8")
    B, C = logits.shape[0], logits.shape[1]
    HW = logits.numel() // (B * C)
    if target.numel() != B * HW:
        raise PylcError("pred/target shape mismatch")
    return logits, target, is_i64, B, C, HW


def multiloss_reduce(logits, target, cfg, class_w=None, partials=None, target_u8_out=None):
    """pylc_multiloss_reduce.  `target_u8_out`: optional [B*HW] u8 CUDA tensor that receives a one-byte copy of
    int64 targets -- hand THAT to multiloss_grad as the target (it then reads 1 B/px instead of 8)."""
    logits, target, is_i64, B, C, HW = _loss_inputs(logits, target)
    if partials is None:
        partials = torch.zeros((2 * C + 3,), dtype=torch.float64, device=logits.device)
    if target_u8_out is not None and (target_u8_out.dtype != torch.uint8 or target_u8_out.numel() != B * HW):
        raise PylcError("target_u8_out must be a uint8 tensor of B*HW elements")
    check(_lib.load().pylc_multiloss_reduce(_p(logits), _p(target), is_i64, B, C, HW, _p(class_w), ctypes.byref(cfg),
                                            _p(partials), _p(target_u8_out), _stream()), "pylc_multiloss_reduce")
    return partials


def multiloss_finalize(partials, n_classes, n_px_total, cfg):
    out = torch.empty((4,), dtype=torch.float32, device=partials.device)
    check(_lib.load().pylc_multiloss_finalize(_p(partials), n_classes, n_px_total, ctypes.byref(cfg), _p(out),
                                              _stream()), "pylc_multiloss_finalize")
    return out


def multiloss_grad(logits, target, cfg, partials, n_px_total, class_w=None, grad_scale=1.0, out=None,
                   grad_scale_dev=None):
    """`grad_scale_dev`: optional CUDA f32 scalar tensor multiplied in on the device (autograd's upstream grad)."""
    logits, target, is_i64, B, C, HW = _loss_inputs(logits, target)
    grad = out if out is not None else torch.empty_like(logits)
    check(_lib.load().pylc_multiloss_grad(_p(logits), _p(target), is_i64, B, C, HW, _p(class_w), ctypes.byref(cfg),
                                          _p(partials), n_px_total, float(grad_scale), _p(grad_scale_dev), _p(grad),
                                          _stream()),
          "pylc_multiloss_grad")
    return grad


def multiloss_fwd_bwd(logits, target, cfg, class_w=None, grad_scale=1.0, out=None, partials=None, target_u8_ws=None,
                      use_u8_ws=True):
    """pylc_multiloss_fwd_bwd: one cooperative launch.  Returns (out4 = loss/ce/dice/focal, grad, partials).
    With int64 targets a [B*HW] u8 workspace (`target_u8_ws`, allocated here unless given or `use_u8_ws` is
    off) carries the targets from the reduce pass to the gradient pass: 1 B/px instead of 8 on the second read."""
    logits, target, is_i64, B, C, HW = _loss_inputs(logits, target)
    grad = out if out is not None else torch.empty_like(logits)
    if partials is None:
        partials = torch.zeros((2 * C + 3,), dtype=torch.float64, device=logits.device)
    if is_i64 and use_u8_ws and target_u8_ws is None:
        target_u8_ws = torch.empty((B * HW,), dtype=torch.uint8, device=logits.device)
    if not (is_i64 and use_u8_ws):
        target_u8_ws = None
    out4 = torch.empty((4,), dtype=torch.float32, device=logits.device)
    check(_lib.load().pylc_multiloss_fwd_bwd(_p(logits), _p(target), is_i64, B, C, HW, _p(class_w), ctypes.byref(cfg),
                                             _p(partials), float(grad_scale), None, _p(grad), _p(out4), _p(target_u8_ws),
                                             _stream()),
          "pylc_multiloss_fwd_bwd")
    return out4, grad, partials


DP_WS_BYTES = 2048          # PYLC_DP_WS_BYTES


def multiloss_fwd_bwd_dp(logits, target, cfg, peer_ws_dev, rank, world, epoch, class_w=None, grad_scale=1.0, out=None,
                         partials=None, target_u8_ws=None):
    """pylc_multiloss_fwd_bwd_dp: the data-parallel training step's loss in one cooperative launch -- the 2C+3
    partials are all-reduced inside the kernel over peer-addressable memory.  `peer_ws_dev`: device address of the
    [world] array of workspace pointers (dist.loss_exchange()); `epoch`: 1, 2, 3, ... the same on every rank.
    Returns (out4, grad, partials) where partials are the global sums."""
    logits, target, is_i64, B, C, HW = _loss_inputs(logits, target)
    grad = out if out is not None else torch.empty_like(logits)
    if partials is None:
        partials = torch.zeros((2 * C + 3,), dtype=torch.float64, device=logits.device)
    if is_i64 and target_u8_ws is None:
        target_u8_ws = torch.empty((B * HW,), dtype=torch.uint8, device=logits.device)
    if not is_i64:
        target_u8_ws = None
    out4 = torch.empty((4,), dtype=torch.float32, device=logits.device)
    check(_lib.load().pylc_multiloss_fwd_bwd_dp(_p(logits), _p(target), is_i64, B, C, HW, _p(class_w), ctypes.byref(cfg),
                                                _p(partials), float(grad_scale), None, _p(grad), _p(out4), _p(target_u8_ws),
                                                ctypes.c_void_p(int(peer_ws_dev)), int(rank), int(world), int(epoch), _stream()),
          "pylc_multiloss_fwd_bwd_dp")
    return out4, grad, partials


def scale_unless_one_(data, scale_dev):
    """In place data *= scale_dev (CUDA f32 scalar) unless it equals 1; no host sync."""
    _need_cuda(data, scale_dev)
    check(_lib.load().pylc_scale_unless_one_f32(_p(data), data.numel(), _p(scale_dev), _stream()), "pylc_scale_unless_one_f32")
    return data


def sample_rate_grid(scores, px_dist, rate_coefs, thresholds, rate_lo, rate_hi):
    """pylc_sample_rate_grid.  scores [N] f64, px_dist [N,C] i64, rate_coefs [R] f64, thresholds [T] f64
    (CUDA) -> (sum_rates [R*T] i64, full_px_dist [R*T, C] i64)."""
    _need_cuda(scores, px_dist, rate_coefs, thresholds)
    if scores.dtype != torch.float64 or px_dist.dtype != torch.int64:
        raise PylcError("sample_rate_grid: scores must be float64 and px_dist int64")
    N, C = px_dist.shape
    G = rate_coefs.numel() * thresholds.numel()
    sum_rates = torch.empty((G,), dtype=torch.int64, device=scores.device)
    full = torch.empty((G, C), dtype=torch.int64, device=scores.device)
    check(_lib.load().pylc_sample_rate_grid(_p(scores.contiguous()), _p(px_dist.contiguous()), N, C,
                                            _p(rate_coefs.contiguous()), rate_coefs.numel(), _p(thresholds.contiguous()),
                                            thresholds.numel(), int(rate_lo), int(rate_hi), _p(sum_rates), _p(full),
                                            _stream()), "pylc_sample_rate_grid")
    return sum_rates, full


def augment_tiles(src_imgs, src_masks, job_src, job_minv, job_shift, out_imgs=None, out_masks=None):
    """pylc_augment_tiles_u8: over-sampled copies of tiles (perspective jitter, crop, resize back, brightness shift),
    bit-identical to the reference's OpenCV chain.  src_imgs [n,ch,T,T] u8, src_masks [n,T,T] u8 (CUDA); job_src
    [J] int, job_minv [J,3,3] / [J,9] f64 (inverse perspective matrices), job_shift [J] int (host arrays or CUDA
    tensors).  Returns (imgs [J,ch,T,T] u8, masks [J,T,T] u8)."""
    _need_cuda(src_imgs, src_masks)
    dev = src_imgs.device
    if src_imgs.dtype != torch.uint8 or src_masks.dtype != torch.uint8 or src_imgs.dim() != 4 or src_masks.dim() != 3:
        raise PylcError("augment_tiles takes u8 tiles [n,ch,T,T] and u8 masks [n,T,T]")
    src_imgs, src_masks = src_imgs.contiguous(), src_masks.contiguous()
    n, ch, T = src_imgs.shape[0], src_imgs.shape[1], src_imgs.shape[2]
    d_src = torch.as_tensor(np.asarray(job_src) if not torch.is_tensor(job_src) else job_src).to(dev, torch.int32).contiguous()
    d_minv = torch.as_tensor(np.asarray(job_minv) if not torch.is_tensor(job_minv) else job_minv).to(dev, torch.float64).reshape(-1, 9).contiguous()
    d_shift = torch.as_tensor(np.asarray(job_shift) if not torch.is_tensor(job_shift) else job_shift).to(dev, torch.int32).contiguous()
    J = d_src.numel()
    if d_minv.shape[0] != J or d_shift.numel() != J:
        raise PylcError("augment_tiles: one source index, matrix and shift per copy")
    if J and (int(d_src.min()) < 0 or int(d_src.max()) >= n):
        raise PylcError("augment_tiles: source index out of range")
    imgs = out_imgs if out_imgs is not None else torch.empty((J, ch, T, T), dtype=torch.uint8, device=dev)
    masks = out_masks if out_masks is not None else torch.empty((J, T, T), dtype=torch.uint8, device=dev)
    check(_lib.load().pylc_augment_tiles_u8(_p(src_imgs), _p(src_masks), n, ch, T, _p(d_src), _p(d_minv), _p(d_shift), J,
                                            _p(imgs), _p(masks), _stream()), "pylc_augment_tiles_u8")
    return imgs, masks


# ---- network glue (channels-last f32 activations) ---------------------------------------------------

def _is_nhwc(t):
    return t.is_cuda and t.dtype == torch.float32 and t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last)


def upsample_concat_nhwc(x, low):
    """pylc_upsample_concat_nhwc_f32: bilinear(align_corners=True) up-sample of x to low's size + channel
    concat, on channels-last tensors.  x [B,Cx,h,w], low [B,Cl,H,W] -> [B,Cx+Cl,H,W] (channels_last)."""
    if not (_is_nhwc(x) and _is_nhwc(low)):
        raise PylcError("upsample_concat_nhwc takes channels-last float32 CUDA tensors")
    B, Cx, h, w = x.shape
    _, Cl, H, W = low.shape
    out = torch.empty((B, Cx + Cl, H, W), dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
    check(_lib.load().pylc_upsample_concat_nhwc_f32(_p(x), B, h, w, Cx, _p(low), H, W, Cl, _p(out), _stream()),
          "pylc_upsample_concat_nhwc_f32")
    return out


def maxpool3x3s2_nhwc(x):
    """pylc_maxpool3x3s2_nhwc_f32: max_pool2d(x, 3, stride=2, padding=1) on a channels-last tensor."""
    if not _is_nhwc(x):
        raise PylcError("maxpool3x3s2_nhwc takes a channels-last float32 CUDA tensor")
    B, C, H, W = x.shape
    out = torch.empty((B, C, (H - 1) // 2 + 1, (W - 1) // 2 + 1), dtype=torch.float32, device=x.device,
                      memory_format=torch.channels_last)
    check(_lib.load().pylc_maxpool3x3s2_nhwc_f32(_p(x), B, H, W, C, _p(out), _stream()), "pylc_maxpool3x3s2_nhwc_f32")
    return out


def tap_combine_relu_(out_bhwo, taps):
    """pylc_tap_combine_relu_f32, in place on `out_bhwo` [B,H,W,O] f32 (contiguous): adds the tap products
    `taps` = [(z [B,m,O] contiguous f32, p0, dy, dx), ...] where their source pixel lies inside the map, then ReLU."""
    _need_cuda(out_bhwo)
    B, H, W, O = out_bhwo.shape
    n = len(taps)
    if not out_bhwo.is_contiguous() or any(not z.is_contiguous() or z.dtype != torch.float32 or z.shape[0] != B or z.shape[2] != O
                                           for z, _, _, _ in taps):
        raise PylcError("tap_combine_relu_ takes contiguous float32 tensors [B,H,W,O] and [B,m,O]")
    zp = (ctypes.c_void_p * max(n, 1))(*[z.data_ptr() for z, _, _, _ in taps])
    i32 = lambda vals: (ctypes.c_int32 * max(n, 1))(*vals)          # noqa: E731
    check(_lib.load().pylc_tap_combine_relu_f32(_p(out_bhwo), B, H, W, O, zp, i32([t[1] for t in taps]), i32([t[0].shape[1] for t in taps]),
                                                i32([t[2] for t in taps]), i32([t[3] for t in taps]), n, _stream()),
          "pylc_tap_combine_relu_f32")
    return out_bhwo


def upsample_nhwc_to_nchw(x, size):
    """pylc_upsample_nhwc_to_nchw_f32: bilinear(align_corners=True) up-sample of a channels-last tensor to
    `size`, returned as a plain contiguous NCHW tensor (the stitch kernel's layout)."""
    if not _is_nhwc(x):
        raise PylcError("upsample_nhwc_to_nchw takes a channels-last float32 CUDA tensor")
    B, C, h, w = x.shape
    H, W = size
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=x.device)
    check(_lib.load().pylc_upsample_nhwc_to_nchw_f32(_p(x), B, h, w, C, _p(out), H, W, _stream()),
          "pylc_upsample_nhwc_to_nchw_f32")
    return out
