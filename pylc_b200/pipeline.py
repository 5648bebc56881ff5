"""
Tiled inference + evaluation pipeline: the GPU-resident form of the loop in PyLC's test.py
(reference test.py:52-115, SURVEY.md 3.2).

Per image, the reference does (host unless noted): fit-resize -> unfold tiles -> float + normalise
-> H2D per 8 tiles -> network (device) -> D2H of ALL logits -> band-merge loops -> argmax ->
colourise -> NN resize -> class_encode(pred), class_encode(GT) -> five scikit-learn passes.

Here, per image (device_fit, the default whenever OpenCV's general area filter applies):
    copy   one pitched H2D of the decoded image and one of the RGB ground truth, straight from the
           caller's (pinned) arrays on the copy engine -- no host-side pass over the pixels
    GPU    pylc_fit_resize_area_u8       cv2.resize(INTER_AREA) of adjust_to_tile, bit-exact (1 launch)
           pylc_tile_gather_norm_f32     tiles, normalised, grayscale replicated   (1 launch)
           DeepLabv3+/ResNet-101         stock PyTorch / cuDNN, batches of `batch_tiles`
           pylc_stitch_probs             logits -> label map, reference band semantics (1 launch)
           pylc_resample_encode_confusion  NN resample + GT encode + [C,C] counts    (1 launch)
With `stitch="mean"` or `confidence=True` the same stitch (pylc_stitch_probs / pylc_stitch_upsample_probs)
gives instead: labels from the mean of the covering tiles' softmaxes ("mean") and / or the u8 confidence plane
of that mean; with keep_masks the plane is also resampled to full resolution (pylc_confidence_resample).
    D2H    nothing per image; the [C,C] i64 matrix (and optional masks) at the end
With `scales` (multi-scale inference, mean stitch only) every image is segmented once per scale s_k: the decoded
image resized by s_k (INTER_AREA) and fitted to the tiles, on the device when both resizes are OpenCV's general
area filter, otherwise with cv2 on the host threads.  Each member's mean-mode probability map P_k stays on the
device; pylc_multiscale_combine samples every P_k onto the full-resolution grid, averages them and writes the
full-resolution labels and confidence, and pylc_resample_encode_confusion counts the confusion from those.
With `temperature` T (post-hoc calibration, mean stitch only) every tile softmax of the mean stitch is softmax(L / T),
in the single-scale stitch and in every multi-scale member alike.
With device_fit off (or for geometries OpenCV resizes with another filter) the fit-resize runs on
host worker threads with cv2 itself and the fitted image is uploaded instead.
Logits never leave the device.  Images are independent, so data-parallel ranks take images
round-robin and all-reduce only the [C,C] matrix (pylc_b200.dist).
"""
import concurrent.futures as cf
import math

import cv2
import numpy as np
import torch

from . import dist as pdist
from . import ops
from .config import defaults
from .utils import tools
from .utils.metrics import scores_from_confusion


class FittedImage(object):
    """A fitted u8 image (and optional RGB ground truth) resident on the device.  Multi-scale: `members` holds one
    (geometry, fitted image, pitch) triple per scale (multiscale_geometry); a fitted image of None means the member
    is fitted from `raw` on the device."""
    __slots__ = ("img", "pitch", "h", "w", "gt", "gt_pitch", "h_full", "w_full", "index", "ready", "raw", "raw_pitch",
                 "members")


MAX_SCALES = 8


def check_scales(scales):
    """The scale list of a multi-scale run, sorted; ValueError for an empty or too long list, a duplicate or a
    non-positive scale."""
    vals = sorted(float(s) for s in scales)
    if not 1 <= len(vals) <= MAX_SCALES:
        raise ValueError("multi-scale inference takes 1 to %d scales, got %d" % (MAX_SCALES, len(vals)))
    if vals[0] <= 0:
        raise ValueError("scales must be positive, got %g" % vals[0])
    if len(set(vals)) != len(vals):
        raise ValueError("duplicate scale in %s" % (vals,))
    return tuple(vals)


def multiscale_geometry(W, H, T, scales):
    """Per scale s of a W x H decoded image: dict(scale, resized=(w, h), fitted=(w, h), device).  The member image is
    cv2.resize(img, (int(s*W), int(s*H)), INTER_AREA) (no resize at s == 1) fitted by adjust_to_tile; `device` is True
    when OpenCV does both resizes with the general area filter that pylc_fit_resize_area_u8 reproduces.  Raises
    ValueError, naming the scale and the size, for a member whose fitted image is less than two tiles high or wide:
    the reference's stitch leaves rows of a one-tile-row image unset, so such a fit is outside its contract."""
    out = []
    for s in check_scales(scales):
        wr, hr = (W, H) if s == 1.0 else (int(s * W), int(s * H))
        wf, hf = tools.fit_dims(wr, hr, T) if wr >= 1 and hr >= 1 else (0, 0)
        if wf < 2 * T or hf < 2 * T:
            raise ValueError("scale %g: the %dx%d image resizes to %dx%d, which fits to %dx%d, less than two %d-pixel "
                             "tiles in a direction" % (s, W, H, wr, hr, wf, hf, T))
        device = (s == 1.0 or ops.area_supported(W, H, wr, hr)) and ops.area_supported(wr, hr, wf, hf)
        out.append({"scale": s, "resized": (wr, hr), "fitted": (wf, hf), "device": bool(device)})
    return out


class TiledSegmenter(object):
    def __init__(self, model, batch_tiles=32, channels_last=True, autocast_dtype=None, host_workers=4,
                 n_inject=None, keep_masks=False, fuse_network=False, device_fit=True, fuse_upsample=True,
                 stitch="reference", confidence=False, scales=None, temperature=1.0):
        self.model = model
        self.meta = model.meta
        self.net = model.net.eval()
        self.device = next(self.net.parameters()).device
        self.T = self.meta.tile_size
        self.S = self.T // 2                      # test.py:63: stride = tile_size // 2
        self.C = self.meta.n_classes
        self.ch = self.meta.ch
        self.batch_tiles = batch_tiles
        self.autocast_dtype = autocast_dtype
        self.channels_last = channels_last
        if channels_last:
            self.net = self.net.to(memory_format=torch.channels_last)
        # inference plan: BatchNorm folded into the convolutions, cuDNN fused conv+bias(+add)+ReLU
        # calls (models/fused.py).  Same network and precision; outputs equal the eager network to
        # fp32 rounding of the folded weights, so it is opt-in.
        self.fused = None
        if fuse_network:
            from .models.fused import FusedDeepLab
            self.fused = FusedDeepLab(self.net, channels_last=channels_last)
        self.mean, self.std, self.post_div, self.out_ch = model.norm_params()
        # space-to-depth stem: the gather writes the tiles in the layout of the rearranged 4x4 stem convolution
        self.s2d = self.fused is not None and self.fused.stem_s2d is not None and self.out_ch == 3 and self.T % 2 == 0
        # SURVEY.md 8f-1: with the inference plan the stitch kernel reads the decoder's [b, T/4, T/4, C] output
        # and evaluates the network's final x4 bilinear up-sample itself (bit-identical to the two-kernel
        # route, 16x less stitch input); `fuse_upsample=False` keeps up-sample and stitch as two launches
        self.fuse_upsample = bool(fuse_upsample and self.fused is not None and self.fused.glue and channels_last
                                  and autocast_dtype is None
                                  and ops.stitch_upsample_supported(self.C, self.T, self.S, self.T // 4, self.T // 4))
        self.palette = self.meta.palette_rgb
        self.lut = tools.colourize_lut(self.C, self.palette)
        self.n_inject = min(len(defaults.class_codes), self.C) if n_inject is None else n_inject
        self.keep_masks = keep_masks
        ops._stitch_mode(stitch)
        self.stitch = stitch                      # "reference": the reference's labels; "mean": argmax of P
        self.confidence = bool(confidence)        # adds res["confidence"] (and res["confidence_full"])
        # multi-scale: labels and confidence from the mean of the members' mean-mode probabilities
        self.scales = None
        if scales is not None:
            if stitch != "mean":
                raise ValueError("multi-scale inference averages the mean stitch's probabilities: it needs stitch='mean'")
            self.scales = check_scales(scales)
        self.temperature = float(temperature)     # softmax(L / T) of every tile in the mean stitch
        if not (math.isfinite(self.temperature) and self.temperature > 0):
            raise ValueError("temperature must be finite and > 0, got %r" % (temperature,))
        if self.temperature != 1.0 and stitch != "mean":
            raise ValueError("temperature scaling applies to the mean stitch's probabilities: it needs stitch='mean'")
        self.device_fit = device_fit
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.pool = cf.ThreadPoolExecutor(max_workers=host_workers)
        self.conf = torch.zeros((self.C, self.C), dtype=torch.int64, device=self.device)

    # ---- host stage ---------------------------------------------------------------------------
    def fit_host(self, img):
        """adjust_to_tile on the host into pinned, 16-byte-pitched memory."""
        fitted, w, h, offset = tools.adjust_to_tile(img, self.T, self.S, self.ch)
        assert offset == 0
        buf, pitch = ops.pinned_pitched(fitted)
        return buf, pitch, h, w

    def stage(self, img, gt=None, index=0):
        """Host fit + async H2D on the copy stream.  Returns a FittedImage; the compute stream must
        wait on `f.ready` before touching its tensors."""
        if torch.is_tensor(img):
            img = img.numpy()
        if self.scales is not None:
            return self._stage_multiscale(img, gt, index, None)
        buf, pitch, h, w = self.fit_host(img)
        f = FittedImage()
        f.index = index
        f.raw, f.raw_pitch = None, 0
        f.h, f.w, f.pitch = h, w, pitch
        f.h_full, f.w_full = img.shape[0], img.shape[1]
        with torch.cuda.stream(self.copy_stream):
            f.img = buf.to(self.device, non_blocking=True)
            if gt is not None:
                if torch.is_tensor(gt) and gt.ndim == 2:      # already a pitched [H, pitch] buffer
                    gbuf, f.gt_pitch = gt, gt.shape[1]
                else:
                    gbuf, f.gt_pitch = ops.pinned_pitched(gt.numpy() if torch.is_tensor(gt) else gt)
                f.gt = gbuf.to(self.device, non_blocking=True)
            else:
                f.gt, f.gt_pitch = None, 0
            f.ready = torch.cuda.Event()
            f.ready.record(self.copy_stream)
        return f

    def can_fit_on_device(self, img):
        H, W = img.shape[:2]
        w, h = tools.fit_dims(W, H, self.T)
        return self.device_fit and h >= self.T and w >= self.T and ops.area_supported(W, H, w, h)

    def stage_device(self, img, gt=None, index=0, after=None):
        """Device fit: pitched H2D of the DECODED image (and ground truth) on the copy stream; the
        INTER_AREA resize itself is launched by segment_fitted on the compute stream.  `after`: an event
        the copy stream waits for first (bounds how far uploads run ahead of the compute stream)."""
        if self.scales is not None:
            return self._stage_multiscale(img, gt, index, after)
        t_img = img if torch.is_tensor(img) else torch.from_numpy(np.ascontiguousarray(img))
        f = FittedImage()
        f.index = index
        f.h_full, f.w_full = t_img.shape[0], t_img.shape[1]
        f.w, f.h = tools.fit_dims(f.w_full, f.h_full, self.T)
        with torch.cuda.stream(self.copy_stream):
            if after is not None:
                self.copy_stream.wait_event(after)
            f.raw, f.raw_pitch = ops.upload_pitched(t_img, device=self.device)
            f.img, f.pitch = None, 0
            if gt is not None:
                t_gt = gt if torch.is_tensor(gt) else torch.from_numpy(np.ascontiguousarray(gt))
                f.gt, f.gt_pitch = ops.upload_pitched(t_gt, device=self.device)
            else:
                f.gt, f.gt_pitch = None, 0
            f.ready = torch.cuda.Event()
            f.ready.record(self.copy_stream)
        return f

    def _stage_multiscale(self, img, gt, index, after):
        """Multi-scale staging on the copy stream: one upload of the decoded image when a member is fitted on the
        device, and for every other member cv2.resize + adjust_to_tile here (a host worker thread under run_host)
        and the upload of the fitted image."""
        img = img.numpy() if torch.is_tensor(img) else np.asarray(img)
        f = FittedImage()
        f.index = index
        f.h_full, f.w_full = img.shape[0], img.shape[1]
        f.w, f.h = tools.fit_dims(f.w_full, f.h_full, self.T)
        f.img, f.pitch = None, 0
        geo = multiscale_geometry(f.w_full, f.h_full, self.T, self.scales)
        on_device = [self.device_fit and g["device"] for g in geo]
        hosted = []
        for g, dev in zip(geo, on_device):
            if dev:
                hosted.append((None, 0))
                continue
            x = img if g["scale"] == 1.0 else cv2.resize(img, g["resized"], interpolation=cv2.INTER_AREA)
            hosted.append(self.fit_host(x)[:2])
        with torch.cuda.stream(self.copy_stream):
            if after is not None:
                self.copy_stream.wait_event(after)
            f.raw, f.raw_pitch = None, 0
            if any(on_device):
                buf, f.raw_pitch = ops.pinned_pitched(img)
                f.raw = buf.to(self.device, non_blocking=True)
            f.members = [(g, None if buf is None else buf.to(self.device, non_blocking=True), pitch)
                         for g, (buf, pitch) in zip(geo, hosted)]
            if gt is not None:
                if torch.is_tensor(gt) and gt.ndim == 2:      # already a pitched [H, pitch] buffer
                    gbuf, f.gt_pitch = gt, gt.shape[1]
                else:
                    gbuf, f.gt_pitch = ops.pinned_pitched(gt.numpy() if torch.is_tensor(gt) else gt)
                f.gt = gbuf.to(self.device, non_blocking=True)
            else:
                f.gt, f.gt_pitch = None, 0
            f.ready = torch.cuda.Event()
            f.ready.record(self.copy_stream)
        return f

    def _release(self, f, stream):
        """Tie the staged buffers of `f` to `stream`, where the device work that reads them was enqueued."""
        for t in [f.img, f.raw, f.gt] + [m[1] for m in (getattr(f, "members", None) or [])]:
            if t is not None:
                t.record_stream(stream)

    # ---- device stage -------------------------------------------------------------------------
    def forward_tiles(self, tiles, s2d=False, decoder_only=False):
        """Network forward over [n,3,T,T] f32 tiles (or their space-to-depth form) in batches; returns
        the list of logit batches [b,C,T,T] -- or, with `decoder_only` (inference plan), of the decoder
        outputs [b,C,T/4,T/4] (channels-last) that the fused stitch up-samples itself."""
        outs = []
        with torch.no_grad():
            for lo in range(0, tiles.shape[0], self.batch_tiles):
                x = tiles[lo:lo + self.batch_tiles]
                if s2d:
                    outs.append(self.fused.decoder_s2d(x) if decoder_only else self.fused.forward_s2d(x))
                    continue
                if self.fused is not None:
                    outs.append(self.fused.decoder(x) if decoder_only else self.fused(x))
                    continue
                if self.channels_last:
                    x = x.contiguous(memory_format=torch.channels_last)
                if self.autocast_dtype is not None:
                    with torch.autocast("cuda", dtype=self.autocast_dtype):
                        y = self.net.features(x)
                else:
                    y = self.net.features(x)
                # the x4 bilinear up-sample of deeplab.py:38, applied to an NCHW copy of the small
                # decoder output so the logits come out NCHW (what the stitch kernel reads)
                y = y.float().contiguous()
                outs.append(torch.nn.functional.interpolate(y, size=x.shape[2:], mode='bilinear', align_corners=True))
        return outs

    def _tiles(self, img, pitch, h, w):
        if self.s2d:
            return ops.tile_gather_norm_s2d(img, h, w, self.ch, pitch, self.T, self.S, self.mean, self.std, self.post_div)
        return ops.tile_gather_norm_f32(img, h, w, self.ch, pitch, self.T, self.S, self.mean, self.std, self.post_div,
                                        self.out_ch)

    def network_output(self, tiles):
        """The network's output for one fitted image's tiles, in the form the probability stitch reads: the list of
        channels-last decoder batches on the fused route, else the logit batches (one tensor for a single batch)."""
        if self.fuse_upsample:
            return self.forward_tiles(tiles, s2d=self.s2d, decoder_only=True)
        src = self.forward_tiles(tiles, s2d=self.s2d)
        return src if len(src) > 1 else src[0]

    def retained_bytes(self, nr, nc):
        """Device bytes of network_output for an nr x nc tile grid: C * T^2 f32 per tile, 16x less on the fused
        route, which keeps the decoder's T/4 x T/4 output."""
        per_tile = self.C * self.T * self.T * 4
        return nr * nc * (per_tile // 16 if self.fuse_upsample else per_tile)

    def stitch_output(self, src, nr, nc, temperature=None, **kw):
        """pylc_stitch_probs (or its fused up-sample form) of a network_output at `temperature` (default: the
        segmenter's)."""
        probs = ops.stitch_upsample_probs if self.fuse_upsample else ops.stitch_probs
        t = self.temperature if temperature is None else temperature
        return probs(src, nr, nc, self.T, self.S, mode=self.stitch, tiles_per_batch=self.batch_tiles, temperature=t, **kw)

    def _stitch_probs(self, tiles, nr, nc, **kw):
        """Network + probability stitch over one fitted image's tiles."""
        return self.stitch_output(self.network_output(tiles), nr, nc, **kw)

    def fitted_tiles(self, f):
        """(tiles, nr, nc) of a single-scale FittedImage; a device-fitted image is resized here first."""
        img, pitch = f.img, f.pitch
        if img is None:        # device fit: INTER_AREA resize of the uploaded decoded image
            img, pitch = ops.fit_resize_area(f.raw, f.h_full, f.w_full, self.ch, f.raw_pitch, f.h, f.w)
        return self._tiles(img, pitch, f.h, f.w), f.h // self.S - 1, f.w // self.S - 1

    def segment_fitted(self, f, inject=None):
        """All device work for one fitted image; accumulates into self.conf when f.gt is set.
        Returns the fitted-resolution label map (and full-res masks when keep_masks)."""
        if self.scales is not None:
            return self._segment_multiscale(f, inject)
        tiles, nr, nc = self.fitted_tiles(f)
        src = self.network_output(tiles)
        conf_fit = None
        if self.stitch != "reference" or self.confidence:
            out = self.stitch_output(src, nr, nc, want_confidence=self.confidence)
            labels, conf_fit = out["labels"], out["confidence"]
        else:
            # looked up on `ops` at call time, so that a wrapper installed there (bench.py's kernel timer) sees it
            stitch = ops.stitch_upsample_argmax_colour if self.fuse_upsample else ops.stitch_argmax_colour
            labels = stitch(src, nr, nc, self.T, self.S, tiles_per_batch=self.batch_tiles)[0]
        n_inject = self.n_inject if inject is None else inject
        res = ops.resample_encode_confusion(
            labels, f.w_full, f.h_full, gt_rgb=f.gt, gt_pitch=f.gt_pitch, palette=self.palette, lut_rgb=self.lut,
            n_classes=self.C, n_inject=n_inject if f.gt is not None else 0, conf=self.conf if f.gt is not None else None,
            want_pred=self.keep_masks, want_rgb=self.keep_masks)
        res["labels"] = labels
        if conf_fit is not None:
            res["confidence"] = conf_fit
            if self.keep_masks:
                res["confidence_full"] = ops.confidence_resample(conf_fit, f.w_full, f.h_full)["confidence_full"]
        return res

    def member_probs(self, f):
        """The mean-mode probability map [C, h_k, w_k] of every scale of a multi-scale FittedImage, in scale order."""
        planes = []
        for g, img, pitch in f.members:
            (wr, hr), (wf, hf) = g["resized"], g["fitted"]
            if img is None and g["scale"] == 1.0:
                img, pitch = ops.fit_resize_area(f.raw, f.h_full, f.w_full, self.ch, f.raw_pitch, hf, wf)
            elif img is None:
                r, rp = ops.fit_resize_area(f.raw, f.h_full, f.w_full, self.ch, f.raw_pitch, hr, wr)
                img, pitch = ops.fit_resize_area(r, hr, wr, self.ch, rp, hf, wf)
            tiles = self._tiles(img, pitch, hf, wf)
            out = self._stitch_probs(tiles, hf // self.S - 1, wf // self.S - 1, want_labels=False, want_confidence=False,
                                     want_probs=True)
            planes.append(out["probs"])
        return planes

    def _segment_multiscale(self, f, inject):
        planes = self.member_probs(f)
        comb = ops.multiscale_combine(planes, f.w_full, f.h_full, want_confidence=self.confidence)
        del planes                     # one image's members are live at a time
        n_inject = self.n_inject if inject is None else inject
        labels = comb["labels"]
        res = ops.resample_encode_confusion(
            labels, f.w_full, f.h_full, gt_rgb=f.gt, gt_pitch=f.gt_pitch, palette=self.palette, lut_rgb=self.lut,
            n_classes=self.C, n_inject=n_inject if f.gt is not None else 0, conf=self.conf if f.gt is not None else None,
            want_pred=self.keep_masks, want_rgb=self.keep_masks)
        res["labels"] = labels
        if comb["confidence"] is not None:
            res["confidence"] = res["confidence_full"] = comb["confidence"]
        return res

    # ---- drivers ------------------------------------------------------------------------------
    def reset(self):
        self.conf.zero_()

    def run_resident(self, fitted_images, results=None):
        """Device-only pass over images already staged in HBM (bench.py `value`).  Returns the last image's
        result; `results`, when given, is a list that receives every image's result in order."""
        out = None
        for f in fitted_images:
            out = self.segment_fitted(f, inject=self.n_inject if f.index == 0 else 0)
            if results is not None:
                results.append(out)
        return out

    def run_host(self, images, masks=None, indices=None, distributed=False, global_offset=None, global_indices=None):
        """End-to-end pass from decoded host arrays (bench.py `e2e`, test.py's loop): host fit and
        H2D of image k+1 overlap the device work of image k.  Returns (conf ndarray, results).

        The coverage injection of Evaluator.validate (reference evaluate.py:172-174) is applied to the
        image whose GLOBAL index is 0 and to no other, so the all-reduced matrix is the same for every
        GPU count.  `images[i]` has global index `global_offset + i`; with `distributed=True` and no
        explicit offset the caller is taken to hold a contiguous shard of equal size per rank
        (offset = rank * len(images)); pass `global_offset`, or `global_indices` (one global index per
        entry of `images`, e.g. dist.shard_indices(n) for a round-robin shard) for any other partition."""
        idx = list(range(len(images))) if indices is None else list(indices)
        if global_indices is not None:
            assert len(global_indices) == len(images)
            self._gidx = [int(g) for g in global_indices]
        else:
            if global_offset is None:
                global_offset = pdist.rank() * len(images) if distributed else 0
            self._gidx = [int(global_offset) + i for i in range(len(images))]
        compute = torch.cuda.current_stream(self.device)
        prefetch = 3
        if self.scales is None and idx and all(self.can_fit_on_device(images[i]) for i in idx):
            return self._run_host_device_fit(images, masks, idx, compute, prefetch, distributed)

        def submit(k):
            i = idx[k]
            return self.pool.submit(self.stage, images[i], None if masks is None else masks[i], self._gidx[i])

        pending = [submit(k) for k in range(min(prefetch, len(idx)))]
        results = []
        for k in range(len(idx)):
            f = pending.pop(0).result()
            if k + prefetch < len(idx):
                pending.append(submit(k + prefetch))
            compute.wait_event(f.ready)
            res = self.segment_fitted(f, inject=self.n_inject if f.index == 0 else 0)
            self._release(f, compute)
            if self.keep_masks:
                results.append(res)
        conf = self.conf
        if distributed:
            conf = pdist.all_reduce_(conf.clone())
        return conf.cpu().numpy(), results           # the step's only D2H: C*C*8 bytes

    def _run_host_device_fit(self, images, masks, idx, compute, prefetch, distributed):
        """run_host without any host-side pixel work: uploads run `prefetch` images ahead on the copy
        stream (throttled by compute-stream events, not by the host), everything else is device work."""
        done = []                     # compute-stream event per finished image
        staged = []
        results = []

        def submit(k):
            i = idx[k]
            after = done[k - prefetch] if k >= prefetch else None
            staged.append(self.stage_device(images[i], None if masks is None else masks[i], self._gidx[i], after=after))

        for k in range(min(prefetch, len(idx))):
            submit(k)
        for k in range(len(idx)):
            f = staged[k]
            staged[k] = None
            compute.wait_event(f.ready)
            res = self.segment_fitted(f, inject=self.n_inject if f.index == 0 else 0)
            f.raw.record_stream(compute)
            if f.gt is not None:
                f.gt.record_stream(compute)
            ev = torch.cuda.Event()
            ev.record(compute)
            done.append(ev)
            if k + prefetch < len(idx):
                submit(k + prefetch)
            if self.keep_masks:
                results.append(res)
        conf = self.conf
        if distributed:
            conf = pdist.all_reduce_(conf.clone())
        return conf.cpu().numpy(), results

    def scores(self, conf):
        labels = defaults.class_codes if self.C == len(defaults.class_codes) else self.meta.class_codes
        return scores_from_confusion(conf, labels)
