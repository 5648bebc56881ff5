"""
Evaluator -- host-side mirror of PyLC's utils/evaluate.py (reference evaluate.py:25-284).

Same interface: Evaluator(params).load(mask_pred, meta, mask_true_path, scale).save_image();
.evaluate(aggregate).save_metrics(); .save_logits(logits); .reset().

What changed underneath: the reference class-encodes the predicted RGB mask and the ground truth
(two tools.class_encode passes), flattens them, overwrites the first len(labels) entries with
(i, i) (validate, evaluate.py:172-174) and hands both vectors to five scikit-learn calls.  Here
load() runs ONE kernel, pylc_resample_encode_confusion, over the ground-truth RGB: it encodes the
truth, gathers / encodes the prediction, applies the coverage injection and adds the pair counts
into an i64 [C,C] matrix on the device.  evaluate() reduces that matrix on the host
(utils/metrics.py).  Aggregate mode sums per-image matrices (and, data-parallel, all-reduces them)
instead of concatenating label vectors; the injection is applied once, to the first image of the
aggregate, exactly where the concatenated vectors would carry it.

`mask_pred` may be the reference's np.float32 [H,W,3] RGB array (it is re-encoded on the GPU) or
the dict returned by tools.reconstruct_device (labels stay on the device; no RGB round trip).

Confidence (an extension): when that dict also carries the fitted u8 confidence plane
(TiledSegmenter(confidence=True)), load() resamples it to full resolution and counts the reliability
table [C,256,2] (predicted class, confidence level, correct) in the same kernel call,
pylc_confidence_resample -- per image and in aggregate, without the coverage injection.  evaluate()
then adds a `calibration` entry (ECE, MCE, reliability bins, per-class confidence / accuracy) to the
metrics, and save_confidence() writes the full-resolution plane as an 8-bit PNG (255 = 1.0).
"""
import json
import os

import cv2
import numpy as np
import torch

from .. import dist as pdist
from .. import ops
from ..config import Parameters, defaults
from . import tools as utils
from .metrics import Metrics, calibration_from_reliability


class Evaluator:
    def __init__(self, params=None, make_dirs=True):
        self.meta = Parameters(params) if params is not None else defaults
        self.metrics = Metrics()
        self._schema = (self.meta.n_classes, self.meta.class_codes)
        self.fid = None
        self.logits = None
        self.mask_pred = None
        self.results = []
        self.y_true = None
        self.y_pred = None
        self.labels = []
        self.aggregate = False
        self.y_true_aggregate = []
        self.y_pred_aggregate = []
        self.conf = None              # device i64 [C,C]: this image, injection applied
        self.conf_aggregate = None    # device i64 [C,C]: all images, injection on the first only
        self.n_aggregated = 0
        self.aggregate_inject = True  # data-parallel: only the rank owning image 0 injects
        self.reliability = None       # device i64 [C,256,2]: this image (confidence runs only)
        self.reliability_aggregate = None
        self.confidence_full = None   # device u8 [H,W]: this image's full-resolution confidence
        self.model_path = None
        self.output_dir = os.path.join(defaults.output_dir, str(self.meta.id))
        if make_dirs:
            self.masks_dir = utils.mk_path(os.path.join(self.output_dir, 'masks'))
            self.logits_dir = utils.mk_path(os.path.join(self.output_dir, 'logits'))
            self.metrics_dir = utils.mk_path(os.path.join(self.output_dir, 'metrics'))
        else:
            self.masks_dir = self.logits_dir = self.metrics_dir = None

    def load(self, mask_pred, meta, mask_true_path=None, scale=None, mask_true=None):
        """Register a prediction (and its ground truth) for evaluation (reference evaluate.py:64-121).
        `mask_true` (extension) passes an already decoded RGB ground truth [H,W,3] u8."""
        self.meta = meta
        self._schema = (meta.n_classes, meta.class_codes)    # survives reset(), which blanks self.meta
        self.fid = self.meta.extract['fid']
        self.mask_pred = mask_pred
        if mask_true_path or mask_true is not None:
            if mask_true is None:
                mask_true, w, h, w_scaled, h_scaled = utils.get_image(
                    mask_true_path, ch=3, scale=scale, interpolate=cv2.INTER_NEAREST)
            else:
                h_scaled, w_scaled = mask_true.shape[:2]
            ex = self.meta.extract
            if not (w_scaled == ex['w_scaled'] and h_scaled == ex['h_scaled']):
                print("Ground truth mask dims ({}px X {}px) do not match predicted mask dims ({}px X {}px).".format(
                    w_scaled, h_scaled, ex['w_scaled'], ex['h_scaled']))
                exit(1)
            self._count(mask_true, w_scaled, h_scaled)
        return self

    def _count(self, mask_true, w_full, h_full):
        dev = utils._device()
        C = self.meta.n_classes
        pal = self.meta.palette_rgb
        n_inject = min(len(defaults.class_codes), C)   # validate(): labels = defaults.class_codes
        if torch.is_tensor(mask_true) and mask_true.is_cuda:
            d_gt = mask_true.view(h_full, -1)            # [H, pitch] u8, rows of interleaved RGB
            pitch = d_gt.shape[1]
        else:
            d_gt, pitch = ops.upload_image(np.asarray(mask_true, dtype=np.uint8), dev)
        pred = self.mask_pred
        if isinstance(pred, dict):
            labels = pred["labels"]                      # fitted-resolution label map on the device
        else:
            # reference route: RGB float mask -> u8 -> class_encode (evaluate.py:104-107)
            rgb = torch.as_tensor(np.ascontiguousarray(pred)).to(torch.uint8)
            assert tuple(rgb.shape[:2]) == (h_full, w_full), "Input dimensions {} not same as target {}.".format(
                tuple(rgb.shape[:2]), (h_full, w_full))
            d_rgb = rgb.pin_memory().to(dev, non_blocking=True)
            labels = ops.class_encode_hwc(d_rgb, h_full, w_full, w_full * 3, pal)[0]
        maps = ops.device_index_maps(labels.shape[1], labels.shape[0], w_full, h_full, dev)

        def count(rows, inject, want=False):
            return ops.resample_encode_confusion(labels, w_full, rows, gt_rgb=d_gt, gt_pitch=pitch, palette=pal,
                                                 n_inject=inject, want_pred=want, want_gt=want, maps=maps)
        res = count(h_full, n_inject, want=True)         # one pass: encode GT, gather pred, inject, count
        self.y_pred = res["pred_full"].view(-1)
        self.y_true = res["gt_full"].view(-1)
        self.conf = res["conf"]
        if self.n_aggregated == 0 and self.aggregate_inject:
            self.conf_aggregate = self.conf.clone()      # the first image carries the injection
        else:
            # the injection only touches flat pixels < n_inject, all in row 0: swap that row's counts
            raw = self.conf - count(1, n_inject)["conf"] + count(1, 0)["conf"]
            self.conf_aggregate = raw if self.conf_aggregate is None else self.conf_aggregate + raw
        self.n_aggregated += 1
        if isinstance(pred, dict) and pred.get("confidence") is not None:
            have_full = pred.get("confidence_full") is not None
            cres = ops.confidence_resample(pred["confidence"], w_full, h_full, y_pred_full=res["pred_full"],
                                           y_true_full=res["gt_full"], n_classes=C, want_full=not have_full, maps=maps)
            self.confidence_full = pred["confidence_full"] if have_full else cres["confidence_full"]
            self.reliability = cres["reliability"]
            self.reliability_aggregate = self.reliability.clone() if self.reliability_aggregate is None \
                else self.reliability_aggregate + self.reliability
        self.y_true_aggregate += [None]                   # placeholders: length = number of masks
        self.y_pred_aggregate += [None]

    def update(self, meta):
        self.meta = meta
        return self

    def evaluate(self, aggregate=False, distributed=False):
        """Compute the evaluation metrics (reference evaluate.py:131-148)."""
        self.aggregate = aggregate
        self.validate()
        counts = self.conf_aggregate if aggregate else self.conf
        assert counts is not None, "Evaluation failed. No ground truth was loaded."
        if aggregate and distributed:
            counts = pdist.all_reduce_(counts.clone())
        self.metrics.set_counts(counts, self.labels)
        self.metrics.f1_score(None, None)
        self.metrics.jaccard(None, None)
        self.metrics.mcc(None, None)
        self.metrics.confusion_matrix(None, None, labels=self.labels)
        self.metrics.report(None, None, labels=self.labels)
        table = self.reliability_aggregate if aggregate else self.reliability
        if table is not None:
            if aggregate and distributed:
                table = pdist.all_reduce_(table.clone())
            self.metrics.results['calibration'] = calibration_from_reliability(table.cpu().numpy(), self.labels)
            print('{:30s}{}'.format('ECE', self.metrics.results['calibration']['ece']))
        return self

    def validate(self):
        """Label list + aggregate bookkeeping (reference evaluate.py:150-176).  The coverage
        injection itself happens inside the confusion kernel (n_inject)."""
        self.labels = defaults.class_codes if self._schema[0] == len(defaults.class_codes) else self._schema[1]
        if self.aggregate:
            self.fid = 'aggregate_metrics'
            assert self.n_aggregated > 0, "Aggregate evaluation failed. Data buffer is empty."
            print("\nReporting aggregate metrics ... ")
            print("\t - Total generated masks: {}".format(self.n_aggregated))
            print()
        return self

    def reset(self):
        self.logits = None
        self.mask_pred = None
        self.results = []
        self.meta = {}
        self.y_true = None
        self.y_pred = None
        self.conf = None
        self.reliability = None
        self.confidence_full = None

    def save_logits(self, logits):
        logits_file = os.path.join(self.logits_dir, self.fid + '_output.pth')
        if utils.confirm_write_file(logits_file):
            torch.save({"results": logits, "meta": self.meta}, logits_file)
            print("Model output data saved to \n\t{}.".format(logits_file))
            return logits_file
        return

    def save_metrics(self):
        metrics_file = os.path.join(self.metrics_dir, self.fid + '_eval.json')
        cmap_img_file = os.path.join(self.metrics_dir, self.fid + '_cmap.pdf')
        cmap_data_file = os.path.join(self.metrics_dir, self.fid + '_cmap.npy')
        if utils.confirm_write_file(metrics_file):
            with open(metrics_file, 'w') as fp:
                json.dump(self.metrics.results, fp, indent=4)
        if utils.confirm_write_file(cmap_img_file):
            self.metrics.cmap.get_figure().savefig(cmap_img_file, format='pdf', dpi=400)
            np.save(cmap_data_file, self.metrics.cmatrix)
        self.metrics.plt.clf()
        return metrics_file, cmap_img_file, cmap_data_file

    def save_confidence(self):
        """Write the full-resolution confidence of the last loaded prediction as an 8-bit gray PNG
        (255 = probability 1.0) to <output>/confidence/<fid>.png; the directory is created on first use."""
        pred = self.mask_pred
        conf = self.confidence_full
        if conf is None and isinstance(pred, dict):
            conf = pred.get("confidence_full")
            if conf is None and pred.get("confidence") is not None:
                ex = self.meta.extract
                conf = ops.confidence_resample(pred["confidence"], ex['w_scaled'], ex['h_scaled'])["confidence_full"]
        if conf is None:
            print("No confidence map was computed. Confidence save cancelled.")
            return
        conf_file = os.path.join(utils.mk_path(os.path.join(self.output_dir, 'confidence')), self.fid + '.png')
        if utils.confirm_write_file(conf_file):
            cv2.imwrite(conf_file, conf.cpu().numpy())
            print("Confidence map saved to: \n\t{}.".format(conf_file))
            return conf_file
        return

    def save_image(self):
        """Write the predicted RGB mask as PNG (reference evaluate.py:262-284)."""
        mask_file = os.path.join(self.masks_dir, self.fid + '.png')
        if self.mask_pred is None:
            print("Mask has not been reconstructed. Image save cancelled.")
            return
        rgb = self.mask_pred
        if isinstance(rgb, dict):
            rgb = rgb["pred_rgb"].cpu().numpy()
        if utils.confirm_write_file(mask_file):
            cv2.imwrite(mask_file, cv2.cvtColor(np.asarray(rgb).astype(np.uint8), cv2.COLOR_RGB2BGR))
            print("Output mask saved to: \n\t{}.".format(mask_file))
            return mask_file
        return
