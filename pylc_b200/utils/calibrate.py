"""
Post-hoc temperature scaling of the mean stitch's probabilities (Guo et al., 2017, "On Calibration of Modern Neural
Networks"): P_T = the mean over the covering tiles of softmax(L / T), with one scalar T fitted by minimising the
negative log-likelihood of the full-resolution ground truth on labelled images.

The network is almost all of a segmentation step, so each image's network output is computed once and kept on the
device (TiledSegmenter.network_output: the logit batches, or the decoder batches on the fused route); every
evaluation of the objective re-runs only the tempered stitch (pylc_stitch_probs) and the score reduction
(pylc_prob_scores), through the same TiledSegmenter.stitch_output that `pylc test` runs.

Search, over u = ln T, of f(u) = sum_images nll_sum(T = exp(u)) / sum_images n_px (the kernels receive f32(exp(u))):
    1. the grid u_i = (i - 12) * ln(20) / 12, i = 0..24 (T from 0.05 to 20, T = 1 exactly at i = 12);
    2. i* = the first argmin on the grid;
    3. golden-section search on [u_max(i*-1, 0), u_min(i*+1, 24)] with invphi = (sqrt(5) - 1) / 2: keep [a, d] when
       f(c) <= f(d), else [c, b]; one interior point is reused per step; stop once b - a < 1e-4;
    4. T* = exp(u) of the evaluated point with the smallest f, the first evaluated on ties;
    5. i* = 0 or 24 flags the result `at_bound`: the minimum may lie outside [0.05, 20].
"""
import math

import numpy as np
import torch

from .. import _lib, ops
from .metrics import calibration_from_reliability

GRID_HALF = 12
GRID_STEP = math.log(20.0) / GRID_HALF
INVPHI = (math.sqrt(5.0) - 1.0) / 2.0
TOL = 1e-4


def fit_temperature(objective):
    """The search of the module docstring over objective(u) -> float.  Returns dict(temperature, u, f, at_bound,
    evals), `evals` = every evaluated (T, f) pair in evaluation order."""
    evals = []

    def f(u):
        v = float(objective(u))
        evals.append((u, v))
        return v
    grid = [(i - GRID_HALF) * GRID_STEP for i in range(2 * GRID_HALF + 1)]
    fg = [f(u) for u in grid]
    i_star = min(range(len(grid)), key=lambda i: (fg[i], i))
    a, b = grid[max(i_star - 1, 0)], grid[min(i_star + 1, len(grid) - 1)]
    c, d = b - INVPHI * (b - a), a + INVPHI * (b - a)
    fc, fd = f(c), f(d)
    while b - a >= TOL:
        if fc <= fd:
            b, d, fd = d, c, fc
            c = b - INVPHI * (b - a)
            fc = f(c)
        else:
            a, c, fc = c, d, fd
            d = a + INVPHI * (b - a)
            fd = f(d)
    best = min(range(len(evals)), key=lambda k: (evals[k][1], k))
    u_best, f_best = evals[best]
    return {"temperature": math.exp(u_best), "u": u_best, "f": f_best, "at_bound": i_star in (0, len(grid) - 1),
            "evals": [(math.exp(u), v) for u, v in evals]}


def write_calibrated_copy(model_path, out_path, calibration):
    """Write a copy of the PyLC model file `model_path` to `out_path` with one extra top-level key, "calibration"
    (Model.load keeps it as model.calibration); every other key is the input's."""
    from ..models.model import _load_model_file
    data = _load_model_file(model_path, "cpu")
    data["calibration"] = dict(calibration)
    torch.save(data, out_path)


class ResidentBudgetError(RuntimeError):
    """The next image's retained network output would pass the device-memory budget."""


class Retained(object):
    """One labelled image kept for the fit: its network output, tile grid, sizes, index maps and encoded
    full-resolution ground truth, all on the device."""
    __slots__ = ("src", "nr", "nc", "h", "w", "h_full", "w_full", "maps", "gt_full")


class TemperatureFit(object):
    """Retains labelled images for a TiledSegmenter(stitch="mean") and fits its temperature.  `budget_bytes` bounds
    the retained network outputs; add() raises ResidentBudgetError before the network pass of an image that would
    pass it."""

    def __init__(self, seg, budget_bytes):
        if seg.stitch != "mean" or seg.scales is not None:
            raise ValueError("temperature fitting needs a single-scale TiledSegmenter(stitch='mean')")
        self.seg = seg
        self.budget = int(budget_bytes)
        self.retained = []
        self.bytes = 0
        self.workspace = torch.empty((_lib.SCORES_WS_DOUBLES,), dtype=torch.float64, device=seg.device)

    def add(self, img, gt_rgb):
        """Stage a decoded image as `pylc test` does, run the network once and keep its output with the encoded
        ground truth (gt_rgb: decoded [H, W, 3] u8 mask of the same size)."""
        seg = self.seg
        h_full, w_full = img.shape[0], img.shape[1]
        if tuple(gt_rgb.shape[:2]) != (h_full, w_full):
            raise ValueError("mask %s and image %s differ in size" % (tuple(gt_rgb.shape[:2]), (h_full, w_full)))
        from . import tools
        w, h = tools.fit_dims(w_full, h_full, seg.T)
        nr, nc = h // seg.S - 1, w // seg.S - 1
        need = seg.retained_bytes(nr, nc)
        if self.bytes + need > self.budget:
            raise ResidentBudgetError(
                "the network outputs of %d image(s) fit in the %.2f GB budget; image %d needs %.2f GB more "
                "(raise --max_resident_gb or pass fewer images)" % (len(self.retained), self.budget / 1e9,
                                                                    len(self.retained) + 1, need / 1e9))
        f = seg.stage(img, None, index=len(self.retained))
        torch.cuda.current_stream().wait_event(f.ready)
        tiles, nr, nc = seg.fitted_tiles(f)
        r = Retained()
        r.src = seg.network_output(tiles)
        del tiles
        seg._release(f, torch.cuda.current_stream())
        r.nr, r.nc, r.h, r.w, r.h_full, r.w_full = nr, nc, f.h, f.w, h_full, w_full
        r.maps = ops.device_index_maps(f.w, f.h, w_full, h_full, seg.device)
        d_gt, pitch = ops.upload_image(np.ascontiguousarray(gt_rgb, dtype=np.uint8), seg.device)
        r.gt_full = ops.class_encode_hwc(d_gt, h_full, w_full, pitch, seg.palette)[0]
        self.retained.append(r)
        self.bytes += need
        return r

    @property
    def n_px(self):
        return sum(r.h_full * r.w_full for r in self.retained)

    def _probs(self, r, temperature, **kw):
        return self.seg.stitch_output(r.src, r.nr, r.nc, temperature=temperature, **kw)

    def nll(self, temperature):
        """Mean NLL over every retained pixel at `temperature` (f32 in the kernels)."""
        total = torch.zeros((2,), dtype=torch.float64, device=self.seg.device)
        for r in self.retained:
            probs = self._probs(r, temperature, want_labels=False, want_confidence=False, want_probs=True)["probs"]
            total += ops.prob_scores(probs, r.gt_full, r.w_full, r.h_full, want_brier=False, maps=r.maps,
                                     workspace=self.workspace)
        return float(total[0].item()) / self.n_px

    def fit(self):
        if not self.retained:
            raise ValueError("no images to fit a temperature on")
        return fit_temperature(lambda u: self.nll(math.exp(u)))

    def report(self, temperature):
        """Mean NLL and Brier score, accuracy, ECE and MCE of the mean stitch at `temperature` over the retained
        images (labels of the full-resolution pixels, no coverage injection)."""
        seg = self.seg
        C = seg.C
        total = torch.zeros((2,), dtype=torch.float64, device=seg.device)
        conf = torch.zeros((C, C), dtype=torch.int64, device=seg.device)
        rel = torch.zeros((C, 256, 2), dtype=torch.int64, device=seg.device)
        for r in self.retained:
            out = self._probs(r, temperature, want_labels=True, want_confidence=True, want_probs=True)
            total += ops.prob_scores(out["probs"], r.gt_full, r.w_full, r.h_full, want_brier=True, maps=r.maps,
                                     workspace=self.workspace)
            pred = ops.resample_encode_confusion(out["labels"], r.w_full, r.h_full, n_classes=C, n_inject=0,
                                                 want_pred=True, maps=r.maps)["pred_full"]
            ops.confusion_u8(r.gt_full, pred, C, conf=conf)
            ops.confidence_resample(out["confidence"], r.w_full, r.h_full, y_pred_full=pred, y_true_full=r.gt_full,
                                    n_classes=C, reliability=rel, want_full=False, maps=r.maps)
        sums = total.cpu().numpy()
        cm = conf.cpu().numpy()
        cal = calibration_from_reliability(rel.cpu().numpy())
        n = self.n_px
        return {"temperature": float(temperature), "nll": float(sums[0] / n), "brier": float(sums[1] / n),
                "accuracy": float(np.trace(cm) / max(cm.sum(), 1)), "ece": cal["ece"], "mce": cal["mce"]}
