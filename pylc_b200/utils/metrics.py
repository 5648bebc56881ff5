"""
Evaluation metrics -- host-side mirror of PyLC's utils/metrics.py (reference metrics.py:24-132).

The reference calls scikit-learn five times per evaluation (weighted F1, weighted Jaccard, MCC,
row-normalised confusion matrix, classification report; metrics.py:45-87) and every call builds
its own confusion matrix from the two flat label vectors.  Here ONE i64 [C,C] matrix is counted on
the GPU (pylc_confusion_u8 / pylc_resample_encode_confusion) and all five results are O(C^2) host
arithmetic on it (SURVEY.md A.6), in float64 like scikit-learn.  `Metrics` keeps the reference's
method names and `.results / .cmatrix / .cmap / .plt` attributes.
"""
import math

import numpy as np
import torch

from .. import ops


def scores_from_confusion(M, labels=None):
    """All reported numbers from one count matrix M[t, p].

    Classes that occur in neither vector are dropped first, which is what scikit-learn's
    `unique_labels` does; with Evaluator.validate's coverage injection every class is present.
    Returns {'f1','iou','mcc','cmatrix'[,'report']} -- cmatrix is M / row-sum (normalize='true').
    """
    M = np.asarray(M, dtype=np.int64)
    present = np.flatnonzero((M.sum(axis=0) + M.sum(axis=1)) > 0)
    K = M[np.ix_(present, present)].astype(np.float64)
    n = K.sum()
    hit = np.diag(K)
    truth = K.sum(axis=1)
    guess = K.sum(axis=0)

    def ratio(a, b):
        out = np.zeros_like(a)
        np.divide(a, b, out=out, where=b > 0)
        return out

    precision = ratio(hit, guess)
    recall = ratio(hit, truth)
    f1 = ratio(2 * hit, truth + guess)
    iou = ratio(hit, truth + guess - hit)
    weighted = lambda v: float((v * truth).sum() / n) if n > 0 else 0.0  # noqa: E731  (np.average's order)
    # Matthews correlation, multiclass form
    cov_tp = hit.sum() * n - np.dot(truth, guess)
    cov_pp = n * n - np.dot(guess, guess)
    cov_tt = n * n - np.dot(truth, truth)
    mcc = 0.0 if cov_pp * cov_tt == 0 else float(cov_tp / math.sqrt(cov_tt * cov_pp))
    out = {'f1': weighted(f1), 'iou': weighted(iou), 'mcc': mcc, 'cmatrix': ratio(K, np.broadcast_to(truth[:, None], K.shape))}
    if labels is not None:
        names = [labels[i] for i in present] if len(labels) >= (present.max() + 1 if len(present) else 0) \
            else [str(i) for i in present]
        report = {}
        for k, name in enumerate(names):
            report[name] = {'precision': float(precision[k]), 'recall': float(recall[k]),
                            'f1-score': float(f1[k]), 'support': float(truth[k])}
        report['accuracy'] = float(hit.sum() / n) if n > 0 else 0.0
        report['macro avg'] = {'precision': float(precision.mean()), 'recall': float(recall.mean()),
                               'f1-score': float(f1.mean()), 'support': float(n)}
        report['weighted avg'] = {'precision': weighted(precision), 'recall': weighted(recall),
                                  'f1-score': weighted(f1), 'support': float(n)}
        out['report'] = report
    return out


def calibration_from_reliability(table, class_codes=None, n_bins=15):
    """Calibration figures from a reliability table [C, 256, 2] of pixel counts (predicted class, confidence
    level q, prediction correct) -- pylc_confidence_resample's table, summed over images and ranks.

    The confidence of level q is q / 255.  Bin b of `n_bins` equal-width bins holds the levels with
    b <= q / 255 * n_bins < b + 1 (the last bin also holds 1.0).  In float64:
        ECE = sum_b n_b / N * |accuracy_b - confidence_b|,   MCE = max over non-empty bins of |accuracy_b - confidence_b|
    and, per predicted class, the mean confidence and the accuracy of its pixels.  Empty bins / classes report
    0.0 with a count of 0.  Returns a JSON-ready dict."""
    t = np.asarray(table, dtype=np.int64)
    if t.ndim != 3 or t.shape[1:] != (256, 2):
        raise ValueError("reliability table must be [C, 256, 2], got %s" % (t.shape,))
    C = t.shape[0]
    level = np.arange(256, dtype=np.float64) / 255.0
    bin_of = np.minimum((level * n_bins).astype(np.int64), n_bins - 1)
    per_q = t.sum(axis=0)                                   # [256, 2] over classes
    n_q = per_q.sum(axis=1).astype(np.float64)
    hit_q = per_q[:, 1].astype(np.float64)
    count = np.bincount(bin_of, weights=n_q, minlength=n_bins)
    hits = np.bincount(bin_of, weights=hit_q, minlength=n_bins)
    conf_sum = np.bincount(bin_of, weights=n_q * level, minlength=n_bins)

    def ratio(a, b):
        out = np.zeros_like(a, dtype=np.float64)
        np.divide(a, b, out=out, where=b > 0)
        return out
    acc_b, conf_b = ratio(hits, count), ratio(conf_sum, count)
    N = count.sum()
    gap = np.abs(acc_b - conf_b)
    ece = float((count * gap).sum() / N) if N > 0 else 0.0
    mce = float(gap[count > 0].max()) if N > 0 else 0.0
    n_c = t.sum(axis=(1, 2)).astype(np.float64)
    hit_c = t[:, :, 1].sum(axis=1).astype(np.float64)
    conf_c = ratio((t.sum(axis=2) * level[None, :]).sum(axis=1), n_c)
    acc_c = ratio(hit_c, n_c)
    names = list(class_codes) if class_codes is not None and len(class_codes) >= C else [str(i) for i in range(C)]
    return {'ece': ece, 'mce': mce, 'n_bins': int(n_bins), 'n_pixels': int(N),
            'bins': {'count': [int(v) for v in count], 'accuracy': [float(v) for v in acc_b],
                     'confidence': [float(v) for v in conf_b]},
            'classes': {str(names[c]): {'count': int(n_c[c]), 'confidence': float(conf_c[c]), 'accuracy': float(acc_c[c])}
                        for c in range(C)}}


def format_report(report):
    """Plain-text table of a classification report dict (what the reference prints, metrics.py:58-64)."""
    rows = [k for k in report if k not in ('accuracy', 'macro avg', 'weighted avg')]
    width = max([len(r) for r in rows] + [len('weighted avg')])
    lines = ['{:>{w}s} {:>9s} {:>9s} {:>9s} {:>9s}'.format('', 'precision', 'recall', 'f1-score', 'support', w=width), '']
    for r in rows:
        v = report[r]
        lines.append('{:>{w}s} {:9.2f} {:9.2f} {:9.2f} {:9d}'.format(
            r, v['precision'], v['recall'], v['f1-score'], int(v['support']), w=width))
    lines.append('')
    total = int(report['weighted avg']['support'])
    lines.append('{:>{w}s} {:>9s} {:>9s} {:9.2f} {:9d}'.format('accuracy', '', '', report['accuracy'], total, w=width))
    for r in ('macro avg', 'weighted avg'):
        v = report[r]
        lines.append('{:>{w}s} {:9.2f} {:9.2f} {:9.2f} {:9d}'.format(
            r, v['precision'], v['recall'], v['f1-score'], int(v['support']), w=width))
    return '\n'.join(lines)


class _Heatmap(object):
    """Stand-in for the seaborn axes the reference keeps in Metrics.cmap (metrics.py:84): renders
    the row-normalised matrix with matplotlib when it is installed, otherwise writes nothing."""

    def __init__(self, matrix, labels):
        self.matrix, self.labels = matrix, labels

    def get_figure(self):
        return self

    def savefig(self, path, **kwargs):
        try:
            import matplotlib
            matplotlib.use('Agg')
            import matplotlib.pyplot as plt
        except Exception:
            return None
        fig, ax = plt.subplots()
        ax.imshow(self.matrix, vmin=0.01, vmax=1.0)
        ax.set_xticks(range(len(self.labels)), self.labels)
        ax.set_yticks(range(len(self.labels)), self.labels)
        ax.set_ylabel('Ground-truth')
        ax.set_xlabel('Predicted')
        fig.savefig(path, **kwargs)
        plt.close(fig)
        return path


class _NoPlot(object):
    def clf(self):
        pass


class Metrics:
    def __init__(self):
        self.font = {'weight': 'bold', 'size': 18}
        self.plt = _NoPlot()
        self.results = {}
        self.cmatrix = None
        self.cmap = None
        self.counts = None          # i64 [C,C] confusion counts of the last evaluation
        self._key = None
        self._scores = None

    # -- confusion matrix plumbing -----------------------------------------------------------
    def set_counts(self, counts, labels=None):
        """Adopt a confusion matrix already counted on the device (or all-reduced across ranks);
        the reference-API methods below may then be called with y_true = y_pred = None."""
        self.counts = counts.cpu().numpy() if torch.is_tensor(counts) else np.asarray(counts, dtype=np.int64)
        self._scores = scores_from_confusion(self.counts, labels)
        self._key = None
        return self

    def _ensure(self, y_true, y_pred, labels=None):
        if y_true is not None and self._key != (id(y_true), id(y_pred)):
            yt, yp = _as_device_u8(y_true), _as_device_u8(y_pred)
            n_classes = len(labels) if labels is not None else int(max(int(yt.max()), int(yp.max()))) + 1
            self.counts = ops.confusion_u8(yt, yp, n_classes).cpu().numpy()
            self._key = (id(y_true), id(y_pred))
            self._scores = None
        if self.counts is None:
            raise ValueError("Metrics: no label vectors and no confusion matrix were given")
        if self._scores is None or (labels is not None and 'report' not in self._scores):
            self._scores = scores_from_confusion(self.counts, labels)
        return self._scores

    # -- reference API (metrics.py:45-87) ----------------------------------------------------
    def report(self, y_true, y_pred, labels):
        self.results['report'] = self._ensure(y_true, y_pred, labels)['report']
        print('\nClassification Report')
        print(format_report(self.results['report']))

    def f1_score(self, y_true, y_pred):
        self.results['f1'] = self._ensure(y_true, y_pred)['f1']
        print('{:30s}{}'.format('Weighted F1 Score', self.results['f1']))

    def jaccard(self, y_true, y_pred):
        self.results['iou'] = self._ensure(y_true, y_pred)['iou']
        print('{:30s}{}'.format('Weighted IoU', self.results['iou']))

    def mcc(self, y_true, y_pred):
        self.results['mcc'] = self._ensure(y_true, y_pred)['mcc']
        print('{:30s}{}'.format('MCC', self.results['mcc']))

    def confusion_matrix(self, y_true, y_pred, labels):
        self.cmatrix = self._ensure(y_true, y_pred, labels)['cmatrix']
        self.cmap = _Heatmap(self.cmatrix, labels)


def _as_device_u8(v):
    t = torch.as_tensor(v)
    if t.dtype != torch.uint8:
        t = t.to(torch.uint8)
    if not t.is_cuda:
        t = t.contiguous().pin_memory().to(torch.device("cuda", torch.cuda.current_device()), non_blocking=True)
    return t


def jsd(p, q):
    """Jensen-Shannon divergence as the reference writes it (metrics.py:107-111)."""
    eps = 1e-8
    m = 0.5 * (p + q + eps)
    return 0.5 * np.sum(np.multiply(p, np.log(p / m + eps))) + 0.5 * np.sum(np.multiply(q, np.log(q / m + eps)))


def m2(p, n_classes):
    """M2 Gibbs index (metrics.py:131-132)."""
    assert n_classes > 1, "M2 variance for multiple classes."
    return (n_classes / (n_classes - 1)) * (1 - np.sum(p ** 2))
