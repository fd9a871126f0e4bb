"""Evaluation of mobile masks on the device: confusion counts for a whole threshold sweep in one pass.

The reference reports accuracy, precision, recall and dice of ``binary_image(mobile, thr)`` (utils.py:100-103) against
moving-object masks, with a binary threshold chosen per mode (README.md:27-33).  Here one kernel pass
(``mdn_mask_confusion``) gives, for every image and threshold, the exact integer counts ``[TP, FP, FN, TN]`` with
``pred >= thr`` in fp32 as the prediction: a prediction equal to a threshold is moving at it, NaN is never moving.
Nothing synchronises with the host, so ``MaskMetrics.update`` can be captured in a CUDA graph.

Metrics are formed from the counts in float64: accuracy = (TP+TN)/(h*w), precision = TP/(TP+FP), recall = TP/(TP+FN),
dice = 2TP/(2TP+FP+FN), iou = TP/(TP+FP+FN); 0/0 is NaN for that image.  Two aggregations: *pooled* (the formulas on
the counts summed over all images) and *per-image mean* (the mean over the images where the value is defined, with the
number of such images).  Neither is claimed to be the reference's: its aggregation (eval_utils.py) is not available,
and its README numbers are not pooled ones -- pooled dice always equals 2PR/(P+R), which is 24.1 % for its SN row,
where the README reports 18.58 %.  Resizing predictions to the ground-truth size is the caller's job.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _cabi

__all__ = ["MAX_THRESHOLDS", "METRICS", "mask_confusion", "mask_metrics", "MaskMetrics"]

MAX_THRESHOLDS = 1024
METRICS = ("accuracy", "precision", "recall", "dice", "iou")


def _host_thresholds(thresholds):
    """-> (K,) float32 numpy array, checked: 1 <= K <= 1024, no NaN, strictly increasing (in fp32)."""
    if isinstance(thresholds, torch.Tensor):
        t = thresholds.detach().to("cpu", torch.float32).numpy()     # one synchronisation for a CUDA tensor
    else:
        t = np.asarray(thresholds, dtype=np.float64).astype(np.float32)
    if t.ndim != 1:
        raise ValueError("mdn_sfm_b200: thresholds must be one-dimensional (got shape %s)" % (t.shape,))
    if not 1 <= t.shape[0] <= MAX_THRESHOLDS:
        raise ValueError("mdn_sfm_b200: 1 to %d thresholds are supported (got %d)" % (MAX_THRESHOLDS, t.shape[0]))
    if np.isnan(t).any():
        raise ValueError("mdn_sfm_b200: thresholds must not be NaN")
    if (np.diff(t) <= 0).any():
        raise ValueError("mdn_sfm_b200: thresholds must be strictly increasing in float32")
    return np.ascontiguousarray(t)


def _aligned(t):
    """Contiguous with a 16-byte aligned base (the C ABI's convention); copies only a tensor that is neither."""
    if not t.is_contiguous() or t.data_ptr() % 16:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


def _maps(pred, gt):
    """(B, h, w) or (B, 1, h, w) pred (fp32) and gt (bool / uint8) -> contiguous (B, h*w)-shaped views and (B, h, w)."""
    if pred.dtype != torch.float32:
        raise TypeError("mdn_sfm_b200: pred must be torch.float32 (got %s)" % pred.dtype)
    _cabi.check_tensor(pred, torch.float32, "pred")
    if gt.dtype not in (torch.bool, torch.uint8):
        raise TypeError("mdn_sfm_b200: gt must be bool or uint8 (got %s)" % gt.dtype)
    if gt.device != pred.device:
        raise ValueError("mdn_sfm_b200: pred on %s, gt on %s" % (pred.device, gt.device))
    shapes = []
    for name, t in (("pred", pred), ("gt", gt)):
        if not (t.dim() == 3 or (t.dim() == 4 and t.shape[1] == 1)):
            raise ValueError("mdn_sfm_b200: %s must be (B, h, w) or (B, 1, h, w) (got %s)" % (name, tuple(t.shape)))
        shapes.append((t.shape[0], t.shape[-2], t.shape[-1]))
    if shapes[0] != shapes[1]:
        raise ValueError("mdn_sfm_b200: pred %s and gt %s differ in size (resize the prediction first)"
                         % (tuple(pred.shape), tuple(gt.shape)))
    B, h, w = shapes[0]
    if not 1 <= B <= 65535 or not 1 <= h * w <= 2 ** 31 - 1:
        raise ValueError("mdn_sfm_b200: batch must be 1..65535 and h*w 1..2^31-1 (got %d, %d)" % (B, h * w))
    gt = _cabi.check_tensor(gt.view(torch.uint8) if gt.dtype == torch.bool else gt, torch.uint8, "gt")
    return _aligned(pred), _aligned(gt), (B, h, w)


def _confusion(pred, gt, thr, library, workspace=None):
    """The launch: thr is an already checked (K,) fp32 tensor on pred's device.  -> (B, K, 4) int64."""
    pred, gt, (B, h, w) = _maps(pred, gt)
    if thr.device != pred.device:
        raise ValueError("mdn_sfm_b200: thresholds on %s, pred on %s" % (thr.device, pred.device))
    library = library or _cabi.lib()
    K = thr.shape[0]
    nbytes = library.cdll.mdn_mask_confusion_workspace_bytes(B, K)
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty(nbytes, dtype=torch.uint8, device=pred.device)
    counts = torch.empty((B, K, 4), dtype=torch.int64, device=pred.device)
    library.call("mdn_mask_confusion", pred.data_ptr(), gt.data_ptr(), thr.data_ptr(), K, counts.data_ptr(), B, h * w,
                 workspace.data_ptr(), nbytes, _cabi.stream_ptr(pred), dev=pred)
    return counts


def _device_thresholds(host, device):
    return torch.from_numpy(host.copy()).to(device)


def mask_confusion(pred, gt, thresholds, library=None):
    """Confusion counts of ``pred >= thr`` against ``gt != 0`` for every image and threshold.

    pred: fp32 mobile probabilities, (B, h, w) or (B, 1, h, w), on a CUDA device.  gt: bool or uint8 of the same
    (B, h, w), on the same device (a bool tensor is read as uint8 without a copy).  thresholds: 1 to 1024 values, strictly
    increasing in fp32, no NaN (+-inf allowed); a host sequence, or a tensor -- checked on the host, so a CUDA tensor
    costs one synchronisation.  -> (B, K, 4) int64 [TP, FP, FN, TN]; every row sums to h*w."""
    host = _host_thresholds(thresholds)
    if isinstance(thresholds, torch.Tensor) and thresholds.dtype == torch.float32 and thresholds.device == pred.device:
        thr = _aligned(thresholds.detach())
    else:
        thr = _device_thresholds(host, pred.device)
    return _confusion(pred, gt, thr, library)


def mask_metrics(counts):
    """(..., K, 4) int64 [TP, FP, FN, TN] -> {name: (..., K) float64} for the names in METRICS, NaN where 0/0."""
    tp, fp, fn, tn = counts.to(torch.float64).unbind(-1)
    return {"accuracy": (tp + tn) / (tp + fp + fn + tn),
            "precision": tp / (tp + fp),
            "recall": tp / (tp + fn),
            "dice": 2 * tp / (2 * tp + fp + fn),
            "iou": tp / (tp + fp + fn)}


class MaskMetrics:
    """Accumulates mask-evaluation results over batches on the device, for a fixed threshold sweep.

    The thresholds are checked and uploaded once.  `update` launches the counting kernel and adds to device accumulators
    -- pooled counts (K, 4), per-image metric sums and the number of images where each metric is defined (K, 5), and the
    number of images -- without synchronising, so a CUDA graph can capture it.  `all_reduce` sums the accumulators over
    the ranks of a process group (DDP validation); `compute` returns host results; `reset` zeroes the accumulators in
    place (a captured graph keeps adding to the same tensors).  See the module docstring for the aggregations."""

    def __init__(self, thresholds, device, library=None):
        self.thresholds = _host_thresholds(thresholds)
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.library = library
        self._thr = _device_thresholds(self.thresholds, self.device)
        self._workspace = {}     # batch size -> workspace of that batch size
        K = self.thresholds.shape[0]
        self.pooled = torch.zeros((K, 4), dtype=torch.int64, device=self.device)
        self.sums = torch.zeros((K, len(METRICS)), dtype=torch.float64, device=self.device)
        self.defined = torch.zeros((K, len(METRICS)), dtype=torch.int64, device=self.device)
        self.images = torch.zeros((), dtype=torch.int64, device=self.device)

    def reset(self):
        for t in (self.pooled, self.sums, self.defined, self.images):
            t.zero_()

    def update(self, pred, gt):
        """Adds a batch: pred / gt as for `mask_confusion`, on this object's device."""
        B = pred.shape[0]
        ws = self._workspace.get(B)
        if ws is None:
            nbytes = (self.library or _cabi.lib()).cdll.mdn_mask_confusion_workspace_bytes(B, self._thr.shape[0])
            ws = self._workspace[B] = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=self.device)
        counts = _confusion(pred, gt, self._thr, self.library, ws)
        m = mask_metrics(counts)
        vals = torch.stack([m[k] for k in METRICS], -1)      # (B, K, 5)
        ok = ~torch.isnan(vals)
        self.pooled += counts.sum(0)
        self.sums += torch.where(ok, vals, torch.zeros_like(vals)).sum(0)
        self.defined += ok.sum(0)
        self.images += B
        return counts

    def all_reduce(self, group=None):
        """Sums every accumulator over the ranks of `group` (torch.distributed must be initialised)."""
        import torch.distributed as dist
        for t in (self.pooled, self.sums, self.defined, self.images):
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return self

    def compute(self):
        """-> {"thresholds": (K,), "pooled": {metric: (K,)}, "per_image": {metric: (K,)}, "defined": {metric: (K,)},
        "images": n, "counts": (K, 4)} as host numpy values (per_image is NaN where no image defines the metric)."""
        host = lambda t: t.to("cpu", copy=True)     # copies: the results outlive a later reset()
        pooled = host(self.pooled)
        sums, defined = host(self.sums).numpy(), host(self.defined).numpy()
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = np.where(defined > 0, sums / np.maximum(defined, 1), np.nan)
        pm = mask_metrics(pooled)
        return {"thresholds": self.thresholds.copy(),
                "pooled": {k: pm[k].numpy() for k in METRICS},
                "per_image": {k: mean[:, i] for i, k in enumerate(METRICS)},
                "defined": {k: defined[:, i] for i, k in enumerate(METRICS)},
                "images": int(self.images.cpu()),
                "counts": pooled.numpy()}
