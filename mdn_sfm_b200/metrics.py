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

Optical flow (``flow_errors``, ``flow_metrics``, ``FlowMetrics``): one kernel pass (``mdn_flow_errors``) up-samples the
network's flow to the ground-truth size the way ``F.interpolate(mode="bilinear", align_corners=False)`` does, scales it
to pixels, and gives per image and region the number of valid pixels, the number of KITTI Fl outliers
(``e > 3 and e / |gt| > 0.05``) and the float64 sum of the end-point errors e.  The per-pixel arithmetic is stated in
include/mdn_loss.h; the sums do not depend on scheduling.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _cabi

__all__ = ["MAX_THRESHOLDS", "METRICS", "mask_confusion", "mask_metrics", "MaskMetrics",
           "MAX_REGIONS", "FLOW_UNITS", "flow_errors", "flow_metrics", "FlowMetrics"]

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


# ----------------------------------------------------------------------------------------------------- optical flow

MAX_REGIONS = 8
FLOW_UNITS = ("normalized", "pixels")


def _flow_scale(units, h, w, H, W):
    """The fp32 (scale_x, scale_y) that take the prediction to pixels of the H x W ground truth."""
    if units == "normalized":      # the nets' output; the loss multiplies it by get_scale_factor
        return np.float32(W), np.float32(H)
    if units == "pixels":          # pixels of the prediction's own h x w
        return np.float32(W) / np.float32(w), np.float32(H) / np.float32(h)
    raise ValueError("mdn_sfm_b200: units must be one of %s (got %r)" % (FLOW_UNITS, units))


def _flow_thresholds(abs_thr, rel_thr):
    out = np.float32(abs_thr), np.float32(rel_thr)
    for name, v in zip(("abs_thr", "rel_thr"), out):
        if not np.isfinite(v) or v < 0:
            raise ValueError("mdn_sfm_b200: %s must be finite and >= 0 (got %r)" % (name, float(v)))
    return out


def _n_regions(n_regions):
    if not isinstance(n_regions, (int, np.integer)) or not 1 <= n_regions <= MAX_REGIONS:
        raise ValueError("mdn_sfm_b200: n_regions must be an integer in 1..%d (got %r)" % (MAX_REGIONS, n_regions))
    return int(n_regions)


def _label_map(t, name, shape, device):
    """bool / uint8 (B, H, W) or (B, 1, H, W) -> contiguous uint8 with a 16-byte aligned base (bool read as uint8)."""
    if t.dtype not in (torch.bool, torch.uint8):
        raise TypeError("mdn_sfm_b200: %s must be bool or uint8 (got %s)" % (name, t.dtype))
    if t.device != device:
        raise ValueError("mdn_sfm_b200: gt_flow on %s, %s on %s" % (device, name, t.device))
    if not (t.dim() == 3 or (t.dim() == 4 and t.shape[1] == 1)):
        raise ValueError("mdn_sfm_b200: %s must be (B, H, W) or (B, 1, H, W) (got %s)" % (name, tuple(t.shape)))
    if (t.shape[0], t.shape[-2], t.shape[-1]) != shape:
        raise ValueError("mdn_sfm_b200: %s %s does not match gt_flow's (B, H, W) = %s" % (name, tuple(t.shape), shape))
    t = _cabi.check_tensor(t.view(torch.uint8) if t.dtype == torch.bool else t, torch.uint8, name)
    return _aligned(t)


def _flow_inputs(flow, gt_flow, gt_valid, region, n_regions):
    """Checks the tensors -> (flow, gt_flow, gt_valid, region or None) ready for the C call, and (B, h, w, H, W)."""
    if region is None and n_regions != 1:
        raise ValueError("mdn_sfm_b200: region=None puts every pixel in region 0, so n_regions must be 1 (got %d)"
                         % n_regions)
    for name, t in (("flow", flow), ("gt_flow", gt_flow)):
        if t.dtype != torch.float32:
            raise TypeError("mdn_sfm_b200: %s must be torch.float32 (got %s; cast it first)" % (name, t.dtype))
        _cabi.check_tensor(t, torch.float32, name)
        if t.dim() != 4 or t.shape[1] != 2:
            raise ValueError("mdn_sfm_b200: %s must be (B, 2, h, w) (got %s)" % (name, tuple(t.shape)))
    if flow.device != gt_flow.device:
        raise ValueError("mdn_sfm_b200: flow on %s, gt_flow on %s" % (flow.device, gt_flow.device))
    B, _, h, w = flow.shape
    H, W = gt_flow.shape[-2:]
    if gt_flow.shape[0] != B:
        raise ValueError("mdn_sfm_b200: flow %s and gt_flow %s differ in batch" % (tuple(flow.shape), tuple(gt_flow.shape)))
    if not 1 <= B <= 65535 or min(h, w, H, W) < 1 or h * w > 2 ** 31 - 1 or H * W > 2 ** 31 - 1:
        raise ValueError("mdn_sfm_b200: batch must be 1..65535 and h*w, H*W 1..2^31-1 (got %d, %d, %d)"
                         % (B, h * w, H * W))
    valid = _label_map(gt_valid, "gt_valid", (B, H, W), gt_flow.device)
    region = None if region is None else _label_map(region, "region", (B, H, W), gt_flow.device)
    return _aligned(flow), _aligned(gt_flow), valid, region, (B, h, w, H, W)


def _flow_call(flow, gt_flow, gt_valid, region, n_regions, units, thr, library, cache=None):
    """The launch on checked scalars: -> (counts (B, R, 2) int64, epe_sum (B, R) float64).  cache: None or a dict
    (B, H, W) -> workspace that keeps the workspace of each shape."""
    flow, gt_flow, gt_valid, region, (B, h, w, H, W) = _flow_inputs(flow, gt_flow, gt_valid, region, n_regions)
    sx, sy = _flow_scale(units, h, w, H, W)
    library = library or _cabi.lib()
    nbytes = library.cdll.mdn_flow_errors_workspace_bytes(B, h, w, H, W, n_regions)
    workspace = None if cache is None else cache.get((B, H, W))
    if workspace is None:
        workspace = torch.empty(nbytes, dtype=torch.uint8, device=flow.device)
        if cache is not None:
            cache[(B, H, W)] = workspace
    counts = torch.empty((B, n_regions, 2), dtype=torch.int64, device=flow.device)
    epe_sum = torch.empty((B, n_regions), dtype=torch.float64, device=flow.device)
    library.call("mdn_flow_errors", flow.data_ptr(), h, w, float(sx), float(sy), gt_flow.data_ptr(), gt_valid.data_ptr(),
                 _cabi.ptr(region), n_regions, H, W, B, float(thr[0]), float(thr[1]), counts.data_ptr(),
                 epe_sum.data_ptr(), workspace.data_ptr(), nbytes, _cabi.stream_ptr(flow), dev=flow)
    return counts, epe_sum


def flow_errors(flow, gt_flow, gt_valid, *, units, region=None, n_regions=1, abs_thr=3.0, rel_thr=0.05, library=None):
    """End-point errors and KITTI Fl outliers of a predicted flow against ground truth, per image and region.

    flow: (B, 2, h, w) fp32 at any resolution, on a CUDA device; it is up-sampled to H x W as
    ``F.interpolate(mode="bilinear", align_corners=False)`` does (the identity at h = H, w = W).  units (required: a wrong
    unit scales every error): "normalized" for the nets' output, which the loss multiplies by ``get_scale_factor`` (scale
    (W, H)); "pixels" for pixels of the prediction's own h x w (scale (W / w, H / h) in fp32).  gt_flow: (B, 2, H, W)
    fp32 in pixels.  gt_valid: bool or uint8 (B, H, W) or (B, 1, H, W), non-zero = valid.  region: None (every pixel in
    region 0; n_regions must be 1) or bool / uint8 labels of the same shape; a label >= n_regions (e.g. 255) is ignored.
    A pixel is an outlier iff ``e > abs_thr and e / |gt| > rel_thr`` (KITTI: 3 px and 5 %).  A bf16 flow is a TypeError:
    cast it.  -> {"valid": (B, R) int64, "outliers": (B, R) int64, "epe_sum": (B, R) float64}."""
    n_regions = _n_regions(n_regions)
    thr = _flow_thresholds(abs_thr, rel_thr)
    counts, epe_sum = _flow_call(flow, gt_flow, gt_valid, region, n_regions, units, thr, library)
    return {"valid": counts[..., 0], "outliers": counts[..., 1], "epe_sum": epe_sum}


def flow_metrics(errors):
    """{"valid", "outliers", "epe_sum"} of `flow_errors` -> {"epe": epe_sum / valid, "fl": outliers / valid} in float64,
    NaN where valid == 0.  Fl is a fraction; KITTI tables print it in percent."""
    valid = errors["valid"].to(torch.float64)
    defined = errors["valid"] > 0
    nan = torch.full_like(valid, float("nan"))
    return {"epe": torch.where(defined, errors["epe_sum"] / valid, nan),
            "fl": torch.where(defined, errors["outliers"].to(torch.float64) / valid, nan)}


class FlowMetrics:
    """Accumulates flow-evaluation results over batches on the device, for n_regions regions plus "all".

    `update` launches `mdn_flow_errors` and adds to device accumulators without synchronising, so a CUDA graph can capture
    it (one workspace is cached per (B, H, W)).  Index r < n_regions of every accumulator is region r and index n_regions
    is "all", the sum over the regions: pooled `valid`, `outliers` (int64) and `epe_sum` (float64); per-image sums of EPE
    and Fl (`image_sums`, float64 (R + 1, 2)) over the images with at least one counted pixel there, and the number of
    such images (`defined`); and the number of images.  `all_reduce` sums every accumulator over the ranks of a process
    group (DDP validation); `compute` returns host results; `reset` zeroes the accumulators in place.

    Two aggregations: *pooled* (epe_sum / valid and outliers / valid of the summed counts: every valid pixel weighs the
    same) and *per-image mean* (the mean of each image's EPE and Fl over the images where they are defined).  Neither is
    claimed to be the reference's: its flow evaluation (eval_utils.py) is not available.  Fl is a fraction; KITTI tables
    print it in percent.  A NaN prediction at a counted pixel makes that image's EPE NaN, and the NaN reaches both
    aggregations rather than being skipped.  Ground-truth images of different sizes go in separate `update` calls.

    Regions, two recipes: static / moving -- the moving-object mask as labels 0 / 1; KITTI noc / occ -- gt_valid = the
    occ validity, region = 0 where noc is valid and 1 elsewhere, so that region 0 gives noc and "all" gives occ."""

    def __init__(self, n_regions, device, *, units, abs_thr=3.0, rel_thr=0.05, library=None):
        self.n_regions = _n_regions(n_regions)
        _flow_scale(units, 1, 1, 1, 1)     # checks the unit
        self.units = units
        self.thresholds = _flow_thresholds(abs_thr, rel_thr)
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.library = library
        self._workspace = {}     # (B, H, W) -> workspace
        R1 = self.n_regions + 1
        self.valid = torch.zeros(R1, dtype=torch.int64, device=self.device)
        self.outliers = torch.zeros(R1, dtype=torch.int64, device=self.device)
        self.epe_sum = torch.zeros(R1, dtype=torch.float64, device=self.device)
        self.image_sums = torch.zeros((R1, 2), dtype=torch.float64, device=self.device)
        self.defined = torch.zeros(R1, dtype=torch.int64, device=self.device)
        self.images = torch.zeros((), dtype=torch.int64, device=self.device)

    def _accumulators(self):
        return (self.valid, self.outliers, self.epe_sum, self.image_sums, self.defined, self.images)

    def reset(self):
        for t in self._accumulators():
            t.zero_()

    def update(self, flow, gt_flow, gt_valid, region=None):
        """Adds a batch: the arguments as for `flow_errors`, on this object's device.  -> the batch's `flow_errors`."""
        counts, epe_sum = _flow_call(flow, gt_flow, gt_valid, region, self.n_regions, self.units, self.thresholds,
                                     self.library, self._workspace)
        counts = torch.cat([counts, counts.sum(1, keepdim=True)], 1)           # (B, R + 1, 2): "all" last
        epe = torch.cat([epe_sum, epe_sum.sum(1, keepdim=True)], 1)
        per = flow_metrics({"valid": counts[..., 0], "outliers": counts[..., 1], "epe_sum": epe})
        defined = counts[..., 0] > 0
        vals = torch.stack([per["epe"], per["fl"]], -1)                          # (B, R + 1, 2)
        self.valid += counts[..., 0].sum(0)
        self.outliers += counts[..., 1].sum(0)
        self.epe_sum += epe.sum(0)
        self.image_sums += torch.where(defined[..., None], vals, torch.zeros_like(vals)).sum(0)
        self.defined += defined.sum(0)
        self.images += flow.shape[0]
        return {"valid": counts[:, :-1, 0], "outliers": counts[:, :-1, 1], "epe_sum": epe_sum}

    def all_reduce(self, group=None):
        """Sums every accumulator over the ranks of `group` (torch.distributed must be initialised)."""
        import torch.distributed as dist
        for t in self._accumulators():
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return self

    def compute(self):
        """-> {"pooled": {"epe", "fl"}, "per_image": {"epe", "fl"}, "defined", "valid", "outliers", "epe_sum": (R + 1,)
        each, "images": n, "regions": R} as host numpy values (index R is "all"; NaN where nothing defines a value)."""
        host = lambda t: t.to("cpu", copy=True)     # copies: the results outlive a later reset()
        valid, outliers, epe_sum = host(self.valid), host(self.outliers), host(self.epe_sum)
        sums, defined = host(self.image_sums).numpy(), host(self.defined).numpy()
        pooled = flow_metrics({"valid": valid, "outliers": outliers, "epe_sum": epe_sum})
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = np.where(defined[:, None] > 0, sums / np.maximum(defined, 1)[:, None], np.nan)
        return {"pooled": {k: pooled[k].numpy() for k in ("epe", "fl")},
                "per_image": {"epe": mean[:, 0], "fl": mean[:, 1]},
                "defined": defined, "valid": valid.numpy(), "outliers": outliers.numpy(), "epe_sum": epe_sum.numpy(),
                "images": int(self.images.cpu()), "regions": self.n_regions}
