"""Drop-in for the reference ``loss_utils.py``: same free functions, same signatures.

The heavy ones (`inverse_warp`, `get_epipolar_new`, `smooth_loss`) call the CUDA kernels through the C ABI;
the per-pixel one-liners that the reference applies to maps it has already materialised
(`post_process_epipolar_*`, `derivable_consistency_loss`, `detectron2_similarity_loss`) are thin torch
expressions on CUDA tensors -- inside ``Loss.forward`` none of them runs, the fused kernel does that work.
"""
from __future__ import annotations

import torch

from . import _cabi, fused
from .ops import EpipolarPointsFn, FlowWarpFn, _c

__all__ = ["inverse_warp", "get_epipolar_new", "detectron2_similarity_loss", "post_pro_epipolar_weighted",
           "post_process_epipolar_1", "get_batch_instance_mask", "post_process_epipolar_2", "create_coords",
           "smooth_loss", "derivable_consistency_loss", "compute_quantiles", "InstanceMaskTable"]


def _arith_flag(arith):
    if arith not in ("cuda", "cpu"):
        raise ValueError("arith must be 'cuda' (the reference's CUDA-eager rounding) or 'cpu'")
    return arith == "cuda"


def inverse_warp(ref_img, flow_map, pix_coords, padding_mode, library=None, arith="cuda"):
    """loss_utils.py:12-36 -> (warped (B,3,H,W), valid_points bool (B,3,H,W)).

    `pix_coords` is accepted for signature compatibility; the kernel derives the grid from the thread index
    (it must be the regular pixel grid, which is what every caller passes).  `arith` picks which of the
    reference's two roundings of `grid /= (w-1)` is replayed: its CUDA-eager one (default) or its CPU one.
    """
    if padding_mode not in _cabi.WARP_PAD:
        raise ValueError("padding_mode must be 'zeros', 'border' or 'reflection' (torch.nn.functional.grid_sample)")
    ref_img, flow_map = _c(ref_img, "ref_img"), _c(flow_map, "flow_map")
    warped, _, valid = FlowWarpFn.apply(ref_img, flow_map, (_cabi.WARP_CUDA_ARITH if _arith_flag(arith) else 0) | _cabi.WARP_PAD[padding_mode],
                                        True, library)
    return warped, valid.bool().unsqueeze(1).expand(-1, ref_img.shape[1], -1, -1)


def get_epipolar_new(p1, p2, inv_K, rotation, translation, library=None):
    """loss_utils.py:39-69 -> signed epipolar distance (B,1,N)."""
    F = fused.fundamental_matrix(inv_K, rotation, translation).contiguous()
    return EpipolarPointsFn.apply(_c(p1, "p1"), _c(p2, "p2"), _c(F, "F"), library)


def get_batch_instance_mask(instances_info):
    """loss_utils.py:102-124 -> int64 {0,1} (B,3,H,W) / (1,3,H,W)."""
    if isinstance(instances_info, list):
        m = torch.stack([(info["instances"].pred_masks.sum(0, keepdim=True) != 0) for info in instances_info], 0)
    else:
        m = (instances_info.pred_masks.sum(0, keepdim=True) != 0).unsqueeze(0)
    return m.to(torch.int64).repeat(1, 3, 1, 1)


def _pred_masks(instances_info):
    if isinstance(instances_info, list):
        return [info["instances"].pred_masks for info in instances_info]
    return [instances_info.pred_masks]


class InstanceMaskTable:
    """A batch's Detectron2 instance masks as a DEVICE table -- B mask pointers (int64) and B instance counts (int32) -- for
    `mdn_instance_mask_union_table`, which reads the table when its kernel runs.  A CUDA graph that captured the union
    therefore follows each new batch: `load` the batch, then replay.  Pass the table where `instances_info` goes
    (`instance_masks_u8`, `Loss.forward`).

    `load` writes the table in the current stream's order (a non-blocking copy from pinned host memory), so work queued
    after it on that stream sees the new batch, and work queued before it the old one.  The table keeps the mask tensors
    alive until the next `load`."""

    def __init__(self, batch, height, width, device):
        if batch < 1 or height < 1 or width < 1:
            raise ValueError("InstanceMaskTable needs batch, height and width >= 1")
        self.batch, self.height, self.width = int(batch), int(height), int(width)
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        # one buffer, one copy per load: B pointers, then B counts (int32, two per int64 slot)
        self._words = self.batch + (self.batch + 1) // 2
        self._table = torch.zeros(self._words, dtype=torch.int64, device=self.device)
        self.ptrs = self._table[:self.batch]
        self.counts = self._table[self.batch:].view(torch.int32)[:self.batch]
        self.masks = []

    def _check(self, m):
        if m.dtype != torch.bool and m.dtype != torch.uint8:
            raise TypeError("mdn_sfm_b200: pred_masks must be bool or uint8 (got %s)" % m.dtype)
        if m.device != self.device:
            raise ValueError("mdn_sfm_b200: pred_masks on %s, the instance table on %s" % (m.device, self.device))
        if m.dim() != 3 or tuple(m.shape[1:]) != (self.height, self.width):
            raise ValueError("mdn_sfm_b200: pred_masks must be (N, %d, %d) (got %s)" % (self.height, self.width, tuple(m.shape)))
        if not m.is_contiguous():
            raise ValueError("mdn_sfm_b200: pred_masks must be contiguous")
        return _cabi.check_tensor(m.view(torch.uint8) if m.dtype == torch.bool else m, dtype=torch.uint8, what="pred_masks")

    def load(self, instances_info):
        """Points the table at this batch's masks: a list of B {"instances": obj} dicts, or one bare `Instances` whose masks
        every sample of the batch uses (the reference's (1,3,H,W) mask broadcast over the batch)."""
        masks = [self._check(m) for m in _pred_masks(instances_info)]
        if isinstance(instances_info, list) and len(masks) != self.batch:
            raise ValueError("instances_info holds %d samples, the instance table %d" % (len(masks), self.batch))
        per_sample = masks if isinstance(instances_info, list) else masks * self.batch
        host = torch.empty(self._words, dtype=torch.int64, pin_memory=self.device.type == "cuda")
        h = host.numpy()
        h[:self.batch] = [m.data_ptr() for m in per_sample]
        h[self.batch:].view("int32")[:self.batch] = [m.shape[0] for m in per_sample]
        if self.device.type == "cuda":
            self._table.copy_(host, non_blocking=True)      # the caching host allocator holds `host` until the copy has run
            stream = torch.cuda.current_stream(self.device)
            for m in masks:
                m.record_stream(stream)
        else:
            self._table.copy_(host)
        self.masks = masks
        return self


def instance_masks_u8(instances_info, sizes, device, library=None, batch=None):
    """One-channel uint8 {0,1} instance masks at every size in `sizes` (a list of (h, w)), from ONE pass over the
    Detectron2 masks: `get_batch_instance_mask` (loss_utils.py:102-124: union of the instances of each sample) and the
    `Resize(size)` of loss_utils.py:73-75 / :135-137 (torchvision bilinear + antialias on the integer mask, rounded
    back to integers) run as two kernels -- `mdn_instance_mask_union`, `mdn_instance_mask_resize` -- instead of the
    reference's per-(frame, scale) int64 (B,3,375,1242) tensors.  The three channels upstream carries are identical;
    one is kept.  -> list of (B, h, w) uint8 tensors.  `batch`: the batch size of the maps the masks will meet; a single
    bare `Instances` (trainer.py:494, evaluate_mix.py:63) then broadcasts over it like the reference's (1,3,H,W) mask.
    `instances_info` may also be an InstanceMaskTable (then `device` is the table's): the union reads it on the device."""
    import ctypes as C
    library = library or _cabi.lib()
    if isinstance(instances_info, InstanceMaskTable):     # the union reads the device table: capturable in a CUDA graph
        T = instances_info
        B, H, W = T.batch, T.height, T.width
        union = torch.empty((B, H, W), dtype=torch.uint8, device=T.device)
        stream = _cabi.stream_ptr(union)
        library.call("mdn_instance_mask_union_table", T.ptrs.data_ptr(), T.counts.data_ptr(), union.data_ptr(), B, H * W,
                     stream, dev=union)
    else:
        masks = []
        for m in _pred_masks(instances_info):
            m = m.to(device)
            if m.dtype != torch.bool and m.dtype != torch.uint8:
                m = m != 0
            m = m.contiguous()
            masks.append(_cabi.check_tensor(m.view(torch.uint8) if m.dtype == torch.bool else m, dtype=torch.uint8, what="pred_masks"))
        B = len(masks)
        H, W = masks[0].shape[-2:]
        if any(tuple(m.shape[-2:]) != (H, W) for m in masks):
            raise ValueError("instance masks of one batch must share their size")
        union = torch.empty((B, H, W), dtype=torch.uint8, device=masks[0].device)
        stream = _cabi.stream_ptr(union)
        counts = (C.c_int32 * B)(*[int(m.shape[0]) if m.dim() == 3 else 1 for m in masks])
        library.call("mdn_instance_mask_union", _cabi.ptr_array(masks), counts, union.data_ptr(), B, H * W, stream, dev=union)
    outs = [torch.empty((B, int(h), int(w)), dtype=torch.uint8, device=union.device) for h, w in sizes]
    for k0 in range(0, len(outs), _cabi.MAX_SCALES):
        chunk = outs[k0:k0 + _cabi.MAX_SCALES]
        oh = (C.c_int32 * len(chunk))(*[o.shape[1] for o in chunk])
        ow = (C.c_int32 * len(chunk))(*[o.shape[2] for o in chunk])
        nbytes = library.cdll.mdn_instance_mask_resize_workspace_bytes(B, H, W, oh, ow, len(chunk))
        ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=union.device)
        library.call("mdn_instance_mask_resize", union.data_ptr(), B, H, W, _cabi.ptr_array(chunk), oh, ow, len(chunk),
                     ws.data_ptr(), nbytes, stream, dev=union)
    if batch is not None and B == 1 and batch > 1:
        outs = [o.expand(batch, -1, -1).contiguous() for o in outs]
    elif batch is not None and B != batch:
        raise ValueError("instances_info holds %d samples, the maps %d" % (B, batch))
    return outs


def instance_mask_u8(instances_info, size, device, library=None, batch=None):
    """Single-size form of instance_masks_u8."""
    return instance_masks_u8(instances_info, [tuple(size)], device, library, batch)[0]


def detectron2_similarity_loss(mobile_mask, instances_info):
    """loss_utils.py:72-78 -> cross-entropy map (B,3,h,w)."""
    from torchvision.transforms import Resize
    mask = Resize(tuple(mobile_mask.size()[2:]))(get_batch_instance_mask(instances_info).to(mobile_mask.device))
    return -(mask * torch.log(mobile_mask + 1e-10) + (1 - mask) * torch.log(1 - mobile_mask + 1e-10))


def post_pro_epipolar_weighted(epipolar_map, weight=None, threshold=None):
    """loss_utils.py:81-89 (T / TG)."""
    post = epipolar_map.clone()
    if threshold is not None:
        post /= threshold
    if weight is not None:
        post /= weight
    return post ** 2


def post_process_epipolar_1(epipolar_map):
    """loss_utils.py:92-99 (SN).  Divides its argument IN PLACE like the reference."""
    b = epipolar_map.size(0)
    norms = torch.max(epipolar_map.view(b, -1), dim=1, keepdim=True)[0]
    epipolar_map /= norms[..., None, None]
    return epipolar_map ** 2


def post_process_epipolar_2(epipolar_map, instances_info):
    """loss_utils.py:127-138 (DS)."""
    from torchvision.transforms import Resize
    mask = Resize(tuple(epipolar_map.size()[2:]))(get_batch_instance_mask(instances_info).to(epipolar_map.device))
    return mask * epipolar_map


def create_coords(batch_size=64, height=128, width=416):
    """loss_utils.py:141-148 -> (B,2,H,W) CPU tensor (ch0 = column, ch1 = row), like the reference."""
    xs = torch.arange(width, dtype=torch.float32).view(1, 1, 1, width).expand(1, 1, height, width)
    ys = torch.arange(height, dtype=torch.float32).view(1, 1, height, 1).expand(1, 1, height, width)
    return torch.cat([xs, ys], 1).repeat(batch_size, 1, 1, 1)


def smooth_loss(target, mobile, library=None):
    """loss_utils.py:151-168 -> scalar."""
    target, mobile = _c(target, "target"), _c(mobile, "mobile")
    b, _, h, w = target.shape
    S = fused.ScaleData(h, w, 1.0, 1.0, 1.0, tgt=target)
    S.mob[0] = mobile
    cfg = fused.FusedConfig(batch=b, n_pairs=1, post=fused.POST_T, mask_mode=_cabi.MASK_SHARED, flags=_cabi.TERM_SMOOTH)
    total, _, _ = fused.fused_loss(cfg, [S], library)
    return total


def derivable_consistency_loss(mobile1, mobile2, threshold=0.5):
    """loss_utils.py:171-177 -> per-pixel map."""
    return (torch.sigmoid(20 * (mobile1 - threshold)) - torch.sigmoid(20 * (mobile2 - threshold))) ** 2


def compute_quantiles(flow, cam_T_cam, inv_K, p1, pix_coords, ones, scale_factor, percentage, i, b):
    """loss_utils.py:197-202."""
    flow_map = scale_factor * flow[("flow", i, 0)]
    p2 = torch.cat([pix_coords + flow_map, ones], 1).view(b, 3, -1)
    e = get_epipolar_new(p1, p2, inv_K[:, :3, :3], cam_T_cam[:, :3, :3], cam_T_cam[:, :3, -1]).view(b, -1).abs()
    return torch.quantile(e, percentage, dim=1)
