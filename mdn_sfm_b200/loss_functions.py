"""Drop-in for the reference ``loss_functions.py`` (``Loss``, ``LossModule``) on top of the fused CUDA path.

Same constructor / method signatures, same returned structures and the same numbers as the reference
(loss_functions.py:11-205); the arithmetic runs in ``libmdn_loss.so``.  Differences, all deliberate:

* ``Loss.forward`` is ONE kernel launch over every (scale, source frame) instead of a Python double loop of
  ATen ops; gradients are produced by the same launch (the loss is a scalar).
* The reference hard-wires DC mode and leaves the photometric term commented out (loss_functions.py:48-50,124,
  132-133,194).  Here ``mode`` in {"SN","T","TG","DS","DC"} (default "DC" == HEAD) and ``photometric``
  (default False == HEAD) select the compositions SURVEY.md section 8a-M defines; both can also be given as
  ``opt.mode`` / ``opt.photometric``.
* ``Loss(opt, no_ssim=True)`` works (upstream raises AttributeError because ``self.ssim`` is never set,
  loss_functions.py:163-164,172): it means "L1 only".
* Only ``losses["loss"]`` carries a grad_fn; the per-term entries are detached values (the reference's are
  differentiable, nobody differentiates them).  The per-pixel ``outputs`` maps are computed lazily on first
  access (they are read every 50 batches for TensorBoard, trainer.py:248-250), and are not differentiable.
* ``padding_mode``: "zeros" (what every upstream caller passes), "border" and "reflection" as in ``F.grid_sample``.
* ``arith="cuda"`` (default) replays the rounding of the reference's CUDA-eager path, ``arith="cpu"`` that of its
  CPU path; they differ where ATen divides a tensor by a Python scalar (a reciprocal multiply on CUDA), which
  moves warp coordinates by an ulp and can flip a bilinear cell (MDN_OPT_CUDA_ARITH in include/mdn_loss.h).
"""
from __future__ import annotations

from collections.abc import Mapping

import torch
from torch import nn

from . import _cabi, fused
from ._cabi import (MASK_MIN, MASK_OWN, MASK_SHARED, OPT_CROSS_ENT, OPT_INST_MASK, OPT_SSIM, OUT_CONSIS, OUT_EPIP,
                    OUT_PHOTO, OUT_SMOOTH, TERM_CONSIS, TERM_EPIPOLAR, TERM_PHOTO, TERM_SMOOTH)
from .layers import SSIM, PoseParameters, get_scale_factor  # noqa: F401  (re-exported like the reference module does)
from .loss_utils import *  # noqa: F401,F403  (the reference does `from loss_utils import *`)
from .loss_utils import create_coords as _create_coords
from .loss_utils import _arith_flag, instance_mask_u8, instance_masks_u8
from .utils import gauss_distance_weight

MODES = ("SN", "T", "TG", "DS", "DC")


def _c(t, what):
    return _cabi.check_tensor(t, what=what).contiguous()


_side_streams = {}


def _side_stream(device):
    """One extra stream per device for work that may overlap the loss call's pre-pass (the DS / DC instance masks)."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device)
    return _side_streams[key]


def _mode_bits(mode, ds_base):
    if mode not in MODES:
        raise ValueError("mode must be one of %s (got %r)" % (MODES, mode))
    base = ds_base if mode == "DS" else ("SN" if mode in ("SN", "DC") else mode)
    if base not in ("SN", "T", "TG"):
        raise ValueError("ds_base must be SN, T or TG")
    bits = TERM_EPIPOLAR
    if mode == "DS":
        bits |= OPT_INST_MASK
    if mode == "DC":
        bits |= OPT_CROSS_ENT
    return fused.POST_OF_MODE[base], bits


class _Lazy(Mapping):
    """Read-only mapping whose values are produced by one shared thunk on first access."""

    def __init__(self, keys, compute, name):
        self._keys, self._compute, self._name = list(keys), compute, name

    def __getitem__(self, k):
        if k not in self._keys:
            raise KeyError(k)
        return self._compute()[self._name][k]

    def __iter__(self):
        return iter(self._keys)

    def __len__(self):
        return len(self._keys)


class LossModule(nn.Module):
    """loss_functions.py:11-157."""

    def __init__(self, opt, batch=None, ssim=None, padding_mode="zeros", cuda=True, *, mode=None, weights=None,
                 ds_base="SN", library=None, arith="cuda"):
        super().__init__()
        if padding_mode not in _cabi.PAD_FLAG:
            raise ValueError("padding_mode must be 'zeros', 'border' or 'reflection' (torch.nn.functional.grid_sample)")
        if not cuda:
            raise RuntimeError("mdn_sfm_b200.LossModule has no CPU path (cuda=False is not supported)")
        self.options = opt
        self.ssim = ssim
        self.alpha = opt.alpha
        self.padding_mode = padding_mode
        self.device = torch.device("cuda")
        self.mode = mode if mode is not None else getattr(opt, "mode", "DC")
        self.ds_base = ds_base
        self.weights = weights
        self._library = library
        self._cuda_arith = _arith_flag(arith)
        self.losses = {"consis": 0, "epip": 0, "smooth": 0}
        self.outputs = {"warps": {}, "diffs": {}, "valids": {}, "epipolars": {}, "flows": {}, "epipolar_ori": {}}
        self._pix_shape = (batch if batch is not None else opt.batch_size, opt.height, opt.width)
        self._pix = None

    # -- pixel grid: kept for API compatibility only; the kernels derive x, y from the thread index
    @property
    def pix_coords(self):
        if self._pix is None or tuple(self._pix.shape[0:1] + self._pix.shape[2:]) != self._pix_shape:
            self._pix = _create_coords(*self._pix_shape).to(self.device)
        return self._pix

    @pix_coords.setter
    def pix_coords(self, v):
        self._pix = v
        self._pix_shape = (v.shape[0], v.shape[2], v.shape[3])

    def create_coords(self, batch_size=64, height=128, width=416):
        """loss_functions.py:150-157."""
        self._pix_shape = (batch_size, height, width)
        self._pix = None
        return self.pix_coords

    # -- helpers
    def _tg_weight(self, h, w, device):
        ws = self.weights
        if ws is None:
            # one table per pyramid level 0 .. max(scales), so that opt.scales = [0, 2] finds its level-2 table
            ws = self.weights = gauss_distance_weight(max(getattr(self.options, "scales", [0, 1, 2, 3])) + 1,
                                                      self.options.height, self.options.width)
        for k, t in enumerate(ws):
            if tuple(t.shape[-2:]) == (h, w):
                if t.device != device:
                    ws[k] = t = t.to(device)
                return t.reshape(h, w).contiguous()
        raise ValueError("no Gaussian weight table of size %dx%d (tables are built from opt.height/width)" % (h, w))

    def _epi_extras(self, post, bits, h, w, device, instances_info, batch=None):
        weight = self._tg_weight(h, w, device) if post == fused.POST_TG else None
        inst = instance_mask_u8(instances_info, (h, w), device, self._library, batch) if bits & (OPT_INST_MASK | OPT_CROSS_ENT) else None
        return weight, inst

    def _frames(self, inputs, frame_ids, flow, mobiles, instances_info, cam_T_cam, scale, mask_mode):
        """One fused launch for `frame_ids` (1 or 2 source frames) at one scale; accumulates like :43-67."""
        o = self.options
        tgt = _c(inputs[("color", 0, scale)], "target image")
        b, _, h, w = tgt.size()
        self._pix_shape, self._pix = (b, h, w), None
        post, bits = _mode_bits(self.mode, self.ds_base)
        inv_K = inputs[("inv_K", scale)][:, :3, :3]
        S = fused.ScaleData(h, w, float(w), float(h), float(2 ** scale), tgt=tgt)
        for p, i in enumerate(frame_ids):
            S.flow[p] = _c(flow[("flow", i, scale)], "flow")
            S.mob[p] = _c(mobiles[p], "mobile mask")
            S.fmat[p] = fused.fundamental_matrix(inv_K, cam_T_cam[i][:, :3, :3], cam_T_cam[i][:, :3, -1]).contiguous()
        S.weight, S.inst = self._epi_extras(post, bits, h, w, tgt.device, instances_info, b)
        thr = getattr(o, "threshold", None) if post != fused.POST_SN else None
        # two launches so that losses["epip"] and losses["smooth"] each own their gradient (the reference
        # keeps them as separate differentiable accumulators); Loss.forward uses a single launch instead
        cfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=len(frame_ids), post=post, mask_mode=mask_mode, flags=bits,
                                threshold=thr, alpha=o.alpha, w_d2_sim=o.w_d2_sim,
                                want_maps=("post_map", "ori_map") if scale == 0 else ())
        epip, _, maps = fused.fused_loss(cfg, [S], self._library)
        self.losses["epip"] = self.losses["epip"] + epip
        if not o.disable_smoothloss:
            scfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=len(frame_ids), post=post, mask_mode=mask_mode, flags=TERM_SMOOTH)
            smooth, _, _ = fused.fused_loss(scfg, [S], self._library)
            self.losses["smooth"] = self.losses["smooth"] + smooth
        if scale == 0:
            for p, i in enumerate(frame_ids):
                self.outputs["epipolars"][(i, scale)] = maps["post_map"][p].expand(b, 3, h, w)
                self.outputs["flows"][(i, scale)] = get_scale_factor(b, h, w).to(tgt.device) * flow[("flow", i, scale)]
                self.outputs["epipolar_ori"][(i, scale)] = maps["ori_map"][p].expand(b, 3, h, w)

    def forward(self, inputs, frame_ids, flow, mobile, instances_info, cam_T_cam, scale):
        """loss_functions.py:27-67: every source frame masked with the same `mobile` map."""
        frame_ids = list(frame_ids)
        for k in range(0, len(frame_ids), 2):
            ids = frame_ids[k:k + 2]
            self._frames(inputs, ids, flow, [mobile] * len(ids), instances_info, cam_T_cam, scale, MASK_SHARED)

    def single_mobile_mask_forward(self, inputs, frame_id, flow, mobile, instances_info, cam_T_cam, scale):
        """loss_functions.py:69-105."""
        self._frames(inputs, [frame_id], flow, [mobile], instances_info, cam_T_cam, scale, MASK_SHARED)

    def photo_metric_loss(self, target, reference, flow_map):
        """loss_functions.py:107-115 -> (loss, warped, diff_map, valid_points (B,3,h,w) bool)."""
        target, reference, flow_map = _c(target, "target"), _c(reference, "reference"), _c(flow_map, "flow_map")
        b, _, h, w = flow_map.size()
        S = fused.ScaleData(h, w, 1.0, 1.0, 1.0, tgt=target)
        S.ref[0], S.flow[0] = reference, flow_map
        cfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=1, post=fused.POST_T, mask_mode=MASK_SHARED,
                                flags=TERM_PHOTO | (OPT_SSIM if self.ssim is not None else 0) | _cabi.PAD_FLAG[self.padding_mode],
                                want_maps=("warped", "diff", "valid"))
        total, _, maps = fused.fused_loss(cfg, [S], self._library)
        valid = maps["valid"][0].bool().expand(b, 3, h, w)
        return total, maps["warped"][0], maps["diff"][0], valid

    def epipolar_loss(self, flow_map, mobile_mask, instances_info, inv_K, ro, tran):
        """loss_functions.py:117-138 -> (loss, post.expand(b,3,h,w), map.expand(b,3,h,w)); flow_map in pixels."""
        flow_map, mobile_mask = _c(flow_map, "flow_map"), _c(mobile_mask, "mobile_mask")
        b, _, h, w = flow_map.size()
        post, bits = _mode_bits(self.mode, self.ds_base)
        S = fused.ScaleData(h, w, 1.0, 1.0, 1.0)
        S.flow[0], S.mob[0] = flow_map, mobile_mask
        S.fmat[0] = fused.fundamental_matrix(inv_K[:, :3, :3], ro, tran).contiguous()
        S.weight, S.inst = self._epi_extras(post, bits, h, w, flow_map.device, instances_info, b)
        o = self.options
        cfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=1, post=post, mask_mode=MASK_SHARED, flags=bits,
                                threshold=getattr(o, "threshold", None) if post != fused.POST_SN else None,
                                alpha=self.alpha, w_d2_sim=o.w_d2_sim, want_maps=("post_map", "ori_map"))
        total, _, maps = fused.fused_loss(cfg, [S], self._library)
        return total, maps["post_map"][0].expand(b, 3, h, w), maps["ori_map"][0].expand(b, 3, h, w)

    def consistency_loss(self, mobile1, mobile2, scale):
        """loss_functions.py:140-147."""
        m1, m2 = _c(mobile1, "mobile1"), _c(mobile2, "mobile2")
        b, _, h, w = m1.size()
        S = fused.ScaleData(h, w, 1.0, 1.0, float(2 ** scale))
        S.mob[0], S.mob[1] = m1, m2
        cfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=1, post=fused.POST_T, mask_mode=MASK_OWN, flags=TERM_CONSIS)
        total, _, _ = fused.fused_loss(cfg, [S], self._library)
        self.losses["consis"] = self.losses["consis"] + total


class Loss(nn.Module):
    """loss_functions.py:160-205."""

    def __init__(self, opt, no_ssim=True, padding_mode="zeros", alpha=1, *, mode=None, photometric=None, weights=None,
                 ds_base="SN", library=None, arith="cuda"):
        super().__init__()
        if padding_mode not in _cabi.PAD_FLAG:
            raise ValueError("padding_mode must be 'zeros', 'border' or 'reflection' (torch.nn.functional.grid_sample)")
        self.ssim = None if no_ssim else SSIM()
        self.opt = opt
        self.alpha = alpha   # stored but unused, as upstream (LossModule reads opt.alpha, loss_functions.py:16)
        self.padding_mode = padding_mode
        self.mode = mode if mode is not None else getattr(opt, "mode", "DC")
        self.photometric = photometric if photometric is not None else bool(getattr(opt, "photometric", False))
        self.ds_base = ds_base
        self.weights = weights
        self._library = library
        self._arith = arith
        self._cuda_arith = _arith_flag(arith)
        self._helper = None

    def _lm(self):
        if self._helper is None:
            self._helper = LossModule(self.opt, ssim=self.ssim, mode=self.mode, weights=self.weights,
                                      ds_base=self.ds_base, library=self._library, arith=self._arith)
        return self._helper

    def _scale_data(self, inputs, frame_id, flow, mobile, instances_info, scales, cam_T_cam, post, bits):
        lm = self._lm()
        ids = list(frame_id)
        poses = None
        params = all(isinstance(cam_T_cam[i], PoseParameters) for i in ids)
        if params and not self._cuda_arith:
            cam_T_cam = {i: cam_T_cam[i].matrix() for i in ids}      # the torch composition of networks/layers.py:16-98
            params = False
        if params:
            # PoseNet's outputs as parameters: the kernels build the pose matrices and F, and return d/d(axisangle, translation)
            F_all = None
            aas = [_c(cam_T_cam[i].axisangle, "axisangle") for i in ids]
            trs = [_c(cam_T_cam[i].translation, "translation") for i in ids]
            inv_Ks = [_c(inputs[("inv_K", s)].detach(), "inv_K") for s in scales]
            poses = ("params", aas, trs, inv_Ks)
        elif self._cuda_arith:
            # the kernels build F themselves from the poses (MdnLossDesc.cam / inv_K: 3x3 products accumulated like the
            # batched SGEMM the reference runs on CUDA) and return the pose gradients
            F_all = None
            cams = [_c(cam_T_cam[i], "cam_T_cam") for i in ids]
            inv_Ks = [_c(inputs[("inv_K", s)].detach(), "inv_K") for s in scales]
            for t in cams + inv_Ks:
                if t.dim() != 3 or tuple(t.shape[1:]) != (4, 4):
                    raise ValueError("inv_K / cam_T_cam must be (B,4,4)")
            poses = ("cam", cams, inv_Ks)
        else:
            # arith="cpu": the reference's own three torch.matmul calls (loss_utils.py:61-62), batched over scales / frames
            R = torch.stack([cam_T_cam[i][:, :3, :3] for i in ids], 0).unsqueeze(0)      # (1,P,B,3,3)
            t = torch.stack([cam_T_cam[i][:, :3, -1] for i in ids], 0).unsqueeze(0)      # (1,P,B,3)
            Kinv = torch.stack([inputs[("inv_K", s)][:, :3, :3] for s in scales], 0).unsqueeze(1)   # (S,1,B,3,3)
            F_all = fused.fundamental_matrix(Kinv, R, t).contiguous()                    # (S,P,B,3,3)
        data = []
        for k, s in enumerate(scales):
            tgt = _c(inputs[("color", 0, s)], "target image")
            b, _, h, w = tgt.size()
            S = fused.ScaleData(h, w, float(w), float(h), float(2 ** s), tgt=tgt)
            for p, i in enumerate(ids):
                S.flow[p] = _c(flow[("flow", i, s)], "flow")
                if F_all is not None:
                    S.fmat[p] = F_all[k, p]
                if self.photometric:
                    pk = inputs.get(("color_packed", i, s)) if hasattr(inputs, "get") else None
                    if pk is not None:      # the pyramid producer already wrote (r, g, b, -) per pixel: no repack launch
                        if tuple(pk.shape) != (b, h, w, 4):
                            raise ValueError("('color_packed', %d, %d) must be (B,h,w,4)" % (i, s))
                        S.ref_packed[p] = _c(pk, "packed source image")
                    else:
                        S.ref[p] = _c(inputs[("color", i, s)], "source image")
            if self.opt.disable_min:   # pair p is masked with its own frame's map (loss_functions.py:183-186)
                # one source frame: its own map masks the pair; the other frame's map is only the consistency term's
                # second operand ((p - r)^2 is symmetric, each map receives its own gradient)
                second = ids[1] if len(ids) == 2 else -ids[0]
                S.mob[0] = _c(mobile[("mobile", ids[0], s)], "mobile mask")
                S.mob[1] = _c(mobile[("mobile", second, s)], "mobile mask")
            else:                                         # torch.cat([m(-1), m(+1)]).min(1): this order breaks ties
                S.mob[0] = _c(mobile[("mobile", -1, s)], "mobile mask")
                S.mob[1] = _c(mobile[("mobile", 1, s)], "mobile mask")
            S.weight, _ = lm._epi_extras(post, 0, h, w, tgt.device, None)
            data.append(S)
        self._inst_ready = None
        if bits & (OPT_INST_MASK | OPT_CROSS_ENT):   # DS / DC: the masks of every pyramid level from one pass (four launches)
            dev = data[0].tgt.device
            sizes = [(S.height, S.width) for S in data]
            if dev.type == "cuda":
                # on a side stream: the fused call launches its pre-pass (source repack, SN maxima) first and waits for the
                # masks only in front of the kernels that read them (MdnLossDesc.inst_ready), so the two overlap
                cur, side = torch.cuda.current_stream(dev), _side_stream(dev)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    insts = instance_masks_u8(instances_info, sizes, dev, self._library, data[0].tgt.shape[0])
                    self._inst_ready = torch.cuda.Event()
                    self._inst_ready.record(side)
                for m in insts:
                    m.record_stream(cur)
            else:
                insts = instance_masks_u8(instances_info, sizes, dev, self._library, data[0].tgt.shape[0])
            for S, m in zip(data, insts):
                S.inst = m
        return data, F_all, poses

    def forward(self, inputs, frame_id, flow, mobile, instances_info, scales, cam_T_cam):
        o = self.opt
        post, bits = _mode_bits(self.mode, self.ds_base)
        scales, ids = list(scales), list(frame_id)
        if len(ids) > 2 or len(scales) > 4:
            raise ValueError("at most 2 source frames and 4 scales")
        flags = bits
        if not o.disable_smoothloss:
            flags |= TERM_SMOOTH
        if not o.disable_consisloss:
            flags |= TERM_CONSIS
        if self.photometric:
            flags |= TERM_PHOTO | (OPT_SSIM if self.ssim is not None else 0) | _cabi.PAD_FLAG[self.padding_mode]
        data, F_all, poses = self._scale_data(inputs, ids, flow, mobile, instances_info, scales, cam_T_cam, post, bits)
        cams = inv_Ks = aas = trs = None
        if poses is not None and poses[0] == "cam":
            _, cams, inv_Ks = poses
        elif poses is not None:
            _, aas, trs, inv_Ks = poses
        b = data[0].tgt.shape[0]
        cfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=len(ids), post=post, mask_mode=MASK_OWN if o.disable_min else MASK_MIN,
                                flags=flags, threshold=getattr(o, "threshold", None) if post != fused.POST_SN else None,
                                alpha=o.alpha, w_d2_sim=o.w_d2_sim, w_e=o.w_e, w_s=o.w_s, w_c=o.w_c,
                                w_p=getattr(o, "w_p", 1.0) if self.photometric else 0.0, inst_ready=self._inst_ready)
        total, terms, _ = fused.fused_loss(cfg, data, self._library, fmat_all=F_all, cams=cams, inv_Ks=inv_Ks, axisangles=aas,
                                           translations=trs)
        losses = {"consis": terms[OUT_CONSIS - 1] if not o.disable_consisloss else 0, "epip": terms[OUT_EPIP - 1],
                  "smooth": terms[OUT_SMOOTH - 1] if not o.disable_smoothloss else 0, "loss": total}
        if self.photometric:
            losses["photo"] = terms[OUT_PHOTO - 1]

        # ---- lazily evaluated per-pixel outputs (scale 0 only, like loss_functions.py:61-67)
        cache = {}

        def compute():
            if cache:
                return cache
            with torch.no_grad():
                S0 = data[0]
                S = fused.ScaleData(S0.height, S0.width, S0.flow_sx, S0.flow_sy, 1.0, tgt=S0.tgt, ref=S0.ref, ref_packed=S0.ref_packed,
                                    flow=[None if f is None else f.detach() for f in S0.flow],
                                    mob=[m.detach() for m in S0.mob],
                                    fmat=[None if f is None else f.detach() for f in S0.fmat],
                                    weight=S0.weight, inst=S0.inst)
                want = ("post_map", "ori_map") + (("warped", "diff", "valid") if self.photometric else ())
                mcfg = fused.FusedConfig(cuda_arith=self._cuda_arith, batch=b, n_pairs=len(ids), post=post, mask_mode=cfg.mask_mode,
                                         flags=flags & ~(TERM_SMOOTH | TERM_CONSIS), threshold=cfg.threshold,
                                         alpha=o.alpha, w_d2_sim=o.w_d2_sim, want_maps=want)
                _, _, maps = fused.fused_loss(mcfg, [S], self._library, cams=None if cams is None else [c.detach() for c in cams],
                                              inv_Ks=None if inv_Ks is None else inv_Ks[:1],
                                              axisangles=None if aas is None else [a.detach() for a in aas],
                                              translations=None if trs is None else [t.detach() for t in trs])
                h, w = S0.height, S0.width
                sf = get_scale_factor(b, h, w).to(S0.tgt.device)
                cache["epipolars"] = {(i, 0): maps["post_map"][p].expand(b, 3, h, w) for p, i in enumerate(ids)}
                cache["epipolar_ori"] = {(i, 0): maps["ori_map"][p].expand(b, 3, h, w) for p, i in enumerate(ids)}
                cache["flows"] = {(i, 0): sf * S0.flow[p].detach() for p, i in enumerate(ids)}
                if self.photometric:
                    cache["warps"] = {(i, 0): maps["warped"][p] for p, i in enumerate(ids)}
                    cache["diffs"] = {(i, 0): maps["diff"][p] for p, i in enumerate(ids)}
                    cache["valids"] = {(i, 0): maps["valid"][p].bool().expand(b, 3, h, w) for p, i in enumerate(ids)}
            return cache

        has0 = 0 in scales and scales[0] == 0
        keys0 = [(i, 0) for i in ids] if has0 else []
        outputs = {name: _Lazy(keys0 if (self.photometric or name not in ("warps", "diffs", "valids")) else [], compute, name)
                   for name in ("warps", "diffs", "valids", "epipolars", "flows", "epipolar_ori")}
        mins = {}

        def min_compute():
            if not mins:
                with torch.no_grad():
                    mins["min_mobiles"] = {s: torch.minimum(mobile[("mobile", -1, s)], mobile[("mobile", 1, s)])
                                           for s in scales}
            return mins

        outputs["min_mobiles"] = _Lazy(scales, min_compute, "min_mobiles")
        return outputs, losses
