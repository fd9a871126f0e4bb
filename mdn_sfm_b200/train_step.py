"""Minimal DDP train-step harness around the loss path (SURVEY.md 8f-N1; BASELINE configs[2]).

Mirrors ``Trainer.process_batch`` + the body of ``Trainer.run_epoch`` (trainer.py:223-287) without Detectron2 / KITTI:

    for each source frame i:  flow, features = flownet(tgt, ref_i);  axisangle, t = posenet(tgt, ref_i)
                              mobiles_i = mobile_decoder(features, axisangle, t);  cam_T_cam[i] = T(axisangle, t)
    outputs, losses = Loss(inputs, frame_ids, flows, mobiles, instances, scales, cam_T_cam)       # trainer.py:280-281
    zero_grad;  losses["loss"].backward();  clip_grad_norm_;  Adam.step                           # trainer.py:233-237

The CNNs are consumers of cuDNN and stay in torch.  The reference's FlowNet_v1 / PoseNet_v3 / MobileDecoder are NOT
re-implemented here: ``StandInNets`` is a compact network family of the same interface (frozen flow + pose nets, a
trainable mobile decoder with four sigmoid output scales), enough to drive the step end to end.  Real nets plug in
through the ``nets`` argument -- any object with ``flownet(tgt, ref, frame_id)``, ``posenet(tgt, ref)`` and
``mobile_decoder(features, axisangle, translation, frame_id)`` of the reference's signatures.

Multi-GPU: one process per GPU, batch sharded by the sampler; the ONLY collectives are DDP's bucketed gradient
all-reduce of the mobile decoder (NCCL over NVLink) and one small all-reduce of the loss scalars for logging
(``distributed.mean_losses``).  The loss kernels communicate nothing (SURVEY.md 8e).
"""
from __future__ import annotations

import torch
import torch.distributed as dist
from torch import nn

from . import distributed as D
from .layers import PoseParameters, transformation_from_parameters


def _conv(cin, cout, stride=1):
    return nn.Sequential(nn.Conv2d(cin, cout, 3, stride, 1), nn.ELU(inplace=True))


class _PairEncoder(nn.Module):
    """Five stride-2 stages on the concatenated (target, source) pair: features at 1/2 ... 1/32 resolution."""

    def __init__(self, width=32):
        super().__init__()
        chans = [6, width, width * 2, width * 4, width * 8, width * 8]
        self.stages = nn.ModuleList([nn.Sequential(_conv(chans[k], chans[k + 1], 2), _conv(chans[k + 1], chans[k + 1]))
                                     for k in range(5)])
        self.chans = chans[1:]

    def forward(self, tgt, ref):
        x = torch.cat([tgt, ref], 1)
        feats = []
        for st in self.stages:
            x = st(x)
            feats.append(x)
        return feats


class _PyramidDecoder(nn.Module):
    """U-Net style decoder with heads at the four finest scales (scale s = 1 / 2**s of the input resolution)."""

    def __init__(self, chans, out_ch, extra=0):
        super().__init__()
        dec = [256, 128, 64, 32, 16]
        self.up, self.fuse, self.heads = nn.ModuleList(), nn.ModuleList(), nn.ModuleDict()
        cin = chans[-1] + extra
        for k in range(5):                       # k = 0 works at 1/16 ... k = 4 at full resolution
            self.up.append(_conv(cin, dec[k]))
            skip = chans[3 - k] if k < 4 else 0
            self.fuse.append(_conv(dec[k] + skip, dec[k]))
            cin = dec[k]
            if k >= 1:
                self.heads[str(4 - k)] = nn.Conv2d(dec[k], out_ch, 3, 1, 1)

    def forward(self, feats, extra=None):
        x = feats[-1]
        if extra is not None:
            x = torch.cat([x, extra.expand(-1, -1, x.shape[2], x.shape[3])], 1)
        outs = {}
        for k in range(5):
            x = nn.functional.interpolate(self.up[k](x), scale_factor=2, mode="nearest")
            if k < 4:
                x = torch.cat([x, feats[3 - k]], 1)
            x = self.fuse[k](x)
            if k >= 1:
                outs[4 - k] = self.heads[str(4 - k)](x)
        return outs


class StandInFlowNet(nn.Module):
    """flownet(tgt, ref, frame_id) -> ({("flow", i, s): (B,2,h,w) normalised flow}, encoder features) (trainer.py:267)."""

    def __init__(self, width=32, flow_scale=0.05):
        super().__init__()
        self.encoder = _PairEncoder(width)
        self.decoder = _PyramidDecoder(self.encoder.chans, 2)
        self.flow_scale = flow_scale

    def forward(self, tgt, ref, frame_id=0):
        feats = self.encoder(tgt, ref)
        outs = self.decoder(feats)
        return {("flow", frame_id, s): self.flow_scale * torch.tanh(o) for s, o in outs.items()}, feats


class StandInPoseNet(nn.Module):
    """posenet(tgt, ref) -> (axisangle (B,1,1,3), translation (B,1,1,3)) (trainer.py:268)."""

    def __init__(self, width=16):
        super().__init__()
        self.encoder = _PairEncoder(width)
        self.head = nn.Conv2d(self.encoder.chans[-1], 6, 1)

    def forward(self, tgt, ref):
        out = 0.01 * self.head(self.encoder(tgt, ref)[-1]).mean((2, 3)).view(-1, 1, 1, 6)
        return out[..., :3], out[..., 3:]


class StandInMobileDecoder(nn.Module):
    """mobile_decoder(features, axisangle, translation, frame_id) -> {("mobile", i, s): (B,1,h,w) in (0,1)} (trainer.py:269)."""

    def __init__(self, chans):
        super().__init__()
        self.decoder = _PyramidDecoder(chans, 1, extra=6)

    def forward(self, features, axisangle, translation, frame_id=0):
        pose = torch.cat([axisangle, translation], -1).view(-1, 6, 1, 1)
        return {("mobile", frame_id, s): torch.sigmoid(o) for s, o in self.decoder(features, pose).items()}


class StandInNets(nn.Module):
    def __init__(self, width=32):
        super().__init__()
        self.flownet = StandInFlowNet(width)
        self.posenet = StandInPoseNet(max(8, width // 2))
        self.mobile_decoder = StandInMobileDecoder(self.flownet.encoder.chans)


class TrainStep:
    """One optimisation step of the mobile decoder, as ``run_epoch`` does it.

    loss_module: a callable with ``Loss.forward``'s signature (default: the CUDA ``mdn_sfm_b200.loss_functions.Loss``;
    the CPU tests pass the oracle).  ``fine_tune_flow_motion`` also trains the flow / pose nets (trainer.py:184-186).
    """

    def __init__(self, opt, nets=None, loss_module=None, device="cuda", lr=1e-4, clip_grad=1.0,
                 fine_tune_flow_motion=False, mode="TG", photometric=True, graph_loss=True, pose_params=True):
        """graph_loss: run the CUDA loss path as one CUDA-graph replay per step (graphs.GraphedLoss; in DS / DC mode the
        batches' new Detectron2 instances replay the same graph).  pose_params: hand PoseNet's (axisangle, translation) to
        the loss as parameters so that the fused call also runs transformation_from_parameters and its adjoint
        (layers.PoseParameters).  Both apply to the default CUDA loss only; a caller-supplied `loss_module` gets the
        reference's (B,4,4) matrices, eagerly."""
        self.opt, self.device = opt, torch.device(device)
        self.nets = (nets or StandInNets()).to(self.device)
        self.fine_tune = fine_tune_flow_motion
        self.pose_params = False
        self.eager_loss = None
        if loss_module is None:
            from .loss_functions import Loss
            loss_module = self.eager_loss = Loss(opt, no_ssim=False, mode=mode, photometric=photometric)
            self.pose_params = pose_params
            if graph_loss and self.device.type == "cuda":
                from .graphs import GraphedLoss
                loss_module = GraphedLoss(loss_module)
        self.loss = loss_module
        self.clip_grad = clip_grad
        trainable = [self.nets.mobile_decoder] + ([self.nets.flownet, self.nets.posenet] if fine_tune_flow_motion else [])
        for m in (self.nets.flownet, self.nets.posenet):
            m.requires_grad_(fine_tune_flow_motion)
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.mobile_decoder = self.nets.mobile_decoder
        if self.world > 1:       # trainer.py:181-183: DDP over the trainable net only
            ids = [self.device.index] if self.device.type == "cuda" else None
            self.mobile_decoder = nn.parallel.DistributedDataParallel(self.nets.mobile_decoder, device_ids=ids)
            if fine_tune_flow_motion:
                self.flownet_ddp = nn.parallel.DistributedDataParallel(self.nets.flownet, device_ids=ids)
                self.posenet_ddp = nn.parallel.DistributedDataParallel(self.nets.posenet, device_ids=ids)
        self.parameters_to_train = [p for m in trainable for p in m.parameters()]
        self.optimizer = torch.optim.Adam(self.parameters_to_train, lr, capturable=self.device.type == "cuda")

    def process_batch(self, inputs, instances=None):
        """trainer.py:256-287 -> (flows, mobiles, cam_T_cam, outputs, losses)."""
        o = self.opt
        ids = list(o.frame_ids)[1:]
        tgt = inputs[("color", 0, 0)]
        flows, mobiles, cams = {}, {}, {}
        flownet = getattr(self, "flownet_ddp", self.nets.flownet)
        posenet = getattr(self, "posenet_ddp", self.nets.posenet)
        for i in ids:
            ref = inputs[("color", i, 0)]
            with torch.set_grad_enabled(self.fine_tune):
                flow, feats = flownet(tgt, ref, frame_id=i)
                axisangle, translation = posenet(tgt, ref)
            flows.update(flow)
            mobiles.update(self.mobile_decoder(feats, axisangle, translation, frame_id=i))
            cams[i] = PoseParameters(axisangle, translation) if self.pose_params else transformation_from_parameters(axisangle, translation)
        outputs, losses = self.loss(inputs, ids, flows, mobiles, instances, list(o.scales), cams)
        return flows, mobiles, cams, outputs, losses

    def step(self, inputs, instances=None):
        """process_batch -> zero_grad -> backward -> clip_grad_norm_ -> Adam (trainer.py:231-237).  Returns the losses dict."""
        _, _, _, _, losses = self.process_batch(inputs, instances)
        self.optimizer.zero_grad(set_to_none=True)
        graphed = hasattr(self.loss, "unit_upstream")
        if graphed:
            self.loss.unit_upstream = True       # loss.backward() below: the upstream gradient is 1
        try:
            losses["loss"].backward()
        finally:
            if graphed:
                self.loss.unit_upstream = False
        torch.nn.utils.clip_grad_norm_(self.parameters_to_train, max_norm=self.clip_grad)
        self.optimizer.step()
        return losses

    def log_losses(self, losses):
        """The one small logging collective: mean of the loss scalars over ranks."""
        return D.mean_losses(losses)
