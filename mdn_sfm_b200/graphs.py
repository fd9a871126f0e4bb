"""CUDA-graph capture of the loss step (SURVEY.md 8f-N1: "with CUDA-graph capture of the loss").

``Loss.forward`` + ``loss.backward()`` is four launches of ours plus autograd's bookkeeping; replayed from a graph the
step costs its kernels and nothing else (bench.py measures exactly this).  ``GraphedLossStep`` captures it once on a set
of STATIC tensors -- the caller refreshes them in place (``tensor.copy_(...)``, or lets the producing nets write into them)
and calls ``replay()``; the loss scalars and the ``.grad`` of the leaf tensors are refreshed by the replay.
"""
from __future__ import annotations

import torch


class GraphedLossStep:
    """Captures ``losses = loss(inputs, frame_ids, flows, mobiles, instances, scales, cams)[1]; losses["loss"].backward()``.

    flows / mobiles / cams whose tensors require grad must be LEAF tensors; after ``replay()`` their ``.grad`` holds the
    gradient of the step (the same graph-owned buffers every time).  ``instances`` (DS / DC) are prepared inside the
    capture: pass a ``loss_utils.InstanceMaskTable`` and ``load`` each batch into it before ``replay()`` (the union kernel
    reads the table when it runs); a list / bare ``Instances`` is replayed with the masks it was captured with."""

    def __init__(self, loss, inputs, frame_ids, flows, mobiles, instances, scales, cams, warmup=3):
        self.loss_module = loss
        self.args = (inputs, list(frame_ids), flows, mobiles, instances, list(scales), cams)
        self.leaves = [t for d in (flows, mobiles) for t in d.values() if t.requires_grad]
        for c in cams.values():      # (B,4,4) matrices, or layers.PoseParameters (axisangle, translation)
            self.leaves += [t for t in ((c.axisangle, c.translation) if hasattr(c, "axisangle") else (c,)) if t.requires_grad]
        for t in self.leaves:
            if not t.is_leaf:
                raise ValueError("tensors that require grad must be leaves of the captured step")
        dev = next(iter(flows.values())).device
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):      # warm-up outside the capture: lazy kernel attributes, allocator pools
            for _ in range(max(1, warmup)):
                self._step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.losses = self._step()
        self.loss = self.losses["loss"]

    def _step(self):
        for t in self.leaves:
            t.grad = None
        with torch.enable_grad():
            self.outputs, losses = self.loss_module(*self.args)
            if losses["loss"].requires_grad:       # (a forward-only capture when nothing is differentiable)
                losses["loss"].backward()
        return {k: (v.detach() if torch.is_tensor(v) else v) for k, v in losses.items()}

    def replay(self):
        """Re-runs the captured step on the current contents of the static tensors; returns the (static) losses dict."""
        self.graph.replay()
        return self.losses


class _ReplayFn(torch.autograd.Function):
    """forward = copy the step's tensors into the static ones + ONE graph replay (which also produced every gradient);
    backward = hand those gradients on (times the upstream gradient unless the caller declared it to be 1)."""

    @staticmethod
    def forward(ctx, owner, *tensors):
        owner._refresh(tensors)
        owner.step.graph.replay()
        ctx.owner = owner
        ctx.leaf = [t.is_leaf for t in tensors]
        return owner.step.loss.clone()

    @staticmethod
    def backward(ctx, g):
        o = ctx.owner
        out = []
        for s, leaf in zip(o.static_diff, ctx.leaf):
            gr = s.grad
            if not o.unit_upstream:
                gr = gr * g
            elif leaf:
                gr = gr.clone()      # AccumulateGrad would adopt the graph-owned buffer as .grad
            out.append(gr)
        return (None,) + tuple(out)


class GraphedLoss:
    """``Loss`` for an EAGER training step whose loss path runs as one CUDA-graph replay (SURVEY.md 8f-N1; trainer.py:280-281).

    Same call signature and return value as ``Loss.forward``.  The first call (and any call with new shapes / keys)
    captures ``Loss.forward + backward`` on static copies of its arguments (GraphedLossStep); every call copies the
    differentiable arguments -- the nets' fresh output tensors -- into the static ones, replays, and returns a loss whose
    autograd node passes the replay's gradients on to the nets.  The (non-differentiable) ``inputs`` are copied only when
    they are not the static tensors themselves: a loader that writes each batch into ``static_inputs`` pays no copy.
    ``unit_upstream`` (set by TrainStep around ``loss.backward()``): the upstream gradient is known to be 1, skip the rescale.
    Detectron2 instances (DS / DC), as a list of ``{"instances": obj}`` or one bare ``Instances``, may hold a different
    number of masks every batch: each call loads their pointers and counts into a device table
    (``loss_utils.InstanceMaskTable``) that the captured union kernel reads at replay.  Their form, the batch size and the
    mask size are part of the capture key; a new mask size captures again."""

    def __init__(self, loss):
        self.loss_module = loss
        self.step = None
        self.key = None
        self.unit_upstream = False

    @staticmethod
    def _pose_tensors(c):
        return (c.axisangle, c.translation) if hasattr(c, "axisangle") else (c,)

    @staticmethod
    def _instance_form(instances, batch):
        """(form, B, H, W, device) of the Detectron2 masks of a batch: everything a capture depends on but the counts."""
        if instances is None:
            return None
        from .loss_utils import _pred_masks
        m = _pred_masks(instances)[0]
        return ("list" if isinstance(instances, list) else "bare", batch, int(m.shape[-2]), int(m.shape[-1]), m.device)

    def _signature(self, inputs, frame_ids, flows, mobiles, scales, cams, inst_form):
        sig = [tuple(frame_ids), tuple(scales), inst_form]
        for d in (inputs, flows, mobiles):
            sig.append(tuple((k, tuple(v.shape), v.requires_grad) for k, v in d.items()))
        sig.append(tuple((k, type(c).__name__, tuple(tuple(t.shape) + (t.requires_grad,) for t in self._pose_tensors(c))) for k, c in cams.items()))
        return tuple(sig)

    def _capture(self, inputs, frame_ids, flows, mobiles, instances, inst_form, scales, cams):
        from .layers import PoseParameters
        from .loss_utils import InstanceMaskTable
        own = lambda t: t.detach().clone().requires_grad_(t.requires_grad)
        self.static_inputs = {k: v.detach().clone() for k, v in inputs.items()}
        s_flows = {k: own(v) for k, v in flows.items()}
        s_mobiles = {k: own(v) for k, v in mobiles.items()}
        s_cams = {k: (PoseParameters(own(c.axisangle), own(c.translation)) if hasattr(c, "axisangle") else own(c)) for k, c in cams.items()}
        self.static_args = (s_flows, s_mobiles, s_cams)
        self.static_diff = [t for t in self._diff_list(s_flows, s_mobiles, s_cams)]
        self.table = None
        if inst_form is not None:      # the capture's warm-up steps already read the first batch's masks
            _, B, H, W, dev = inst_form
            self.table = InstanceMaskTable(B, H, W, dev).load(instances)
        self.step = GraphedLossStep(self.loss_module, self.static_inputs, frame_ids, s_flows, s_mobiles, self.table, scales, s_cams)

    def _diff_list(self, flows, mobiles, cams):
        out = [t for d in (flows, mobiles) for t in d.values() if t.requires_grad]
        for c in cams.values():
            out += [t for t in self._pose_tensors(c) if t.requires_grad]
        return out

    def _refresh(self, tensors):
        with torch.no_grad():
            torch._foreach_copy_([s for s in self.static_diff], [t.detach() for t in tensors])

    def __call__(self, inputs, frame_ids, flows, mobiles, instances, scales, cams):
        inst_form = self._instance_form(instances, next(iter(flows.values())).shape[0])
        key = self._signature(inputs, frame_ids, flows, mobiles, scales, cams, inst_form)
        if self.step is None or key != self.key:
            self._capture(inputs, list(frame_ids), flows, mobiles, instances, inst_form, list(scales), cams)
            self.key = key
        elif instances is not None:
            self.table.load(instances)      # this batch's masks: written ahead of the replay in stream order
        with torch.no_grad():      # the batch itself: copied only when the caller did not write it into static_inputs
            src = [(self.static_inputs[k], v) for k, v in inputs.items() if v.data_ptr() != self.static_inputs[k].data_ptr()]
            if src:
                torch._foreach_copy_([a for a, _ in src], [b for _, b in src])
            # non-differentiable flows / maps / poses (frozen nets under no_grad)
            s_flows, s_mobiles, s_cams = self.static_args
            fixed = [(s_flows[k], v) for k, v in flows.items() if not v.requires_grad] + [(s_mobiles[k], v) for k, v in mobiles.items() if not v.requires_grad]
            for k, c in cams.items():
                fixed += [(a, b) for a, b in zip(self._pose_tensors(s_cams[k]), self._pose_tensors(c)) if not b.requires_grad]
            if fixed:
                torch._foreach_copy_([a for a, _ in fixed], [b for _, b in fixed])
        diff = self._diff_list(flows, mobiles, cams)
        if diff and torch.is_grad_enabled():
            total = _ReplayFn.apply(self, *diff)
        else:
            self._refresh(diff)
            self.step.graph.replay()
            total = self.step.loss.clone()
        losses = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in self.step.losses.items()}
        losses["loss"] = total
        return self.step.outputs, losses
