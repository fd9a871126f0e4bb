"""Times the DS / DC loss step with a new set of Detectron2 instances every batch, one GPU, one process.

    python scripts/time_graphed_instances.py [--steps 200] [--train-steps 30] [--out FILE]

1. The two union kernels on the same 12 x 375 x 1242 masks, alternating blocks of launches (CUDA events):
   mdn_instance_mask_union (pointer table in the kernel parameters) and mdn_instance_mask_union_table (table in device memory).
2. The DC loss step at BASELINE configs[3] (B = 12, 192 x 640, 4 scales, photometric term on), forward + backward over
   `--steps` steps rotating 4 instance sets with different counts: the eager Loss against GraphedLoss.  GPU time per step
   (events around the loop) and host time per step (host clock around the enqueue of the loop, no synchronise inside),
   and a bit-for-bit check of both paths on every set.
3. TrainStep in DC (HEAD: no photometric term) with graph_loss on and off, frames/s.

Prints one JSON line, with the card's name and power limit read through NVML in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

DEV = "cuda"


def card():
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        name = pynvml.nvmlDeviceGetName(h)
        return {"name": name.decode() if isinstance(name, bytes) else name,
                "power_limit_w": pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0,
                "sm_max_mhz": pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)}
    except Exception as e:          # (NVML missing: the numbers still print, the card is named by torch)
        return {"name": torch.cuda.get_device_name(), "power_limit_w": None, "nvml_error": str(e)}


def instance_sets(B, counts_per_set, seed=0):
    from mdn_sfm_b200 import synthetic
    H, W = synthetic.INSTANCE_HW
    g = torch.Generator().manual_seed(seed)
    sets = []
    for counts in counts_per_set:
        out = []
        for n in counts:
            m = torch.rand(n, H, W, generator=g) > 0.95
            for k in range(n):
                y0, x0 = int(torch.randint(0, H - 80, (1,), generator=g)), int(torch.randint(0, W - 250, (1,), generator=g))
                m[k, y0:y0 + 80, x0:x0 + 250] = True
            out.append({"instances": synthetic.SyntheticInstances(m.to(DEV))})
        sets.append(out)
    return sets


def time_unions(lib, blocks=10, per_block=200):
    """Median and spread of µs per launch over alternating blocks of launches of the two union entry points."""
    from mdn_sfm_b200 import _cabi, loss_utils
    B, (H, W) = 12, (375, 1242)
    inst = instance_sets(B, [[3] * B], seed=1)[0]
    masks = [d["instances"].pred_masks.view(torch.uint8) for d in inst]
    table = loss_utils.InstanceMaskTable(B, H, W, DEV).load(inst)
    out_old = torch.empty(B, H, W, dtype=torch.uint8, device=DEV)
    out_new = torch.empty_like(out_old)
    stream = _cabi.stream_ptr(out_old)
    ptrs, counts = _cabi.ptr_array(masks), (C.c_int32 * B)(*[m.shape[0] for m in masks])
    old = lambda: lib.call("mdn_instance_mask_union", ptrs, counts, out_old.data_ptr(), B, H * W, stream, dev=out_old)
    new = lambda: lib.call("mdn_instance_mask_union_table", table.ptrs.data_ptr(), table.counts.data_ptr(), out_new.data_ptr(), B,
                           H * W, stream, dev=out_new)
    for fn in (old, new):
        for _ in range(20):
            fn()
    torch.cuda.synchronize()
    res = {"old": [], "new": []}
    for blk in range(blocks):
        for name, fn in (("old", old), ("new", new)) if blk % 2 == 0 else (("new", new), ("old", old)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_block):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[name].append(1000.0 * e0.elapsed_time(e1) / per_block)
    same = torch.equal(out_old, out_new)
    summ = lambda v: {"median_us": round(statistics.median(v), 3), "min_us": round(min(v), 3), "max_us": round(max(v), 3)}
    return {"masks": "12 x 3 x 375 x 1242 bool", "launches_per_block": per_block, "blocks_each": blocks,
            "mdn_instance_mask_union": summ(res["old"]), "mdn_instance_mask_union_table": summ(res["new"]),
            "outputs_equal": same}


def time_loss_step(steps, B=12, H=192, W=640, scales=(0, 1, 2, 3)):
    from mdn_sfm_b200 import synthetic
    from mdn_sfm_b200.graphs import GraphedLoss
    from mdn_sfm_b200.layers import PoseParameters
    from mdn_sfm_b200.loss_functions import Loss
    opt = synthetic.default_opt(B, H, W)
    eager = Loss(opt, no_ssim=False, mode="DC", photometric=True)
    graphed = GraphedLoss(Loss(opt, no_ssim=False, mode="DC", photometric=True))
    counts = [[(b + s) % 4 for b in range(B)] for s in range(4)]          # 0-3 instances, another pattern per set
    insts = instance_sets(B, counts, seed=2)
    sets = []
    for s in range(4):
        inputs, flows, mobiles, _, _ = synthetic.make_batch(B, H, W, scales=scales, seed=42 + 1000 * s, flow_std=0.05,
                                                            with_instances=False, device=DEV)
        g = torch.Generator().manual_seed(s)
        leaf = lambda t: t.to(DEV).requires_grad_(True)
        cams = {i: PoseParameters(leaf(0.02 * torch.randn(B, 1, 1, 3, generator=g)), leaf(0.3 * torch.randn(B, 1, 1, 3, generator=g)))
                for i in (-1, 1)}
        sets.append((inputs, {k: v.requires_grad_(True) for k, v in flows.items()},
                     {k: v.requires_grad_(True) for k, v in mobiles.items()}, cams, insts[s]))

    def leaves(s):
        return list(s[1].values()) + list(s[2].values()) + [t for c in s[3].values() for t in (c.axisangle, c.translation)]

    def step(loss, s):
        for t in leaves(s):
            t.grad = None
        _, losses = loss(s[0], [-1, 1], s[1], s[2], s[4], list(scales), s[3])
        losses["loss"].backward()
        return losses

    agree = True
    for s in sets:                     # outputs of both paths on every set: total, terms, every gradient
        le = step(eager, s)
        ge = [t.grad.clone() for t in leaves(s)]
        lg = step(graphed, s)
        gg = [t.grad for t in leaves(s)]
        agree &= all(torch.equal(torch.as_tensor(le[k]), torch.as_tensor(lg[k])) for k in ("loss", "epip", "smooth", "consis", "photo"))
        agree &= all(torch.equal(a, b) for a, b in zip(ge, gg))
    capture = graphed.step
    out = {"config": "DC, B=%d, %dx%d, scales %s, photometric, %d steps over 4 instance sets (counts 0-3 per sample)" % (
        B, H, W, list(scales), steps), "outputs_equal": bool(agree)}
    for name, loss in (("eager", eager), ("graphed", graphed), ("eager_again", eager), ("graphed_again", graphed)):
        for k in range(8):
            step(loss, sets[k % 4])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for k in range(steps):
            step(loss, sets[k % 4])
        t1 = time.perf_counter()
        e1.record()
        torch.cuda.synchronize()
        out[name] = {"gpu_us_per_step": round(1000.0 * e0.elapsed_time(e1) / steps, 2),
                     "host_us_per_step": round(1e6 * (t1 - t0) / steps, 2)}
    out["one_capture"] = graphed.step is capture
    return out


def time_train_step(n, B=12, H=192, W=640):
    from mdn_sfm_b200 import synthetic
    from mdn_sfm_b200.train_step import TrainStep
    opt = synthetic.default_opt(B, H, W)
    inputs = [synthetic.make_batch(B, H, W, seed=s, with_instances=False, device=DEV)[0] for s in (1, 2)]
    insts = instance_sets(B, [[(b + s) % 4 for b in range(B)] for s in range(4)], seed=3)
    out = {"config": "TrainStep DC (no photometric term), B=%d, %dx%d, 4 scales, stand-in nets, %d steps x 3 chunks" % (B, H, W, n)}
    for graph in (False, True, False, True):
        torch.manual_seed(0)
        ts = TrainStep(opt, device=DEV, mode="DC", photometric=False, graph_loss=graph)
        for k in range(5):
            ts.step(inputs[k % 2], insts[k % 4])
        torch.cuda.synchronize()
        chunks = []
        for c in range(3):
            t0 = time.perf_counter()
            for k in range(n):
                ts.step(inputs[k % 2], insts[k % 4])
            torch.cuda.synchronize()
            chunks.append(B * n / (time.perf_counter() - t0))
        key = "graph_loss_%s" % ("on" if graph else "off")
        out.setdefault(key, []).append(round(statistics.median(chunks), 1))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--train-steps", type=int, default=30)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_graphed_instances.py needs a CUDA device")
    from mdn_sfm_b200 import _cabi
    res = {"card": card(), "torch": torch.__version__}
    res["union_kernels"] = time_unions(_cabi.lib())
    res["dc_loss_step"] = time_loss_step(args.steps)
    res["train_step_frames_per_s"] = time_train_step(args.train_steps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
