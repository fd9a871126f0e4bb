"""Kernel-variant timing: python scripts/kbench.py lib1.so [lib2.so ...] [--shape HxW] [--batch B] [--mode T] [--iters N]

Times Loss.forward (= fundamental prologue + mdn_loss_fused) with CUDA events over 4 rotating input sets for each
library build given on the command line (any builds of libmdn_loss.so, for example of two commits).  Experiment
tooling: bench.py is the number of record.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mdn_sfm_b200 import _cabi, synthetic
from mdn_sfm_b200.loss_functions import Loss


def arg(name, default):
    return sys.argv[sys.argv.index(name) + 1] if name in sys.argv else default


def main():
    libs = [a for a in sys.argv[1:] if a.endswith(".so")]
    H, W = map(int, arg("--shape", "192x640").split("x"))
    B, mode, iters = int(arg("--batch", "12")), arg("--mode", "T"), int(arg("--iters", "200"))
    flow_kind = arg("--flow", "iid")
    scales = (0, 1, 2, 3) if H % 8 == 0 and W % 8 == 0 else (0,)
    opt = synthetic.default_opt(B, H, W)
    sets = []
    for i in range(4):
        inputs, flows, mobiles, cams, inst = synthetic.make_batch(B, H, W, scales=scales, seed=42 + i, flow_std=0.05, device="cuda", flow_kind=flow_kind,
                                                                  with_instances=mode in ("DS", "DC"))
        flows = {k: v.requires_grad_(True) for k, v in flows.items()}
        mobiles = {k: v.requires_grad_(True) for k, v in mobiles.items()}
        sets.append((inputs, flows, mobiles, cams, inst))
    for path in libs:
        _cabi._lib = _cabi.Library(os.path.abspath(path))
        loss = Loss(opt, no_ssim=False, mode=mode, photometric=True)

        bwd = "--bwd" in sys.argv
        reps = int(arg("--reps", "1"))    # rotations of the 4 input sets per graph

        def step(i):
            inputs, flows, mobiles, cams, inst = sets[i % 4]
            if bwd:
                for d in (flows, mobiles):
                    for v in d.values():
                        v.grad = None
            _, losses = loss(inputs, [-1, 1], flows, mobiles, inst, list(scales), cams)
            if bwd:
                losses["loss"].backward()
            return losses["loss"]

        for i in range(20):
            step(i)
        torch.cuda.synchronize()
        # the Python layer adds launch overhead between kernels: time many steps and also report the best single step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(4 * reps):
                step(i)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters // (4 * reps)):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / (iters // (4 * reps) * 4 * reps)
        print(f"{path} [{flow_kind}]: {ms * 1e3:8.1f} us / forward+grads step   loss {float(step(0)):.6f}", flush=True)


if __name__ == "__main__":
    main()
