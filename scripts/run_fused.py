"""Runs the fused loss launch a few times on one GPU (for ncu / compute-sanitizer): python scripts/run_fused.py [HxW] [B] [mode] [n]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mdn_sfm_b200 import synthetic
from mdn_sfm_b200.loss_functions import Loss

shape = sys.argv[1] if len(sys.argv) > 1 else "192x640"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 12
mode = sys.argv[3] if len(sys.argv) > 3 else "T"
n = int(sys.argv[4]) if len(sys.argv) > 4 else 6
flow_kind = sys.argv[5] if len(sys.argv) > 5 else "iid"
H, W = map(int, shape.split("x"))
scales = (0, 1, 2, 3) if H % 8 == 0 and W % 8 == 0 else (0,)
opt = synthetic.default_opt(B, H, W)
inputs, flows, mobiles, cams, inst = synthetic.make_batch(B, H, W, scales=scales, seed=42, flow_std=0.05, device="cuda", flow_kind=flow_kind,
                                                          with_instances=mode in ("DS", "DC"))
flows = {k: v.requires_grad_(True) for k, v in flows.items()}
mobiles = {k: v.requires_grad_(True) for k, v in mobiles.items()}
if "--lib" in sys.argv:   # another build of libmdn_loss.so instead of the in-tree library
    from mdn_sfm_b200 import _cabi
    _cabi._lib = _cabi.Library(os.path.abspath(sys.argv[sys.argv.index("--lib") + 1]))
loss = Loss(opt, no_ssim=False, mode=mode, photometric=True)
for i in range(n):
    for d in (flows, mobiles):
        for v in d.values():
            v.grad = None
    _, losses = loss(inputs, [-1, 1], flows, mobiles, inst, list(scales), cams)
    losses["loss"].backward()
torch.cuda.synchronize()
print("ok", float(losses["loss"].detach()))
