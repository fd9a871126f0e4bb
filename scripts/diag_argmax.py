"""For fuzz case 3248 (DC, level 1, pair -1, sample 0): the oracle's |e| map on the GPU, its top values, and the oracle / product gradients there."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch, common
from mdn_sfm_b200 import synthetic
from oracle import restate
c = {'kind': 'inst', 'B': 2, 'H': 112, 'W': 160, 'scales': (0, 1), 'mode': 'DC', 'photo': True, 'ssim': False, 'dmin': False, 'dsm': False, 'dcs': True, 'fstd': 0.01, 'pad': 'zeros', 'seed': 360869}
B, H, W, scales, mode = c["B"], c["H"], c["W"], c["scales"], c["mode"]
opt = synthetic.default_opt(B, H, W, disable_min=c["dmin"], disable_smoothloss=c["dsm"], disable_consisloss=c["dcs"], scales=list(scales))
batch = synthetic.make_batch(B, H, W, scales=scales, seed=c["seed"], flow_std=c["fstd"], with_instances=True)
ref = common.oracle_run(opt, batch, mode, True, False, device="cuda", pose_grad=True)
got = common.product_run(opt, batch, mode, True, False, "cuda", pose_grad=True)
inputs, flows, mobiles, cams, inst = batch
s, i = 1, -1
h, w = H // 2, W // 2
dev = "cuda"
pix = restate.create_coords(B, h, w, dev)
f = (restate.get_scale_factor(B, h, w, dev) * flows[("flow", i, s)].to(dev)).contiguous()
ones = torch.ones(B, 1, h, w, device=dev)
p1 = torch.cat([pix, ones], 1).view(B, 3, -1)
p2 = torch.cat([pix + f, ones], 1).view(B, 3, -1)
cam = cams[i].to(dev)
for tag, dt in (("fp32", torch.float32), ("fp64", torch.float64)):
    e = restate.get_epipolar_new(p1.to(dt), p2.to(dt), inputs[("inv_K", s)].to(dev)[:, :3, :3].to(dt), cam[:, :3, :3].to(dt), cam[:, :3, -1].to(dt)).view(B, h * w).abs()
    v, ix = e[0].topk(4)
    print(tag, "top |e| of sample 0:", [(int(k) // w, int(k) % w, float(x)) for x, k in zip(v, ix)])
a, b = ref[2][("flow", i, s)].grad, got[2][("flow", i, s)].grad
d = (a - b).abs()
print("pixels where product != oracle by > 1e-6 abs:", [(tuple(t.tolist()), float(a[tuple(t.tolist())]), float(b[tuple(t.tolist())])) for t in (d > 1e-6).nonzero()[:8]])
print("max |grad| oracle", float(a.abs().max()))
# the L1 kink: tgt - warped at the differing pixel, oracle vs product (standalone warp kernel = the fused kernel's gather)
from mdn_sfm_b200 import loss_utils
tgt = inputs[("color", 0, s)].to(dev)
refimg = inputs[("color", i, s)].to(dev)
fl = flows[("flow", i, s)].to(dev)
pixn = restate.create_coords(B, h, w, dev)
fpx = (restate.get_scale_factor(B, h, w, dev) * fl).contiguous()
wo, vo = restate.inverse_warp(refimg, fpx, pixn)
wg, vg = loss_utils.inverse_warp(refimg, fpx, pixn, "zeros")
y, x = 49, 67
print("tgt - warped at (49,67), oracle :", [float(tgt[0, ch, y, x] - wo[0, ch, y, x]) for ch in range(3)])
print("tgt - warped at (49,67), product:", [float(tgt[0, ch, y, x] - wg[0, ch, y, x]) for ch in range(3)])
print("warped oracle / product:", [(float(wo[0, ch, y, x]), float(wg[0, ch, y, x])) for ch in range(3)], "tgt", [float(tgt[0, ch, y, x]) for ch in range(3)])
