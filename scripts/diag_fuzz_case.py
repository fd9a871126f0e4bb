"""Re-runs one case printed by scripts/fuzz_gpu.py and shows WHERE the product and the oracle differ: python scripts/diag_fuzz_case.py "<case dict>" """
import ast
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch

import common
from mdn_sfm_b200 import synthetic

c = ast.literal_eval(sys.argv[1])
B, H, W, scales, mode = c["B"], c["H"], c["W"], c["scales"], c["mode"]
opt = synthetic.default_opt(B, H, W, disable_min=c["dmin"], disable_smoothloss=c["dsm"], disable_consisloss=c["dcs"], scales=list(scales))
batch = synthetic.make_batch(B, H, W, scales=scales, seed=c["seed"], flow_std=c["fstd"], with_instances=c["kind"] == "inst")
if c["kind"] != "inst":
    batch = batch[:4] + (None,)
ref = common.oracle_run(opt, batch, mode, c["photo"], c["ssim"], device="cuda", pose_grad=True, padding_mode=c["pad"])
got = common.product_run(opt, batch, mode, c["photo"], c["ssim"], "cuda", pose_grad=True, padding_mode=c["pad"])
# float64 oracle for the pose gradients (the reference's own fp32 noise floor)
torch.set_default_dtype(torch.float64)
b64 = tuple(({k: v.double() for k, v in d.items()} if isinstance(d, dict) else d) for d in batch)
try:
    ref64 = common.oracle_run(opt, b64, mode, c["photo"], c["ssim"], device="cuda", pose_grad=True, padding_mode=c["pad"], rule_ties=False)
except Exception as e:
    ref64 = None
    print("float64 oracle failed:", type(e).__name__, str(e)[:200])
torch.set_default_dtype(torch.float32)
for name, i in (("flows", 2), ("mobiles", 3), ("poses", 4)):
    for k in ref[i]:
        a, b = ref[i][k].grad, got[i][k].grad
        if a is None:
            continue
        d = (a - b).abs()
        scale = float(a.abs().max())
        big = d > 1e-4 * scale
        line = "%-8s %-16s rel max %.3g  pixels beyond 1e-4: %d of %d" % (name, str(k), float(d.max()) / scale, int(big.sum()), d.numel())
        if ref64 is not None:
            a64 = ref64[i][k].grad
            s64 = float(a64.abs().max())
            line += "   | vs float64 oracle: reference fp32 %.3g, product %.3g" % (float((a.double() - a64).abs().max()) / s64, float((b.double() - a64).abs().max()) / s64)
        print(line)
        if 0 < int(big.sum()) <= 6:
            for idx in big.nonzero()[:6]:
                idx = tuple(idx.tolist())
                print("      at", idx, "oracle", float(a[idx]), "product", float(b[idx]))
