"""GPU fuzz campaign: random shapes / modes / switches, the CUDA path through the C ABI against the oracle run eagerly on the same
GPU (tests/common.compare: forward 1e-5, gradients 1e-4, masks bit-exact).  python scripts/fuzz_gpu.py [N] [seed0]
Prints one line per failing case (the case is reproducible from its line) and a summary; exit code 1 if anything failed."""
import os
import random
import sys
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch

import common
from mdn_sfm_b200 import synthetic


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    seed0 = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    rng = random.Random(seed0)
    fails = 0
    for it in range(n):
        kind = rng.choice(["tiny", "tiny", "mid", "pyr", "inst"])
        if kind == "tiny":
            B, H, W, scales = rng.randint(1, 3), rng.randint(3, 40), rng.randint(3, 150), (0,)
        elif kind == "mid":
            B, H, W, scales = rng.randint(1, 2), rng.randint(17, 200), rng.randint(60, 400), (0,)
        elif kind == "pyr":
            B, H, W = rng.randint(1, 2), 8 * rng.randint(3, 20), 8 * rng.randint(8, 40)
            scales = (0, 1, 2, 3)[:rng.randint(2, 4)]
        else:
            B, H, W = rng.randint(1, 2), 8 * rng.randint(4, 16), 8 * rng.randint(8, 30)
            scales = (0, 1)
        mode = rng.choice(["DS", "DC"]) if kind == "inst" else rng.choice(["SN", "T", "TG"])
        if mode == "TG" and (H < 8 * 2 ** (len(scales) - 1) or W < 8 * 2 ** (len(scales) - 1)):
            mode = "T"
        photo, ssim = rng.random() < 0.8, rng.random() < 0.7
        dmin, dsm, dcs = rng.random() < 0.3, rng.random() < 0.2, rng.random() < 0.2
        fstd = rng.choice([0.01, 0.05, 0.2, 0.6])
        pad = rng.choice(["zeros", "zeros", "zeros", "border", "reflection"])
        seed = rng.randint(0, 10 ** 6)
        case = dict(kind=kind, B=B, H=H, W=W, scales=scales, mode=mode, photo=photo, ssim=ssim, dmin=dmin, dsm=dsm, dcs=dcs, fstd=fstd,
                    pad=pad, seed=seed)
        try:
            opt = synthetic.default_opt(B, H, W, disable_min=dmin, disable_smoothloss=dsm, disable_consisloss=dcs, scales=list(scales))
            batch = synthetic.make_batch(B, H, W, scales=scales, seed=seed, flow_std=fstd, with_instances=kind == "inst")
            if kind != "inst":
                batch = batch[:4] + (None,)
            ref = common.oracle_run(opt, batch, mode, photo, ssim, device="cuda", pose_grad=True, padding_mode=pad)
            got = common.product_run(opt, batch, mode, photo, ssim, "cuda", pose_grad=True, padding_mode=pad)
            # B = 1: the reference's own CUDA result depends on the batch size there (torch.matmul runs gemm for one batch, bgemm for
            # more; scripts/diag_batch1.py: its distance maps differ by 2e-5 ... 5e-5 between B = 1 and the same sample in a batch
            # of two).  The product follows the B >= 2 rounding at every batch size, so B = 1 is compared at that noise floor.
            if B == 1:
                common.compare(ref, got, photo, fwd_tol=2e-4, grad_tol=4e-4)
            else:
                common.compare(ref, got, photo)
        except AssertionError as e:
            fails += 1
            print("FAIL", it, case, "->", str(e)[:300], flush=True)
        except Exception as e:
            fails += 1
            print("ERROR", it, case, "->", type(e).__name__, str(e)[:300], flush=True)
            traceback.print_exc(limit=3)
        if (it + 1) % 50 == 0:
            print("...", it + 1, "cases,", fails, "failures", flush=True)
    print("fuzz: %d cases, %d failures" % (n, fails))
    sys.exit(1 if fails else 0)


if __name__ == "__main__":
    main()
