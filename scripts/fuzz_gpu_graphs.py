"""GPU fuzz of graphs.GraphedLoss: for random shapes / modes, one GraphedLoss object is called with a sequence of batches whose
shapes CHANGE (re-capture) and repeat (replay on new contents); every call must equal the eager Loss bit for bit (loss, every
gradient).  DS / DC cases get a new set of Detectron2 instances every call, 0-6 per sample (now and then one bare Instances
for the whole batch), replayed from the same capture.  python scripts/fuzz_gpu_graphs.py [N] [seed0]"""
import os
import random
import sys
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch

from mdn_sfm_b200 import synthetic
from mdn_sfm_b200.graphs import GraphedLoss
from mdn_sfm_b200.loss_functions import Loss

DEV = "cuda"


def instances(rng, B, gen):
    """0-6 Detectron2-style masks per sample at the size the reference feeds Detectron2; one time in five a bare Instances."""
    H, W = synthetic.INSTANCE_HW
    bare, out = rng.random() < 0.2, []
    for _ in range(1 if bare else B):
        n = rng.randint(0, 6)
        m = torch.rand(n, H, W, generator=gen) > rng.choice([0.9, 0.99])
        for k in range(n):
            y0, x0 = rng.randrange(H - 60), rng.randrange(W - 200)
            m[k, y0:y0 + rng.randint(20, 60), x0:x0 + rng.randint(40, 200)] = True
        out.append({"instances": synthetic.SyntheticInstances(m.to(DEV))})
    return out[0]["instances"] if bare else out


def run(loss, batch, scales, inst=None):
    inputs, flows, mobiles, cams, _ = batch
    f = {k: v.clone().requires_grad_(True) for k, v in flows.items()}
    m = {k: v.clone().requires_grad_(True) for k, v in mobiles.items()}
    c = {k: v.clone().requires_grad_(True) for k, v in cams.items()}
    _, losses = loss(inputs, [-1, 1], f, m, inst, list(scales), c)
    losses["loss"].backward()
    return losses, f, m, c


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    rng = random.Random(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    fails = 0
    for it in range(n):
        # two GraphedLoss objects of different shapes / modes alive at once, called alternately with fresh contents: every call
        # (the captures, then replays) must equal the eager Loss bit for bit -- the graphs share the process-wide workspace cache
        objs = []
        for _ in range(2):
            B, H, W = rng.randint(1, 3), 8 * rng.randint(2, 14), 8 * rng.randint(4, 34)
            scales = (0, 1, 2, 3)[:rng.randint(1, 3)]
            mode, photo = rng.choice(["SN", "T", "TG", "DS", "DC"]), rng.random() < 0.8
            opt = synthetic.default_opt(B, H, W, scales=list(scales), threshold=0.8625 if mode == "TG" else 9.22)
            objs.append(dict(B=B, H=H, W=W, scales=scales, mode=mode, photo=photo, opt=opt,
                             eager=Loss(opt, no_ssim=False, mode=mode, photometric=photo),
                             graphed=GraphedLoss(Loss(opt, no_ssim=False, mode=mode, photometric=photo))))
        case = [{k: o[k] for k in ("B", "H", "W", "scales", "mode", "photo")} for o in objs]
        try:
            for k in range(7):
                o = objs[(k * 3 // 2) % 2] if k else objs[1]       # 1 0 1 0 1 1 0 ...: the larger may come first or second
                batch = synthetic.make_batch(o["B"], o["H"], o["W"], scales=o["scales"], seed=rng.randint(0, 10 ** 6),
                                             flow_std=rng.choice([0.02, 0.1]), with_instances=False, device=DEV)
                inst = instances(rng, o["B"], torch.Generator().manual_seed(rng.randint(0, 10 ** 6))) if o["mode"] in ("DS", "DC") else None
                le, fe, me, ce = run(o["eager"], batch, o["scales"], inst)
                lg, fg, mg, cg = run(o["graphed"], batch, o["scales"], inst)
                assert torch.equal(le["loss"].detach(), lg["loss"].detach()), ("loss", k, float(le["loss"]), float(lg["loss"]))
                for da, db, what in ((fe, fg, "d/dflow"), (me, mg, "d/dmobile"), (ce, cg, "d/dpose")):
                    for key in da:
                        assert torch.equal(da[key].grad, db[key].grad), (what, key, k)
        except AssertionError as e:
            fails += 1
            print("FAIL", it, case, "->", str(e)[:300], flush=True)
        except Exception as e:
            fails += 1
            print("ERROR", it, case, "->", type(e).__name__, str(e)[:300], flush=True)
            traceback.print_exc(limit=5)
    print("fuzz (graphs): %d pairs of graphed losses x 7 interleaved calls, %d failures" % (n, fails))
    sys.exit(1 if fails else 0)


if __name__ == "__main__":
    main()
