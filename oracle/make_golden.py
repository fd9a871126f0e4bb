"""Writes tests/golden/*.npz from the UPSTREAM REFERENCE itself (build container only) -- TEST INFRASTRUCTURE.

    python -m oracle.make_golden

The reference has no golden vectors (SURVEY.md section 4), so these fixtures are the pin: outputs of the
reference's own `Loss.forward` / `LossModule` (imported in place from /root/reference, with each non-HEAD
mode composed from the reference's own functions by oracle/ref_modes.py) on

  netinit_*   inputs produced by the reference's random-init FlowNet_v1 / PoseNet_v3 / MobileDecoder
              (trainer.py:139-142,152) on synthetic images, B=2, 64x128, 4 scales -- inputs AND outputs stored;
  stress_*    seeded synthetic tensors from mdn_sfm_b200.synthetic (regenerated identically at test time) --
              only the seed and the outputs are stored.

Both the oracle (CPU, not-gpu tests) and the CUDA path (gpu tests) are checked against these files.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mdn_sfm_b200 import synthetic  # noqa: E402
from oracle import ref_loader, ref_modes  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SCALES = [0, 1, 2, 3]
MODES = [("SN", True, True, False), ("T", True, True, False), ("TG", True, True, False), ("DC", False, False, False),
         ("DS", False, False, True)]


def key(k):
    return "_".join(str(x) for x in k).replace("-1", "m1")


def netinit_inputs(B=2, H=64, W=128, seed=42):
    ref = ref_loader.load()
    flow_net, pose_net, mdn = ref_loader.load_networks()
    torch.manual_seed(seed)
    flownet = flow_net.FlowNet_v1(use_elu=True, pretrained=False).eval()
    posenet = pose_net.PoseNet_v3(18, False).eval()
    decoder = mdn.MobileDecoder(use_elu=True)
    decoder.init_weights()
    decoder.eval()
    inputs, _, _, _, inst = synthetic.make_batch(B, H, W, scales=SCALES, seed=seed)
    flows, mobiles, cams = {}, {}, {}
    with torch.no_grad():
        tgt = inputs[("color", 0, 0)]
        for i in (-1, 1):
            refimg = inputs[("color", i, 0)]
            flow, feats = flownet(tgt, refimg, frame_id=i)
            aa, tt = posenet(tgt, refimg)
            mob = decoder(feats, aa, tt, frame_id=i)
            flows.update({k: v.clone() for k, v in flow.items()})
            mobiles.update({k: v.clone() for k, v in mob.items()})
            cams[i] = ref.layers.transformation_from_parameters(aa, tt)
    return inputs, flows, mobiles, cams, inst


def save_split(name, arrays, part, moved_prefixes):
    """Keeps each file under 1 MB: the arrays named with `moved_prefixes` go to `part`.npz (tests/golden_util.PARTS)."""
    moved = {k: v for k, v in arrays.items() if k.startswith(moved_prefixes)}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **{k: v for k, v in arrays.items() if k not in moved})
    np.savez_compressed(os.path.join(OUT, part + ".npz"), **moved)


def run_reference(opt, batch, mode, photo, ssim_on, weights):
    inputs, flows, mobiles, cams, inst = batch
    f = {k: v.clone().requires_grad_(True) for k, v in flows.items()}
    m = {k: v.clone().requires_grad_(True) for k, v in mobiles.items()}
    c = {k: v.clone().requires_grad_(True) for k, v in cams.items()}
    out, losses = ref_modes.reference_loss_forward(opt, inputs, [-1, 1], f, m, inst, SCALES, c, mode=mode, weights=weights,
                                                   photometric=photo, ssim_on=ssim_on)
    losses["loss"].backward()
    rec = {}
    for k in ("loss", "epip", "smooth", "consis") + (("photo",) if photo else ()):
        rec["loss_" + k] = np.float32(float(losses[k].detach()))
    return out, rec, f, m, c


def main():
    assert ref_loader.available(), "needs /root/reference"
    os.makedirs(OUT, exist_ok=True)
    ref = ref_loader.load()

    # ---- netinit: store inputs once, outputs per mode (full gradients: the tensors are small)
    B, H, W = 2, 64, 128
    batch = netinit_inputs(B, H, W)
    inputs, flows, mobiles, cams, inst = batch
    store = {}
    for d, pre in ((inputs, "in"), (flows, "flow"), (mobiles, "mob")):
        for k, v in d.items():
            store["%s_%s" % (pre, key(k))] = v.numpy()
    for i, v in cams.items():
        store["cam_%s" % key((i,))] = v.numpy()
    for b, d in enumerate(inst):
        store["inst_%d" % b] = np.packbits(d["instances"].pred_masks.numpy(), axis=-1)
    save_split("netinit_inputs", store, "netinit_inputs_nets", ("flow_", "mob_", "cam_", "inst_"))
    weights = ref.gauss_distance_weight(4, H, W)
    for mode, photo, ssim_on, dmin in MODES:
        opt = synthetic.default_opt(B, H, W, disable_min=dmin)
        out, rec, f, m, c = run_reference(opt, batch, mode, photo, ssim_on, weights if mode == "TG" else None)
        for k, v in f.items():
            rec["gflow_" + key(k[1:])] = v.grad.numpy()
        for k, v in m.items():
            rec["gmob_" + key(k[1:])] = v.grad.numpy()
        for k, v in c.items():
            rec["gcam_" + key((k,))] = v.grad.numpy()
        for i in (-1, 1):
            rec["epipolars_" + key((i,))] = out["epipolars"][(i, 0)][:, :1].detach().numpy()
            rec["epipolar_ori_" + key((i,))] = out["epipolar_ori"][(i, 0)][:, :1].detach().numpy()
            if photo and mode == "T":   # the warp does not depend on the mode: stored once
                rec["warps_" + key((i,))] = out["warps"][(i, 0)].detach().numpy()
            if photo:
                rec["valids_" + key((i,))] = np.packbits(out["valids"][(i, 0)][:, :1].numpy(), axis=-1)
        if mode == "T":
            save_split("netinit_T", rec, "netinit_T_warps", ("warps_",))
        else:
            np.savez_compressed(os.path.join(OUT, "netinit_%s.npz" % mode), **rec)
        print("netinit", mode, {k: float(v) for k, v in rec.items() if k.startswith("loss_")})

    # ---- stress: BASELINE configs[0] shape (B=4, 192x640); scalars + strided gradient samples
    B, H, W = 4, 192, 640
    weights = ref.gauss_distance_weight(4, H, W)
    for seed, flow_std in ((42, 0.01), (43, 0.05)):
        batch = synthetic.make_batch(B, H, W, scales=SCALES, seed=seed, flow_std=flow_std)
        for mode, photo, ssim_on, dmin in MODES[:4]:
            opt = synthetic.default_opt(B, H, W, disable_min=dmin)
            out, rec, f, m, c = run_reference(opt, batch, mode, photo, ssim_on, weights if mode == "TG" else None)
            rec["seed"], rec["flow_std"] = np.int64(seed), np.float64(flow_std)
            for k, v in f.items():
                g = v.grad.reshape(-1)
                rec["gflow_" + key(k[1:])] = g[::97].numpy()
                rec["gflow_absmax_" + key(k[1:])] = np.float32(g.abs().max())
                rec["gflow_sum_" + key(k[1:])] = np.float64(g.double().sum())
            for k, v in m.items():
                g = v.grad.reshape(-1)
                rec["gmob_" + key(k[1:])] = g[::97].numpy()
                rec["gmob_absmax_" + key(k[1:])] = np.float32(g.abs().max())
                rec["gmob_sum_" + key(k[1:])] = np.float64(g.double().sum())
            for k, v in c.items():
                rec["gcam_" + key((k,))] = v.grad.numpy()
            np.savez_compressed(os.path.join(OUT, "stress_%s_seed%d.npz" % (mode, seed)), **rec)
            print("stress", mode, seed, {k: float(v) for k, v in rec.items() if k.startswith("loss_")})


if __name__ == "__main__":
    main()
