"""Loads tests/golden/*.npz (written by oracle/make_golden.py from the upstream reference itself)."""
import os

import numpy as np
import torch

from mdn_sfm_b200 import synthetic

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SCALES = [0, 1, 2, 3]
NETINIT_MODES = {"SN": (True, True, False), "T": (True, True, False), "TG": (True, True, False),
                 "DC": (False, False, False), "DS": (False, False, True)}
STRESS_MODES = {"SN": (True, True, False), "T": (True, True, False), "TG": (True, True, False), "DC": (False, False, False)}
# fixtures stored in more than one file (each file stays under 1 MB): name -> its further parts
PARTS = {"netinit_inputs": ["netinit_inputs_nets"], "netinit_T": ["netinit_T_warps"]}


class Fixture(dict):
    """The arrays of one fixture, gathered from all its files; `.files` lists the names like np.load's result."""

    @property
    def files(self):
        return list(self)


def key(k):
    return "_".join(str(x) for x in k).replace("-1", "m1")


def load_netinit_batch():
    z = load_outputs("netinit_inputs")
    B, H, W = 2, 64, 128
    inputs, flows, mobiles, cams = {}, {}, {}, {}
    for i in (0, -1, 1):
        for s in SCALES:
            inputs[("color", i, s)] = torch.from_numpy(z["in_" + key(("color", i, s))])
    for s in SCALES:
        inputs[("inv_K", s)] = torch.from_numpy(z["in_" + key(("inv_K", s))])
    for i in (-1, 1):
        for s in SCALES:
            flows[("flow", i, s)] = torch.from_numpy(z["flow_" + key(("flow", i, s))])
            mobiles[("mobile", i, s)] = torch.from_numpy(z["mob_" + key(("mobile", i, s))])
        cams[i] = torch.from_numpy(z["cam_" + key((i,))])
    inst = []
    for b in range(B):
        m = np.unpackbits(z["inst_%d" % b], axis=-1)[..., :synthetic.INSTANCE_HW[1]].astype(bool)
        inst.append({"instances": synthetic.SyntheticInstances(torch.from_numpy(m))})
    return (B, H, W), (inputs, flows, mobiles, cams, inst)


def load_outputs(name):
    z = Fixture()
    for part in [name] + PARTS.get(name, []):
        with np.load(os.path.join(GOLD, part + ".npz")) as f:
            z.update((k, f[k]) for k in f.files)
    return z


def check_against_golden(z, got, photo, fwd_tol, grad_tol, full=True, check_maps=True, map_tol=None):
    """`got` = (outputs, losses, flows, mobiles, cams) as returned by common.product_run / oracle_run."""
    out, losses, f, m, c = got

    def rel(a, b):
        a = torch.as_tensor(np.asarray(a)).double()
        b = b.detach().double().cpu()
        return ((a - b).abs().max() / a.abs().max().clamp_min(1e-30)).item()

    for k in ("loss", "epip", "smooth", "consis") + (("photo",) if photo else ()):
        a, b = float(z["loss_" + k]), float(losses[k])
        assert abs(a - b) <= fwd_tol * max(abs(a), 1e-12), (k, a, b)
    for k, v in f.items():
        g = v.grad if full else v.grad.reshape(-1)[::97]
        scale = 1.0 if full else float(z["gflow_absmax_" + key(k[1:])])
        a = torch.as_tensor(z["gflow_" + key(k[1:])]).double()
        err = (a - g.detach().double().cpu()).abs().max().item() / max(a.abs().max().item() if full else scale, 1e-30)
        assert err <= grad_tol, ("d/dflow", k, err)
    for k, v in m.items():
        g = v.grad if full else v.grad.reshape(-1)[::97]
        a = torch.as_tensor(z["gmob_" + key(k[1:])]).double()
        scale = a.abs().max().item() if full else float(z["gmob_absmax_" + key(k[1:])])
        err = (a - g.detach().double().cpu()).abs().max().item() / max(scale, 1e-30)
        assert err <= grad_tol, ("d/dmobile", k, err)
    for k, v in c.items():
        if v.grad is not None:
            assert rel(z["gcam_" + key((k,))], v.grad) <= grad_tol, ("d/dpose", k, rel(z["gcam_" + key((k,))], v.grad))
    map_tol = fwd_tol if map_tol is None else map_tol
    if check_maps and full:
        fwd_tol = map_tol
        for i in (-1, 1):
            assert rel(z["epipolars_" + key((i,))], out["epipolars"][(i, 0)][:, :1]) <= fwd_tol, ("epipolars", i)
            assert rel(z["epipolar_ori_" + key((i,))], out["epipolar_ori"][(i, 0)][:, :1]) <= fwd_tol, ("epipolar_ori", i)
            if "warps_" + key((i,)) in z.files:
                assert rel(z["warps_" + key((i,))], out["warps"][(i, 0)]) <= fwd_tol, ("warps", i)
            if photo:
                v = out["valids"][(i, 0)][:, :1].cpu().numpy()
                assert np.array_equal(np.packbits(v, axis=-1), z["valids_" + key((i,))]), ("valids", i)


def map_noise_floor(z, ref_run):
    """Largest max-norm deviation of the epipolar maps of `ref_run` (the oracle on some device) from the fixture."""
    out = ref_run[0]
    worst = 0.0
    for i in (-1, 1):
        for name in ("epipolars", "epipolar_ori"):
            a = torch.as_tensor(z[name + "_" + key((i,))]).double()
            b = out[name][(i, 0)][:, :1].detach().double().cpu()
            worst = max(worst, ((a - b).abs().max() / a.abs().max().clamp_min(1e-30)).item())
    return worst
