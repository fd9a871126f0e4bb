"""Pins oracle/restate.py bit for bit against the upstream MDN_SfM reference.

Every array these tests compare is stored in tests/golden/oracle_pins_grads.npz and oracle_pins_maps.npz (each distinct
array once, with an index from `<case>/<name>` to it), and restate's results must equal the stored arrays bit for bit,
so the pin holds in any checkout.  Where the reference tree is present (MDN_REFERENCE_ROOT, see oracle/ref_loader.py)
each test also runs the reference itself and requires the same bits from it, which re-checks the stored arrays too.

    python tests/test_oracle_vs_reference.py --write                 records the arrays from the reference tree
    python tests/test_oracle_vs_reference.py --write --from-oracle   records them from oracle/restate.py

The stored files name their source (`source`).  They were recorded from oracle/restate.py with no reference tree at
hand, at a commit where restate.py was unchanged since it was pinned bit-exactly against the reference by this module's
live comparisons.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__":
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import pytest  # noqa: E402
import torch  # noqa: E402

from mdn_sfm_b200 import synthetic  # noqa: E402
from oracle import ref_loader, ref_modes, restate  # noqa: E402

B, H, W = 2, 32, 64
GOLD = os.path.join(ROOT, "tests", "golden")
PIN_FILES = {"grads": "oracle_pins_grads.npz", "maps": "oracle_pins_maps.npz"}
CASES = [("DC", False, False, False), ("SN", True, True, False), ("T", True, True, False), ("TG", True, False, True),
         ("DS", False, False, False), ("DC", True, True, True)]


def case_id(mode, photo, ssim_on, disable_min):
    return "%s-photo%d-ssim%d-dmin%d" % (mode, photo, ssim_on, disable_min)


def _leafify(flows, mobiles):
    flows = {k: v.clone().requires_grad_(True) for k, v in flows.items()}
    mobiles = {k: v.clone().requires_grad_(True) for k, v in mobiles.items()}
    return flows, mobiles


def _numpy(d):
    return {k: v.detach().numpy() for k, v in d.items()}


def loss_arrays(forward, mode, photo, ssim_on, disable_min):
    """forward = restate.loss_forward or ref_modes.reference_loss_forward -> {name: array} of every compared output."""
    opt = synthetic.default_opt(B, H, W, disable_min=disable_min)
    inputs, flows, mobiles, cams, inst = synthetic.make_batch(B, H, W, seed=7, flow_std=0.05)
    weights = restate.gauss_distance_weight(4, H, W) if mode == "TG" else None
    f, m = _leafify(flows, mobiles)
    o, losses = forward(opt, inputs, [-1, 1], f, m, inst, [0, 1, 2, 3], cams, mode=mode, weights=weights,
                        photometric=photo, ssim_on=ssim_on)
    out = {"loss_" + k: losses[k] for k in ("loss", "epip", "smooth", "consis")}
    losses["loss"].backward()
    for d in (f, m):
        for (kind, i, s), v in d.items():
            out["grad_%s_%d_%d" % (kind, i, s)] = v.grad
    for name in ("epipolars", "epipolar_ori", "flows") + (("warps", "diffs", "valids") if photo else ()):
        for (i, s) in o[name]:
            out["%s_%d_%d" % (name, i, s)] = o[name][(i, s)]
    for s in o["min_mobiles"]:
        out["min_mobiles_%d" % s] = o["min_mobiles"][s]
    return _numpy(out)


def free_function_arrays(tfp, scale_factor, coords, ssim, binary_image, flow_warp, gauss_weight, smooth, consistency):
    g = torch.Generator().manual_seed(3)
    aa = torch.randn(3, 1, 1, 3, generator=g) * 0.3
    tt = torch.randn(3, 1, 1, 3, generator=g)
    out = {"transformation_inv%d" % inv: tfp(aa, tt, inv) for inv in (False, True)}
    out["scale_factor"] = scale_factor(2, 5, 7).contiguous()
    out["coords"] = coords(2, 5, 7)
    x = torch.rand(2, 3, 9, 11, generator=g)
    y = torch.rand(2, 3, 9, 11, generator=g)
    out["ssim"] = ssim(x, y)
    out["binary_image"] = binary_image(x, 0.4)
    fl = torch.randn(2, 2, 9, 11, generator=g) * 3
    for k, t in enumerate(flow_warp(fl)):
        out["flow_warp_%d" % k] = t
    for k, t in enumerate(gauss_weight(3, 32, 64)):
        out["gauss_distance_weight_%d" % k] = t
    m = torch.rand(2, 1, 9, 11, generator=g)
    out["smooth_loss"] = smooth(x, m)
    out["consistency_loss"] = consistency(m, 1 - m)
    return _numpy(out)


def oracle_free_functions():
    return free_function_arrays(restate.transformation_from_parameters, restate.get_scale_factor, restate.create_coords,
                                restate.ssim, restate.binary_image, restate.flow_warp_grid, restate.gauss_distance_weight,
                                restate.smooth_loss, restate.derivable_consistency_loss)


def reference_free_functions():
    ref = ref_loader.load()
    return free_function_arrays(ref.layers.transformation_from_parameters, ref.layers.get_scale_factor,
                                ref.loss_utils.create_coords, lambda x, y: ref.layers.SSIM()(x, y), ref.binary_image,
                                lambda fl: ref.FlowWarp(2, 9, 11)(fl), ref.gauss_distance_weight, ref.loss_utils.smooth_loss,
                                ref.loss_utils.derivable_consistency_loss)


def instance_mask_arrays(get_batch_instance_mask):
    inst = synthetic.make_instances(1, torch.Generator().manual_seed(5))[0]["instances"]
    return _numpy({"batch_instance_mask": get_batch_instance_mask(inst)})


def all_arrays(from_reference):
    """{`<case>/<name>`: array} of everything the tests compare, from the reference or from restate."""
    forward = ref_modes.reference_loss_forward if from_reference else restate.loss_forward
    groups = {case_id(*c): loss_arrays(forward, *c) for c in CASES}
    groups["free_functions"] = reference_free_functions() if from_reference else oracle_free_functions()
    groups["instances"] = instance_mask_arrays(ref_loader.load().loss_utils.get_batch_instance_mask if from_reference
                                               else restate.get_batch_instance_mask)
    return {"%s/%s" % (g, k): v for g, d in groups.items() for k, v in d.items()}


def write_pins(arrays, source):
    """Gradients go to one file, everything else to the other; an array equal (dtype, shape, bits) to one already
    stored in the same file is stored once."""
    for part, fname in PIN_FILES.items():
        blobs, index, seen = {}, {}, {}
        for key, a in arrays.items():
            if (key.split("/", 1)[1].startswith("grad_")) != (part == "grads"):
                continue
            a = a.copy(order="C")
            sig = (a.dtype.str, a.shape, a.tobytes())
            if sig not in seen:
                seen[sig] = "a%d" % len(blobs)
                blobs[seen[sig]] = a
            index[key] = seen[sig]
        np.savez_compressed(os.path.join(GOLD, fname), index=np.array(json.dumps(index, sort_keys=True)),
                            source=np.array(source), **blobs)


_pins = None


def pins():
    global _pins
    if _pins is None:
        _pins = {}
        for fname in PIN_FILES.values():
            with np.load(os.path.join(GOLD, fname)) as z:
                _pins.update({k: z[b] for k, b in json.loads(str(z["index"])).items()})
    return _pins


def assert_bit_equal(want, got, what):
    assert sorted(want) == sorted(got), (what, sorted(set(want) ^ set(got)))
    for k in want:
        assert want[k].dtype == got[k].dtype and want[k].shape == got[k].shape, (what, k, want[k].dtype, got[k].dtype,
                                                                                want[k].shape, got[k].shape)
        assert np.array_equal(want[k], got[k]), (what, k)


def check(group, got, reference_run):
    stored = {k.split("/", 1)[1]: v for k, v in pins().items() if k.split("/", 1)[0] == group}
    assert_bit_equal(stored, got, (group, "restate vs stored"))
    if ref_loader.available():
        assert_bit_equal(reference_run(), got, (group, "restate vs the reference tree"))


@pytest.mark.parametrize("mode,photo,ssim_on,disable_min", CASES)
def test_loss_forward_and_grads_bit_exact(mode, photo, ssim_on, disable_min):
    got = loss_arrays(restate.loss_forward, mode, photo, ssim_on, disable_min)
    check(case_id(mode, photo, ssim_on, disable_min), got,
          lambda: loss_arrays(ref_modes.reference_loss_forward, mode, photo, ssim_on, disable_min))


def test_free_functions_bit_exact():
    check("free_functions", oracle_free_functions(), reference_free_functions)


def test_bare_instances_branch():
    check("instances", instance_mask_arrays(restate.get_batch_instance_mask),
          lambda: instance_mask_arrays(ref_loader.load().loss_utils.get_batch_instance_mask))


if __name__ == "__main__":
    if "--write" not in sys.argv:
        sys.exit(__doc__)
    from_reference = "--from-oracle" not in sys.argv
    assert not from_reference or ref_loader.available(), "no reference tree at %s (or pass --from-oracle)" % ref_loader.REF
    write_pins(all_arrays(from_reference), "reference tree (oracle/ref_loader.py)" if from_reference else "oracle/restate.py")
