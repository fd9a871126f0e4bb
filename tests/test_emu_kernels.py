"""CPU-side execution of the UNMODIFIED kernel source under the SIMT emulator (tests/emu) vs the oracle.

This is what catches tile / halo / reflection / adjoint bugs without a GPU.  It says nothing about speed and
the product never takes this route (see tests/emu/cuda_emu.h).
"""
import os

import pytest
import torch

import common
from emu_harness import emulated
from mdn_sfm_b200 import synthetic
from oracle import restate


@pytest.mark.parametrize("mode,photo,ssim_on,disable_min", common.CASES)
def test_fused_loss_matches_oracle(mode, photo, ssim_on, disable_min):
    opt, batch = common.make(2, 32, 64, disable_min=disable_min)
    with emulated():
        ref = common.oracle_run(opt, batch, mode, photo, ssim_on)      # (inside: the DS / DC tie ruling runs the emulated kernels)
        got = common.product_run(opt, batch, mode, photo, ssim_on, "cpu")
        common.compare(ref, got, photo)


def test_ragged_tiles_and_pose_gradient():
    # 23x45: not a multiple of the 32x16 tile in either direction, odd sizes; single scale like config 5 (375x1242)
    opt, batch = common.make(2, 23, 45, scales=(0,), seed=5, flow_std=0.08)
    for mode in ("SN", "T"):
        ref = common.oracle_run(opt, batch, mode, True, True, pose_grad=True)
        with emulated():
            got = common.product_run(opt, batch, mode, True, True, "cpu", pose_grad=True)
            common.compare(ref, got, True)


def test_large_flow_out_of_bounds_and_disabled_terms():
    opt, batch = common.make(1, 32, 64, scales=(0, 1), seed=9, flow_std=0.6, disable_smoothloss=True,
                             disable_consisloss=True)
    ref = common.oracle_run(opt, batch, "T", True, True)
    with emulated():
        got = common.product_run(opt, batch, "T", True, True, "cpu")
        common.compare(ref, got, True)
    assert float(got[1]["loss"]) == pytest.approx(float(ref[1]["loss"]), rel=1e-5)
    assert got[1]["smooth"] == 0 and got[1]["consis"] == 0


def test_upstream_gradient_scaling():
    opt, batch = common.make(1, 16, 32, scales=(0,), seed=3)
    inputs, flows, mobiles, cams, inst = batch
    from mdn_sfm_b200.loss_functions import Loss
    with emulated():
        f1, m1 = common.leaf(flows), common.leaf(mobiles)
        _, l1 = Loss(opt, no_ssim=False, mode="T", photometric=True, arith="cpu")(inputs, [-1, 1], f1, m1, inst, [0], cams)
        l1["loss"].backward()
        f2, m2 = common.leaf(flows), common.leaf(mobiles)
        _, l2 = Loss(opt, no_ssim=False, mode="T", photometric=True, arith="cpu")(inputs, [-1, 1], f2, m2, inst, [0], cams)
        (l2["loss"] * 3.5).backward()
    for k in f1:
        assert torch.allclose(f1[k].grad * 3.5, f2[k].grad, rtol=1e-6, atol=0)
    for k in m1:
        assert torch.allclose(m1[k].grad * 3.5, m2[k].grad, rtol=1e-6, atol=0)


def test_loss_module_methods():
    opt, batch = common.make(2, 32, 64, seed=13)
    inputs, flows, mobiles, cams, inst = batch
    from mdn_sfm_b200.loss_functions import LossModule
    from mdn_sfm_b200.layers import SSIM
    pix = restate.create_coords(2, 32, 64)
    f = (restate.get_scale_factor(2, 32, 64) * flows[("flow", 1, 0)]).contiguous()
    m = mobiles[("mobile", 1, 0)]
    R, t = cams[1][:, :3, :3], cams[1][:, :3, -1]
    with emulated():
        for mode in ("SN", "T", "TG", "DS", "DC"):
            fo, mo = f.clone().requires_grad_(True), m.clone().requires_grad_(True)
            weights = restate.gauss_distance_weight(4, 32, 64)
            lo, po, eo = restate.epipolar_loss(fo, mo, inst, inputs[("inv_K", 0)], R, t, pix, mode=mode, alpha=opt.alpha,
                                               w_d2_sim=opt.w_d2_sim, threshold=opt.threshold,
                                               weight=weights[0] if mode == "TG" else None)
            lo.backward()
            fg, mg = f.clone().requires_grad_(True), m.clone().requires_grad_(True)
            lm = LossModule(opt, batch=2, ssim=SSIM(), mode=mode, arith="cpu")
            lg, pg, eg = lm.epipolar_loss(fg, mg, inst, inputs[("inv_K", 0)], R, t)
            lg.backward()
            assert float(lg) == pytest.approx(float(lo), rel=1e-5), mode
            assert pg.shape == po.shape and eg.shape == eo.shape
            assert common.rel_max(po, pg) < 1e-5 and common.rel_max(eo, eg) < 1e-5, mode
            assert common.rel_max(fo.grad, fg.grad) < 1e-4 and common.rel_max(mo.grad, mg.grad) < 1e-4, mode
        # photometric
        fo = f.clone().requires_grad_(True)
        lo, wo, do, vo = restate.photo_metric_loss(inputs[("color", 0, 0)], inputs[("color", 1, 0)], fo, pix, True)
        lo.backward()
        fg = f.clone().requires_grad_(True)
        lm = LossModule(opt, batch=2, ssim=SSIM(), arith="cpu")
        lg, wg, dg, vg = lm.photo_metric_loss(inputs[("color", 0, 0)], inputs[("color", 1, 0)], fg)
        lg.backward()
        assert float(lg) == pytest.approx(float(lo), rel=1e-5)
        assert common.rel_max(wo, wg) < 1e-5 and common.rel_max(do, dg) < 1e-5 and torch.equal(vo, vg)
        assert common.rel_max(fo.grad, fg.grad) < 1e-4
        # forward()/consistency accumulate like the reference
        lm = LossModule(opt, batch=2, mode="DC", arith="cpu")
        lm.consistency_loss(mobiles[("mobile", -1, 1)], mobiles[("mobile", 1, 1)], 1)
        lm(inputs, [-1, 1], flows, mobiles[("mobile", 1, 1)], inst, cams, 1)
        olm = restate.LossModule(opt, mode="DC")
        olm.consistency_loss(mobiles[("mobile", -1, 1)], mobiles[("mobile", 1, 1)], 1)
        for i in (-1, 1):
            olm.frame_terms(inputs, i, flows, mobiles[("mobile", 1, 1)], inst, cams, 1)
        for k in ("consis", "epip", "smooth"):
            assert float(lm.losses[k]) == pytest.approx(float(olm.losses[k]), rel=1e-5), k


@pytest.mark.parametrize("padding_mode", ["border", "reflection"])
def test_padding_modes_of_the_flow_warp(padding_mode):
    """Loss(padding_mode=...) / inverse_warp(..., padding_mode): grid_sample's border and reflection modes (the ctor argument of
    loss_functions.py:12,161; upstream callers pass "zeros").  Large flows, so that many samples leave the image and are
    clipped / folded back -- values, validity and the gradient through the clipped coordinate against the oracle."""
    from mdn_sfm_b200 import loss_utils
    opt, batch = common.make(2, 24, 72, scales=(0, 1), seed=17, flow_std=0.4)
    ref = common.oracle_run(opt, batch, "T", True, True, padding_mode=padding_mode)
    with emulated():
        got = common.product_run(opt, batch, "T", True, True, "cpu", padding_mode=padding_mode)
        common.compare(ref, got, True)
        g = torch.Generator().manual_seed(22)
        B, h, w = 2, 19, 37
        img, x = torch.rand(B, 3, h, w, generator=g), torch.rand(B, 3, h, w, generator=g)
        flow = torch.randn(B, 2, h, w, generator=g) * 25
        pix = restate.create_coords(B, h, w)
        fo = flow.clone().requires_grad_(True)
        wo, vo = restate.inverse_warp(img, fo, pix, padding_mode)
        (wo * x).sum().backward()
        fg = flow.clone().requires_grad_(True)
        wg, vg = loss_utils.inverse_warp(img, fg, pix, padding_mode, arith="cpu")
        (wg * x).sum().backward()
        assert common.rel_max(wo, wg) < 1e-5 and torch.equal(vo, vg)
        assert common.rel_max(fo.grad, fg.grad) < 1e-4
    with pytest.raises(ValueError):
        loss_utils.inverse_warp(img, flow, pix, "circular")


def test_free_functions():
    from mdn_sfm_b200 import layers, loss_utils, utils
    g = torch.Generator().manual_seed(21)
    B, h, w = 2, 19, 37
    ref = torch.rand(B, 3, h, w, generator=g)
    x = torch.rand(B, 3, h, w, generator=g)
    flow = torch.randn(B, 2, h, w, generator=g) * 6
    pix = restate.create_coords(B, h, w)
    with emulated():
        # inverse_warp fwd + bwd, valid mask bit exact
        fo = flow.clone().requires_grad_(True)
        wo, vo = restate.inverse_warp(ref, fo, pix)
        (wo * x).sum().backward()
        fg = flow.clone().requires_grad_(True)
        wg, vg = loss_utils.inverse_warp(ref, fg, pix, "zeros", arith="cpu")
        (wg * x).sum().backward()
        assert common.rel_max(wo, wg) < 1e-5 and torch.equal(vo, vg)
        assert common.rel_max(fo.grad, fg.grad) < 1e-4
        # SSIM module fwd + bwd to both arguments
        xo, yo = x.clone().requires_grad_(True), ref.clone().requires_grad_(True)
        (restate.ssim(xo, yo) * flow[:, :1].abs()).sum().backward()
        xg, yg = x.clone().requires_grad_(True), ref.clone().requires_grad_(True)
        sg = layers.SSIM()(xg, yg)
        (sg * flow[:, :1].abs()).sum().backward()
        assert common.rel_max(restate.ssim(x, ref), sg) < 1e-5
        assert common.rel_max(xo.grad, xg.grad) < 1e-4 and common.rel_max(yo.grad, yg.grad) < 1e-4
        # get_epipolar_new on arbitrary point sets, with gradients to p2 and pose
        p1 = torch.cat([pix, torch.ones(B, 1, h, w)], 1).view(B, 3, -1)
        p2 = torch.cat([pix + flow, torch.ones(B, 1, h, w)], 1).view(B, 3, -1)
        K = torch.tensor([[0.58 * w, 0, 0.5 * w], [0, 1.92 * h, 0.5 * h], [0, 0, 1]])
        invK = torch.linalg.inv(K).unsqueeze(0).repeat(B, 1, 1)
        M = synthetic.make_pose(torch.randn(B, 1, 1, 3, generator=g) * 0.02, torch.randn(B, 1, 1, 3, generator=g) * 0.1)
        R, t = M[:, :3, :3].contiguous(), M[:, :3, 3].contiguous()
        p2o, to = p2.clone().requires_grad_(True), t.clone().requires_grad_(True)
        eo = restate.get_epipolar_new(p1, p2o, invK, R, to)
        eo.abs().sum().backward()
        p2g, tg = p2.clone().requires_grad_(True), t.clone().requires_grad_(True)
        eg = loss_utils.get_epipolar_new(p1, p2g, invK, R, tg)
        eg.abs().sum().backward()
        assert eg.shape == eo.shape and common.rel_max(eo, eg) < 1e-5
        assert common.rel_max(p2o.grad, p2g.grad) < 1e-4 and common.rel_max(to.grad, tg.grad) < 1e-4
        # smooth_loss, binary_image, FlowWarp
        m = torch.rand(B, 1, h, w, generator=g)
        assert float(loss_utils.smooth_loss(x, m)) == pytest.approx(float(restate.smooth_loss(x, m)), rel=1e-5)
        assert torch.equal(utils.binary_image(m, 0.4), restate.binary_image(m, 0.4))
        a, b = utils.FlowWarp(B, h, w, arith="cpu")(flow), restate.flow_warp_grid(flow)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    # pure host helpers
    for wa, wb in zip(utils.gauss_distance_weight(4, 64, 96), restate.gauss_distance_weight(4, 64, 96)):
        assert torch.equal(wa, wb)
    aa, tt = torch.randn(3, 1, 1, 3, generator=g) * 0.3, torch.randn(3, 1, 1, 3, generator=g)
    for inv in (False, True):
        assert torch.equal(layers.transformation_from_parameters(aa, tt, inv), restate.transformation_from_parameters(aa, tt, inv))
    assert torch.equal(layers.get_scale_factor(2, 5, 7).contiguous(), restate.get_scale_factor(2, 5, 7).contiguous())
    assert torch.equal(loss_utils.create_coords(2, 5, 7), restate.create_coords(2, 5, 7))


def test_multiple_tiles_in_x_and_vector_staging():
    # 136 = two full 64-wide tiles + a ragged one (w % 4 == 0: 16-byte staging path); 68 at scale 1; heights 24 / 12
    opt, batch = common.make(1, 24, 136, scales=(0, 1), seed=17, flow_std=0.06)
    for mode in ("T", "SN"):
        ref = common.oracle_run(opt, batch, mode, True, True)
        with emulated():
            got = common.product_run(opt, batch, mode, True, True, "cpu")
            common.compare(ref, got, True)


@pytest.mark.parametrize("mode", ["SN", "T"])
def test_poses_inside_the_call_match_the_oracle(mode):
    """MdnLossDesc.cam / inv_K: F and the pose adjoint computed inside mdn_loss_fused, two scales, ragged tiles, SN fix-up
    included.  d/dcam (the g_cam write of the finish kernel) and the loss scalars against the CPU oracle."""
    opt, batch = common.make(2, 24, 72, scales=(0, 1), seed=13, flow_std=0.08)
    with emulated():
        a = common.product_run(opt, batch, mode, True, True, "cpu", pose_grad=True, arith="cuda")
    assert all(c.grad is not None and float(c.grad.abs().sum()) > 0 for c in a[4].values())
    ref = common.oracle_run(opt, batch, mode, True, True, pose_grad=True)
    for k in ref[4]:
        assert common.rel_max(ref[4][k].grad, a[4][k].grad) <= common.GRAD_TOL, ("d/dcam", k, common.rel_max(ref[4][k].grad, a[4][k].grad))
    # the CUDA-eager arithmetic stays within tolerance of the CPU oracle away from flipped bilinear cells (scalars only)
    for k in ("loss", "epip", "smooth", "consis", "photo"):
        assert float(a[1][k]) == pytest.approx(float(ref[1][k]), rel=1e-4), k


def _ref_resized_masks(inst, sizes):
    from oracle import restate
    return [restate.resized_instance_mask(inst, s)[:, 0].to(torch.uint8) for s in sizes]


def assert_masks_equal_up_to_exact_ties(got, inst, sizes):
    """Bit-exact against Resize(size)(get_batch_instance_mask(.)), except where the resized value is an exact 0.5 tie
    in exact arithmetic (|float64 value - 0.5| < 1e-6): there the reference's own answer depends on the last-bit
    rounding path of the ATen build (its CPU and CUDA kernels differ), which BASELINE.json's tolerance exempts."""
    import torch.nn.functional as F
    from oracle import restate
    ref = _ref_resized_masks(inst, sizes)
    full = restate.get_batch_instance_mask(inst)[:, :1].double()
    n_bad = 0
    for g_, r_, s in zip(got, ref, sizes):
        assert g_.dtype == torch.uint8 and tuple(g_.shape) == tuple(r_.shape)
        bad = (g_.cpu() != r_)
        if bad.any():
            v64 = F.interpolate(full, size=tuple(s), mode="bilinear", align_corners=False, antialias=True)[:, 0]
            assert float((v64[bad] - 0.5).abs().max()) < 1e-6, (s, int(bad.sum()))
            n_bad += int(bad.sum())
        assert 0 < int(r_.sum()) < r_.numel()
    assert n_bad <= 1e-5 * sum(r.numel() for r in ref) + 1, n_bad
    return n_bad


@pytest.mark.parametrize("src_hw,sizes", [((375, 1242), [(192, 640), (96, 320), (48, 160), (24, 80)]),
                                          ((61, 97), [(64, 128), (61, 97), (17, 200)]), ((375, 1242), [(8, 12), (3, 640)]), ((64, 96), [(32, 48), (64, 96)])])
def test_instance_mask_union_and_resize_match_torchvision(src_hw, sizes):
    """mdn_instance_mask_union + mdn_instance_mask_resize == Resize(size)(get_batch_instance_mask(.)) of the reference
    (loss_utils.py:73-75,102-124,135-137; torchvision bilinear + antialias on int64, rounded), bit for bit except at
    exact 0.5 ties: KITTI-sized
    Detectron2-style masks down to the four pyramid levels; up-scaling, identity and mixed factors; list and bare forms."""
    from mdn_sfm_b200 import loss_utils, synthetic
    g = torch.Generator().manual_seed(7)
    H, W = src_hw
    inst = []
    for n_inst in (3, 2):      # Detectron2-style: sparse speckle plus filled boxes, a different instance count per sample
        m = torch.rand(n_inst, H, W, generator=g) > 0.9
        for n in range(n_inst):
            y0, x0 = int(torch.randint(0, H // 2, (1,), generator=g)), int(torch.randint(0, W // 2, (1,), generator=g))
            m[n, y0:y0 + H // 4, x0:x0 + W // 3] = True
        inst.append({"instances": synthetic.SyntheticInstances(m)})
    with emulated() as lib:
        got = loss_utils.instance_masks_u8(inst, sizes, "cpu", lib)
        bare = loss_utils.instance_masks_u8(inst[0]["instances"], sizes[:1], "cpu", lib)
    assert assert_masks_equal_up_to_exact_ties(got, inst, sizes) == 0      # (this seed has no tie)
    assert_masks_equal_up_to_exact_ties(bare, inst[0]["instances"], sizes[:1])
    # the fused pass over bit-packed rows (the default where a block's source window fits) and the two separable passes
    # through the global temporary perform the same fp32 operations in the same order
    os.environ["MDN_RESIZE_TWO_PASS"] = "1"
    try:
        with emulated() as lib:
            two = loss_utils.instance_masks_u8(inst, sizes, "cpu", lib)
    finally:
        del os.environ["MDN_RESIZE_TWO_PASS"]
    assert all(torch.equal(a, b) for a, b in zip(got, two))


def test_fused_mask_resize_equals_the_two_passes_on_random_shapes():
    """The bit-packed fused resize against the two separable passes (same fp32 operations, same order) over random source /
    output sizes, batch sizes, level counts and mask densities: up- and down-scaling, factors on both sides of the fused
    path's limits (a block's 48 source rows / 56 packed words), sizes that are not multiples of anything."""
    import random
    from mdn_sfm_b200 import loss_utils, synthetic
    rnd = random.Random(11)
    g = torch.Generator().manual_seed(3)
    with emulated() as lib:
        for _ in range(12):
            H, W = rnd.randint(3, 120), rnd.randint(3, 260)
            sizes = [(rnd.randint(1, 130), rnd.randint(1, 290)) for _ in range(rnd.randint(1, 4))]
            inst = [{"instances": synthetic.SyntheticInstances(torch.rand(rnd.randint(1, 3), H, W, generator=g) > rnd.choice([0.5, 0.9, 0.99]))}
                    for _ in range(rnd.randint(1, 2))]
            one = loss_utils.instance_masks_u8(inst, sizes, "cpu", lib)
            os.environ["MDN_RESIZE_TWO_PASS"] = "1"
            try:
                two = loss_utils.instance_masks_u8(inst, sizes, "cpu", lib)
            finally:
                del os.environ["MDN_RESIZE_TWO_PASS"]
            assert all(torch.equal(a, b) for a, b in zip(one, two)), ((H, W), sizes)


def test_image_pyramid_matches_torchvision_resize():
    """SURVEY 8f-N3: mdn_image_pyramid == torchvision Resize((H/2**s, W/2**s)) of an fp32 image (bilinear + antialias),
    the three lower pyramid levels in one call; fp32 round-off only (the separable sums run in the library's order)."""
    from torchvision.transforms import Resize
    from mdn_sfm_b200 import pyramid
    g = torch.Generator().manual_seed(3)
    img = (torch.rand(2, 3, 48, 80, generator=g) - 0.45) / 0.225
    sizes = [(48, 80), (24, 40), (12, 20), (6, 10), (17, 33)]
    with emulated() as lib:
        got = pyramid.image_pyramid(img, sizes, lib)
    assert got[0] is img
    for t, s in zip(got, sizes):
        ref = Resize(s)(img)
        assert tuple(t.shape) == tuple(ref.shape)
        assert float((t - ref).abs().max()) <= 2e-6 * float(ref.abs().max()), (s, float((t - ref).abs().max()))


FUZZ = [  # B, H, W, scales, mode, photometric, ssim, opt overrides, flow std  (drawn once at random; odd / tiny / ragged shapes)
    (2, 30, 3, (0,), "DS", True, False, dict(disable_smoothloss=True), 0.01),
    (1, 37, 5, (0,), "T", False, False, {}, 0.3),
    (1, 25, 62, (0, 1), "T", False, False, {}, 0.3),
    (2, 14, 96, (0, 1), "TG", True, True, dict(disable_min=True, disable_smoothloss=True), 0.05),
    (1, 3, 54, (0,), "DC", True, True, {}, 0.05),
    (3, 38, 4, (0,), "DC", False, True, dict(disable_consisloss=True), 0.05),
    (3, 17, 135, (0,), "T", True, True, {}, 0.05),
    (3, 34, 139, (0,), "SN", False, True, dict(disable_min=True), 0.05),
    (1, 20, 134, (0,), "T", True, True, {}, 0.05),      # even width, not a multiple of 4: the 8-byte staging path (1242)
]


@pytest.mark.parametrize("case", FUZZ, ids=lambda c: "%dx%dx%d-%s" % (c[0], c[1], c[2], c[4]))
def test_odd_tiny_and_ragged_shapes_all_modes(case):
    """Edge shapes the tile geometry does not divide (3-pixel-wide images, 3 rows, widths just past a tile, odd sizes),
    every mode and term switch, pose gradients: product (kernel source under the SIMT emulator) vs the oracle."""
    B, H, W, scales, mode, photo, ssim, over, fstd = case
    opt, batch = common.make(B, H, W, scales=scales, seed=100 + H + W, flow_std=fstd, **over)
    with emulated():
        ref = common.oracle_run(opt, batch, mode, photo, ssim, pose_grad=True)
        got = common.product_run(opt, batch, mode, photo, ssim, "cpu", pose_grad=True)
        common.compare(ref, got, photo)


def test_epipolar_statistics_match_the_reference_quantiles():
    """SURVEY 8f-N4: per-sample quantiles of |e| over batches == loss_utils.compute_quantiles (:197-202) of the oracle."""
    from mdn_sfm_b200 import layers, statistics
    opt, batch = common.make(2, 24, 72, scales=(0,), seed=19, flow_std=0.05)
    inputs, flows, _, cams, _ = batch
    B, h, w = 2, 24, 72
    pix = restate.create_coords(B, h, w)
    ones = torch.ones(B, 1, h, w)
    p1 = torch.cat([pix, ones], 1).view(B, 3, -1)
    q = torch.linspace(0, 1, 50)
    with emulated() as lib:
        st = statistics.EpipolarStatistics(num_quantile=50, library=lib, arith="cpu")
        st.update(flows, inputs[("inv_K", 0)], cams)
        st.update(flows, inputs[("inv_K", 0)], cams)
        per, thr = st.result()
    assert per.shape == (2, 50, 4) and thr.shape == (8,)
    sf = layers.get_scale_factor(B, h, w)
    for k, i in enumerate((-1, 1)):
        ref = restate.compute_quantiles(flows, cams[i], inputs[("inv_K", 0)], p1, pix, ones, sf, q, i, B)
        got = torch.from_numpy(per[k, :, :B])
        assert float((got - ref).abs().max()) <= 1e-5 * float(ref.abs().max()), i


def test_packed_source_pyramid_feeds_the_loss_without_a_repack():
    """SURVEY 8f-N3, second half: source frames handed over as ('color_packed', i, s) -- (B,h,w,4), what
    mdn_image_pyramid_packed writes -- give bit-identical losses, gradients and maps to the NCHW form (which the call
    repacks itself), and the packed pyramid made from the full-resolution frame equals torchvision's Resize."""
    from torchvision.transforms import Resize
    from mdn_sfm_b200 import pyramid
    from mdn_sfm_b200.loss_functions import Loss
    opt, batch = common.make(2, 32, 80, scales=(0, 1), seed=29, flow_std=0.08)
    inputs, flows, mobiles, cams, _ = batch
    with emulated() as lib:
        a = common.product_run(opt, batch, "T", True, True, "cpu", pose_grad=True, arith="cuda")
        packed = dict(inputs)
        for i in (-1, 1):
            for s in (0, 1):
                lvl = inputs[("color", i, s)]
                packed[("color_packed", i, s)] = pyramid.image_pyramid(lvl, [tuple(lvl.shape[-2:])], lib, packed=True)[0]
                del packed[("color", i, s)]          # the NCHW source levels are not read any more
        b = common.product_run(opt, (packed, flows, mobiles, cams, None), "T", True, True, "cpu", pose_grad=True, arith="cuda")
        common.assert_identical_runs(a, b, maps=("epipolars", "epipolar_ori", "warps", "diffs"))
        pk = pyramid.image_pyramid(inputs[("color", 1, 0)], [(32, 80), (16, 40), (9, 21)], lib, packed=True)
    for t, sz in zip(pk, [(32, 80), (16, 40), (9, 21)]):
        ref = Resize(sz)(inputs[("color", 1, 0)]).permute(0, 2, 3, 1)
        assert tuple(t.shape) == (2,) + sz + (4,)
        assert float((t[..., :3] - ref).abs().max()) <= 2e-6 * float(ref.abs().max()) and float(t[..., 3].abs().max()) == 0.0


def test_uint8_frames_normalised_on_the_device_equal_the_dataset_transforms():
    """mdn_normalize_u8 == ArrayToTensor + Normalize of the reference's dataset (custom_transforms.py:72-80,103-112), bit for bit."""
    from mdn_sfm_b200 import pyramid
    g = torch.Generator().manual_seed(2)
    u8 = torch.randint(0, 256, (2, 13, 37, 3), dtype=torch.uint8, generator=g)
    ref = u8.permute(0, 3, 1, 2).float() / 255
    for t, m, s in zip(ref.unbind(1), (0.45, 0.45, 0.45), (0.225, 0.225, 0.225)):
        t.sub_(m).div_(s)
    with emulated() as lib:
        got = pyramid.frames_from_u8(u8, library=lib)
    assert torch.equal(got, ref.contiguous())


@pytest.mark.parametrize("mode", ["T", "SN"])
def test_pose_parameters_inside_the_call(mode):
    """SURVEY 8f-N1, fused pose prologue: cam_T_cam[i] = PoseParameters(axisangle, translation) -- the kernels run
    transformation_from_parameters (networks/layers.py:16-98) themselves and return d/d(axisangle), d/d(translation) --
    against the oracle's torch composition + autograd.  (Epipolar terms only: the parameter path needs the CUDA-eager
    arithmetic flag, whose warp rounding the CPU oracle does not share.)"""
    from mdn_sfm_b200.layers import PoseParameters
    from mdn_sfm_b200.loss_functions import Loss
    B, H, W = 2, 32, 64
    opt, batch = common.make(B, H, W, seed=23, flow_std=0.05)
    inputs, flows, mobiles, _, _ = batch
    g = torch.Generator().manual_seed(5)
    aa = {i: torch.randn(B, 1, 1, 3, generator=g) * 0.05 for i in (-1, 1)}
    tt = {i: torch.randn(B, 1, 1, 3, generator=g) * 0.2 for i in (-1, 1)}
    aa[1][0] = 0.0      # a zero rotation: the 1e-7 guard and the norm's zero sub-gradient
    ao, to = common.leaf(aa), common.leaf(tt)
    fo, mo = common.leaf(flows), common.leaf(mobiles)
    cams = {i: restate.transformation_from_parameters(ao[i], to[i]) for i in (-1, 1)}
    _, lo = restate.loss_forward(opt, inputs, [-1, 1], fo, mo, None, [0, 1, 2, 3], cams, mode=mode)
    lo["loss"].backward()
    with emulated():
        ag, tg = common.leaf(aa), common.leaf(tt)
        fg, mg = common.leaf(flows), common.leaf(mobiles)
        _, lg = Loss(opt, mode=mode, arith="cuda")(inputs, [-1, 1], fg, mg, None, [0, 1, 2, 3],
                                                  {i: PoseParameters(ag[i], tg[i]) for i in (-1, 1)})
        lg["loss"].backward()
    assert float(lg["loss"]) == pytest.approx(float(lo["loss"]), rel=common.FWD_TOL)
    for i in (-1, 1):
        assert common.rel_max(ao[i].grad, ag[i].grad) <= common.GRAD_TOL, ("d/daxisangle", i)
        assert common.rel_max(to[i].grad, tg[i].grad) <= common.GRAD_TOL, ("d/dtranslation", i)
    for k in fo:
        assert common.rel_max(fo[k].grad, fg[k].grad) <= common.GRAD_TOL, k
