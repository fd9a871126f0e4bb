"""-m gpu: the PIECEWISE API the reference's callers use, on the GPU against the oracle run eagerly on the same GPU.

`Loss.forward` is covered by test_gpu_parity.py.  Here are the call sites around it:
  LossModule.epipolar_loss called directly        trainer.py:312-314,494-497, evaluate_mix.py:70-72
  LossModule.forward / single_mobile_mask_forward / consistency_loss   loss_functions.py:27-105,140-147
  get_epipolar_new on arbitrary point sets        evaluate_flow.py:105-113
  compute_quantiles                               loss_utils.py:197-202
and BASELINE.json's own batch sizes for TG (configs[2]), DS / DC (configs[3]) and 375x1242 in T mode (configs[4]).
Only the GPU sees the real rcp / sqrt / ex2 / lg2 approximations (the emulator maps them to exact math).
"""
import pytest
import torch

import common
from mdn_sfm_b200 import synthetic
from oracle import restate

pytestmark = pytest.mark.gpu
DEV = "cuda"
MODES = ("SN", "T", "TG", "DS", "DC")
SMALL = False     # scratch runs of this file under the CPU emulator shrink the shapes (scripts/emu_piecewise.py)


def _shape(B, H, W):
    return (min(B, 2), 32, 64) if SMALL else (B, H, W)


def _dev(d):
    return {k: v.to(DEV) for k, v in d.items()}


def _inst_dev(inst):
    return [{"instances": d["instances"].to(DEV)} for d in inst]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("form", ["list", "bare"])
def test_epipolar_loss_called_directly(mode, form):
    """What Trainer.val / log_hyper / evaluate_mix call: one (flow, mask) pair at scale 0, flow in PIXELS, the Detectron2
    output either as the list of {"instances": ...} dicts (trainer.py:312-314) or as one bare Instances
    (trainer.py:494, evaluate_mix.py:63), loss_utils.py:110-120."""
    from mdn_sfm_b200.layers import SSIM
    from mdn_sfm_b200.loss_functions import LossModule
    B, H, W = _shape(4, 192, 640) if form == "list" else _shape(1, 128, 416)     # evaluate_mix runs B=1 at 128x416
    opt, batch = common.make(B, H, W, scales=(0,), seed=13, flow_std=0.02)
    inputs, flows, mobiles, cams, inst = batch
    inputs, cams = _dev(inputs), _dev(cams)
    inst = _inst_dev(inst)
    info = inst if form == "list" else inst[0]["instances"]
    pix = restate.create_coords(B, H, W, DEV)
    f = (restate.get_scale_factor(B, H, W, DEV) * flows[("flow", 1, 0)].to(DEV)).contiguous()
    m = mobiles[("mobile", 1, 0)].to(DEV)
    R, t = cams[1][:, :3, :3], cams[1][:, :3, -1]
    weights = restate.gauss_distance_weight(1, H, W)
    fo, mo = f.clone().requires_grad_(True), m.clone().requires_grad_(True)
    with common.tie_ruling(DEV):      # DS / DC: the product's mask at PROVEN exact 0.5 ties of the resize, nothing exempted
        lo, po, eo = restate.epipolar_loss(fo, mo, info, inputs[("inv_K", 0)], R, t, pix, mode=mode, alpha=opt.alpha,
                                           w_d2_sim=opt.w_d2_sim, threshold=opt.threshold,
                                           weight=weights[0].to(DEV) if mode == "TG" else None)
    lo.backward()
    fg, mg = f.clone().requires_grad_(True), m.clone().requires_grad_(True)
    lm = LossModule(opt, batch=B, ssim=SSIM(), mode=mode)
    lg, pg, eg = lm.epipolar_loss(fg, mg, info, inputs[("inv_K", 0)], R, t)
    lg.backward()
    assert float(lg) == pytest.approx(float(lo), rel=common.FWD_TOL), mode
    assert pg.shape == po.shape == (B, 3, H, W) and eg.shape == eo.shape
    assert common.rel_max(po, pg) <= common.FWD_TOL and common.rel_max(eo, eg) <= common.FWD_TOL, mode
    assert common.rel_max(fo.grad, fg.grad) <= common.GRAD_TOL, mode
    assert common.rel_max(mo.grad, mg.grad) <= common.GRAD_TOL, mode


def test_bare_instances_broadcast_over_a_batch():
    """A single Instances object with a batch of maps: the reference's (1,3,H,W) mask broadcasts (loss_utils.py:116-120,138)."""
    from mdn_sfm_b200.loss_functions import LossModule
    B, H, W = 3, 64, 96
    if SMALL:
        H, W = 32, 64
    opt, batch = common.make(B, H, W, scales=(0,), seed=14, flow_std=0.02)
    inputs, flows, mobiles, cams, inst = batch
    inputs, cams = _dev(inputs), _dev(cams)
    info = inst[1]["instances"].to(DEV)
    pix = restate.create_coords(B, H, W, DEV)
    f = (restate.get_scale_factor(B, H, W, DEV) * flows[("flow", -1, 0)].to(DEV)).contiguous()
    m = mobiles[("mobile", -1, 0)].to(DEV)
    R, t = cams[-1][:, :3, :3], cams[-1][:, :3, -1]
    for mode in ("DS", "DC"):
        with common.tie_ruling(DEV):
            lo, po, _ = restate.epipolar_loss(f, m, info, inputs[("inv_K", 0)], R, t, pix, mode=mode, alpha=opt.alpha,
                                              w_d2_sim=opt.w_d2_sim, threshold=opt.threshold)
        lg, pg, _ = LossModule(opt, batch=B, mode=mode).epipolar_loss(f, m, info, inputs[("inv_K", 0)], R, t)
        assert float(lg) == pytest.approx(float(lo), rel=common.FWD_TOL), mode
        assert common.rel_max(po, pg) <= common.FWD_TOL, mode


@pytest.mark.parametrize("mode", ["DC", "SN", "TG", "DS"])
def test_loss_module_forward_and_accumulators(mode):
    """LossModule.forward (shared mask, smooth counted per source frame), single_mobile_mask_forward and consistency_loss
    accumulate into .losses like loss_functions.py:27-105,140-147, with gradients to the flows and the mask."""
    from mdn_sfm_b200.loss_functions import LossModule
    B, H, W = _shape(4, 96, 320)
    opt, batch = common.make(B, H, W, scales=(0, 1), seed=15, flow_std=0.03)
    inputs, flows, mobiles, cams, inst = batch
    inputs, cams, inst = _dev(inputs), _dev(cams), _inst_dev(inst)
    weights = restate.gauss_distance_weight(2, H, W)

    def run(product):
        fl = {k: v.to(DEV).requires_grad_(True) for k, v in flows.items()}
        mo = {k: v.to(DEV).requires_grad_(True) for k, v in mobiles.items()}
        if product:
            lm = LossModule(opt, batch=B, mode=mode, weights=[w.to(DEV) for w in weights])
        else:
            lm = restate.LossModule(opt, mode=mode, weights=[w.to(DEV) for w in weights])
        for s in (0, 1):
            lm.consistency_loss(mo[("mobile", -1, s)], mo[("mobile", 1, s)], s)
            shared = mo[("mobile", 1, s)]
            if product:
                lm(inputs, [-1, 1], fl, shared, inst, cams, s)
                lm.single_mobile_mask_forward(inputs, -1, fl, mo[("mobile", -1, s)], inst, cams, s)
            else:
                for i in (-1, 1):
                    lm.frame_terms(inputs, i, fl, shared, inst, cams, s)
                lm.frame_terms(inputs, -1, fl, mo[("mobile", -1, s)], inst, cams, s)
        total = lm.losses["epip"] + 0.7 * lm.losses["smooth"] + 0.3 * lm.losses["consis"]
        total.backward()
        return lm, fl, mo

    with common.tie_ruling(DEV):
        olm, fo, mo_ = run(False)
    glm, fg, mg = run(True)
    for k in ("consis", "epip", "smooth"):
        assert float(glm.losses[k]) == pytest.approx(float(olm.losses[k]), rel=common.FWD_TOL), k
    for k in fo:
        assert common.rel_max(fo[k].grad, fg[k].grad) <= common.GRAD_TOL, k
    for k in mo_:
        assert common.rel_max(mo_[k].grad, mg[k].grad) <= common.GRAD_TOL, k
    # the scale-0 visualisation tensors the reference stashes (loss_functions.py:61-67,99-105)
    for name in ("epipolars", "epipolar_ori", "flows"):
        assert set(glm.outputs[name].keys()) == {(-1, 0), (1, 0)}, name
        for key, ref in olm.outputs[name].items():
            assert glm.outputs[name][key].shape == ref.shape
            assert common.rel_max(ref, glm.outputs[name][key]) <= common.FWD_TOL, (name, key)


def test_get_epipolar_new_on_point_sets():
    """evaluate_flow.py:105-113: arbitrary correspondences (not the pixel grid), gradients to p1, p2, R and t."""
    from mdn_sfm_b200 import loss_utils
    g = torch.Generator().manual_seed(22)
    for B, n in ((3, 1000), (1, 7)) if SMALL else ((3, 1000), (12, 192 * 640), (1, 7)):
        p1 = torch.cat([torch.rand(B, 2, n, generator=g) * 600, torch.ones(B, 1, n)], 1).to(DEV)
        p2 = (p1.cpu() + torch.cat([torch.randn(B, 2, n, generator=g) * 8, torch.zeros(B, 1, n)], 1)).to(DEV)
        K = torch.tensor([[0.58 * 640, 0, 320.], [0, 1.92 * 192, 96.], [0, 0, 1]])
        invK = torch.linalg.inv(K).unsqueeze(0).repeat(B, 1, 1).to(DEV)
        M = synthetic.make_pose(torch.randn(B, 1, 1, 3, generator=g) * 0.02, torch.randn(B, 1, 1, 3, generator=g) * 0.1)
        R, t = M[:, :3, :3].contiguous().to(DEV), M[:, :3, 3].contiguous().to(DEV)
        wgt = torch.randn(B, 1, n, generator=g).to(DEV)
        outs = []
        for fn in (restate.get_epipolar_new, loss_utils.get_epipolar_new):
            a, b, r_, t_ = (x.clone().requires_grad_(True) for x in (p1, p2, R, t))
            e = fn(a, b, invK, r_, t_)
            (e * wgt).sum().backward()
            outs.append((e, a.grad, b.grad, r_.grad, t_.grad))
        (eo, *go), (eg, *gg) = outs
        assert eg.shape == eo.shape == (B, 1, n)
        assert common.rel_max(eo, eg) <= common.FWD_TOL
        for a, b, what in zip(go, gg, ("p1", "p2", "R", "t")):
            assert common.rel_max(a, b) <= common.GRAD_TOL, (what, B, n)


def test_compute_quantiles_product_function():
    """loss_utils.compute_quantiles (the corrected form of Trainer.epipolar_statics, loss_utils.py:197-202)."""
    from mdn_sfm_b200 import layers, loss_utils
    B, H, W = _shape(4, 192, 640)
    opt, batch = common.make(B, H, W, scales=(0,), seed=23, flow_std=0.02)
    inputs, flows, _, cams, _ = batch
    inputs, flows, cams = _dev(inputs), _dev(flows), _dev(cams)
    pix = restate.create_coords(B, H, W, DEV)
    ones = torch.ones(B, 1, H, W, device=DEV)
    p1 = torch.cat([pix, ones], 1).view(B, 3, -1)
    q = torch.linspace(0, 1, 1000, device=DEV)
    for i in (-1, 1):
        ref = restate.compute_quantiles(flows, cams[i], inputs[("inv_K", 0)], p1, pix, ones, restate.get_scale_factor(B, H, W, DEV), q, i, B)
        got = loss_utils.compute_quantiles(flows, cams[i], inputs[("inv_K", 0)], p1, pix, ones, layers.get_scale_factor(B, H, W).to(DEV), q, i, B)
        assert got.shape == ref.shape == (1000, B)
        assert common.rel_max(ref, got) <= common.FWD_TOL, i


# ---- BASELINE.json's own batch sizes
def test_tg_mode_at_config2_batch():
    opt, batch = common.make(12, 192, 640, seed=52, flow_std=0.03, threshold=0.8625)
    got = common.product_run(opt, batch, "TG", True, True, DEV, pose_grad=True)
    common.compare(common.oracle_run(opt, batch, "TG", True, True, DEV, pose_grad=True), got, True)


@pytest.mark.parametrize("mode", ["DS", "DC"])
def test_ds_dc_at_config3_batch(mode):
    opt, batch = common.make(12, 192, 640, seed=53, flow_std=0.03)
    got = common.product_run(opt, batch, mode, True, True, DEV, pose_grad=True)
    common.compare(common.oracle_run(opt, batch, mode, True, True, DEV, pose_grad=True), got, True)


def test_t_mode_full_res_at_config4_batch():
    opt, batch = common.make(12, 375, 1242, scales=(0,), seed=54, flow_std=0.02)
    got = common.product_run(opt, batch, "T", True, True, DEV, pose_grad=True)
    common.compare(common.oracle_run(opt, batch, "T", True, True, DEV, pose_grad=True), got, True)


def test_single_source_frame_with_disable_min():
    """frame_id = [1] with --disable_min: the pair is masked with mobile(+1) (loss_functions.py:183-186), the consistency
    term still reads both maps (:176-181)."""
    from mdn_sfm_b200.loss_functions import Loss
    B, H, W = 2, 64, 96
    opt, batch = common.make(B, H, W, seed=16, flow_std=0.03, disable_min=True)
    inputs, flows, mobiles, cams, inst = batch
    inputs, cams = _dev(inputs), _dev(cams)
    for ids in ([1], [-1]):
        res = []
        for product in (False, True):
            fl = {k: v.to(DEV).requires_grad_(True) for k, v in flows.items()}
            mo = {k: v.to(DEV).requires_grad_(True) for k, v in mobiles.items()}
            if product:
                _, losses = Loss(opt, no_ssim=False, mode="T", photometric=True)(inputs, ids, fl, mo, None, [0, 1, 2, 3], cams)
            else:
                _, losses = restate.loss_forward(opt, inputs, ids, fl, mo, None, [0, 1, 2, 3], cams, mode="T", photometric=True, ssim_on=True)
            losses["loss"].backward()
            res.append((losses, fl, mo))
        (lo, fo, mo_), (lg, fg, mg) = res
        for k in ("loss", "epip", "smooth", "consis", "photo"):
            assert float(lg[k]) == pytest.approx(float(lo[k]), rel=common.FWD_TOL), (ids, k)
        for k in fo:
            if fo[k].grad is not None:
                assert common.rel_max(fo[k].grad, fg[k].grad) <= common.GRAD_TOL, (ids, k)
        for k in mo_:
            if mo_[k].grad is not None:
                assert common.rel_max(mo_[k].grad, mg[k].grad) <= common.GRAD_TOL, (ids, k)
            else:     # a map the reference never touched gets no (or an all-zero) gradient
                assert mg[k].grad is None or not bool(mg[k].grad.abs().sum() > 0), (ids, k)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_every_entry_point_on_a_non_current_device():
    """cuda:0 is current, the tensors live on cuda:1: DC / DS (instance-mask kernels), the pyramid producer, uint8
    frames, the standalone ops -- every launch must go to the tensors' device."""
    from mdn_sfm_b200 import loss_utils, pyramid, utils
    torch.cuda.set_device(0)
    opt, batch = common.make(2, 64, 128, seed=5)
    for mode in ("DC", "DS"):
        a = common.product_run(opt, batch, mode, True, True, "cuda:0", pose_grad=True)
        b = common.product_run(opt, batch, mode, True, True, "cuda:1", pose_grad=True)
        assert torch.equal(a[1]["loss"].cpu(), b[1]["loss"].cpu()), mode
        for k in a[2]:
            assert torch.equal(a[2][k].grad.cpu(), b[2][k].grad.cpu()), (mode, k)
    img = batch[0][("color", 0, 0)]
    p0 = pyramid.image_pyramid(img.to("cuda:0"), [(32, 64), (16, 32)])
    p1 = pyramid.image_pyramid(img.to("cuda:1"), [(32, 64), (16, 32)])
    assert all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(p0, p1))
    q0 = pyramid.image_pyramid(img.to("cuda:0"), [(64, 128), (32, 64)], packed=True)
    q1 = pyramid.image_pyramid(img.to("cuda:1"), [(64, 128), (32, 64)], packed=True)
    assert all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(q0, q1))
    u8 = torch.randint(0, 256, (2, 64, 128, 3), dtype=torch.uint8)
    assert torch.equal(pyramid.frames_from_u8(u8.to("cuda:0")).cpu(), pyramid.frames_from_u8(u8.to("cuda:1")).cpu())
    m = batch[2][("mobile", 1, 0)]
    assert torch.equal(utils.binary_image(m.to("cuda:0"), 0.4).cpu(), utils.binary_image(m.to("cuda:1"), 0.4).cpu())
    fl = batch[1][("flow", 1, 0)] * 50
    pix = loss_utils.create_coords(2, 64, 128)
    w0, v0 = loss_utils.inverse_warp(img.to("cuda:0"), fl.to("cuda:0"), pix, "zeros")
    w1, v1 = loss_utils.inverse_warp(img.to("cuda:1"), fl.to("cuda:1"), pix, "zeros")
    assert torch.equal(w0.cpu(), w1.cpu()) and torch.equal(v0.cpu(), v1.cpu())
    assert float(loss_utils.smooth_loss(img.to("cuda:0"), m.to("cuda:0"))) == float(loss_utils.smooth_loss(img.to("cuda:1"), m.to("cuda:1")))


# ---- SURVEY 8f-N1: the train step around the loss
def _train_steps(fine_tune):
    from mdn_sfm_b200.train_step import StandInNets, TrainStep
    B, H, W = 2, 64, 96
    opt = synthetic.default_opt(B, H, W, threshold=0.8625)
    inputs, _, _, _, _ = synthetic.make_batch(B, H, W, seed=1, with_instances=False)
    inputs = _dev(inputs)
    weights = [w.to(DEV) for w in restate.gauss_distance_weight(4, H, W)]

    def oracle_loss(inp, ids, flows, mobiles, inst, scales, cams):
        return restate.loss_forward(opt, inp, ids, flows, mobiles, inst, scales, cams, mode="TG", weights=weights,
                                    photometric=True, ssim_on=True)

    def build(**kw):
        torch.manual_seed(0)
        nets = StandInNets(width=8)
        with torch.no_grad():      # a random-init pose head emits |t| ~ 1e-3: scaled to KITTI-like magnitudes (|t| ~ 0.1), where the
            nets.posenet.head.weight.mul_(40.0)     # epipolar geometry is not degenerate and fp32 gradients are meaningful
            nets.posenet.head.bias.add_(torch.tensor([0.3, -0.2, 0.5, 4.0, -6.0, 9.0]))
        return TrainStep(opt, nets=nets, device=DEV, lr=1e-3, fine_tune_flow_motion=fine_tune, **kw)

    return inputs, build, oracle_loss


@pytest.mark.parametrize("fine_tune", [False, True])
def test_train_step_with_the_cuda_loss_equals_the_step_with_the_oracle_loss(fine_tune):
    """One optimisation step (nets -> loss -> backward -> clip -> Adam, trainer.py:223-287) with the CUDA loss -- graph
    replay, PoseNet's outputs handed over as parameters -- against the same step with the oracle as the loss (the
    reference's transformation_from_parameters + ATen composition + autograd): loss 1e-5, every trainable gradient 1e-4.
    fine_tune=True also trains the flow / pose nets, so d/dflow and d/d(axisangle, translation) reach their weights."""
    inputs, build, oracle_loss = _train_steps(fine_tune)
    ts_g = build(mode="TG", photometric=True)                      # graphed loss, pose parameters (the defaults)
    ts_o = build(loss_module=oracle_loss)
    lg, lo = ts_g.step(inputs), ts_o.step(inputs)
    assert float(lg["loss"]) == pytest.approx(float(lo["loss"]), rel=common.FWD_TOL)
    for (n, a), (_, b) in zip(ts_o.nets.named_parameters(), ts_g.nets.named_parameters()):
        if a.grad is None:
            assert b.grad is None, n
            continue
        # PoseNet's weights see the loss through a six-number bottleneck per sample: the 1e-4 the loss is held to on
        # d/d(axisangle, translation) (checked directly below) reaches them amplified by the net's own Jacobian
        tol = 10 * common.GRAD_TOL if n.startswith("posenet") else common.GRAD_TOL
        assert common.rel_max(a.grad, b.grad) <= tol, (n, common.rel_max(a.grad, b.grad))
    if fine_tune:
        assert ts_g.nets.posenet.head.weight.grad is not None and float(ts_g.nets.posenet.head.weight.grad.abs().sum()) > 0
        # the loss itself on the nets' outputs: d/d(axisangle), d/d(translation), d/dflow, d/dmobile at the plain tolerance
        from mdn_sfm_b200.layers import PoseParameters
        flows, mobiles, cams, _, _ = ts_g.process_batch(inputs)
        res = {}
        for which in ("oracle64", "oracle", "product"):
            dt = torch.float64 if which == "oracle64" else torch.float32
            own = lambda v: v.detach().to(dt).clone().requires_grad_(True)
            fl, mo = {k: own(v) for k, v in flows.items()}, {k: own(v) for k, v in mobiles.items()}
            aa, tt = {k: own(c.axisangle) for k, c in cams.items()}, {k: own(c.translation) for k, c in cams.items()}
            if which == "product":
                _, losses = ts_g.eager_loss(inputs, [-1, 1], fl, mo, None, [0, 1, 2, 3], {k: PoseParameters(aa[k], tt[k]) for k in aa})
            else:
                inp = {k: v.to(dt) for k, v in inputs.items()}
                # (the reference allocates its pose matrices with torch.zeros: the default dtype decides their precision)
                torch.set_default_dtype(dt)
                try:
                    _, losses = oracle_loss(inp, [-1, 1], fl, mo, None, [0, 1, 2, 3],
                                            {k: restate.transformation_from_parameters(aa[k], tt[k]) for k in aa})
                finally:
                    torch.set_default_dtype(torch.float32)
            losses["loss"].backward()
            res[which] = (fl, mo, aa, tt)
        for d64, do, dg, what in zip(res["oracle64"], res["oracle"], res["product"], ("d/dflow", "d/dmobile", "d/daxisangle", "d/dtranslation")):
            for k in do:
                if what in ("d/dflow", "d/dmobile"):       # per-pixel gradients: against the reference's own fp32 arithmetic
                    assert common.rel_max(do[k].grad, dg[k].grad) <= common.GRAD_TOL, (what, k, common.rel_max(do[k].grad, dg[k].grad))
                else:
                    # the six pose gradients are sums over every pixel of terms of both signs: in fp32 the REFERENCE's own
                    # result is only good to a few 1e-4 of the float64 value here.  The product is held to the float64 truth,
                    # to the plain tolerance or twice the reference's own fp32 error, whichever is larger.
                    floor = common.rel_max(d64[k].grad, do[k].grad)
                    err = common.rel_max(d64[k].grad, dg[k].grad)
                    assert err <= max(common.GRAD_TOL, 2 * floor), (what, k, err, floor)


def test_graphed_train_step_equals_the_eager_one_bit_for_bit():
    """graphs.GraphedLoss inside TrainStep: three steps (capture, then two replays on new net outputs) leave the nets with
    exactly the parameters of three steps through the eager Loss; so do pose parameters vs pose matrices built by torch."""
    det, bench_ = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False     # (the nets' cuDNN kernels, not ours)
    try:
        _graphed_vs_eager()
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = det, bench_


def _graphed_vs_eager():
    inputs, build, _ = _train_steps(True)
    inputs2 = {k: (v.flip(0) if k[0] == "color" else v) for k, v in inputs.items()}
    ts_a = build(mode="TG", photometric=True, graph_loss=True)
    ts_b = build(mode="TG", photometric=True, graph_loss=False)
    for n, batch in enumerate((inputs, inputs2, inputs)):
        la, lb = ts_a.step(batch), ts_b.step(batch)
        assert torch.equal(la["loss"].detach(), lb["loss"].detach()), (n, float(la["loss"]), float(lb["loss"]))
    for (n, a), (_, b) in zip(ts_a.nets.named_parameters(), ts_b.nets.named_parameters()):
        assert torch.equal(a, b), n


@pytest.mark.parametrize("mode", ["T", "SN"])
def test_batch_of_one_at_the_references_own_noise_floor(mode):
    """Found by the GPU fuzz campaign (scripts/fuzz_gpu.py, 3 400 random cases): at B = 1 the reference's CUDA path rounds
    differently from itself at B >= 2 -- torch.matmul runs gemm for one batch and bgemm for more, so F and F p1 move in the last
    bits and the (cancelling) epipolar numerator with them: 2e-5 ... 5e-5 of the map's maximum (scripts/diag_batch1.py).  The
    product rounds the same way at every batch size.  Pinned here: (1) the product's per-pixel maps of a sample are bit-identical
    whether it runs alone or as sample 0 of a batch of two, (2) the batch-of-two run meets the 1e-5 contract against the
    oracle, (3) the oracle at B = 1 stays within 2e-4 of the oracle at B = 2 -- the floor the B = 1 comparison is held to."""
    H, W = 25, 18
    opt1, b1 = common.make(1, H, W, scales=(0,), seed=573554, flow_std=0.01)
    b1 = b1[:4] + (None,)
    dup = lambda d: {k: v.repeat(2, *([1] * (v.dim() - 1))) for k, v in d.items()}
    b2 = tuple(dup(d) for d in b1[:4]) + (None,)
    opt2 = synthetic.default_opt(2, H, W, scales=[0])
    g1 = common.product_run(opt1, b1, mode, True, True, DEV, pose_grad=True)
    g2 = common.product_run(opt2, b2, mode, True, True, DEV, pose_grad=True)
    o1 = common.oracle_run(opt1, b1, mode, True, True, device=DEV, pose_grad=True)
    o2 = common.oracle_run(opt2, b2, mode, True, True, device=DEV, pose_grad=True)
    for name in ("epipolars", "epipolar_ori", "warps", "diffs"):
        for key in g1[0][name]:
            assert torch.equal(g1[0][name][key][:1], g2[0][name][key][:1]), (name, key)      # (1)
    common.compare(o2, g2, True)                                                             # (2)
    for name in ("epipolars", "epipolar_ori"):
        for key in o1[0][name]:
            assert common.rel_max(o1[0][name][key][:1], o2[0][name][key][:1]) <= 2e-4, (name, key)   # (3)
    common.compare(o1, g1, True, fwd_tol=2e-4, grad_tol=4e-4)
