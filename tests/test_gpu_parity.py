"""-m gpu: the CUDA path, called through the C ABI, against the oracle on identical seeded inputs.

Comparators: the oracle run eagerly on the same GPU (the reference's own CUDA-eager arithmetic) and on the host CPU.
"""
import pytest
import torch

import common
from mdn_sfm_b200 import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("mode,photo,ssim_on,disable_min", common.CASES)
def test_fused_vs_oracle_small(mode, photo, ssim_on, disable_min):
    opt, batch = common.make(2, 64, 96, disable_min=disable_min)
    # against the reference arithmetic run eagerly on this GPU ...
    got = common.product_run(opt, batch, mode, photo, ssim_on, DEV, arith="cuda")
    common.compare(common.oracle_run(opt, batch, mode, photo, ssim_on, DEV), got, photo)
    # ... and against the same code on the host CPU (whose `tensor /= scalar` rounds differently: arith="cpu")
    got = common.product_run(opt, batch, mode, photo, ssim_on, DEV, arith="cpu")
    common.compare(common.oracle_run(opt, batch, mode, photo, ssim_on, "cpu", product_device=DEV), got, photo)


@pytest.mark.parametrize("mode", ["SN", "T", "TG", "DC"])
def test_fused_vs_oracle_config1_shape(mode):
    # BASELINE configs[0]: B=4, 3x192x640, 4 scales; the pose gradient of the in-call F (fused kernel) and its adjoint
    # (finish kernel) too
    opt, batch = common.make(4, 192, 640, seed=42, flow_std=0.01)
    got = common.product_run(opt, batch, mode, True, True, DEV, pose_grad=True)
    common.compare(common.oracle_run(opt, batch, mode, True, True, DEV, pose_grad=True), got, True)


def test_fused_vs_oracle_headline_shape():
    # BASELINE configs[1]: T mode + photometric, B=12, 192x640, 4 scales
    opt, batch = common.make(12, 192, 640, seed=42, flow_std=0.05)
    got = common.product_run(opt, batch, "T", True, True, DEV, pose_grad=True)
    common.compare(common.oracle_run(opt, batch, "T", True, True, DEV, pose_grad=True), got, True)


def test_fused_vs_oracle_full_res_kitti():
    # BASELINE configs[4]: 375x1242, scale 0 only (ragged tiles)
    opt, batch = common.make(2, 375, 1242, scales=(0,), seed=42, flow_std=0.02)
    for mode in ("SN", "TG"):
        got = common.product_run(opt, batch, mode, True, True, DEV)
        common.compare(common.oracle_run(opt, batch, mode, True, True, DEV), got, True)


def test_deterministic_and_repeatable():
    opt, batch = common.make(3, 96, 160, seed=1)
    a = common.product_run(opt, batch, "SN", True, True, DEV)
    b = common.product_run(opt, batch, "SN", True, True, DEV)
    assert torch.equal(a[1]["loss"], b[1]["loss"])
    for k in a[2]:
        assert torch.equal(a[2][k].grad, b[2][k].grad)
    for k in a[3]:
        assert torch.equal(a[3][k].grad, b[3][k].grad)


def test_batch_linearity_property():
    """Size-independent property: every term is a mean over the batch, so the loss of a batch made of the same
    sample repeated equals the loss of that sample (T mode has no cross-pixel coupling) and gradients scale by 1/B."""
    opt1, b1 = common.make(1, 192, 640, seed=8)
    opt6 = synthetic.default_opt(6, 192, 640)
    rep = lambda d: {k: v.repeat(6, *([1] * (v.dim() - 1))) for k, v in d.items()}
    b6 = (rep(b1[0]), rep(b1[1]), rep(b1[2]), rep(b1[3]), None)
    b1 = b1[:4] + (None,)
    g1 = common.product_run(opt1, b1, "T", True, True, DEV)
    g6 = common.product_run(opt6, b6, "T", True, True, DEV)
    assert float(g6[1]["loss"]) == pytest.approx(float(g1[1]["loss"]), rel=1e-5)
    for k in g1[2]:
        assert common.rel_max(g1[2][k].grad / 6, g6[2][k].grad[2:3]) < 1e-5


def test_zero_flow_valid_mask_and_identity_quirk():
    """valid mask is all-true for zero flow and the warp is NOT the identity (SURVEY.md section 7): both must match."""
    from mdn_sfm_b200.loss_functions import LossModule
    from mdn_sfm_b200.layers import SSIM
    from oracle import restate
    opt = synthetic.default_opt(2, 192, 640)
    g = torch.Generator().manual_seed(0)
    tgt = torch.rand(2, 3, 192, 640, generator=g).to(DEV)
    flow = torch.zeros(2, 2, 192, 640, device=DEV)
    lo, wo, do, vo = restate.photo_metric_loss(tgt, tgt, flow, restate.create_coords(2, 192, 640, DEV), True)
    lg, wg, dg, vg = LossModule(opt, ssim=SSIM()).photo_metric_loss(tgt, tgt, flow)
    assert torch.equal(vo, vg) and bool(vg.all())
    assert common.rel_max(wo, wg) < 1e-6
    assert float(lg) == pytest.approx(float(lo), rel=1e-5, abs=2e-8)   # the loss itself is ~3e-7: pure rounding noise of 1 - n/d


def test_standalone_ops_on_gpu():
    from mdn_sfm_b200 import layers, loss_utils, utils
    from oracle import restate
    g = torch.Generator().manual_seed(21)
    B, h, w = 3, 75, 131
    ref = torch.rand(B, 3, h, w, generator=g).to(DEV)
    x = torch.rand(B, 3, h, w, generator=g).to(DEV)
    flow = (torch.randn(B, 2, h, w, generator=g) * 9).to(DEV)
    pix = restate.create_coords(B, h, w, DEV)
    fo = flow.clone().requires_grad_(True)
    wo, vo = restate.inverse_warp(ref, fo, pix)
    (wo * x).sum().backward()
    fg = flow.clone().requires_grad_(True)
    wg, vg = loss_utils.inverse_warp(ref, fg, pix, "zeros")
    (wg * x).sum().backward()
    assert common.rel_max(wo, wg) < 1e-5 and torch.equal(vo, vg) and common.rel_max(fo.grad, fg.grad) < 1e-4
    xo, yo = x.clone().requires_grad_(True), ref.clone().requires_grad_(True)
    (restate.ssim(xo, yo) * flow[:, :1].abs()).sum().backward()
    xg, yg = x.clone().requires_grad_(True), ref.clone().requires_grad_(True)
    sg = layers.SSIM()(xg, yg)
    (sg * flow[:, :1].abs()).sum().backward()
    assert common.rel_max(restate.ssim(x, ref), sg) < 1e-5
    assert common.rel_max(xo.grad, xg.grad) < 1e-4 and common.rel_max(yo.grad, yg.grad) < 1e-4
    m = torch.rand(B, 1, h, w, generator=g).to(DEV)
    assert float(loss_utils.smooth_loss(x, m)) == pytest.approx(float(restate.smooth_loss(x, m)), rel=1e-5)
    assert torch.equal(utils.binary_image(m, 0.4), restate.binary_image(m, 0.4))
    a, b = utils.FlowWarp(B, h, w)(flow), restate.flow_warp_grid(flow)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


def test_native_library_is_what_ran():
    """Guards against a silent fallback: the in-tree .so must be mapped into this process."""
    from mdn_sfm_b200 import _cabi
    _cabi.lib()
    maps = open("/proc/self/maps").read()
    assert "libmdn_loss.so" in maps


@pytest.mark.gpu
def test_batch_stager_uploads_what_the_loader_wrote():
    """mdn_sfm_b200.staging.BatchStager: one pinned slab -> one copy; the device views equal the loader's tensors,
    are 256-byte aligned and feed Loss.forward unchanged (same loss as the per-key .to(device) upload)."""
    from mdn_sfm_b200.loss_functions import Loss
    from mdn_sfm_b200.staging import BatchStager
    opt, batch = common.make(2, 64, 96, seed=3)
    inputs, flows, mobiles, cams, inst = batch
    st = BatchStager([inputs, flows, mobiles, cams], DEV, n_buffers=2)
    for k in range(3):   # buffer 0 is reused on the third round
        st.fill(k, [inputs, flows, mobiles, cams])
        views = st.upload(k)
        st.wait(k)
        for src, dst in zip([inputs, flows, mobiles, cams], views):
            for key in src:
                assert dst[key].data_ptr() % 256 == 0 and dst[key].is_contiguous()
                assert torch.equal(dst[key].cpu(), src[key]), key
        st.release(k)
    loss = Loss(opt, no_ssim=False, mode="T", photometric=True)
    _, a = loss(views[0], [-1, 1], views[1], views[2], None, [0, 1, 2, 3], views[3])
    mv = lambda d: {k: v.to(DEV) for k, v in d.items()}
    _, b = loss(mv(inputs), [-1, 1], mv(flows), mv(mobiles), None, [0, 1, 2, 3], mv(cams))
    assert torch.equal(a["loss"], b["loss"])


@pytest.mark.gpu
@pytest.mark.parametrize("padding_mode", ["border", "reflection"])
def test_padding_modes_on_gpu(padding_mode):
    """grid_sample's other padding modes through Loss(padding_mode=...) (loss_functions.py:12,161) against the oracle run
    eagerly on the same GPU, flows large enough that a fifth of the samples leave the image; multi-tile shape, 4 scales."""
    opt, batch = common.make(2, 64, 192, seed=23, flow_std=0.3)
    ref = common.oracle_run(opt, batch, "TG", True, True, DEV, padding_mode=padding_mode)
    got = common.product_run(opt, batch, "TG", True, True, DEV, padding_mode=padding_mode)
    common.compare(ref, got, True)


@pytest.mark.gpu
def test_instance_mask_prep_on_gpu_matches_torchvision():
    """SURVEY 8f-N2: mdn_instance_mask_union + mdn_instance_mask_resize on the GPU == the reference's
    Resize(size)(get_batch_instance_mask(.)) (torchvision on the CPU, int64), all four pyramid levels from one pass,
    bit for bit except at exact 0.5 ties; B=12 KITTI-sized Detectron2-style masks (config 4's input)."""
    from test_emu_kernels import assert_masks_equal_up_to_exact_ties
    from mdn_sfm_b200 import loss_utils
    g = torch.Generator().manual_seed(5)
    inst = synthetic.make_instances(12, g)
    sizes = [(192, 640), (96, 320), (48, 160), (24, 80)]
    got = loss_utils.instance_masks_u8([{"instances": d["instances"].to(DEV)} for d in inst], sizes, DEV)
    assert all(m.is_cuda for m in got)
    assert_masks_equal_up_to_exact_ties(got, inst, sizes)
    # fused pass (bit-packed rows, no global temporary) == the two separable passes, bit for bit; so does a shape whose
    # smallest level falls back to the two passes (factor 47 > a block's 64 source rows)
    import os
    for szs in (sizes, [(192, 640), (8, 12)]):
        one = loss_utils.instance_masks_u8([{"instances": d["instances"].to(DEV)} for d in inst], szs, DEV)
        os.environ["MDN_RESIZE_TWO_PASS"] = "1"
        try:
            two = loss_utils.instance_masks_u8([{"instances": d["instances"].to(DEV)} for d in inst], szs, DEV)
        finally:
            del os.environ["MDN_RESIZE_TWO_PASS"]
        assert all(torch.equal(a, b) for a, b in zip(one, two))


@pytest.mark.gpu
def test_train_step_harness_runs_on_the_cuda_loss():
    """SURVEY 8f-N1: nets -> Loss (CUDA, TG mode) -> backward -> clip -> Adam; the loss falls over a few steps on a fixed
    batch, only the mobile decoder moves, pose / flow nets stay frozen."""
    from mdn_sfm_b200.train_step import StandInNets, TrainStep
    opt = synthetic.default_opt(2, 64, 96, threshold=0.8625)
    torch.manual_seed(0)
    ts = TrainStep(opt, nets=StandInNets(width=8), device=DEV, mode="TG", photometric=True, lr=1e-3)
    inputs, _, _, _, _ = synthetic.make_batch(2, 64, 96, seed=1, with_instances=False)
    inputs = {k: v.to(DEV) for k, v in inputs.items()}
    frozen = [p.detach().clone() for p in ts.nets.flownet.parameters()]
    first = float(ts.step(inputs)["loss"].detach())
    for _ in range(10):
        last = float(ts.step(inputs)["loss"].detach())
    assert last == last and last < first
    assert all(torch.equal(a, b) for a, b in zip(frozen, ts.nets.flownet.parameters()))


@pytest.mark.gpu
def test_image_pyramid_on_gpu_matches_torchvision():
    """SURVEY 8f-N3: the lower pyramid levels made on the GPU equal torchvision's Resize of the fp32 frame (CPU), and the
    loss on a device-made pyramid equals the loss on the dataset-made one to 1e-5."""
    from torchvision.transforms import Resize
    from mdn_sfm_b200 import pyramid
    from mdn_sfm_b200.loss_functions import Loss
    opt, batch = common.make(2, 192, 640, seed=8)
    inputs, flows, mobiles, cams, _ = batch
    img = inputs[("color", -1, 0)]
    got = pyramid.image_pyramid(img.to(DEV), [(96, 320), (48, 160), (24, 80)])
    for t, s in zip(got, [(96, 320), (48, 160), (24, 80)]):
        ref = Resize(s)(img)
        assert float((t.cpu() - ref).abs().max()) <= 2e-6 * float(ref.abs().max())
    mv = lambda d: {k: v.to(DEV) for k, v in d.items()}
    loss = Loss(opt, no_ssim=False, mode="T", photometric=True)
    a = loss(mv(inputs), [-1, 1], mv(flows), mv(mobiles), None, [0, 1, 2, 3], mv(cams))[1]["loss"]
    dev_in = {k: v.to(DEV) for k, v in inputs.items() if not (k[0] == "color" and k[2] != 0)}
    pyramid.add_pyramid_levels(dev_in, [0, -1, 1], [0, 1, 2, 3])
    b = loss(dev_in, [-1, 1], mv(flows), mv(mobiles), None, [0, 1, 2, 3], mv(cams))[1]["loss"]
    assert float(b) == pytest.approx(float(a), rel=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 6, 8), (1, 17, 20), (2, 16, 64), (1, 40, 132), (3, 21, 76), (1, 2, 4), (2, 19, 45), (1, 8, 9)])
def test_tma_staging_on_images_smaller_than_the_box(shape):
    """The TMA box (72 x 20) is larger than these images / their edge tiles: out-of-tensor elements must arrive as zeros and
    the reflected ring must be patched from inside the tile -- every mode family against the oracle on the same GPU."""
    B, H, W = shape
    for mode, photo in (("T", True), ("SN", True), ("TG", False)):
        if mode == "TG" and (H < 8 or W < 8):
            continue        # (the reference's Gaussian weight table needs at least 8 pixels over its 4 scales)
        opt, batch = common.make(B, H, W, scales=(0,), seed=31, flow_std=0.1)
        got = common.product_run(opt, batch, mode, photo, True, DEV, pose_grad=True)
        common.compare(common.oracle_run(opt, batch, mode, photo, True, DEV, pose_grad=True), got, photo)


@pytest.mark.gpu
def test_epipolar_statistics_on_gpu():
    """SURVEY 8f-N4 on the GPU (poses into the maps-only launch): quantiles of |e| == the oracle's compute_quantiles run on the
    same GPU, and the thresholds come out ordered."""
    from oracle import restate
    from mdn_sfm_b200 import layers, statistics
    opt, batch = common.make(4, 192, 640, scales=(0,), seed=19, flow_std=0.02)
    inputs, flows, _, cams, _ = batch
    mv = lambda d: {k: v.to(DEV) for k, v in d.items()}
    inputs, flows, cams = mv(inputs), mv(flows), mv(cams)
    B, h, w = 4, 192, 640
    st = statistics.EpipolarStatistics(num_quantile=100)
    st.update(flows, inputs[("inv_K", 0)], cams)
    per, thr = st.result()
    pix = restate.create_coords(B, h, w, DEV)
    ones = torch.ones(B, 1, h, w, device=DEV)
    p1 = torch.cat([pix, ones], 1).view(B, 3, -1)
    q = torch.linspace(0, 1, 100, device=DEV)
    sf = layers.get_scale_factor(B, h, w).to(DEV)
    for k, i in enumerate((-1, 1)):
        ref = restate.compute_quantiles(flows, cams[i], inputs[("inv_K", 0)], p1, pix, ones, sf, q, i, B).cpu()
        assert float((torch.from_numpy(per[k]) - ref).abs().max()) <= 1e-5 * float(ref.abs().max()), i
    assert (thr[1:] >= thr[:-1]).all()


@pytest.mark.gpu
def test_packed_source_pyramid_on_gpu():
    """SURVEY 8f-N3, second half, on the GPU at configs[0]'s shape: ('color_packed', i, s) sources == NCHW sources bit for
    bit (the call's own repack is skipped), and the packed pyramid equals torchvision's Resize of the fp32 frame."""
    from torchvision.transforms import Resize
    from mdn_sfm_b200 import pyramid
    opt, batch = common.make(4, 192, 640, seed=29)
    inputs, flows, mobiles, cams, _ = batch
    a = common.product_run(opt, batch, "T", True, True, DEV, pose_grad=True)
    packed = {k: v for k, v in inputs.items()}
    for i in (-1, 1):
        for s in range(4):
            lvl = packed.pop(("color", i, s)).to(DEV)
            packed[("color_packed", i, s)] = pyramid.image_pyramid(lvl, [tuple(lvl.shape[-2:])], packed=True)[0]
    b = common.product_run(opt, (packed, flows, mobiles, cams, None), "T", True, True, DEV, pose_grad=True)
    common.assert_identical_runs(a, b, maps=("epipolars", "epipolar_ori", "warps", "diffs"))
    sizes = [(192, 640), (96, 320), (48, 160), (24, 80)]
    pk = pyramid.image_pyramid(inputs[("color", 1, 0)].to(DEV), sizes, packed=True)
    for t, sz in zip(pk, sizes):
        ref = Resize(sz)(inputs[("color", 1, 0)]).permute(0, 2, 3, 1)
        assert float((t[..., :3].cpu() - ref).abs().max()) <= 2e-6 * float(ref.abs().max())


@pytest.mark.gpu
def test_graphed_loss_step_replays_on_refreshed_inputs():
    """mdn_sfm_b200.graphs.GraphedLossStep: the captured forward + backward, replayed after the static tensors were
    refreshed in place, equals the eager step on the same values bit for bit (losses and every gradient)."""
    from mdn_sfm_b200.graphs import GraphedLossStep
    from mdn_sfm_b200.loss_functions import Loss
    opt, b1 = common.make(2, 64, 128, seed=3)
    _, b2 = common.make(2, 64, 128, seed=4)
    dev = lambda d, g=False: {k: v.to(DEV).requires_grad_(g) for k, v in d.items()}
    inputs, flows, mobiles, cams = dev(b1[0]), dev(b1[1], True), dev(b1[2], True), dev(b1[3], True)
    loss = Loss(opt, no_ssim=False, mode="TG", photometric=True)
    step = GraphedLossStep(loss, inputs, [-1, 1], flows, mobiles, None, [0, 1, 2, 3], cams)
    with torch.no_grad():        # refresh every static tensor with the second batch
        for dst, src in ((inputs, b2[0]), (flows, b2[1]), (mobiles, b2[2]), (cams, b2[3])):
            for k in dst:
                dst[k].copy_(src[k])
    got = step.replay()
    ref = common.product_run(opt, b2, "TG", True, True, DEV, pose_grad=True)
    assert torch.equal(got["loss"], ref[1]["loss"].detach())
    for mine, theirs in ((flows, ref[2]), (mobiles, ref[3]), (cams, ref[4])):
        for k in mine:
            assert torch.equal(mine[k].grad, theirs[k].grad), k


@pytest.mark.gpu
def test_uint8_frames_on_gpu_equal_the_dataset_transforms():
    """mdn_normalize_u8 on the GPU == ArrayToTensor + Normalize of the reference's dataset run on the CPU, bit for bit."""
    from mdn_sfm_b200 import pyramid
    g = torch.Generator().manual_seed(2)
    u8 = torch.randint(0, 256, (3, 192, 640, 3), dtype=torch.uint8, generator=g)
    ref = u8.permute(0, 3, 1, 2).float() / 255
    for t, m, s in zip(ref.unbind(1), (0.45, 0.45, 0.45), (0.225, 0.225, 0.225)):
        t.sub_(m).div_(s)
    assert torch.equal(pyramid.frames_from_u8(u8.to(DEV)).cpu(), ref.contiguous())


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_second_device_in_the_same_process():
    """The loss launched on cuda:1 while cuda:0 is current (and after cuda:0 was used) equals the cuda:0 result."""
    opt, batch = common.make(2, 64, 128, seed=5)
    a = common.product_run(opt, batch, "T", True, True, "cuda:0", pose_grad=True)
    b = common.product_run(opt, batch, "T", True, True, "cuda:1", pose_grad=True)
    assert torch.equal(a[1]["loss"].cpu(), b[1]["loss"].cpu())
    for k in a[2]:
        assert torch.equal(a[2][k].grad.cpu(), b[2][k].grad.cpu()), k
