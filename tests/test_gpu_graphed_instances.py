"""-m gpu: DS / DC loss steps replayed from ONE CUDA graph while the Detectron2 instances change every batch
(graphs.GraphedLoss + loss_utils.InstanceMaskTable + mdn_instance_mask_union_table), bit for bit against the eager Loss."""
import pytest
import torch

from mdn_sfm_b200 import synthetic
from mdn_sfm_b200.graphs import GraphedLoss
from mdn_sfm_b200.layers import PoseParameters
from mdn_sfm_b200.loss_functions import Loss

pytestmark = pytest.mark.gpu
DEV = "cuda"
TERMS = ("loss", "epip", "smooth", "consis", "photo")


def _instances(counts, H=375, W=1242, seed=0):
    """Detectron2-style masks (speckle plus a filled box per instance), counts[b] of them for sample b, on the GPU."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for n in counts:
        m = torch.rand(n, H, W, generator=g) > 0.95
        for k in range(n):
            y0, x0 = int(torch.randint(0, H // 2, (1,), generator=g)), int(torch.randint(0, W // 2, (1,), generator=g))
            m[k, y0:y0 + H // 5, x0:x0 + W // 6] = True
        out.append({"instances": synthetic.SyntheticInstances(m.to(DEV))})
    return out


def _batch(B, H, W, scales, seed):
    inputs, flows, mobiles, _, _ = synthetic.make_batch(B, H, W, scales=scales, seed=seed, flow_std=0.05, with_instances=False,
                                                        device=DEV)
    g = torch.Generator().manual_seed(seed)
    poses = {i: (0.02 * torch.randn(B, 1, 1, 3, generator=g), torch.randn(B, 1, 1, 3, generator=g) * 0.3) for i in (-1, 1)}
    return inputs, flows, mobiles, {i: (a.to(DEV), t.to(DEV)) for i, (a, t) in poses.items()}


def _run(loss, batch, inst, scales):
    inputs, flows, mobiles, poses = batch
    leaf = lambda t: t.detach().clone().requires_grad_(True)
    f = {k: leaf(v) for k, v in flows.items()}
    m = {k: leaf(v) for k, v in mobiles.items()}
    p = {k: PoseParameters(leaf(a), leaf(t)) for k, (a, t) in poses.items()}
    _, losses = loss(inputs, [-1, 1], f, m, inst, list(scales), p)
    losses["loss"].backward()
    grads = [t.grad for d in (f, m) for t in d.values()] + [t.grad for c in p.values() for t in (c.axisangle, c.translation)]
    return losses, grads


def _assert_same(eager, graphed, what):
    (le, ge), (lg, gg) = eager, graphed
    for k in TERMS:
        if k in le:
            assert torch.equal(torch.as_tensor(le[k]).detach(), torch.as_tensor(lg[k]).detach()), (what, k, float(le[k]), float(lg[k]))
    assert len(ge) == len(gg)
    for n, (a, b) in enumerate(zip(ge, gg)):
        assert a is not None and torch.equal(a, b), (what, "gradient", n)


def _pair(mode, B, H, W, scales):
    opt = synthetic.default_opt(B, H, W, scales=list(scales))
    return Loss(opt, no_ssim=False, mode=mode, photometric=True), GraphedLoss(Loss(opt, no_ssim=False, mode=mode, photometric=True))


@pytest.mark.parametrize("mode", ["DS", "DC"])
def test_new_instances_every_call_replay_one_capture(mode):
    """Four calls at B = 4, 192 x 640, 4 scales, with other instance counts per sample every call (zeros included):
    each equals the eager Loss bit for bit (total, four terms, every gradient), and all four run from the first capture."""
    scales = (0, 1, 2, 3)
    eager, graphed = _pair(mode, 4, 192, 640, scales)
    step = None
    for n, counts in enumerate(([3, 1, 0, 2], [1, 5, 2, 0], [0, 0, 0, 0], [2, 2, 2, 2])):
        batch, inst = _batch(4, 192, 640, scales, seed=10 + n), _instances(counts, seed=n)
        _assert_same(_run(eager, batch, inst, scales), _run(graphed, batch, inst, scales), (mode, counts))
        step = step or graphed.step
        assert graphed.step is step, "recaptured at call %d" % n


def test_a_new_mask_size_recaptures():
    """Masks of another frame size (another KITTI raw resolution) capture a new graph; the results stay equal to eager."""
    scales = (0, 1)
    eager, graphed = _pair("DC", 2, 96, 320, scales)
    steps = []
    for n, (hw, counts) in enumerate((((375, 1242), [2, 1]), ((370, 1224), [0, 3]), ((370, 1224), [1, 1]))):
        batch, inst = _batch(2, 96, 320, scales, seed=30 + n), _instances(counts, *hw, seed=20 + n)
        _assert_same(_run(eager, batch, inst, scales), _run(graphed, batch, inst, scales), (hw, counts))
        steps.append(graphed.step)
    assert steps[1] is not steps[0] and steps[2] is steps[1]


@pytest.mark.parametrize("mode", ["DS", "DC"])
def test_bare_instances_equal_the_eager_broadcast(mode):
    """One bare Instances (trainer.py:494, evaluate_mix.py:63) masks every sample, as the eager (1, 3, H, W) broadcast does."""
    scales = (0, 1, 2)
    eager, graphed = _pair(mode, 3, 64, 160, scales)
    for n, count in enumerate((2, 0, 4)):
        batch, bare = _batch(3, 64, 160, scales, seed=40 + n), _instances([count], seed=40 + n)[0]["instances"]
        _assert_same(_run(eager, batch, bare, scales), _run(graphed, batch, bare, scales), (mode, count))
    assert graphed.step is not None


def _train_step_builder(mode):
    from mdn_sfm_b200.train_step import StandInNets, TrainStep
    B, H, W = 2, 64, 96
    opt = synthetic.default_opt(B, H, W, threshold=0.8625)
    inputs, _, _, _, _ = synthetic.make_batch(B, H, W, seed=1, with_instances=False, device=DEV)

    def build(**kw):
        torch.manual_seed(0)
        nets = StandInNets(width=8)
        with torch.no_grad():      # KITTI-like pose magnitudes, as the TG train-step test sets them
            nets.posenet.head.weight.mul_(40.0)
            nets.posenet.head.bias.add_(torch.tensor([0.3, -0.2, 0.5, 4.0, -6.0, 9.0]))
        return TrainStep(opt, nets=nets, device=DEV, lr=1e-3, mode=mode, photometric=False, **kw)

    return inputs, build


@pytest.mark.parametrize("mode", ["DC", "DS"])
def test_graphed_train_step_with_new_instances_equals_the_eager_one(mode):
    """TrainStep with graph_loss=True against graph_loss=False (HEAD's DC mode: no photometric term; and DS): three steps, a
    different instance set each time, leave the nets with bit-identical parameters, and the graphed loss never recaptures."""
    det, bench_ = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False     # (the nets' cuDNN kernels, not ours)
    try:
        inputs, build = _train_step_builder(mode)
        inputs2 = {k: (v.flip(0) if k[0] == "color" else v) for k, v in inputs.items()}
        ts_a, ts_b = build(graph_loss=True), build(graph_loss=False)
        assert isinstance(ts_a.loss, GraphedLoss) and not isinstance(ts_b.loss, GraphedLoss)
        step = None
        for n, (batch, counts) in enumerate(((inputs, [2, 1]), (inputs2, [0, 4]), (inputs, [3, 0]))):
            inst = _instances(counts, seed=50 + n)
            la, lb = ts_a.step(batch, inst), ts_b.step(batch, inst)
            assert torch.equal(la["loss"].detach(), lb["loss"].detach()), (n, float(la["loss"]), float(lb["loss"]))
            step = step or ts_a.loss.step
            assert ts_a.loss.step is step
        for (n, a), (_, b) in zip(ts_a.nets.named_parameters(), ts_b.nets.named_parameters()):
            assert torch.equal(a, b), n
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = det, bench_
