"""-m gpu: mask evaluation (mdn_mask_confusion, metrics.MaskMetrics) on the device -- the counts against a torch oracle on
the same GPU at the evaluation shapes, MaskMetrics.update replayed from a CUDA graph against eager updates, and
run-to-run identity."""
import numpy as np
import pytest
import torch

from mdn_sfm_b200 import metrics

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHAPES = [(375, 1242), (192, 640)]


def torch_confusion(pred, gt, thr):
    """bucketize(right=True) gives j = #{k : thr[k] <= pred}; one bincount over (sample, label, j) keys; suffix sums.
    NaN-free inputs only (bucketize puts NaN in the last bin)."""
    B, K = pred.shape[0], thr.numel()
    j = torch.bucketize(pred.reshape(B, -1), thr, right=True)
    key = j + (gt.reshape(B, -1) != 0).long() * (K + 1) + torch.arange(B, device=pred.device)[:, None] * (2 * (K + 1))
    h = torch.bincount(key.reshape(-1), minlength=B * 2 * (K + 1)).view(B, 2, K + 1)
    s = h.flip(-1).cumsum(-1).flip(-1)                     # s[..., j] = pixels in bins >= j
    tp, fp = s[:, 1, 1:], s[:, 0, 1:]
    return torch.stack([tp, fp, s[:, 1, :1] - tp, s[:, 0, :1] - fp], -1)


def direct_confusion(pred, gt, thr):
    """(pred >= thr) & label counted image by image: NaN-correct."""
    out = []
    for p, g in zip(pred, gt):
        m = p.reshape(-1, 1) >= thr.reshape(1, -1)
        lab = (g.reshape(-1, 1) != 0)
        out.append(torch.stack([(m & lab).sum(0), (m & ~lab).sum(0), (~m & lab).sum(0), (~m & ~lab).sum(0)], -1))
    return torch.stack(out)


def make(B, H, W, kind, seed, thr=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    if kind == "skewed":      # a mobile map: a sigmoid of mostly very negative logits, so most pixels lie near 0
        pred = torch.sigmoid(torch.randn(B, 1, H, W, generator=g, device=DEV) * 1.5 - 4.0)
    else:
        pred = torch.rand(B, 1, H, W, generator=g, device=DEV)
    if thr is not None:       # 2 % of the pixels exactly on a threshold
        hit = torch.rand(B, 1, H, W, generator=g, device=DEV) < 0.02
        idx = torch.randint(0, thr.numel(), (B, 1, H, W), generator=g, device=DEV)
        pred = torch.where(hit, thr[idx], pred)
    gt = torch.rand(B, H, W, generator=g, device=DEV) < 0.15
    return pred.contiguous(), gt


@pytest.mark.parametrize("kind", ["skewed", "uniform"])
@pytest.mark.parametrize("K", [101, 1024])
@pytest.mark.parametrize("H,W", SHAPES, ids=["375x1242", "192x640"])
def test_counts_equal_the_torch_composition(H, W, K, kind):
    thr = torch.linspace(0, 1, K, device=DEV)
    pred, gt = make(12, H, W, kind, seed=H + K, thr=thr)
    got = metrics.mask_confusion(pred, gt, thr)
    want = torch_confusion(pred, gt, thr)
    assert torch.equal(got.sum(-1), torch.full_like(got[..., 0], H * W))
    assert torch.equal(got, want)
    # the same as uint8 labels with arbitrary non-zero values
    gt8 = gt.to(torch.uint8) * torch.randint(1, 256, gt.shape, device=DEV, dtype=torch.uint8)
    assert torch.equal(metrics.mask_confusion(pred, gt8, thr), want)


def test_nan_and_infinities_against_the_direct_comparison():
    thr = torch.cat([torch.tensor([-float("inf")]), torch.linspace(0, 1, 99), torch.tensor([float("inf")])]).to(DEV)
    pred, gt = make(12, 192, 640, "skewed", seed=5, thr=thr)
    g = torch.Generator(device=DEV).manual_seed(6)
    r = torch.rand(pred.shape, generator=g, device=DEV)
    pred = torch.where(r < 0.01, torch.full_like(pred, float("nan")), pred)
    pred = torch.where((r >= 0.01) & (r < 0.02), torch.full_like(pred, float("inf")), pred)
    pred = torch.where((r >= 0.02) & (r < 0.03), torch.full_like(pred, -float("inf")), pred)
    pred = torch.where((r >= 0.03) & (r < 0.04), torch.full_like(pred, -0.0), pred)
    got = metrics.mask_confusion(pred, gt, thr)
    assert torch.equal(got, direct_confusion(pred, gt, thr))
    assert torch.equal(got.sum(-1), torch.full_like(got[..., 0], 192 * 640))


def test_update_replayed_from_a_cuda_graph_equals_eager_updates():
    thr = torch.linspace(0, 1, 101)
    batches = [make(12, 375, 1242, kind, seed=s) for s, kind in enumerate(("skewed", "uniform", "skewed"))]
    graphed = metrics.MaskMetrics(thr, DEV)
    static_pred, static_gt = torch.empty_like(batches[0][0]), torch.empty_like(batches[0][1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):            # warm-up: caches the workspace of this batch size
        static_pred.copy_(batches[0][0]); static_gt.copy_(batches[0][1])
        graphed.update(static_pred, static_gt)
    torch.cuda.current_stream().wait_stream(side)
    graphed.reset()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.update(static_pred, static_gt)
    for p, g in batches:
        static_pred.copy_(p); static_gt.copy_(g)
        graph.replay()
    eager = metrics.MaskMetrics(thr, DEV)
    for p, g in batches:
        eager.update(p, g)
    a, b = graphed.compute(), eager.compute()
    assert a["images"] == b["images"] == 36 and np.array_equal(a["counts"], b["counts"])
    for agg in ("pooled", "per_image", "defined"):
        for k in metrics.METRICS:
            assert np.array_equal(a[agg][k], b[agg][k], equal_nan=True), (agg, k)
    want = sum(torch_confusion(p, g, graphed._thr).sum(0) for p, g in batches)
    assert np.array_equal(a["counts"], want.cpu().numpy())


def test_identical_over_two_runs():
    thr = torch.linspace(0, 1, 1024, device=DEV)
    pred, gt = make(12, 375, 1242, "skewed", seed=9, thr=thr)
    runs = []
    for _ in range(2):
        m = metrics.MaskMetrics(thr, DEV)
        counts = m.update(pred, gt)
        runs.append((counts.clone(), m.compute()))
    assert torch.equal(runs[0][0], runs[1][0])
    for agg in ("pooled", "per_image", "defined"):
        for k in metrics.METRICS:
            assert np.array_equal(runs[0][1][agg][k], runs[1][1][agg][k], equal_nan=True), (agg, k)
