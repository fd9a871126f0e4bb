"""-m gpu: flow evaluation (mdn_flow_errors, metrics.FlowMetrics) on the device at B = 12 -- counts and EPE sums against
the replay of the per-pixel arithmetic (flow_replay.py) on the same GPU, against the natural torch composition
(F.interpolate + the same formulas) within that function's rounding, FlowMetrics.update replayed from a CUDA graph
against eager updates, and run-to-run identity."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from flow_replay import reduce, replay, sqrt_rn, upsample
from mdn_sfm_b200 import metrics

pytestmark = pytest.mark.gpu
DEV = "cuda"
CONFIGS = [(192, 640, 375, 1242), (375, 1242, 375, 1242), (192, 640, 370, 1224)]
IDS = ["192x640-375x1242", "375x1242-same", "192x640-370x1224"]


def make(B, h, w, H, W, seed, R):
    """Normalized flow; ground truth = its up-sampled pixels + mixed noise with 10-40 % outliers per image, about 30 %
    valid, and pixels placed on the abs (e = 3) and rel (e / m = 0.05) boundaries -- only where the replay's up-sampling
    and F.interpolate agree bit for bit, so that the boundary pixels cannot flip between the two."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    flow = torch.randn(B, 2, h, w, generator=g, device=DEV) * 0.04
    sx, sy = metrics._flow_scale("normalized", h, w, H, W)
    f = upsample(flow, H, W)
    agree = (F.interpolate(flow, size=(H, W), mode="bilinear", align_corners=False) == f).all(1)
    u, v = f[:, 0] * torch.tensor(sx, device=DEV), f[:, 1] * torch.tensor(sy, device=DEV)
    p_out = torch.linspace(0.1, 0.4, B, device=DEV).view(B, 1, 1)
    big = torch.rand(B, H, W, generator=g, device=DEV) < p_out
    noise = torch.randn(B, 2, H, W, generator=g, device=DEV) * torch.where(big, 20.0, 0.8)[:, None]
    gu, gv = u + noise[:, 0], v + noise[:, 1]
    pick = torch.rand(B, H, W, generator=g, device=DEV)
    on_abs = agree & (pick < 0.004)
    gu, gv = torch.where(on_abs, u - 3.0, gu), torch.where(on_abs, v, gv)
    k = 1.0 / 1.05          # gt = k (u, v): e / m = (1 - k) / k = 0.05, and e > 3 where |(u, v)| > 63
    on_rel = agree & (pick >= 0.004) & (pick < 0.03) & (u * u + v * v > 70.0 ** 2)
    gu = torch.where(on_rel, (u.double() * k).float(), gu)
    gv = torch.where(on_rel, (v.double() * k).float(), gv)
    valid = torch.rand(B, H, W, generator=g, device=DEV) < 0.3
    gt = torch.stack([gu, gv], 1)
    gt = torch.where(valid[:, None], gt, torch.full_like(gt, float("nan")))      # loaders that store NaN there
    region = torch.randint(0, R + 1, (B, H, W), generator=g, device=DEV, dtype=torch.uint8) if R > 1 else None
    return flow.contiguous(), gt.contiguous(), valid, region, (sx, sy)


@pytest.mark.parametrize("R", [1, 4])
@pytest.mark.parametrize("h,w,H,W", CONFIGS, ids=IDS)
def test_counts_and_sums_equal_the_replay(h, w, H, W, R):
    flow, gt, valid, region, scale = make(12, h, w, H, W, seed=h + H + R, R=R)
    got = metrics.flow_errors(flow, gt, valid, units="normalized", region=region, n_regions=R)
    want = replay(flow, gt, valid, region, R, scale, 3.0, 0.05, pixels=True)
    assert torch.equal(got["valid"], want["valid"]) and torch.equal(got["outliers"], want["outliers"])
    assert np.allclose(got["epe_sum"].cpu().numpy(), want["epe_sum"].cpu().numpy(), rtol=1e-12, atol=0, equal_nan=True)
    fl = got["outliers"].sum(-1).double() / got["valid"].sum(-1).double()
    assert 0.05 < float(fl.min()) and float(fl.max()) < 0.5
    # the boundaries are exercised: counted pixels with e exactly 3 and with e / m exactly rel_thr
    e = want["e"]
    ratio = e / sqrt_rn(gt[:, 0] * gt[:, 0] + gt[:, 1] * gt[:, 1])
    assert int((valid & (e == 3.0)).sum()) > 0
    assert int((valid & (ratio == torch.tensor(0.05, device=DEV)) & (e > 3)).sum()) > 0


@pytest.mark.parametrize("R", [1, 4])
@pytest.mark.parametrize("h,w,H,W", CONFIGS, ids=IDS)
def test_against_the_natural_torch_composition(h, w, H, W, R):
    flow, gt, valid, region, (sx, sy) = make(12, h, w, H, W, seed=7 * h + H + R, R=R)
    got = metrics.flow_errors(flow, gt, valid, units="normalized", region=region, n_regions=R)
    up = F.interpolate(flow, size=(H, W), mode="bilinear", align_corners=False)
    scaled = up * torch.tensor([float(sx), float(sy)], device=DEV).view(1, 2, 1, 1)
    du, dv = scaled[:, 0] - gt[:, 0], scaled[:, 1] - gt[:, 1]
    e = torch.sqrt(du * du + dv * dv)
    m = torch.sqrt(gt[:, 0] * gt[:, 0] + gt[:, 1] * gt[:, 1])
    out = (e > 3.0) & (e / m > 0.05)
    comp = reduce(e, out, valid, region, R)
    assert torch.equal(got["valid"], comp["valid"])
    assert np.allclose(got["epe_sum"].cpu().numpy(), comp["epe_sum"].cpu().numpy(), rtol=1e-5, atol=0)
    rep = replay(flow, gt, valid, region, R, (sx, sy), 3.0, 0.05, pixels=True)
    counted = valid & ((region.long() < R) if region is not None else True)
    flipped = counted & (rep["out"] != out)
    same_up = (rep["f"] == up).all(1)
    assert not bool((flipped & same_up).any()), "an outlier flag differs where the two up-samplings agree"
    assert int(flipped.sum()) <= 1e-5 * int(counted.sum())
    # the kernel's outliers are the replay's, not the composition's
    assert torch.equal(got["outliers"], rep["outliers"])


def test_update_replayed_from_a_cuda_graph_equals_eager_updates():
    batches = [make(12, 192, 640, 375, 1242, seed=s, R=3)[:4] for s in range(3)]
    graphed = metrics.FlowMetrics(3, DEV, units="normalized")
    static = [torch.empty_like(t) for t in batches[0]]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):            # warm-up: caches the workspace of this shape
        for s, t in zip(static, batches[0]):
            s.copy_(t)
        graphed.update(*static)
    torch.cuda.current_stream().wait_stream(side)
    graphed.reset()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.update(*static)
    for b in batches:
        for s, t in zip(static, b):
            s.copy_(t)
        graph.replay()
    eager = metrics.FlowMetrics(3, DEV, units="normalized")
    for b in batches:
        eager.update(*b)
    a, c = graphed.compute(), eager.compute()
    assert a["images"] == c["images"] == 36
    for k in ("valid", "outliers", "defined", "epe_sum"):
        assert np.array_equal(a[k], c[k]), k
    for agg in ("pooled", "per_image"):
        for k in ("epe", "fl"):
            assert np.array_equal(a[agg][k], c[agg][k], equal_nan=True), (agg, k)
    assert a["valid"][3] == a["valid"][:3].sum() and a["valid"][3] > 0


def test_identical_over_two_runs():
    flow, gt, valid, region, _ = make(12, 192, 640, 375, 1242, seed=9, R=8)
    runs = []
    for _ in range(2):
        m = metrics.FlowMetrics(8, DEV, units="normalized")
        errs = m.update(flow, gt, valid, region)
        runs.append(({k: v.clone() for k, v in errs.items()}, m.compute()))
    for k in ("valid", "outliers", "epe_sum"):
        assert torch.equal(runs[0][0][k], runs[1][0][k]), k
    for k in ("valid", "outliers", "defined", "epe_sum"):
        assert np.array_equal(runs[0][1][k], runs[1][1][k]), k
