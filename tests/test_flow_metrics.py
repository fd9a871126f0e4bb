"""Flow evaluation (mdn_sfm_b200.metrics.flow_errors / FlowMetrics, mdn_flow_errors) under the SIMT emulator: counts and
EPE sums against the torch replay of the per-pixel arithmetic (flow_replay.py) over up-, down- and same-size resizes,
every sample alignment and region count; special values and one hand-checked image; the metrics and both aggregations
against a float64 numpy restatement; the Python checks, the entry point's error codes in the real library (no GPU
needed) and a two-rank all_reduce over gloo."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from emu_harness import emu_library, emulated
from flow_replay import replay, upsample
from mdn_sfm_b200 import metrics

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INF, NAN = float("inf"), float("nan")


def make(B, h, w, H, W, seed, R=1, units="pixels", p_valid=0.6, junk=True):
    """A prediction, ground truth = its up-sampled pixels + mixed noise (a share of outliers, a few pixels within an ulp or
    so of e = 3), validity, labels 0 .. R+1 (some >= R) and 255.  Invalid pixels hold 0, NaN or inf when `junk`."""
    g = torch.Generator().manual_seed(seed)
    flow = torch.randn(B, 2, h, w, generator=g) * (0.02 if units == "normalized" else 4.0)
    sx, sy = metrics._flow_scale(units, h, w, H, W)
    f = upsample(flow, H, W)
    u, v = f[:, 0] * torch.tensor(sx), f[:, 1] * torch.tensor(sy)
    big = torch.rand(B, H, W, generator=g) < 0.25
    noise = torch.randn(B, 2, H, W, generator=g) * torch.where(big, 12.0, 0.8)[:, None]
    gt = torch.stack([u, v], 1) + noise
    edge = torch.rand(B, H, W, generator=g) < 0.05             # e = 3 up to the rounding of u - 3
    gt[:, 0] = torch.where(edge, u - 3.0, gt[:, 0])
    gt[:, 1] = torch.where(edge, v, gt[:, 1])
    valid = torch.rand(B, H, W, generator=g) < p_valid
    if junk:
        pick = torch.randint(0, 3, (B, 2, H, W), generator=g)
        bad = torch.tensor([0.0, NAN, INF])[pick]
        gt = torch.where(valid[:, None], gt, bad)
    region = torch.randint(0, R + 2, (B, H, W), generator=g, dtype=torch.uint8)
    region = torch.where(torch.rand(B, H, W, generator=g) < 0.05, torch.full_like(region, 255), region)
    return flow.contiguous(), gt.contiguous(), valid, region


def run(flow, gt, valid, region=None, R=1, units="pixels", abs_thr=3.0, rel_thr=0.05):
    with emulated() as lib:
        return metrics.flow_errors(flow, gt, valid, units=units, region=region, n_regions=R, abs_thr=abs_thr,
                                   rel_thr=rel_thr, library=lib)


def check(flow, gt, valid, region=None, R=1, units="pixels", abs_thr=3.0, rel_thr=0.05):
    """flow_errors under the emulator held to the replay: counts equal, epe_sum to rtol 1e-12 (NaN == NaN)."""
    got = run(flow, gt, valid, region, R, units, abs_thr, rel_thr)
    scale = metrics._flow_scale(units, flow.shape[-2], flow.shape[-1], gt.shape[-2], gt.shape[-1])
    want = replay(flow, gt, valid, region, R, scale, abs_thr, rel_thr)
    B = flow.shape[0]
    assert got["valid"].dtype == got["outliers"].dtype == torch.int64 and got["epe_sum"].dtype == torch.float64
    assert got["valid"].shape == got["outliers"].shape == got["epe_sum"].shape == (B, R)
    assert torch.equal(got["valid"], want["valid"])
    assert torch.equal(got["outliers"], want["outliers"])
    assert np.allclose(got["epe_sum"].numpy(), want["epe_sum"].numpy(), rtol=1e-12, atol=0, equal_nan=True)
    return got


@pytest.mark.parametrize("h,w,H,W", [(9, 13, 9, 13), (6, 10, 12, 20), (12, 40, 23, 77), (23, 41, 10, 17),
                                     (1, 1, 5, 7), (1, 9, 4, 9), (7, 1, 7, 5), (3, 4, 1, 1)],
                         ids=["same", "x2", "12x40-23x77", "down", "h=w=1", "h=1", "w=1", "to-1x1"])
@pytest.mark.parametrize("units", ["pixels", "normalized"])
def test_counts_and_sums_over_resizes(h, w, H, W, units):
    flow, gt, valid, region = make(3, h, w, H, W, seed=h * 100 + W, R=2, units=units)
    check(flow, gt, valid, region, R=2, units=units)


@pytest.mark.parametrize("H,W", [(4, 6), (5, 5), (3, 10), (3, 9), (1, 3), (1, 1)],
                         ids=["HW%4==0", "HW%4==1", "HW%4==2", "HW%4==3", "HW=3", "HW=1"])
def test_every_sample_alignment(H, W):
    """B = 5 samples back to back: with H*W % 4 != 0 the samples start at every offset mod 4, so the scalar head, the
    vector body with every gt_flow plane offset, and the scalar tail all run."""
    flow, gt, valid, region = make(5, 3, 4, H, W, seed=H * W, R=2)
    check(flow, gt, valid, region, R=2)


@pytest.mark.parametrize("R", [1, 2, 3, 8])
def test_region_counts_and_ignored_labels(R):
    flow, gt, valid, region = make(4, 7, 11, 13, 29, seed=R, R=R)
    assert (region >= R).any() and (region == 255).any()
    got = check(flow, gt, valid, region, R=R)
    assert int(got["valid"].sum()) < int(valid.sum())              # labels >= R are not counted


def test_region_none_is_region_zero():
    flow, gt, valid, _ = make(3, 8, 12, 15, 22, seed=4)
    a = check(flow, gt, valid, None, R=1)
    b = check(flow, gt, valid, torch.zeros(3, 15, 22, dtype=torch.uint8), R=1)
    assert torch.equal(a["valid"], b["valid"]) and torch.equal(a["outliers"], b["outliers"])
    assert torch.equal(a["epe_sum"], b["epe_sum"])
    assert torch.equal(a["valid"][:, 0], valid.reshape(3, -1).sum(1))


def test_kitti_size():
    flow, gt, valid, region = make(2, 192, 640, 375, 1242, seed=11, R=2, units="normalized", p_valid=0.3)
    got = check(flow, gt, valid, region, R=2, units="normalized")
    assert int(got["outliers"].sum()) > 0.05 * int(got["valid"].sum())


def test_invalid_ground_truth_never_reaches_a_sum():
    """The same inputs with 0, NaN or +-inf in the invalid pixels' ground truth give identical outputs, bit for bit."""
    flow, gt, valid, region = make(3, 9, 14, 17, 30, seed=21, R=2, junk=False)
    outs = []
    for fill in (0.0, NAN, INF, -INF):
        g = torch.where(valid[:, None], gt, torch.full_like(gt, fill))
        outs.append(check(flow, g, valid, region, R=2))
    for o in outs[1:]:
        for k in ("valid", "outliers", "epe_sum"):
            assert torch.equal(o[k], outs[0][k]), k
    assert torch.isfinite(outs[0]["epe_sum"]).all()


def test_nan_prediction_reaches_epe_but_is_never_an_outlier():
    flow, gt, valid, _ = make(2, 6, 8, 6, 8, seed=22, junk=False)
    valid[:] = True
    flow[0, 0, 2, 3] = NAN
    got = check(flow, gt, valid)
    assert torch.isnan(got["epe_sum"][0, 0]) and torch.isfinite(got["epe_sum"][1, 0])
    # the NaN pixels themselves: counted, not outliers
    only = torch.zeros_like(valid)
    only[0, 2, 3] = True
    one = check(flow, gt, only)
    assert one["valid"][0, 0] == 1 and one["outliers"][0, 0] == 0 and torch.isnan(one["epe_sum"][0, 0])


def hand_image():
    """One 2 x 4 image at its own size in pixels (the up-sampling is the identity, scale 1):
    p0 gt (3, 0), pred 0          e = 3 exactly: not an outlier (e > 3 is false)          region 0
    p1 gt (nextafter(3), 0)       e = 3.0000002, ratio 1: outlier                         region 0
    p2 gt (0, 0), pred (4, 0)     e = 4, m = 0, ratio inf: outlier                        region 0
    p3 gt (80, 0), pred (84, 0)   e = 4, ratio fl(4 / 80) = fl(0.05) = rel_thr: not        region 1
    p4 invalid, gt NaN                                                                  region 0
    p5 gt (0, 0), pred 0          e = 0, m = 0, ratio NaN: not                             region 1
    p6 valid, label 255           ignored                                               (255)
    p7 gt (-6, 8), pred 0         e = 10, ratio 1: outlier                                region 1"""
    flow = torch.zeros(1, 2, 2, 4)
    flow[0, 0, 0, 2], flow[0, 0, 0, 3] = 4.0, 84.0
    n3 = float(np.nextafter(np.float32(3), np.float32(np.inf)))
    gu = torch.tensor([[3.0, n3, 0.0, 80.0], [NAN, 0.0, 100.0, -6.0]])
    gv = torch.tensor([[0.0, 0.0, 0.0, 0.0], [NAN, 0.0, 0.0, 8.0]])
    valid = torch.tensor([[[1, 1, 1, 1], [0, 1, 1, 1]]], dtype=torch.uint8)
    region = torch.tensor([[[0, 0, 0, 1], [0, 1, 255, 1]]], dtype=torch.uint8)
    return flow, torch.stack([gu, gv])[None], valid, region


def test_hand_checked_image_and_threshold_edges():
    flow, gt, valid, region = hand_image()
    got = check(flow, gt, valid, region, R=2)
    assert got["valid"].tolist() == [[3, 3]] and got["outliers"].tolist() == [[2, 1]]
    n3 = float(np.float32(np.nextafter(np.float32(3), np.float32(np.inf))))
    assert got["epe_sum"].tolist() == [[3.0 + n3 + 4.0, 4.0 + 0.0 + 10.0]]
    # a ratio just above rel_thr is an outlier; at rel_thr = 0.5 the ratio 0.5 of p3' is not
    flow2 = flow.clone()
    flow2[0, 0, 0, 3] = float(np.nextafter(np.float32(84), np.float32(np.inf)))
    assert check(flow2, gt, valid, region, R=2)["outliers"].tolist() == [[2, 2]]
    gt3 = gt.clone()
    gt3[0, 0, 0, 3] = 8.0
    flow3 = flow.clone()
    flow3[0, 0, 0, 3] = 12.0
    assert check(flow3, gt3, valid, region, R=2, rel_thr=0.5)["outliers"].tolist() == [[2, 1]]
    m = metrics.flow_metrics(got)
    assert m["epe"].dtype == torch.float64 and m["epe"][0, 1] == 14.0 / 3 and m["fl"][0, 0] == 2.0 / 3


def np_metrics(valid, outliers, epe_sum):
    valid = np.asarray(valid, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return {"epe": np.where(valid > 0, np.asarray(epe_sum) / valid, np.nan),
                "fl": np.where(valid > 0, np.asarray(outliers) / valid, np.nan)}


def same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def batches():
    """Three batches of R = 3 regions at one ground-truth size; image 1 of the first has no valid pixel and region 2 has
    none anywhere in the second."""
    parts = []
    for k, B in enumerate((3, 1, 4)):
        flow, gt, valid, region = make(B, 6, 9, 11, 17, seed=50 + k, R=3)
        region = torch.where(region == 255, region, region % 3)
        if k == 0:
            valid[1] = False
        if k == 1:
            region = torch.where(region == 2, torch.zeros_like(region), region)
        parts.append((flow, gt, valid, region))
    return parts


def test_flow_metrics_and_both_aggregations():
    parts = batches()
    with emulated() as lib:
        acc = metrics.FlowMetrics(3, "cpu", units="pixels", library=lib)
        errs = [acc.update(*p) for p in parts]
        r = acc.compute()
    n = np.concatenate([e["valid"].numpy() for e in errs])
    o = np.concatenate([e["outliers"].numpy() for e in errs])
    s = np.concatenate([e["epe_sum"].numpy() for e in errs])
    per = metrics.flow_metrics({"valid": torch.from_numpy(n), "outliers": torch.from_numpy(o),
                                "epe_sum": torch.from_numpy(s)})
    ref = np_metrics(n, o, s)
    assert same(per["epe"].numpy(), ref["epe"]) and same(per["fl"].numpy(), ref["fl"])
    assert np.isnan(ref["epe"][1]).all() and np.isnan(ref["epe"][3, 2])
    # "all" = the sum over the regions, appended as index R
    n, o, s = (np.concatenate([x, x.sum(1, keepdims=True)], 1) for x in (n, o, s))
    assert r["images"] == 8 and r["regions"] == 3
    assert np.array_equal(r["valid"], n.sum(0)) and np.array_equal(r["outliers"], o.sum(0))
    assert np.allclose(r["epe_sum"], s.sum(0), rtol=1e-14, atol=0)
    pooled = np_metrics(n.sum(0), o.sum(0), r["epe_sum"])
    assert same(r["pooled"]["epe"], pooled["epe"]) and same(r["pooled"]["fl"], pooled["fl"])
    img = np_metrics(n, o, s)
    ok = n > 0
    assert np.array_equal(r["defined"], ok.sum(0)) and r["defined"].tolist()[0] == 7
    for k in ("epe", "fl"):
        want = np.where(ok, img[k], 0).sum(0) / ok.sum(0)
        assert np.allclose(r["per_image"][k], want, rtol=1e-13, atol=0), k


def test_several_updates_equal_one_update_and_reset():
    parts = batches()
    cat = [torch.cat([p[i] for p in parts]) for i in range(4)]
    with emulated() as lib:
        many = metrics.FlowMetrics(3, "cpu", units="pixels", library=lib)
        for p in parts:
            many.update(*p)
        one = metrics.FlowMetrics(3, "cpu", units="pixels", library=lib)
        one.update(*cat)
        a, b = many.compute(), one.compute()
        many.reset()
        assert int(many.images) == 0 and not many.valid.any() and not many.epe_sum.any() and not many.defined.any()
        # a region with no valid pixel anywhere: NaN in both aggregations
        empty = metrics.FlowMetrics(2, "cpu", units="pixels", library=lib)
        flow, gt, valid, region = parts[1]
        empty.update(flow, gt, valid, torch.zeros_like(region))
        e = empty.compute()
    assert e["valid"][1] == 0 and np.isnan(e["pooled"]["epe"][1]) and np.isnan(e["per_image"]["fl"][1])
    assert e["defined"][1] == 0
    assert a["images"] == b["images"] == 8
    for k in ("valid", "outliers", "defined"):
        assert np.array_equal(a[k], b[k]), k
    assert np.allclose(a["epe_sum"], b["epe_sum"], rtol=1e-14, atol=0)
    for agg in ("pooled", "per_image"):
        for k in ("epe", "fl"):
            assert np.allclose(a[agg][k], b[agg][k], rtol=1e-14, atol=0, equal_nan=True), (agg, k)


def test_bool_and_channel_layouts_and_misaligned_views():
    flow, gt, valid, region = make(5, 4, 6, 7, 9, seed=31, R=2)
    a = check(flow, gt, valid, region, R=2)
    b = run(flow, gt, valid.unsqueeze(1).to(torch.uint8) * 7, region.unsqueeze(1), R=2)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    check(flow[1:], gt[1:], valid[1:], region[1:], R=2)          # base offsets not 16-byte aligned: copied
    check(flow.transpose(2, 3).contiguous().transpose(2, 3), gt, valid, region, R=2)


def test_python_checks():
    flow, gt, valid, region = make(2, 4, 6, 5, 7, seed=1, R=2)
    with emulated() as lib:
        def call(f=flow, g=gt, v=valid, r=region, R=2, **kw):
            kw.setdefault("units", "pixels")
            return metrics.flow_errors(f, g, v, region=r, n_regions=R, library=lib, **kw)
        call()
        with pytest.raises(TypeError, match="units"):
            metrics.flow_errors(flow, gt, valid, library=lib)
        with pytest.raises(ValueError, match="units must be"):
            call(units="px")
        with pytest.raises(TypeError, match="float32"):
            call(f=flow.to(torch.bfloat16))
        with pytest.raises(TypeError, match="float32"):
            call(g=gt.double())
        with pytest.raises(TypeError, match="bool or uint8"):
            call(v=valid.float())
        with pytest.raises(TypeError, match="bool or uint8"):
            call(r=region.long())
        with pytest.raises(ValueError, match=r"\(B, 2, h, w\)"):
            call(f=flow[:, :1].contiguous())
        with pytest.raises(ValueError, match=r"\(B, 2, h, w\)"):
            call(g=gt[:, 0].contiguous())
        with pytest.raises(ValueError, match="differ in batch"):
            call(g=gt[:1].contiguous())
        with pytest.raises(ValueError, match="does not match"):
            call(v=valid[:, :, :3])
        with pytest.raises(ValueError, match="does not match"):
            call(r=region[:1])
        with pytest.raises(ValueError, match=r"\(B, H, W\) or \(B, 1, H, W\)"):
            call(v=valid.view(2, 1, 1, 5, 7))
        for R in (0, 9, 1.0):
            with pytest.raises(ValueError, match="n_regions"):
                call(R=R)
            with pytest.raises(ValueError, match="n_regions"):
                metrics.FlowMetrics(R, "cpu", units="pixels", library=lib)
        with pytest.raises(ValueError, match="region=None"):
            call(r=None)
        with pytest.raises(ValueError, match="region=None"):
            metrics.FlowMetrics(2, "cpu", units="pixels", library=lib).update(flow, gt, valid)
        for kw in (dict(abs_thr=-1.0), dict(rel_thr=NAN), dict(abs_thr=INF), dict(rel_thr=-0.01)):
            with pytest.raises(ValueError, match="finite and >= 0"):
                call(**kw)
        with pytest.raises(ValueError, match="units must be"):
            metrics.FlowMetrics(1, "cpu", units="normalised", library=lib)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        metrics.flow_errors(flow, gt, valid, units="pixels")      # the product refuses host tensors


def test_error_codes_of_the_flow_errors():
    """Argument checks of mdn_flow_errors return status codes before any launch."""
    from mdn_sfm_b200 import _cabi, build
    lib = _cabi.Library(build.build())
    ws = lib.cdll.mdn_flow_errors_workspace_bytes
    # 375 x 1242: 116438 quads -> 114 blocks per sample of 4096 pixels; 24 bytes per (block, region)
    assert ws(12, 192, 640, 375, 1242, 4) == 12 * 114 * 4 * 24 and ws(1, 1, 1, 1, 1, 1) == 24
    for args in ((0, 1, 1, 1, 1, 1), (65536, 1, 1, 1, 1, 1), (1, 0, 1, 1, 1, 1), (1, 1, 0, 1, 1, 1),
                 (1, 1, 1, 0, 1, 1), (1, 1, 1, 1, 0, 1), (1, 1, 1, 65536, 32768, 1), (1, 65536, 32768, 1, 1, 1),
                 (1, 1, 1, 1, 1, 0), (1, 1, 1, 1, 1, 9)):
        assert ws(*args) == 0, args
    big = 1 << 20
    ok = dict(flow=16, h=4, w=6, sx=1.0, sy=1.0, gt=16, valid=16, region=16, R=2, H=8, W=12, B=2, abs_thr=3.0,
              rel_thr=0.05, counts=16, epe=16, ws=16, nbytes=big)
    call = lambda **kw: lib.call("mdn_flow_errors", *dict(ok, **kw).values(), None)
    for name in ("flow", "gt", "valid", "counts", "epe", "ws"):
        with pytest.raises(RuntimeError, match=r"\(-2\).*NULL"):
            call(**{name: None})
    with pytest.raises(RuntimeError, match=r"\(-2\).*region is NULL"):
        call(region=None)
    for kw in (dict(B=0), dict(B=65536), dict(h=0), dict(w=-1), dict(H=0), dict(W=0), dict(H=65536, W=32768),
               dict(h=65536, w=32768), dict(R=0), dict(R=9)):
        with pytest.raises(RuntimeError, match=r"\(-1\).*out of range"):
            call(**kw)
    for kw in (dict(sx=INF), dict(sy=NAN), dict(abs_thr=-1.0), dict(rel_thr=-0.0001), dict(abs_thr=NAN),
               dict(rel_thr=INF)):
        with pytest.raises(RuntimeError, match=r"\(-1\).*threshold"):
            call(**kw)
    for name in ("flow", "gt", "valid", "region", "counts", "epe", "ws"):
        with pytest.raises(RuntimeError, match=r"\(-3\).*16-byte"):
            call(**{name: 24})
    with pytest.raises(RuntimeError, match=r"\(-5\).*workspace too small"):
        call(nbytes=2 * 1 * 2 * 24 - 1)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    torch.set_num_threads(1)
    from emu_harness import emulated
    from mdn_sfm_b200 import metrics
    from test_flow_metrics import batches
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    parts = batches()
    mine = parts[:1] if rank == 0 else parts[1:]
    with emulated() as lib:
        m = metrics.FlowMetrics(3, "cpu", units="pixels", library=lib)
        for p in mine:
            m.update(*p)
    m.all_reduce()
    if rank == 0:
        q.put(m.compute())
    dist.barrier()
    dist.destroy_process_group()


def test_all_reduce_over_two_ranks_equals_one_process():
    emu_library()      # build the emulated library once, before the ranks load it
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    parts = batches()
    with emulated() as lib:
        m = metrics.FlowMetrics(3, "cpu", units="pixels", library=lib)
        m.update(*parts[0])
        rest = metrics.FlowMetrics(3, "cpu", units="pixels", library=lib)
        for p in parts[1:]:
            rest.update(*p)
        for a, b in zip(m._accumulators(), rest._accumulators()):
            a += b
        want = m.compute()
    assert got["images"] == want["images"] == 8
    for k in ("valid", "outliers", "defined", "epe_sum"):
        assert same(got[k], want[k]), k
    for agg in ("pooled", "per_image"):
        for k in ("epe", "fl"):
            assert same(got[agg][k], want[agg][k]), (agg, k)
