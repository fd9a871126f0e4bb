"""Mask evaluation (mdn_sfm_b200.metrics, mdn_mask_confusion) under the SIMT emulator: the confusion counts against a
direct count of `(pred >= thr) & label` (exact and NaN-correct at these sizes), the metrics and both aggregations
against a float64 numpy restatement, the Python checks, a two-rank all_reduce over gloo, and the entry point's error
codes in the real library (no GPU needed)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from emu_harness import emu_library, emulated
from mdn_sfm_b200 import metrics

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle(pred, gt, thr):
    """(B, ...) fp32 pred, (B, ...) gt (non-zero = moving), (K,) fp32 thresholds -> (B, K, 4) int64 [TP, FP, FN, TN]."""
    B = pred.shape[0]
    p = pred.reshape(B, -1, 1) >= thr.reshape(1, 1, -1)
    lab = (gt.reshape(B, -1, 1) != 0)
    out = [(p & lab).sum(1), (p & ~lab).sum(1), (~p & lab).sum(1), (~p & ~lab).sum(1)]
    return torch.stack(out, -1).to(torch.int64)


def check(pred, gt, thr):
    """Runs mask_confusion under the emulator and holds it to the oracle; -> the counts."""
    thr = torch.as_tensor(thr, dtype=torch.float32)
    with emulated() as lib:
        got = metrics.mask_confusion(pred, gt, thr, library=lib)
    want = oracle(pred, gt, thr)
    hw = pred.shape[-1] * pred.shape[-2]
    assert got.dtype == torch.int64 and got.shape == (pred.shape[0], thr.numel(), 4)
    assert torch.equal(got.sum(-1), torch.full_like(got[..., 0], hw))
    assert torch.equal(got, want)
    return got


def sweep(K, seed=0):
    g = torch.Generator().manual_seed(seed)
    t = torch.unique(torch.rand(4 * K + 8, generator=g))[:K]
    assert t.numel() == K
    return t.sort().values


def maps(B, H, W, seed, K_thr=None, p_moving=0.3):
    g = torch.Generator().manual_seed(seed)
    pred = torch.rand(B, H, W, generator=g)
    gt = torch.rand(B, H, W, generator=g) < p_moving
    if K_thr is not None:   # some predictions land exactly on a threshold or just below it
        idx = torch.randint(0, K_thr.numel(), (B, H, W), generator=g)
        pick = torch.rand(B, H, W, generator=g)
        pred = torch.where(pick < 0.2, K_thr[idx], pred)
        pred = torch.where((pick >= 0.2) & (pick < 0.4), torch.nextafter(K_thr[idx], torch.tensor(-float("inf"))), pred)
    return pred.contiguous(), gt.contiguous()


@pytest.mark.parametrize("H,W", [(4, 6), (5, 5), (3, 10), (3, 9), (1, 3), (1, 1)],
                         ids=["hw%4==0", "hw%4==1", "hw%4==2", "hw%4==3", "hw=3", "hw=1"])
def test_counts_at_every_sample_alignment(H, W):
    """B = 5 samples back to back: with h*w % 4 != 0 the samples start at every offset mod 4, so the scalar head, the
    vector body and the scalar tail all run."""
    thr = sweep(7, seed=H * W)
    pred, gt = maps(5, H, W, seed=H + W, K_thr=thr)
    check(pred, gt, thr)


@pytest.mark.parametrize("K", [1, 7, 101, 1024])
def test_counts_for_each_sweep_length(K):
    thr = sweep(K, seed=K)
    pred, gt = maps(4, 13, 29, seed=K, K_thr=thr)
    check(pred, gt, thr)


def test_special_values_and_infinite_thresholds():
    """Exact hits, nextafter(thr, -inf), NaN, +-inf and -0.0 against thresholds that contain 0.0 and +-inf: NaN is never
    moving, a prediction equal to a threshold is moving at it, -0.0 >= 0.0, -inf >= -inf."""
    inf, nan = float("inf"), float("nan")
    thr = torch.tensor([-inf, -0.5, 0.0, 0.25, 0.5, 1.0, inf])
    specials = torch.tensor([nan, inf, -inf, -0.0, 0.0, 0.5, 0.49999997, 1.0, 0.99999994, -0.5, 1e-45, -1e-45, 0.25, 2.0])
    g = torch.Generator().manual_seed(3)
    pred = specials[torch.randint(0, specials.numel(), (6, 7, 11), generator=g)]
    gt = torch.randint(0, 2, (6, 7, 11), generator=g).bool()
    got = check(pred, gt, thr)
    # one hand-checked image: every special value once, all moving
    one = torch.tensor([[nan, 0.5, 0.49999997, -0.0, inf, -inf]])
    c = check(one.view(1, 1, 6), torch.ones(1, 1, 6, dtype=torch.bool), torch.tensor([0.1, 0.5, 0.9]))
    assert c[0, :, 0].tolist() == [3, 2, 1]       # TP per threshold: {0.5, 0.49999997, inf}, {0.5, inf}, {inf}
    assert got.shape == (6, 7, 4)


@pytest.mark.parametrize("kind", ["bool", "u8"])
def test_gt_as_bool_and_as_uint8(kind):
    thr = sweep(9, seed=5)
    pred, gt = maps(4, 9, 14, seed=6, K_thr=thr)
    if kind == "u8":
        vals = torch.tensor([0, 1, 7, 255], dtype=torch.uint8)
        gt = vals[torch.randint(0, 4, gt.shape, generator=torch.Generator().manual_seed(7))]
    check(pred, gt, thr)


def test_channel_layout_and_host_sequence_thresholds():
    thr = sweep(5, seed=8)
    pred, gt = maps(3, 10, 15, seed=9, K_thr=thr)
    a = check(pred.unsqueeze(1), gt.unsqueeze(1), thr)
    with emulated() as lib:
        b = metrics.mask_confusion(pred, gt.unsqueeze(1), thr.tolist(), library=lib)
    assert torch.equal(a, b)


def test_kitti_size():
    thr = torch.linspace(0, 1, 7)
    g = torch.Generator().manual_seed(11)
    pred = torch.rand(2, 375, 1242, generator=g) ** 4          # skewed towards 0, like a mobile map
    gt = torch.rand(2, 375, 1242, generator=g) < 0.1
    check(pred, gt, thr)


def test_misaligned_views_are_copied_to_an_aligned_base():
    thr = sweep(4, seed=12)
    pred, gt = maps(5, 3, 7, seed=13, K_thr=thr)
    check(pred[1:], gt[1:], thr)                 # base offset 21 elements: not 16-byte aligned
    check(pred.transpose(1, 2), gt.transpose(1, 2), thr)


def np_metrics(c):
    """float64 numpy restatement of the five metrics from [TP, FP, FN, TN]."""
    tp, fp, fn, tn = (np.asarray(c)[..., i].astype(np.float64) for i in range(4))
    with np.errstate(invalid="ignore", divide="ignore"):
        return {"accuracy": (tp + tn) / (tp + fp + fn + tn), "precision": tp / (tp + fp), "recall": tp / (tp + fn),
                "dice": 2 * tp / (2 * tp + fp + fn), "iou": tp / (tp + fp + fn)}


def hand_built():
    """Four 2 x 4 images at thresholds [0.5, 0.8]: a mixed one (TP 2, FP 1, FN 1, TN 4 at 0.5), one with no moving pixels,
    one with no predicted pixels, one with neither."""
    pred = torch.tensor([[[0.9, 0.6, 0.7, 0.1], [0.2, 0.3, 0.0, 0.4]],
                         [[0.9, 0.1, 0.1, 0.1], [0.1, 0.1, 0.1, 0.1]],
                         [[0.1, 0.1, 0.1, 0.1], [0.2, 0.3, 0.0, 0.4]],
                         [[0.0, 0.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0]]])
    gt = torch.tensor([[[1, 1, 0, 1], [0, 0, 0, 0]],
                       [[0, 0, 0, 0], [0, 0, 0, 0]],
                       [[1, 1, 0, 0], [0, 0, 0, 0]],
                       [[0, 0, 0, 0], [0, 0, 0, 0]]], dtype=torch.uint8)
    return pred, gt, [0.5, 0.8]


def same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def test_metrics_and_both_aggregations_on_hand_built_images():
    pred, gt, thr = hand_built()
    counts = check(pred, gt, thr)
    assert counts[0, 0].tolist() == [2, 1, 1, 4] and counts[0, 1].tolist() == [1, 0, 2, 5]
    assert counts[1, 0].tolist() == [0, 1, 0, 7] and counts[2, 0].tolist() == [0, 0, 2, 6]
    assert counts[3, 0].tolist() == [0, 0, 0, 8]
    m = metrics.mask_metrics(counts)
    ref = np_metrics(counts.numpy())
    for k in metrics.METRICS:
        assert m[k].dtype == torch.float64 and same(m[k].numpy(), ref[k]), k
    assert m["precision"][0, 0] == 2 / 3 and m["iou"][0, 0] == 0.5 and m["accuracy"][0, 0] == 0.75
    assert m["dice"][1, 0] == 0 and np.isnan(float(m["recall"][1, 0])) and np.isnan(float(m["precision"][2, 0]))
    assert all(np.isnan(float(m[k][3, 0])) for k in ("precision", "recall", "dice", "iou")) and m["accuracy"][3, 0] == 1

    with emulated() as lib:
        acc = metrics.MaskMetrics(thr, "cpu", library=lib)
        acc.update(pred, gt)
        r = acc.compute()
    assert r["images"] == 4 and same(r["thresholds"], np.float32(thr))
    pooled = counts.numpy().sum(0)
    assert np.array_equal(r["counts"], pooled)
    ref_pooled = np_metrics(pooled)
    for k in metrics.METRICS:
        assert same(r["pooled"][k], ref_pooled[k]), k
        v = ref[k]
        ok = ~np.isnan(v)
        assert np.array_equal(r["defined"][k], ok.sum(0)), k
        with np.errstate(invalid="ignore"):
            want = np.where(ok.sum(0) > 0, np.where(ok, v, 0).sum(0) / np.maximum(ok.sum(0), 1), np.nan)
        assert np.allclose(r["per_image"][k], want, rtol=1e-15, atol=0, equal_nan=True), k
    # pooled dice is 2PR / (P + R) of the pooled precision and recall
    P, R = r["pooled"]["precision"], r["pooled"]["recall"]
    assert np.allclose(r["pooled"]["dice"], 2 * P * R / (P + R), rtol=1e-15)
    assert r["defined"]["precision"].tolist() == [2, 2] and r["defined"]["accuracy"].tolist() == [4, 4]


def test_several_updates_equal_one_update_of_the_concatenated_batch():
    thr = sweep(13, seed=20)
    parts = [maps(b, 11, 17, seed=30 + b, K_thr=thr) for b in (3, 1, 4)]
    with emulated() as lib:
        many = metrics.MaskMetrics(thr, "cpu", library=lib)
        for p, g in parts:
            many.update(p, g)
        one = metrics.MaskMetrics(thr, "cpu", library=lib)
        one.update(torch.cat([p for p, _ in parts]), torch.cat([g for _, g in parts]))
        a, b = many.compute(), one.compute()
        many.reset()
        assert int(many.images) == 0 and not many.pooled.any() and not many.sums.any() and not many.defined.any()
    assert a["images"] == b["images"] == 8 and np.array_equal(a["counts"], b["counts"])
    for k in metrics.METRICS:
        assert same(a["pooled"][k], b["pooled"][k]) and np.array_equal(a["defined"][k], b["defined"][k])
        assert np.allclose(a["per_image"][k], b["per_image"][k], rtol=1e-14, atol=0, equal_nan=True)


def test_python_checks():
    pred, gt = maps(2, 4, 8, seed=1)
    with emulated() as lib:
        call = lambda p=pred, g=gt, t=(0.1, 0.5): metrics.mask_confusion(p, g, t, library=lib)
        for bad, msg in (([0.5, 0.1], "strictly increasing"), ([0.1, 0.1], "strictly increasing"),
                         ([0.1, float("nan")], "NaN"), ([], "1 to 1024"), (np.linspace(0, 1, 1025), "1 to 1024"),
                         ([[0.1, 0.2]], "one-dimensional"), ([0.5, 0.5 + 1e-12], "strictly increasing")):
            with pytest.raises(ValueError, match=msg):
                call(t=bad)
            with pytest.raises(ValueError, match=msg):
                metrics.MaskMetrics(bad, "cpu", library=lib)
        call(t=np.linspace(0, 1, 1024))
        with pytest.raises(ValueError, match="differ in size"):
            call(g=gt[:, :, :4].contiguous())
        with pytest.raises(ValueError, match="differ in size"):
            call(g=gt[:1])
        with pytest.raises(ValueError, match=r"\(B, h, w\) or \(B, 1, h, w\)"):
            call(p=pred.view(2, 1, 1, 4, 8))
        with pytest.raises(ValueError, match=r"\(B, h, w\) or \(B, 1, h, w\)"):
            call(p=pred.view(1, 2, 4, 8), g=gt.view(1, 2, 4, 8))
        with pytest.raises(TypeError, match="bool or uint8"):
            call(g=gt.float())
        with pytest.raises(TypeError, match="float32"):
            call(p=pred.double())
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        metrics.mask_confusion(pred, gt, [0.5])        # the product refuses host tensors


def test_error_codes_of_the_mask_confusion():
    """Argument checks of mdn_mask_confusion return status codes before any launch."""
    from mdn_sfm_b200 import _cabi, build
    lib = _cabi.Library(build.build())
    ws = lib.cdll.mdn_mask_confusion_workspace_bytes
    assert ws(12, 101) == 12 * 2 * 102 * 4 and ws(1, 1024) == 2 * 1025 * 4
    for b, k in ((0, 5), (65536, 5), (1, 0), (1, 1025)):
        assert ws(b, k) == 0
    big = 1 << 20
    ok = dict(pred=16, gt=16, thr=16, K=5, counts=16, B=2, hw=64, ws=16, nbytes=big)
    call = lambda **kw: lib.call("mdn_mask_confusion", *dict(ok, **kw).values(), None)
    for name in ("pred", "gt", "thr", "counts", "ws"):
        with pytest.raises(RuntimeError, match=r"\(-2\).*NULL"):
            call(**{name: None})
    for kw in (dict(B=0), dict(B=65536), dict(hw=0), dict(hw=1 << 31), dict(K=0), dict(K=1025), dict(B=-1, hw=-1)):
        with pytest.raises(RuntimeError, match=r"\(-1\).*out of range"):
            call(**kw)
    for name in ("pred", "gt", "thr", "counts", "ws"):
        with pytest.raises(RuntimeError, match=r"\(-3\).*16-byte"):
            call(**{name: 24})
    with pytest.raises(RuntimeError, match=r"\(-5\).*workspace too small"):
        call(nbytes=2 * 2 * 6 * 4 - 1)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    torch.set_num_threads(1)
    from emu_harness import emulated
    from mdn_sfm_b200 import metrics
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    pred, gt, thr = _global_batch()
    half = pred.shape[0] // world
    with emulated() as lib:
        m = metrics.MaskMetrics(thr, "cpu", library=lib)
        m.update(pred[rank * half:(rank + 1) * half], gt[rank * half:(rank + 1) * half])
    m.all_reduce()
    if rank == 0:
        q.put(m.compute())
    dist.barrier()
    dist.destroy_process_group()


def _global_batch():
    g = torch.Generator().manual_seed(99)
    pred = torch.rand(6, 9, 13, generator=g) ** 3
    gt = torch.rand(6, 9, 13, generator=g) < 0.2
    pred[1] = 0.0      # an image with no predicted pixels at any positive threshold
    gt[4] = False      # an image with no moving pixels
    return pred, gt, [0.0, 0.05, 0.1, 0.3, 0.6, 0.9]


def test_all_reduce_over_two_ranks_equals_one_process():
    emu_library()      # build the emulated library once, before the ranks load it
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    pred, gt, thr = _global_batch()
    with emulated() as lib:
        m = metrics.MaskMetrics(thr, "cpu", library=lib)
        m.update(pred[:3], gt[:3])
        m.update(pred[3:], gt[3:])
        want = m.compute()
    assert got["images"] == want["images"] == 6 and np.array_equal(got["counts"], want["counts"])
    for k in metrics.METRICS:
        for agg in ("pooled", "per_image", "defined"):
            assert same(got[agg][k], want[agg][k]), (agg, k)
