"""Times flow evaluation on one GPU: mdn_flow_errors against the torch composition of the same numbers.

    python scripts/time_flow_metrics.py [--blocks 7] [--per-block 200] [--out FILE]

For B = 12, ground truth at 375 x 1242, the prediction at 192 x 640 or at 375 x 1242, and R = 1 (region=None) or R = 4
(uint8 labels):
- `mdn_flow_errors` alone: the C call (main kernel + finish kernel) with preallocated buffers;
- the torch composition: F.interpolate(bilinear, align_corners=False) * scale, the elementwise EPE / Fl formulas, and
  per-(sample, region) sums by index_add_ on an int64 key (uncounted pixels go to a spare bin; no host synchronisation).
Each is timed with CUDA events around a block of `--per-block` calls after a warm-up; the two alternate for `--blocks`
blocks and the median block gives the time per call.  Each block rotates over enough input sets to exceed the 126 MB L2,
so every call reads its inputs from HBM.  Effective bandwidth = the compulsory bytes (gt_flow 8 B, gt_valid 1 B and
region 1 B per ground-truth pixel, the prediction 8 B per pixel) over the time per call.  Before timing, the valid counts
of both must be equal and the outlier counts may differ only by the pixels where F.interpolate rounds differently.

Prints one JSON line (also written to --out), with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.nn.functional as F

DEV = "cuda"
L2_BYTES = 126 * 2 ** 20
ABS_THR, REL_THR = 3.0, 0.05


def card():
    out = {"torch_name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip() or q.stderr.strip()
    except Exception as e:      # (the numbers still print; the card is named by torch)
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def torch_flow_errors(flow, gt, valid, region, R, scale):
    """-> (counts (B, R, 2) int64, epe_sum (B, R) float64), the composition a user would write."""
    B, H, W = valid.shape
    up = F.interpolate(flow, size=(H, W), mode="bilinear", align_corners=False) * scale
    du, dv = up[:, 0] - gt[:, 0], up[:, 1] - gt[:, 1]
    e = torch.sqrt(du * du + dv * dv)
    m = torch.sqrt(gt[:, 0] * gt[:, 0] + gt[:, 1] * gt[:, 1])
    out = (e > ABS_THR) & (e / m > REL_THR)
    base = torch.arange(B, device=flow.device).view(B, 1, 1) * R
    if region is None:
        counted = valid
        key = torch.where(counted, base, B * R)
    else:
        lab = region.long()
        counted = valid & (lab < R)
        key = torch.where(counted, base + lab, B * R)
    key = key.reshape(-1)
    n = torch.zeros(B * R + 1, dtype=torch.int64, device=flow.device).index_add_(0, key, counted.reshape(-1).long())
    o = torch.zeros(B * R + 1, dtype=torch.int64, device=flow.device).index_add_(0, key, (out & counted).reshape(-1).long())
    s = torch.zeros(B * R + 1, dtype=torch.float64, device=flow.device).index_add_(
        0, key, torch.where(counted, e, torch.zeros_like(e)).reshape(-1).double())
    return torch.stack([n[:-1], o[:-1]], -1).view(B, R, 2), s[:-1].view(B, R)


def inputs(B, h, w, H, W, R, n_sets, seed, scale):
    g = torch.Generator(device=DEV).manual_seed(seed)
    sets = []
    for _ in range(n_sets):
        flow = torch.randn(B, 2, h, w, generator=g, device=DEV) * 0.04
        up = F.interpolate(flow, size=(H, W), mode="bilinear", align_corners=False) * scale
        big = torch.rand(B, 1, H, W, generator=g, device=DEV) < 0.25
        gt = (up + torch.randn(B, 2, H, W, generator=g, device=DEV) * torch.where(big, 20.0, 0.8)).contiguous()
        valid = torch.rand(B, H, W, generator=g, device=DEV) < 0.3
        region = torch.randint(0, R + 1, (B, H, W), generator=g, device=DEV, dtype=torch.uint8) if R > 1 else None
        sets.append((flow, gt, valid, region))
    return sets


def time_block(fn, sets, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(*sets[i % len(sets)])
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / n       # µs per call


def run_config(lib, B, h, w, H, W, R, blocks, per_block):
    from mdn_sfm_b200 import _cabi, metrics
    sx, sy = metrics._flow_scale("normalized", h, w, H, W)
    scale = torch.tensor([float(sx), float(sy)], device=DEV).view(1, 2, 1, 1)
    set_bytes = B * (H * W * (8 + 1 + (1 if R > 1 else 0)) + h * w * 8)
    n_sets = max(2, -(-int(1.25 * L2_BYTES) // set_bytes))
    sets = inputs(B, h, w, H, W, R, n_sets, seed=h + R, scale=scale)
    nbytes = lib.cdll.mdn_flow_errors_workspace_bytes(B, h, w, H, W, R)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    counts = torch.empty(B, R, 2, dtype=torch.int64, device=DEV)
    epe = torch.empty(B, R, dtype=torch.float64, device=DEV)
    stream = _cabi.stream_ptr(counts)

    def kernel(flow, gt, valid, region):
        lib.call("mdn_flow_errors", flow.data_ptr(), h, w, float(sx), float(sy), gt.data_ptr(), valid.data_ptr(),
                 _cabi.ptr(region), R, H, W, B, ABS_THR, REL_THR, counts.data_ptr(), epe.data_ptr(), ws.data_ptr(),
                 nbytes, stream, dev=counts)

    composition = lambda flow, gt, valid, region: torch_flow_errors(flow, gt, valid, region, R, scale)
    kernel(*sets[0])
    c_ref, e_ref = composition(*sets[0])
    valid_equal = bool(torch.equal(counts[..., 0], c_ref[..., 0]))
    outlier_diff = int((counts[..., 1] - c_ref[..., 1]).abs().sum())
    epe_rel = float(((epe - e_ref).abs() / e_ref.abs()).max())
    if not valid_equal or outlier_diff > 1e-5 * int(c_ref[..., 0].sum()) or not epe_rel < 1e-5:
        raise SystemExit("the kernel and the composition disagree: valid_equal=%s outlier_diff=%d epe_rel=%g"
                         % (valid_equal, outlier_diff, epe_rel))
    for fn in (kernel, composition):
        time_block(fn, sets, 20)
    res = {"kernel": [], "torch": []}
    for _ in range(blocks):
        res["kernel"].append(time_block(kernel, sets, per_block))
        res["torch"].append(time_block(composition, sets, per_block))
    out = {"B": B, "h": h, "w": w, "H": H, "W": W, "R": R, "input_sets": n_sets,
           "rotated_MB": round(n_sets * set_bytes / 2 ** 20, 1), "compulsory_MB": round(set_bytes / 1e6, 1),
           "valid_equal": valid_equal, "outlier_diff": outlier_diff, "epe_sum_max_rel_diff": epe_rel}
    for name, v in res.items():
        med = statistics.median(v)
        out[name + "_us"] = round(med, 2)
        out[name + "_us_range"] = [round(min(v), 2), round(max(v), 2)]
        out[name + "_GBps"] = round(set_bytes / (med * 1e-6) / 1e9, 1)
    out["speedup"] = round(out["torch_us"] / out["kernel_us"], 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=7)
    ap.add_argument("--per-block", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_flow_metrics.py needs a CUDA device")
    from mdn_sfm_b200 import _cabi
    lib = _cabi.lib()
    rows = []
    for (h, w) in ((192, 640), (375, 1242)):
        for R in (1, 4):
            r = run_config(lib, 12, h, w, 375, 1242, R, a.blocks, a.per_block)
            rows.append(r)
            print("B=12 %4dx%-4d -> 375x1242 R=%d  kernel %8.2f us (%6.1f GB/s)  torch %9.2f us  x%.1f  outlier_diff=%d"
                  % (h, w, R, r["kernel_us"], r["kernel_GBps"], r["torch_us"], r["speedup"], r["outlier_diff"]),
                  flush=True)
    line = json.dumps({"card": card(), "blocks": a.blocks, "per_block": a.per_block, "configs": rows})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
