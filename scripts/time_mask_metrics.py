"""Times mask evaluation on one GPU: mdn_mask_confusion against the torch composition of the same counts.

    python scripts/time_mask_metrics.py [--blocks 7] [--per-block 200] [--out FILE]

For B = 12 at 375 x 1242 and at 192 x 640, K in {101, 1024} and skewed (a mobile map: sigmoid of logits around -4) or
uniform predictions:
- `mdn_mask_confusion` alone: the C call (workspace memset, counting kernel, finish kernel) with preallocated buffers;
- the torch composition of the same counts: bucketize(right=True) -> int64 key (sample, label, bin) -> bincount -> suffix
  sums (torch.bincount on CUDA reads the key maximum back to the host, one synchronisation per call).
Each is timed with CUDA events around a block of `--per-block` calls after a warm-up; the two alternate for `--blocks`
blocks and the median block gives the time per call.  Each block rotates over enough input sets (pred fp32 + gt uint8)
to exceed the 126 MB L2, so every call reads its inputs from HBM.  Effective bandwidth = 5 bytes per pixel over the
time per call.  The results of both are checked equal once per configuration.

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

DEV = "cuda"
L2_BYTES = 126 * 2 ** 20


def card():
    out = {"torch_name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip() or q.stderr.strip()
    except Exception as e:      # (the numbers still print; the card is named by torch)
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def torch_confusion(pred, gt, thr):
    B, K = pred.shape[0], thr.numel()
    j = torch.bucketize(pred.reshape(B, -1), thr, right=True)
    key = j + (gt.reshape(B, -1) != 0).long() * (K + 1) + torch.arange(B, device=pred.device)[:, None] * (2 * (K + 1))
    h = torch.bincount(key.reshape(-1), minlength=B * 2 * (K + 1)).view(B, 2, K + 1)
    s = h.flip(-1).cumsum(-1).flip(-1)
    tp, fp = s[:, 1, 1:], s[:, 0, 1:]
    return torch.stack([tp, fp, s[:, 1, :1] - tp, s[:, 0, :1] - fp], -1)


def inputs(B, H, W, kind, n_sets, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    sets = []
    for _ in range(n_sets):
        if kind == "skewed":
            pred = torch.sigmoid(torch.randn(B, H, W, generator=g, device=DEV) * 1.5 - 4.0)
        else:
            pred = torch.rand(B, H, W, generator=g, device=DEV)
        gt = (torch.rand(B, H, W, generator=g, device=DEV) < 0.15).to(torch.uint8)
        sets.append((pred, gt))
    return sets


def time_block(fn, sets, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(*sets[i % len(sets)])
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / n       # µs per call


def run_config(lib, B, H, W, K, kind, blocks, per_block):
    from mdn_sfm_b200 import _cabi
    set_bytes = B * H * W * 5
    n_sets = max(2, -(-int(1.25 * L2_BYTES) // set_bytes))
    sets = inputs(B, H, W, kind, n_sets, seed=H + K)
    thr = torch.linspace(0, 1, K, device=DEV)
    nbytes = lib.cdll.mdn_mask_confusion_workspace_bytes(B, K)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    counts = torch.empty(B, K, 4, dtype=torch.int64, device=DEV)
    stream = _cabi.stream_ptr(counts)

    def kernel(pred, gt):
        lib.call("mdn_mask_confusion", pred.data_ptr(), gt.data_ptr(), thr.data_ptr(), K, counts.data_ptr(), B, H * W,
                 ws.data_ptr(), nbytes, stream, dev=counts)

    composition = lambda pred, gt: torch_confusion(pred, gt, thr)
    kernel(*sets[0])
    same = bool(torch.equal(counts, composition(*sets[0])))
    for fn in (kernel, composition):
        time_block(fn, sets, 20)
    res = {"kernel": [], "torch": []}
    for _ in range(blocks):
        res["kernel"].append(time_block(kernel, sets, per_block))
        res["torch"].append(time_block(composition, sets, per_block))
    out = {"B": B, "H": H, "W": W, "K": K, "pred": kind, "input_sets": n_sets, "rotated_MB": round(n_sets * set_bytes / 2 ** 20, 1),
           "equal": same}
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
        raise SystemExit("time_mask_metrics.py needs a CUDA device")
    from mdn_sfm_b200 import _cabi
    lib = _cabi.lib()
    rows = []
    for (H, W) in ((375, 1242), (192, 640)):
        for K in (101, 1024):
            for kind in ("skewed", "uniform"):
                r = run_config(lib, 12, H, W, K, kind, a.blocks, a.per_block)
                rows.append(r)
                print("B=12 %4dx%-4d K=%4d %-7s  kernel %8.2f us (%6.1f GB/s)  torch %9.2f us  x%.1f  equal=%s"
                      % (H, W, K, kind, r["kernel_us"], r["kernel_GBps"], r["torch_us"], r["speedup"], r["equal"]), flush=True)
    line = json.dumps({"card": card(), "blocks": a.blocks, "per_block": a.per_block, "configs": rows})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
