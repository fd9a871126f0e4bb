#!/usr/bin/env python
"""bench.py -- loss-path frames/s, forward + backward, @192x640 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape 192x640|375x1242] [--mode T]
                    [--dump-outputs DIR]

A *step* is one pass of the whole configured loss path over one batch: `Loss.forward` (all scales, both
source frames: epipolar map + post-processing, flow warp, SSIM + L1, smoothness, consistency, min mask) followed
by `losses["loss"].backward()` down to d/dflow, d/dmobile and d/dpose.  Workload at every N: BASELINE configs[1],
T mode + photometric, batch 12 per GPU (weak scaling), 3x192x640, 4 scales, synthetic KITTI-shaped inputs.

`value`   whole-job frames/s with inputs resident in HBM, the step replayed from a CUDA graph, `--sets` input
          sets rotated so the working set (inputs + gradients) is several times the 126 MB L2.
`e2e`     the same step through the public Python API with HOST inputs: one pinned host -> device copy of the batch
          per step (frames as uint8, normalised and turned into pyramids on the device) and a device -> host read of
          the loss inside the timed region; median of five runs, beside the measured host-copy ceiling.
`other_configs`  BASELINE configs[3] (DS, DC) and configs[4] (375x1242) at the same N.
`gpu_eager_baseline`  the reference's op sequence run eagerly on the same GPU (upstream's default cuda=True path).
`roofline` algorithmic bytes of one fused launch / its measured duration (CUDA events) vs MEASURED_PEAKS.json.
`cpu_baseline` the oracle port (oracle/restate.py, eager torch, the reference's own op sequence) on the host cores.
`--impl reference` prints the reference arm: the same oracle port timed on the host CPU with all threads.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "loss-path frames/s fwd+bwd @192x640"
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 64 * 10 ** 6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="192x640")
    ap.add_argument("--mode", default="T", choices=["SN", "T", "TG", "DS", "DC"])
    ap.add_argument("--batch", type=int, default=12)
    ap.add_argument("--sets", type=int, default=4, help="rotating input sets (defeats L2 reuse between steps)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 100)")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--flow", default="iid", choices=["iid", "smooth"],
                    help="synthetic flow field: iid = white noise N(0, 0.05^2) per pixel (stress: every pixel gathers from an "
                         "unrelated place), smooth = network-like field of the same magnitude")
    ap.add_argument("--no-second-flow", action="store_true", help="skip the short extra measurement on the other flow kind")
    ap.add_argument("--no-train-step", action="store_true", help="skip the short whole-train-step measurement (configs[2])")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the DS / DC / 375x1242 lines (BASELINE configs[3], [4])")
    ap.add_argument("--train-steps", type=int, default=30)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss terms and gradients of the last timed step as DIR/<name>.npy "
                         "(float32; an array is replaced by a fixed seeded sample of its elements when all of them would "
                         "exceed %d MB); with several GPUs, rank 0's step" % (DUMP_BYTES // 10 ** 6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


FLOW_DESC = {"iid": "normalised flow ~ N(0, 0.05^2) i.i.d. per pixel (+-32 px at 640: stress case, no locality in the warp gather)",
             "smooth": "network-like smooth flow field, total std 0.05 (mdn_sfm_b200.synthetic.smooth_flow)"}


def workload(args):
    H, W = map(int, args.shape.split("x"))
    scales = (0, 1, 2, 3) if (H % 8 == 0 and W % 8 == 0) else (0,)
    return H, W, scales


def algorithmic_bytes_per_frame(H, W, scales, with_inst=False):
    """One-pass variant A1 of SURVEY.md section 8d: every input read once, every gradient written once.
    per scale-pixel: tgt 12 + mob 4+4 + 2 x (flow 8 + ref 12) = 60 read, g_flow 2x8 + g_mob 2x4 = 24 written."""
    px = sum((H >> s) * (W >> s) for s in scales)
    return px * (84 + (1 if with_inst else 0))


def config_dict(args, H, W, scales, n_gpus):
    return {"workload": "BASELINE configs[1]: %s-mode epipolar map + flow-warp SSIM/L1 photometric + smooth + consistency, "
                        "fwd+bwd, batch %d/GPU x %d GPU, 3x%dx%d, %d scales, 2 source frames" % (
                            args.mode, args.batch, n_gpus, H, W, len(scales)),
            "mode": args.mode, "batch_per_gpu": args.batch, "global_batch": args.batch * n_gpus, "height": H, "width": W,
            "scales": list(scales), "frame_ids": [0, -1, 1], "photometric": True, "ssim": True,
            "flow": FLOW_DESC[args.flow],
            # (how the GPU arm keeps L2 from serving one step's inputs to the next; the CPU reference arm carries the same
            # config so that the driver can match the two lines)
            "l2": "%d rotating input sets (%.0f MB inputs+grads per set vs 126 MB L2)" % (
                args.sets, algorithmic_bytes_per_frame(H, W, scales, args.mode in ("DS", "DC")) * args.batch / 1e6)}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the GPU is under load."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.stop_flag = index, period, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_step_fn(args, H, W, scales, seed=42):
    """The oracle port on the host CPU: same workload, fwd + backward, all host threads."""
    from mdn_sfm_b200 import synthetic
    from oracle import restate
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    opt = synthetic.default_opt(args.batch, H, W)
    inputs, flows, mobiles, cams, inst = synthetic.make_batch(args.batch, H, W, scales=scales, seed=seed, flow_std=0.05,
                                                              with_instances=args.mode in ("DS", "DC"), flow_kind=args.flow)
    weights = restate.gauss_distance_weight(4, H, W) if args.mode == "TG" else None

    def step():
        f = {k: v.clone().requires_grad_(True) for k, v in flows.items()}
        m = {k: v.clone().requires_grad_(True) for k, v in mobiles.items()}
        c = {k: v.clone().requires_grad_(True) for k, v in cams.items()}
        _, losses = restate.loss_forward(opt, inputs, [-1, 1], f, m, inst, list(scales), c, mode=args.mode,
                                         weights=weights, photometric=True, ssim_on=True)
        losses["loss"].backward()
        return float(losses["loss"].detach())

    return step, threads


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    H, W, scales = workload(args)
    step, threads = cpu_reference_step_fn(args, H, W, scales)
    warm = max(1, args.warmup)              # the driver's W, as given (each CPU step is ~0.2 s at the headline shape)
    steps = max(1, min(args.steps, 20))     # bounded sample: ~1-2 s of CPU work per step
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    fps = args.batch * steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args, H, W, scales, args.gpus),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": "%d steps of one batch of %d frames (the N=1 workload) on the host CPU, torch %d threads; "
                                       "requested steps=%d were capped at 20" % (steps, args.batch, threads, args.steps)},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ train step (configs[2])
def measure_train_step(args, dev, world, rank, H, W, scales):
    """TG-mode full train step, batch `--batch` per GPU: mdn_sfm_b200.train_step.TrainStep (SURVEY 8f-N1) with the stand-in
    nets (the reference's FlowNet / PoseNet / MobileDecoder are cuDNN consumers outside the path; random init either way),
    frozen flow + pose nets, DDP on the mobile decoder when N > 1.  Eager launches, CUDA events, max over ranks."""
    import torch.distributed as dist
    from mdn_sfm_b200 import synthetic
    from mdn_sfm_b200.train_step import TrainStep
    B = args.batch
    opt = synthetic.default_opt(B, H, W, threshold=0.8625, scales=list(scales))   # options_eval.py:55-58 (weighted 95 %)
    torch.manual_seed(1234)     # identical initial weights on every rank, like DDP's broadcast would leave them
    ts = TrainStep(opt, device=dev, mode="TG", photometric=True)
    sets = []
    for k in range(2):
        inputs, _, _, _, _ = synthetic.make_batch(B, H, W, scales=scales, seed=4242 + rank + 1000 * k, with_instances=False)
        sets.append({kk: v.to(dev) for kk, v in inputs.items()})
    for i in range(5):
        losses = ts.step(sets[i % 2])
    torch.cuda.synchronize()
    # loss path alone inside this step (forward + backward of the loss on the nets' outputs), for the share: as the step runs
    # it (one CUDA-graph replay, PoseNet's outputs as parameters) and through the eager public API
    from mdn_sfm_b200.layers import PoseParameters
    flows, mobiles, cams, _, _ = ts.process_batch(sets[0])
    fl = {k: v.detach() for k, v in flows.items()}
    mo = {k: v.detach().requires_grad_(True) for k, v in mobiles.items()}
    ca = {k: PoseParameters(c.axisangle.detach(), c.translation.detach()) for k, c in cams.items()}
    ids = list(opt.frame_ids)[1:]

    def loss_only(loss_fn):
        for v in mo.values():
            v.grad = None
        total = loss_fn(sets[0], ids, fl, mo, None, list(scales), ca)[1]["loss"]
        if hasattr(loss_fn, "unit_upstream"):
            loss_fn.unit_upstream = True
        total.backward()
        if hasattr(loss_fn, "unit_upstream"):
            loss_fn.unit_upstream = False

    def time_loss(loss_fn, n=20):
        for _ in range(3):
            loss_only(loss_fn)
        torch.cuda.synchronize()
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record()
        for _ in range(n):
            loss_only(loss_fn)
        l1.record()
        torch.cuda.synchronize()
        return l0.elapsed_time(l1) / n

    loss_ms = time_loss(ts.loss)
    loss_ms_eager = time_loss(ts.eager_loss)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    # three equal chunks, the median chunk reported: the step is ~30 eager cuDNN / optimizer launches per net, and a host hiccup
    # inside a single 30-step window used to move the figure by 2x between runs
    n_total = args.train_steps
    n = max(1, n_total // 3)
    chunk_ms = []
    for c in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            losses = ts.step(sets[i % 2])
        e1.record()
        torch.cuda.synchronize()
        ms_c = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms_c], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_c = float(t.item())
        chunk_ms.append(ms_c)
    ms = sorted(chunk_ms)[1]
    logged = ts.log_losses(losses)
    n_par = sum(p.numel() for p in ts.parameters_to_train)
    return {"workload": "BASELINE configs[2]: TG-mode full train step (stand-in flow / pose / mobile-decoder CNNs on cuDNN, frozen flow + "
                        "pose, %s on the mobile decoder, clip_grad_norm_, Adam), batch %d/GPU x %d GPU; nets eager, the loss path as one CUDA-graph "
                        "replay with PoseNet's outputs as parameters (graphs.GraphedLoss, layers.PoseParameters)" % (
                            "DDP (NCCL all-reduce)" if world > 1 else "single process", B, world),
            "value": world * B * n / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms / n, "steps": n,
            "statistic": "median of 3 chunks of %d steps (max over ranks per chunk)" % n, "chunks_ms_per_step": [c / n for c in chunk_ms],
            "loss_path_ms_per_step": loss_ms, "loss_path_ms_per_step_eager": loss_ms_eager, "trainable_parameters": n_par,
            "loss": logged.get("loss")}


# ------------------------------------------------------------------------------------------------ GPU arm
def source_hash():
    """Hash of the kernel sources the in-tree library is built from: ties profiles/traffic.json (ncu numbers) to a build."""
    import hashlib
    hsh = hashlib.sha256()
    for rel in ("mdn_sfm_b200/csrc/mdn_loss.cu", "mdn_sfm_b200/csrc/mdn_fused.cuh", "mdn_sfm_b200/csrc/mdn_common.cuh",
                "mdn_sfm_b200/csrc/mdn_resize.cuh", "include/mdn_loss.h"):
        with open(os.path.join(ROOT, rel), "rb") as f:
            hsh.update(f.read())
    return hsh.hexdigest()[:16]


class Workload:
    """One (mode, shape, batch) configuration of the loss path on this rank: the public `Loss`, rotating input sets, the
    graph-replayed timing of K steps and the dominant kernel timed alone."""

    def __init__(self, args, mode, H, W, scales, dev, world, rank, flow_kind, n_sets):
        from mdn_sfm_b200 import synthetic
        from mdn_sfm_b200.loss_functions import Loss
        self.args, self.mode, self.H, self.W, self.scales, self.dev, self.world, self.rank = args, mode, H, W, tuple(scales), dev, world, rank
        self.B = args.batch
        self.opt = synthetic.default_opt(self.B, H, W)
        self.with_inst = mode in ("DS", "DC")
        self.loss_mod = Loss(self.opt, no_ssim=False, mode=mode, photometric=True)
        self.ids = [-1, 1]
        self.host_sets, self.dev_sets = [], []
        for k in range(n_sets):   # pinned host masters + device-resident copies
            inputs, flows, mobiles, cams, inst = synthetic.make_batch(self.B, H, W, scales=self.scales, seed=42 + rank + 1000 * k, flow_std=0.05,
                                                                      with_instances=self.with_inst, flow_kind=flow_kind)
            pin = lambda d: {kk: v.pin_memory() for kk, v in d.items()}
            self.host_sets.append((pin(inputs), pin(flows), pin(mobiles), pin(cams), inst))
            to = lambda d, g=False: {kk: v.to(dev).requires_grad_(g) for kk, v in d.items()}
            inst_d = [{"instances": d["instances"].to(dev)} for d in inst] if inst is not None else None
            self.dev_sets.append((to(inputs), to(flows, True), to(mobiles, True), to(cams, True), inst_d))

    def step_on(self, s):
        """One forward + backward on input set `s`; returns the losses dict (the gradients land in the leaves' .grad)."""
        inputs, flows, mobiles, cams, inst = s
        for d in (flows, mobiles, cams):
            for v in d.values():
                v.grad = None
        _, losses = self.loss_mod(inputs, self.ids, flows, mobiles, inst, list(self.scales), cams)
        losses["loss"].backward()
        return losses

    def timed_steps(self, dev_sets, steps, warmup, ramp_s):
        """fwd+bwd steps replayed from CUDA graphs over rotating input sets; returns (total ms, graph_ok).
        `self.last_step` is left as (input set, losses dict) of the last timed step."""
        import torch.distributed as dist
        step_on, world, dev = self.step_on, self.world, self.dev
        for s in dev_sets:   # eager warm-up (also sets the kernel attributes outside any capture)
            step_on(s)
        torch.cuda.synchronize()
        # One graph holds a whole rotation (one step per input set), so the launch latency of the graph itself is paid
        # once per `len(dev_sets)` steps; a remainder of the requested step count runs from single-step graphs.
        group, singles, graph_ok = None, [], not self.args.no_graph
        n_sets = len(dev_sets)
        q, r = divmod(steps, n_sets)
        if graph_ok:
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for s in dev_sets:
                        step_on(s)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                group = torch.cuda.CUDAGraph()
                with torch.cuda.graph(group):
                    outs = [step_on(s) for s in dev_sets]
                for s in dev_sets[:r]:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        out = step_on(s)
                    singles.append((g, out))
                torch.cuda.synchronize()
            except Exception as e:   # keep measuring, but say so
                graph_ok, group, singles = False, None, []
                print("bench: CUDA graph capture failed (%r); timing eager launches" % (e,), file=sys.stderr)
                torch.cuda.synchronize()

        def run_rotation():
            if graph_ok:
                group.replay()
                return outs[-1]
            for s in dev_sets:
                losses = step_on(s)
            return losses

        # clock ramp (untimed) so a short timed region does not run at idle clocks
        t_end = time.perf_counter() + ramp_s
        while time.perf_counter() < t_end:
            run_rotation()
        for _ in range((warmup + n_sets - 1) // n_sets):
            run_rotation()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(q):                      # q * n_sets + r == steps, exactly
            last = run_rotation()
        for i in range(r):
            if graph_ok:
                singles[i][0].replay()
                last = singles[i][1]
            else:
                last = step_on(dev_sets[i])
        e1.record()
        torch.cuda.synchronize()
        self.last_step = (dev_sets[r - 1] if r else dev_sets[-1], last)
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, graph_ok

    def kernel_alone(self, n_p=200, clocks_mhz=None):
        """The dominant kernel (mdn::fused_tile_kernel) timed ALONE: CUDA events recorded around its launch on the launching
        stream inside the library (mdn_loss_fused_profile), rotating input sets -> the `roofline` object."""
        from mdn_sfm_b200 import _cabi, fused as fz
        from mdn_sfm_b200.loss_functions import _mode_bits
        args, opt, dev, B = self.args, self.opt, self.dev, self.B
        post, bits = _mode_bits(self.mode, "SN")
        flags = bits | _cabi.TERM_SMOOTH | _cabi.TERM_CONSIS | _cabi.TERM_PHOTO | _cabi.OPT_SSIM
        lib = _cabi.lib()
        stream = torch.cuda.current_stream().cuda_stream
        calls = []
        for s in self.dev_sets:
            inputs, flows, mobiles, cams, inst = s
            with torch.no_grad():
                data, _, poses = self.loss_mod._scale_data(inputs, self.ids, flows, mobiles, inst, list(self.scales), cams, post, bits)
            cfg = fz.FusedConfig(batch=B, n_pairs=2, post=post, mask_mode=_cabi.MASK_MIN, flags=flags,
                                 threshold=opt.threshold if post != 0 else None, alpha=opt.alpha, w_d2_sim=opt.w_d2_sim,
                                 w_e=opt.w_e, w_s=opt.w_s, w_c=opt.w_c, w_p=opt.w_p, inst_ready=self.loss_mod._inst_ready)
            need = [{"flow": [True, True], "mob": [True, True], "fmat": [False, False]} for _ in data]
            g_cams = [torch.empty_like(c) for c in poses[1]]
            loss_out, grads, _, call = fz.run_fused(cfg, data, need, lib, poses=([c.detach() for c in poses[1]], poses[2]), g_cams=g_cams)
            ws = fz._workspace(dev, call.workspace_bytes(lib))
            calls.append((call, loss_out, ws, grads))
        torch.cuda.synchronize()
        n_k = max(100, min(args.steps, 1000)) if n_p >= 200 else n_p
        for i in range(20):
            c = calls[i % len(calls)]
            c[0].run(lib, c[1], c[2], stream)
            c[0].keep = c[0].keep[:-2]
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for i in range(n_k):
            c = calls[i % len(calls)]
            c[0].run(lib, c[1], c[2], stream)
            c[0].keep = c[0].keep[:-2]
        k1.record()
        torch.cuda.synchronize()
        call_ms = k0.elapsed_time(k1) / n_k          # whole mdn_loss_fused call: repack + fused + finish, back to back
        parts = [0.0, 0.0, 0.0]
        for i in range(n_p):
            c = calls[i % len(calls)]
            pm = c[0].profile(lib, c[1], c[2], stream)
            for j in range(3):
                parts[j] += pm[j] / n_p
        repack_ms, kernel_ms, finish_ms = parts
        del calls
        alg_bytes = algorithmic_bytes_per_frame(self.H, self.W, self.scales, self.with_inst) * B
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        # ncu numbers of this exact kernel build (profiles/traffic.json carries the hash of the sources it was captured from);
        # a different build prints null rather than a stale number
        traffic = winst = None
        shape_key = "%dx%d" % (self.H, self.W)
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tj.get("source_hash") == source_hash() and self.mode in tj.get("modes", ["T"]):
                ent = tj.get(shape_key) or {}
                traffic, winst = ent.get("dram_bytes"), ent.get("warp_instructions")
        except Exception:
            pass
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": "mdn::fused_tile_kernel, timed alone with CUDA events around its launch (mdn_loss_fused_profile), mean of %d launches on rotating input sets" % n_p,
                "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "other_kernels_of_the_call_ms": {"mdn::ref_pack_kernel": repack_ms, "mdn::finish_kernel": finish_ms,
                                                 "whole mdn_loss_fused call, back to back": call_ms},
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"}
        if winst and clocks_mhz:
            # what actually bounds the kernel (DESIGN.md section 4): issued warp-instructions (ncu smsp__inst_executed.sum of this
            # build) against 148 SMs x 4 schedulers x 1 instruction / clock at the SM clock sampled during the run
            issue_peak = 148 * 4 * clocks_mhz * 1e6
            roof["issue_roofline"] = {"warp_instructions_per_launch": winst, "achieved_ginst_s": winst / (kernel_ms * 1e-3) / 1e9,
                                      "peak_ginst_s": issue_peak / 1e9, "frac": winst / (kernel_ms * 1e-3) / issue_peak,
                                      "sm_mhz": clocks_mhz}
        return roof


def dump_outputs(directory, last_step):
    """Writes what one step of the loss path hands its caller -- the loss terms and d/dflow, d/dmobile, d/dpose -- as
    float32 `directory/<name>.npy`, so that two builds run with the same arguments can be compared output for output.
    When the gradients together exceed DUMP_BYTES, each one larger than 4096 elements is replaced by the same fixed
    fraction of its elements, taken at indices drawn (sorted) from numpy's default_rng(0): the same indices in every run."""
    import numpy as np
    (_, flows, mobiles, cams, _), losses = last_step
    tag = lambda v: str(v).replace("-", "m")
    arrays = {("loss" if k == "loss" else "loss_" + k): v for k, v in losses.items() if torch.is_tensor(v)}
    for prefix, d in (("grad_flow", flows), ("grad_mobile", mobiles)):
        for (_, i, s), v in d.items():
            arrays["%s_%s_s%d" % (prefix, tag(i), s)] = v.grad
    for i, v in cams.items():
        arrays["grad_cam_%s" % tag(i)] = v.grad
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    large = {k for k, a in arrays.items() if a.size > 4096}
    large_bytes = sum(arrays[k].nbytes for k in large)
    small_bytes = sum(a.nbytes for a in arrays.values()) - large_bytes
    headers = 1024 * len(arrays)     # an .npy header takes 128 bytes for arrays of this rank; the files stay under the cap
    keep = min(1.0, (DUMP_BYTES - headers - small_bytes) / max(large_bytes, 1))
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        if keep < 1.0 and k in large:
            idx = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(directory, k + ".npy"), a)
    return keep


def host_copy_ceiling(dev, world, nbytes=256 << 20, reps=4):
    """Pinned host -> device bandwidth of plain `reps` x 256 MB cudaMemcpyAsync on every rank AT THE SAME TIME (GB/s of this
    rank, min over ranks): what the host's PCIe / memory system gives the e2e upload when all ranks pull together.
    (Measured on this pool, scratch runs of round 2: the same copy lands anywhere between 14 and 55 GB/s from one pinned
    allocation to the next -- NUMA placement of the pinned pages on a shared host -- and small copies scatter most; large
    copies, the best of five rounds, give the stable upper figure.)"""
    import torch.distributed as dist
    from mdn_sfm_b200.staging import pinned_empty
    h = pinned_empty(nbytes, dev)          # on the GPU's own NUMA node, like BatchStager's slabs
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    for _ in range(4):
        d.copy_(h, non_blocking=True)
    torch.cuda.synchronize()
    gbs = 0.0
    for _ in range(5):
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            d.copy_(h, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        gbs = max(gbs, reps * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    if world > 1:
        t = torch.tensor([gbs], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        gbs = float(t.item())
    return gbs


def gpu_eager_baseline(args, wl, n=5):
    """BASELINE.md section 3's second comparator: the reference's own op sequence (oracle/restate.py, eager ATen launches)
    on THIS GPU -- what upstream's default `cuda=True` path (loss_functions.py:12,18,172) costs -- same workload, same inputs,
    forward + backward, CUDA events."""
    from oracle import restate
    inputs, flows, mobiles, cams, inst = wl.dev_sets[0]
    weights = [w.to(wl.dev) for w in restate.gauss_distance_weight(4, wl.H, wl.W)] if wl.mode == "TG" else None

    def step():
        for d in (flows, mobiles, cams):
            for v in d.values():
                v.grad = None
        _, losses = restate.loss_forward(wl.opt, inputs, [-1, 1], flows, mobiles, inst, list(wl.scales), cams, mode=wl.mode,
                                         weights=weights, photometric=True, ssim_on=True)
        losses["loss"].backward()

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    return {"value": wl.B / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "steps": n, "kind": "port",
            "what": "oracle/restate.py (the reference's ATen op sequence, pinned bit-exactly to the reference) run eagerly on this GPU: "
                    "the upstream default cuda=True path, same workload and inputs, fwd + bwd, anomaly detection off"}


def run_ours(args):
    import torch.distributed as dist
    from mdn_sfm_b200 import _cabi, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _cabi.lib()   # fail loudly right here if the extension is missing

    H, W, scales = workload(args)
    B = args.batch
    wl = Workload(args, args.mode, H, W, scales, dev, world, rank, args.flow, args.sets)
    host_sets, dev_sets, ids, with_inst, step_on = wl.host_sets, wl.dev_sets, wl.ids, wl.with_inst, wl.step_on
    sampler = ClockSampler(local)
    sampler.start()
    ms, graph_ok = wl.timed_steps(dev_sets, args.steps, args.warmup, 1.0)
    ms_per_step = ms / args.steps
    value = world * B * args.steps / (ms * 1e-3)
    clocks_now = sampler.summary()
    if args.dump_outputs and rank == 0:
        keep = dump_outputs(args.dump_outputs, wl.last_step)
        print("bench: last timed step's outputs written to %s%s" % (
            args.dump_outputs, "" if keep == 1.0 else " (gradients sampled: %.3g of their elements)" % keep), file=sys.stderr)

    # ---- dominant kernel alone
    roofline = wl.kernel_alone(200, clocks_now.get("sm_mhz"))
    alg_bytes = roofline["algorithmic_bytes_per_launch"]

    # ---- e2e: public API, host buffers in, loss out, every step.
    # The batch lives in ONE pinned slab (the loader writes there); per step one cudaMemcpyAsync on a copy stream brings it to
    # the device, multi-buffered so the copy of step i+1 overlaps the kernels of step i.  DEFAULT path: the three full-resolution
    # frames cross PCIe as the loader holds them -- (B,H,W,3) uint8 -- and are normalised on the device (mdn_normalize_u8 = the
    # dataset's ArrayToTensor + Normalize, bit-identical); the pyramid levels are made on the device, the source frames directly
    # in the packed layout of the warp gather (no ref_pack_kernel in the step).  `e2e_fp32_frames` is the same step with the
    # fp32 NCHW frames the reference's loader produces (100 MB instead of 60 MB per step).
    from mdn_sfm_b200 import pyramid
    from mdn_sfm_b200.staging import BatchStager
    n_e2e = args.e2e_steps or min(args.steps, 100)
    host_loss = torch.empty((), dtype=torch.float32).pin_memory()
    leaf = lambda d: {kk: v.detach().requires_grad_(True) for kk, v in d.items()}
    # DS / DC: the Detectron2-style boolean instance masks of the batch cross PCIe every step too
    up_inst = lambda inst: {("inst", j): d["instances"].pred_masks for j, d in enumerate(inst)} if inst is not None else {}
    to_u8 = lambda x: ((x * 0.225 + 0.45) * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    u8_part = lambda d: {kk: to_u8(v) for kk, v in d.items() if kk[0] == "color" and kk[2] == 0}
    f32_part = lambda d: {kk: v for kk, v in d.items() if kk[0] == "color" and kk[2] == 0}
    rest_part = lambda d: {kk: v for kk, v in d.items() if kk[0] != "color"}

    def make_e2e(frames_part, from_frames, packed):
        st = BatchStager([frames_part(host_sets[0][0]), rest_part(host_sets[0][0])] + list(host_sets[0][1:4]) + [up_inst(host_sets[0][4])],
                         dev, n_buffers=len(host_sets))
        for k, hs in enumerate(host_sets):   # untimed: producing the batch in pinned memory is the loader's part
            st.fill(k, [frames_part(hs[0]), rest_part(hs[0])] + list(hs[1:4]) + [up_inst(hs[4])])

        def run(n, start_event=None):
            if start_event is not None:
                st.copy_stream.wait_event(start_event)
            st.upload(0)
            for i in range(n):
                if i + 1 < n:
                    st.upload(i + 1)
                st.wait(i)
                v = st._dev_views[i % st.n_buffers]
                inputs_i = dict(v[1])
                for kk, fr in v[0].items():
                    inputs_i[kk] = from_frames(fr)
                pyramid.add_pyramid_levels(inputs_i, [0] + ids, list(scales), packed_sources=packed)
                inst_i = [{"instances": synthetic.SyntheticInstances(v[5][("inst", j)])} for j in range(len(v[5]))] if with_inst else None
                loss = step_on((inputs_i, leaf(v[2]), leaf(v[3]), leaf(v[4]), inst_i))["loss"]
                st.release(i)
                host_loss.copy_(loss.detach(), non_blocking=True)
        return st, run

    def time_e2e(run, n_runs):
        run(2 * len(host_sets) + 4)            # warm-up: every buffer, the allocator pools and the copy stream have been through once
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        runs = []
        for _ in range(n_runs):
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            run(n_e2e, f0)
            f1.record()
            torch.cuda.synchronize()
            ms_run = f0.elapsed_time(f1)
            if world > 1:
                t = torch.tensor([ms_run], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_run = float(t.item())
            runs.append(ms_run / n_e2e)
        return sorted(runs)

    ceiling = host_copy_ceiling(dev, world)
    st8, run8 = make_e2e(u8_part, pyramid.frames_from_u8, True)
    runs8 = time_e2e(run8, 5)
    e2e_ms = runs8[len(runs8) // 2]            # median of 5 runs of n_e2e steps (max over ranks each)
    e2e_value = world * B / (e2e_ms * 1e-3)
    h2d_bytes = st8.nbytes
    e2e = {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4, "steps": n_e2e,
           "ms_per_step": e2e_ms, "runs_ms_per_step_sorted": runs8, "statistic": "median of 5 runs of %d steps (max over ranks per run)" % n_e2e,
           "h2d_gbs_achieved": h2d_bytes / (e2e_ms * 1e-3) / 1e9, "host_copy_ceiling_gbs": ceiling,
           "frac_of_host_copy_ceiling": h2d_bytes / (e2e_ms * 1e-3) / 1e9 / ceiling,
           "host_copy_ceiling": "4 x 256 MB pinned cudaMemcpyAsync on every rank at the same time, best of 5 rounds, min over ranks",
           "path": "mdn_sfm_b200.staging.BatchStager (one pinned slab -> one H2D copy per step on a copy stream, %d buffers: three "
                   "full-resolution frames as (B,H,W,3) uint8, flows, mobile maps, poses, intrinsics) + pyramid.frames_from_u8 "
                   "(ArrayToTensor + Normalize on the device) + pyramid.add_pyramid_levels(packed_sources=True) + "
                   "loss_functions.Loss.forward + backward (eager public API) + loss read back to pinned host memory" % len(host_sets)}
    del st8
    e2e_f32 = None
    if not args.no_second_flow:
        try:
            st32, run32 = make_e2e(f32_part, lambda fr: fr, False)
            runs32 = time_e2e(run32, 3)
            m32 = runs32[len(runs32) // 2]
            e2e_f32 = {"value": world * B / (m32 * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": st32.nbytes, "d2h_bytes_per_step": 4,
                       "steps": n_e2e, "ms_per_step": m32, "runs_ms_per_step_sorted": runs32,
                       "path": "as e2e, but the frames cross PCIe as fp32 NCHW (what the reference's loader holds after Normalize) and the "
                               "loss repacks the source frames itself (round 1's e2e)"}
            del st32
        except Exception as e:
            e2e_f32 = {"error": repr(e)}
    sampler.stop_flag = True
    sampler.join(timeout=1.0)

    # ---- the same workload on the other flow kind (short run, reported beside the headline, never instead of it)
    second = None
    if not args.no_second_flow and world == 1:
        other = "smooth" if args.flow == "iid" else "iid"
        wl2 = Workload(args, args.mode, H, W, scales, dev, world, rank, other, 2)
        n2 = max(50, args.steps // 4)
        ms2, _ = wl2.timed_steps(wl2.dev_sets, n2, max(3, args.warmup // 4), 0.3)
        second = {"flow": FLOW_DESC[other], "value": B * n2 / (ms2 * 1e-3), "unit": "frames/s", "ms_per_step": ms2 / n2, "steps": n2}
        del wl2

    # ---- the same step when the data side hands the source frames over already packed (SURVEY 8f-N3: the pyramid
    # producer writes (r, g, b, -) per pixel, ('color_packed', i, s)): no repack kernel inside the step.  Reported beside
    # the headline, never instead of it -- the headline takes the reference's NCHW inputs.
    packed_run = None
    if not args.no_second_flow and world == 1:
        try:
            pk_sets = []
            for s in dev_sets[:2]:
                inp = dict(s[0])
                for i in ids:
                    for sc in scales:
                        lvl = inp.pop(("color", i, sc))
                        inp[("color_packed", i, sc)] = pyramid.image_pyramid(lvl, [tuple(lvl.shape[-2:])], packed=True)[0]
                pk_sets.append((inp,) + tuple(s[1:]))
            n3 = max(50, args.steps // 4)
            ms3, _ = wl.timed_steps(pk_sets, n3, max(3, args.warmup // 4), 0.3)
            packed_run = {"inputs": "source frames as ('color_packed', i, s) from mdn_sfm_b200.pyramid (no ref_pack_kernel in the step)",
                          "value": B * n3 / (ms3 * 1e-3), "unit": "frames/s", "ms_per_step": ms3 / n3, "steps": n3}
            del pk_sets
        except Exception as e:
            packed_run = {"error": repr(e)}

    # ---- the reference's op sequence run eagerly on this GPU (N = 1)
    gpu_eager = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            gpu_eager = gpu_eager_baseline(args, wl)
        except Exception as e:
            gpu_eager = {"error": repr(e)}
    del wl, dev_sets, host_sets
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations, at every N (weak scaling, max over ranks like the headline): configs[3]
    # DS / DC with synthetic Detectron2-style instance masks, configs[4] full-resolution KITTI 375x1242 (scale 0 only)
    others = []
    if not args.no_other_configs and args.shape == "192x640" and args.mode == "T":
        for label, mode, shp in (("BASELINE configs[3]: DS mode", "DS", "192x640"), ("BASELINE configs[3]: DC mode", "DC", "192x640"),
                                 ("BASELINE configs[4]: T mode, 375x1242, scale 0", "T", "375x1242")):
            try:
                Ho, Wo = map(int, shp.split("x"))
                sc = (0, 1, 2, 3) if (Ho % 8 == 0 and Wo % 8 == 0) else (0,)
                wo = Workload(args, mode, Ho, Wo, sc, dev, world, rank, args.flow, 2)
                n_o = max(40, min(args.steps, 400) // 2)
                ms_o, _ = wo.timed_steps(wo.dev_sets, n_o, max(3, min(args.warmup, 40)), 0.2)
                ro = wo.kernel_alone(40, clocks_now.get("sm_mhz"))
                others.append({"workload": "%s + photometric + smooth + consistency, fwd+bwd, batch %d/GPU x %d GPU, 3x%dx%d, %d scale(s)" % (
                                   label, B, world, Ho, Wo, len(sc)),
                               "mode": mode, "height": Ho, "width": Wo, "value": world * B * n_o / (ms_o * 1e-3), "unit": "frames/s",
                               "ms_per_step": ms_o / n_o, "steps": n_o,
                               "roofline": {k: ro[k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "kernel_ms",
                                                               "algorithmic_bytes_per_launch", "other_kernels_of_the_call_ms")}})
                del wo
                torch.cuda.empty_cache()
            except Exception as e:
                others.append({"workload": label, "error": repr(e)})

    # ---- BASELINE configs[2]: the whole train step (stand-in nets on cuDNN -> TG loss -> backward -> DDP -> clip -> Adam)
    train = None
    if not args.no_train_step:
        try:
            train = measure_train_step(args, dev, world, rank, H, W, scales)
        except Exception as e:   # reported, never fatal for the headline line
            train = {"error": repr(e)}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        step, threads = cpu_reference_step_fn(args, H, W, scales)
        step()
        best = 1e30
        for _ in range(args.cpu_steps):
            t0 = time.perf_counter()
            step()
            best = min(best, time.perf_counter() - t0)
        cpu_base = {"value": B / best, "unit": "frames/s", "cores": threads, "kind": "port",
                    "sample": "best of %d steps of the same batch of %d frames (oracle/restate.py, eager torch on the host CPU, "
                              "%d threads, anomaly detection off)" % (args.cpu_steps, B, threads)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config_dict(args, H, W, scales, world),
                "cuda_graph": ("%d steps (one per input set) per graph launch" % args.sets) if graph_ok else False,
                "clocks": sampler.summary(),
                "e2e": e2e,
                "gpu_launches": 4 * args.steps,
                "launches_per_step": "mdn::ref_pack_kernel, mdn::fused_tile_kernel (builds the fundamental matrices from the poses), "
                                     "mdn::finish_kernel (loss scalars, d/dF, pose adjoint), mdn::scale_grads_kernel; "
                                     "(+ torch's ones_like fill for the upstream gradient)",
                "e2e_fp32_frames": e2e_f32, "other_flow": second, "packed_sources": packed_run, "other_configs": others,
                "train_step": train, "roofline": roofline, "cpu_baseline": cpu_base, "gpu_eager_baseline": gpu_eager,
                "kernel_source_hash": source_hash()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)
