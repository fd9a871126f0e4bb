"""The per-pixel arithmetic of mdn_flow_errors (include/mdn_loss.h) restated with torch elementwise ops, shared by the flow
evaluation tests.  Same operations in the same order, one rounding per op, so it reproduces the kernel bit for bit on the
CPU and on the GPU: the scalars are 0-dim fp32 tensors on the data's device (ATen's CUDA `tensor / python_scalar`
multiplies by a reciprocal; tensor / tensor divides), gathers use index tensors, sums are float64.  torch's fp32 sqrt on
the CPU is not always correctly rounded (it is on the GPU), so `sqrt_rn` takes it in float64 and rounds once, which for
the square root of an fp32 number is the correctly rounded fp32 result."""
import torch


def _f32(v, dev):
    return torch.tensor(v, dtype=torch.float32, device=dev)


def taps(n_out, n_in, dev):
    """Source index pair and weights of ATen's upsample_bilinear2d (align_corners=False) along one axis."""
    r = _f32(float(n_in), dev) / _f32(float(n_out), dev)
    i = torch.arange(n_out, device=dev, dtype=torch.float32)
    s = r * (i + _f32(0.5, dev)) - _f32(0.5, dev)
    s = torch.where(s < 0, torch.zeros_like(s), s)
    i0 = torch.clamp(s.to(torch.int64), max=n_in - 1)
    i1 = i0 + (i0 < n_in - 1).to(torch.int64)
    l1 = s - i0.to(torch.float32)
    l0 = _f32(1.0, dev) - l1
    return i0, i1, l0, l1


def upsample(flow, H, W):
    """(B, C, h, w) -> (B, C, H, W): ly0*(lx0*F00 + lx1*F01) + ly1*(lx0*F10 + lx1*F11), each op rounded on its own."""
    dev = flow.device
    y0, y1, ly0, ly1 = taps(H, flow.shape[-2], dev)
    x0, x1, lx0, lx1 = taps(W, flow.shape[-1], dev)
    Y0, Y1, X0, X1 = y0[:, None], y1[:, None], x0[None, :], x1[None, :]
    LY0, LY1 = ly0.view(1, 1, H, 1), ly1.view(1, 1, H, 1)
    LX0, LX1 = lx0.view(1, 1, 1, W), lx1.view(1, 1, 1, W)
    a = LX0 * flow[:, :, Y0, X0] + LX1 * flow[:, :, Y0, X1]
    b = LX0 * flow[:, :, Y1, X0] + LX1 * flow[:, :, Y1, X1]
    return LY0 * a + LY1 * b


def sqrt_rn(x):
    return torch.sqrt(x.to(torch.float64)).to(torch.float32)


def pixel_errors(u, v, gu, gv, abs_thr, rel_thr):
    """e, m and the outlier flag from flows already in pixels (steps 4-5)."""
    dev = u.device
    du, dv = u - gu, v - gv
    e = sqrt_rn(du * du + dv * dv)
    m = sqrt_rn(gu * gu + gv * gv)
    out = (e > _f32(abs_thr, dev)) & ((e / m) > _f32(rel_thr, dev))
    return e, out


def reduce(e, out, valid, region, R):
    """Step 6: per (sample, region) [valid, outliers] and the float64 sum of e over the counted pixels."""
    B, dev = e.shape[0], e.device
    lab = torch.zeros_like(e, dtype=torch.int64) if region is None else region.reshape(e.shape).to(torch.int64)
    counted = (valid.reshape(e.shape) != 0) & (lab < R)
    key = (torch.arange(B, device=dev).view(B, 1, 1) * R + lab)[counted]
    n = torch.bincount(key, minlength=B * R)
    o = torch.bincount(key[out[counted]], minlength=B * R)
    s = torch.zeros(B * R, dtype=torch.float64, device=dev).index_add_(0, key, e[counted].to(torch.float64))
    return {"valid": n.view(B, R), "outliers": o.view(B, R), "epe_sum": s.view(B, R)}


def replay(flow, gt, valid, region, R, scale, abs_thr, rel_thr, pixels=False):
    """flow (B, 2, h, w), gt (B, 2, H, W) fp32; valid / region (B, H, W); scale = (sx, sy) fp32 values.
    -> {"valid", "outliers", "epe_sum"} as flow_errors returns them (plus "f", "e", "out" per pixel with pixels=True)."""
    H, W = gt.shape[-2:]
    dev = flow.device
    f = upsample(flow, H, W)
    u = f[:, 0] * _f32(float(scale[0]), dev)
    v = f[:, 1] * _f32(float(scale[1]), dev)
    e, out = pixel_errors(u, v, gt[:, 0], gt[:, 1], abs_thr, rel_thr)
    res = reduce(e, out, valid, region, R)
    if pixels:
        res.update(f=f, e=e, out=out)
    return res
