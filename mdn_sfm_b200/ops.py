"""autograd nodes over the standalone C-ABI kernels (warp, point-set epipolar distance, SSIM)."""
from __future__ import annotations

import torch

from . import _cabi


def _c(t, what, dtype=torch.float32):
    return _cabi.check_tensor(t, dtype=dtype, what=what).contiguous()


class FlowWarpFn(torch.autograd.Function):
    """inverse_warp's sampling (loss_utils.py:27-34): flow in pixels -> (warped, grid, valid)."""

    @staticmethod
    def forward(ctx, ref, flow, warp_flags, want_warp, library):
        library = library or _cabi.lib()
        B, _, h, w = flow.shape
        C = ref.shape[1] if want_warp else 0
        warped = torch.empty((B, C, h, w), dtype=torch.float32, device=flow.device) if want_warp else None
        grid = torch.empty((B, h, w, 2), dtype=torch.float32, device=flow.device)
        valid = torch.empty((B, h, w), dtype=torch.uint8, device=flow.device)
        library.call("mdn_flow_warp_fwd", _cabi.ptr(ref) if want_warp else None, flow.data_ptr(), _cabi.ptr(warped),
                     grid.data_ptr(), valid.data_ptr(), B, C, h, w, int(warp_flags), _cabi.stream_ptr(flow), dev=flow)
        ctx.library, ctx.warp_flags = library, int(warp_flags)
        ctx.save_for_backward(ref, flow)
        ctx.mark_non_differentiable(grid, valid)
        if not want_warp:
            warped = torch.empty(0, device=flow.device)
            ctx.mark_non_differentiable(warped)
        return warped, grid, valid

    @staticmethod
    def backward(ctx, g_warped, _g1, _g2):
        ref, flow = ctx.saved_tensors
        if ctx.needs_input_grad[0]:
            raise NotImplementedError("mdn_sfm_b200: gradient w.r.t. the sampled image is not implemented "
                                      "(images are data in the MDN_SfM loss path)")
        B, C, h, w = ref.shape
        g_flow = torch.empty_like(flow)
        ctx.library.call("mdn_flow_warp_bwd", ref.data_ptr(), flow.data_ptr(), g_warped.contiguous().data_ptr(),
                         g_flow.data_ptr(), B, C, h, w, ctx.warp_flags, _cabi.stream_ptr(flow), dev=flow)
        return None, g_flow, None, None, None


class EpipolarPointsFn(torch.autograd.Function):
    """Signed epipolar distance of arbitrary point sets given F (loss_utils.py:64-67)."""

    @staticmethod
    def forward(ctx, p1, p2, fmat, library):
        library = library or _cabi.lib()
        B, _, n = p1.shape
        out = torch.empty((B, 1, n), dtype=torch.float32, device=p1.device)
        library.call("mdn_epipolar_points_fwd", p1.data_ptr(), p2.data_ptr(), fmat.data_ptr(), out.data_ptr(), B, n,
                     _cabi.stream_ptr(p1), dev=p1)
        ctx.library = library
        ctx.save_for_backward(p1, p2, fmat)
        return out

    @staticmethod
    def backward(ctx, g_out):
        p1, p2, fmat = ctx.saved_tensors
        B, _, n = p1.shape
        lib = ctx.library
        g1 = torch.empty_like(p1) if ctx.needs_input_grad[0] else None
        g2 = torch.empty_like(p2) if ctx.needs_input_grad[1] else None
        gF = torch.empty_like(fmat) if ctx.needs_input_grad[2] else None
        nbytes = lib.cdll.mdn_epipolar_points_workspace_bytes(B, n)
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=p1.device)
        lib.call("mdn_epipolar_points_bwd", p1.data_ptr(), p2.data_ptr(), fmat.data_ptr(), g_out.contiguous().data_ptr(),
                 _cabi.ptr(g1), _cabi.ptr(g2), _cabi.ptr(gF), B, n, ws.data_ptr(), nbytes, _cabi.stream_ptr(p1), dev=p1)
        return g1, g2, gF, None


class SsimFn(torch.autograd.Function):
    """networks/layers.py:164-178."""

    @staticmethod
    def forward(ctx, x, y, library):
        library = library or _cabi.lib()
        out = torch.empty_like(x)
        h, w = x.shape[-2:]
        planes = x.numel() // (h * w)
        library.call("mdn_ssim_fwd", x.data_ptr(), y.data_ptr(), out.data_ptr(), planes, h, w, _cabi.stream_ptr(x), dev=x)
        ctx.library = library
        ctx.save_for_backward(x, y)
        return out

    @staticmethod
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        h, w = x.shape[-2:]
        planes = x.numel() // (h * w)
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(y) if ctx.needs_input_grad[1] else None
        ctx.library.call("mdn_ssim_bwd", x.data_ptr(), y.data_ptr(), g.contiguous().data_ptr(), _cabi.ptr(gx),
                         _cabi.ptr(gy), planes, h, w, _cabi.stream_ptr(x), dev=x)
        return gx, gy, None

