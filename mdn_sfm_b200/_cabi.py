"""ctypes binding of include/mdn_loss.h -- the only door between Python and the CUDA kernels.

There is no CPU path: if ``libmdn_loss.so`` is missing or a tensor is not a CUDA tensor the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

MAX_SCALES, MAX_PAIRS = 4, 2
POST_SN, POST_T, POST_TG = 0, 1, 2
MASK_MIN, MASK_OWN, MASK_SHARED = 0, 1, 2
TERM_EPIPOLAR, TERM_PHOTO, TERM_SMOOTH, TERM_CONSIS = 1, 2, 4, 8
OPT_SSIM, OPT_INST_MASK, OPT_CROSS_ENT, OPT_GRADS, OPT_CUDA_ARITH = 16, 32, 64, 128, 256
OPT_PAD_BORDER, OPT_PAD_REFLECTION = 512, 1024
PAD_FLAG = {"zeros": 0, "border": OPT_PAD_BORDER, "reflection": OPT_PAD_REFLECTION}      # grid_sample padding_mode -> MdnFlags
WARP_FLOWWARP_NORM, WARP_CUDA_ARITH = 1, 2
WARP_PAD = {"zeros": 0, "border": 4, "reflection": 8}      # bits 2-3 of warp_flags
OUT_LOSS, OUT_EPIP, OUT_SMOOTH, OUT_CONSIS, OUT_PHOTO, OUT_APPLIED, OUT_COUNT = 0, 1, 2, 3, 4, 5, 8

ABI_VERSION = 4

_P = C.c_void_p
_PAIR = _P * MAX_PAIRS


class MdnScale(C.Structure):
    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("flow_sx", C.c_float), ("flow_sy", C.c_float),
                ("scale_div", C.c_float), ("pad_", C.c_float),
                ("tgt", _P), ("ref", _PAIR), ("flow", _PAIR), ("mob", _PAIR), ("fmat", _PAIR),
                ("weight", _P), ("inst", _P),
                ("g_flow", _PAIR), ("g_mob", _PAIR), ("g_fmat", _PAIR),
                ("post_map", _PAIR), ("ori_map", _PAIR), ("warped", _PAIR), ("diff", _PAIR), ("valid", _PAIR),
                ("ssim_map", _PAIR), ("ref_packed", _PAIR)]


class MdnLossDesc(C.Structure):
    _fields_ = [("batch", C.c_int32), ("n_scales", C.c_int32), ("n_pairs", C.c_int32), ("post", C.c_int32),
                ("mask_mode", C.c_int32), ("flags", C.c_int32), ("threshold", C.c_double), ("alpha", C.c_float),
                ("w_d2_sim", C.c_float), ("w_e", C.c_float), ("w_s", C.c_float), ("w_c", C.c_float),
                ("w_p", C.c_float), ("scale", MdnScale * MAX_SCALES),
                ("cam", _PAIR), ("g_cam", _PAIR), ("inv_K", _P * MAX_SCALES),
                ("axisangle", _PAIR), ("translation", _PAIR), ("g_axisangle", _PAIR), ("g_translation", _PAIR),
                ("inst_ready", _P)]


LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib", "libmdn_loss.so")

EXPORTS = ("mdn_version", "mdn_last_error_string", "mdn_loss_workspace_bytes", "mdn_loss_fused", "mdn_loss_fused_profile",
           "mdn_loss_scale_grads",
           "mdn_epipolar_points_fwd", "mdn_epipolar_points_bwd", "mdn_epipolar_points_workspace_bytes",
           "mdn_flow_warp_fwd", "mdn_flow_warp_bwd", "mdn_ssim_fwd", "mdn_ssim_bwd", "mdn_binary_image",
           "mdn_instance_mask_union", "mdn_instance_mask_union_table", "mdn_instance_mask_resize", "mdn_instance_mask_resize_workspace_bytes", "mdn_image_pyramid", "mdn_image_pyramid_packed", "mdn_normalize_u8",
           "mdn_mask_confusion", "mdn_mask_confusion_workspace_bytes", "mdn_flow_errors", "mdn_flow_errors_workspace_bytes")


class Library:
    """A loaded libmdn_loss.so with typed entry points; every call checks the status code."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise RuntimeError("%s not found: build it with `python -m mdn_sfm_b200.build` "
                               "(there is no CPU fallback for the loss path)" % path)
        self.path = path
        d = self.cdll = C.CDLL(path)
        i32, i64, sz, f32 = C.c_int32, C.c_int64, C.c_size_t, C.c_float
        D = C.POINTER(MdnLossDesc)
        sig = {
            "mdn_version": (C.c_int, []),
            "mdn_last_error_string": (C.c_char_p, []),
            "mdn_loss_workspace_bytes": (sz, [D]),
            "mdn_loss_fused": (C.c_int, [D, _P, _P, sz, _P]),
            "mdn_loss_fused_profile": (C.c_int, [D, _P, _P, sz, _P, C.POINTER(C.c_float)]),
            "mdn_loss_scale_grads": (C.c_int, [D, _P, _P, _P]),
            "mdn_epipolar_points_fwd": (C.c_int, [_P, _P, _P, _P, i32, i64, _P]),
            "mdn_epipolar_points_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, i32, i64, _P, sz, _P]),
            "mdn_epipolar_points_workspace_bytes": (sz, [i32, i64]),
            "mdn_flow_warp_fwd": (C.c_int, [_P, _P, _P, _P, _P, i32, i32, i32, i32, i32, _P]),
            "mdn_flow_warp_bwd": (C.c_int, [_P, _P, _P, _P, i32, i32, i32, i32, i32, _P]),
            "mdn_ssim_fwd": (C.c_int, [_P, _P, _P, i32, i32, i32, _P]),
            "mdn_ssim_bwd": (C.c_int, [_P, _P, _P, _P, _P, i32, i32, i32, _P]),
            "mdn_binary_image": (C.c_int, [_P, _P, i64, f32, _P]),
            "mdn_instance_mask_union": (C.c_int, [C.POINTER(_P), C.POINTER(i32), _P, i32, i64, _P]),
            "mdn_instance_mask_union_table": (C.c_int, [_P, _P, _P, i32, i64, _P]),
            "mdn_instance_mask_resize": (C.c_int, [_P, i32, i32, i32, C.POINTER(_P), C.POINTER(i32), C.POINTER(i32), i32, _P, sz, _P]),
            "mdn_image_pyramid": (C.c_int, [_P, i32, i32, i32, C.POINTER(_P), C.POINTER(i32), C.POINTER(i32), i32, _P, sz, _P]),
            "mdn_normalize_u8": (C.c_int, [_P, _P, i32, i32, i32, C.POINTER(f32), C.POINTER(f32), _P]),
            "mdn_image_pyramid_packed": (C.c_int, [_P, i32, i32, i32, C.POINTER(_P), C.POINTER(i32), C.POINTER(i32), i32, _P, sz, _P]),
            "mdn_instance_mask_resize_workspace_bytes": (sz, [i32, i32, i32, C.POINTER(i32), C.POINTER(i32), i32]),
            "mdn_mask_confusion": (C.c_int, [_P, _P, _P, i32, _P, i32, i64, _P, sz, _P]),
            "mdn_mask_confusion_workspace_bytes": (sz, [i32, i32]),
            "mdn_flow_errors": (C.c_int, [_P, i32, i32, f32, f32, _P, _P, _P, i32, i32, i32, i32, f32, f32, _P, _P, _P, sz, _P]),
            "mdn_flow_errors_workspace_bytes": (sz, [i32, i32, i32, i32, i32, i32]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(d, name)
            fn.restype, fn.argtypes = res, args
        if d.mdn_version() != ABI_VERSION:
            raise RuntimeError("libmdn_loss ABI version mismatch")

    def call(self, name, *args, dev=None):
        """Calls an entry point and raises on a non-zero status.  `dev` (a tensor or a device) names the CUDA device the
        launches belong to: it is made current for the duration of the call, so a stream of that device is never used
        from another current device (every call site passes one of the tensors it hands over)."""
        if dev is not None:
            dev = getattr(dev, "device", dev)
            if getattr(dev, "type", None) == "cuda":
                with torch.cuda.device(dev):
                    rc = getattr(self.cdll, name)(*args)
            else:
                rc = getattr(self.cdll, name)(*args)
        else:
            rc = getattr(self.cdll, name)(*args)
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (name, rc, self.cdll.mdn_last_error_string().decode()))


_lib = None


def lib() -> Library:
    global _lib
    if _lib is None:
        _lib = Library()
    return _lib


def check_tensor(t, dtype=torch.float32, what="tensor"):
    """The product only accepts CUDA tensors; anything else is an error, never a silent CPU path."""
    if not t.is_cuda:
        raise RuntimeError("mdn_sfm_b200: %s must be a CUDA tensor (got %s); the loss path has no CPU implementation"
                           % (what, t.device))
    if t.dtype != dtype:
        raise TypeError("mdn_sfm_b200: %s must be %s (got %s)" % (what, dtype, t.dtype))
    return t


def stream_ptr(ref_tensor):
    return torch.cuda.current_stream(ref_tensor.device).cuda_stream if ref_tensor.is_cuda else 0


def ptr_array(tensors):
    """Host array of device pointers (the `const float* const*` arguments of the C ABI)."""
    return (_P * len(tensors))(*[t.data_ptr() for t in tensors])


def ptr(t):
    return None if t is None else t.data_ptr()


class FusedCall:
    """Fills an MdnLossDesc from tensors and keeps them alive for the duration of the (asynchronous) call."""

    PAIR_FIELDS = ("ref", "flow", "mob", "fmat", "g_flow", "g_mob", "g_fmat", "post_map", "ori_map", "warped", "diff",
                   "valid", "ssim_map", "ref_packed")
    ONE_FIELDS = ("tgt", "weight", "inst")

    def __init__(self, *, batch, n_pairs, post, mask_mode, flags, threshold=0.0, alpha=0.0, w_d2_sim=0.0, w_e=1.0,
                 w_s=1.0, w_c=1.0, w_p=1.0):
        d = self.desc = MdnLossDesc()
        d.batch, d.n_scales, d.n_pairs, d.post, d.mask_mode, d.flags = batch, 0, n_pairs, post, mask_mode, flags
        d.threshold = 0.0 if threshold is None else float(threshold)
        d.alpha, d.w_d2_sim, d.w_e, d.w_s, d.w_c, d.w_p = alpha, w_d2_sim, w_e, w_s, w_c, w_p
        self.keep = []

    def add_scale(self, height, width, flow_sx, flow_sy, scale_div, **tensors):
        d = self.desc
        S = d.scale[d.n_scales]
        d.n_scales += 1
        S.height, S.width, S.flow_sx, S.flow_sy, S.scale_div = height, width, flow_sx, flow_sy, scale_div
        for name in self.ONE_FIELDS:
            t = tensors.pop(name, None)
            if t is not None:
                setattr(S, name, t.data_ptr())
                self.keep.append(t)
        for name in self.PAIR_FIELDS:
            seq = tensors.pop(name, None)
            if seq is None:
                continue
            arr = getattr(S, name)
            for k, t in enumerate(seq):
                if t is not None:
                    arr[k] = t.data_ptr()
                    self.keep.append(t)
        if tensors:
            raise TypeError("unknown scale tensors: %s" % sorted(tensors))
        return self

    def set_poses(self, cams, inv_Ks, g_cams=None):
        """Poses instead of fundamental matrices (MdnLossDesc.cam / inv_K / g_cam): cams = one (B,4,4) tensor per pair,
        inv_Ks = one (B,4,4) tensor per scale (in add_scale order), g_cams = gradient buffers or None."""
        d = self.desc
        for p, t in enumerate(cams):
            d.cam[p] = t.data_ptr()
        for k, t in enumerate(inv_Ks):
            d.inv_K[k] = t.data_ptr()
        self.keep += list(cams) + list(inv_Ks)
        if g_cams is not None:
            for p, t in enumerate(g_cams):
                if t is not None:
                    d.g_cam[p] = t.data_ptr()
                    self.keep.append(t)
        return self

    def set_pose_params(self, axisangles, translations, inv_Ks, g_axisangles=None, g_translations=None):
        """Pose PARAMETERS instead of pose matrices (MdnLossDesc.axisangle / translation, ABI 3): one (B,1,1,3) tensor per
        pair each, as PoseNet emits them; the kernels run transformation_from_parameters themselves and return
        d(loss)/d(axisangle), d(loss)/d(translation) into the given buffers."""
        d = self.desc
        for p, (a, t) in enumerate(zip(axisangles, translations)):
            d.axisangle[p], d.translation[p] = a.data_ptr(), t.data_ptr()
        for k, t in enumerate(inv_Ks):
            d.inv_K[k] = t.data_ptr()
        self.keep += list(axisangles) + list(translations) + list(inv_Ks)
        for name, seq in (("g_axisangle", g_axisangles), ("g_translation", g_translations)):
            if seq is not None:
                arr = getattr(d, name)
                for p, t in enumerate(seq):
                    if t is not None:
                        arr[p] = t.data_ptr()
                        self.keep.append(t)
        return self

    def workspace_bytes(self, library):
        n = library.cdll.mdn_loss_workspace_bytes(C.byref(self.desc))
        if n == 0:
            raise RuntimeError("mdn_loss_workspace_bytes: %s" % library.cdll.mdn_last_error_string().decode())
        return n

    def run(self, library, loss_out, workspace, stream):
        self.keep += [loss_out, workspace]
        # launches go to the tensors' device even when it is not the current one
        library.call("mdn_loss_fused", C.byref(self.desc), loss_out.data_ptr(), workspace.data_ptr(),
                     workspace.numel() * workspace.element_size(), stream, dev=loss_out)

    def profile(self, library, loss_out, workspace, stream):
        """Blocking measurement aid: returns (repack_ms, fused_kernel_ms, finish_ms) of one call (mdn_loss_fused_profile)."""
        ms = (C.c_float * 3)()
        library.call("mdn_loss_fused_profile", C.byref(self.desc), loss_out.data_ptr(), workspace.data_ptr(),
                     workspace.numel() * workspace.element_size(), stream, ms, dev=loss_out)
        return float(ms[0]), float(ms[1]), float(ms[2])

    def scale_grads(self, library, g, applied, stream):
        library.call("mdn_loss_scale_grads", C.byref(self.desc), g.data_ptr(), applied.data_ptr(), stream, dev=applied)
