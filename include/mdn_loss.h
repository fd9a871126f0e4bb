/*
 * mdn_loss.h -- C ABI of the B200-native MDN_SfM loss path (libmdn_loss.so).
 *
 * The upstream project (chenluchu/MDN_SfM) has no FFI / plugin layer: its loss path is a set of Python
 * callables (loss_functions.py, loss_utils.py, networks/layers.py, utils.py) made of ATen ops.  This header
 * is the boundary a maintainer binds INSTEAD of those ATen compositions; each entry point cites the
 * upstream lines it replaces.  The binding the reference side would add is a ctypes stub -- see
 * INTEGRATION.md and mdn_sfm_b200/_cabi.py.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name says host
 *   - all tensors are contiguous fp32 NCHW (instance masks / validity are uint8), 16-byte aligned
 *   - the caller owns every buffer including the workspace; entry points enqueue work on `stream`
 *     (a cudaStream_t passed as void*), never allocate, never synchronise, and are CUDA-graph capturable
 *   - return 0 on success, a negative MdnStatus otherwise; mdn_last_error_string() explains (thread local)
 *   - reductions are deterministic (two-stage, fixed order, no floating-point atomics)
 */
#ifndef MDN_LOSS_H_
#define MDN_LOSS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MDN_API __attribute__((visibility("default")))
#else
#define MDN_API
#endif

#define MDN_ABI_VERSION 3
#define MDN_MAX_SCALES 4
#define MDN_MAX_PAIRS 2

typedef enum MdnStatus {
  MDN_OK = 0,
  MDN_ERR_BAD_SHAPE = -1,      /* batch/height/width/n_scales/n_pairs out of range (h,w >= 2 required)      */
  MDN_ERR_NULL_POINTER = -2,   /* a tensor the requested terms need is NULL                                 */
  MDN_ERR_MISALIGNED = -3,     /* a tensor pointer is not 16-byte aligned                                   */
  MDN_ERR_UNSUPPORTED = -4,    /* unknown mode / mask mode / padding mode                                   */
  MDN_ERR_WORKSPACE = -5,      /* workspace too small (see mdn_loss_workspace_bytes)                        */
  MDN_ERR_CUDA = -6            /* a CUDA runtime call failed                                                */
} MdnStatus;

/* Epipolar post-processing of |e| (SURVEY.md section 8a-M):
 *   SN  post_process_epipolar_1        loss_utils.py:92-99   (per-sample max normalise, square)
 *   T   post_pro_epipolar_weighted     loss_utils.py:81-89   (divide by threshold, square)
 *   TG  same with the Gaussian distance weight of utils.py:355-379 (threshold, then weight, square) */
typedef enum MdnPost { MDN_POST_SN = 0, MDN_POST_T = 1, MDN_POST_TG = 2 } MdnPost;

/* Which mobile mask a (target, source) pair is masked with:
 *   MIN     m = min(mob[0], mob[1]) for both pairs, gradient to the arg-min (first on ties) -- loss_functions.py:176-178,188
 *   OWN     pair i uses mob[i]                                                             -- --disable_min, loss_functions.py:183-186
 *   SHARED  both pairs use mob[0] as given (LossModule.forward called directly with a mask) -- loss_functions.py:27            */
typedef enum MdnMaskMode { MDN_MASK_MIN = 0, MDN_MASK_OWN = 1, MDN_MASK_SHARED = 2 } MdnMaskMode;

enum MdnFlags {
  MDN_TERM_EPIPOLAR   = 1 << 0,  /* LossModule.epipolar_loss          loss_functions.py:117-138              */
  MDN_TERM_PHOTO      = 1 << 1,  /* LossModule.photo_metric_loss      loss_functions.py:107-115              */
  MDN_TERM_SMOOTH     = 1 << 2,  /* smooth_loss                       loss_utils.py:151-168                  */
  MDN_TERM_CONSIS     = 1 << 3,  /* derivable_consistency_loss        loss_utils.py:171-177                  */
  MDN_OPT_SSIM        = 1 << 4,  /* photo = 0.15*L1 + 0.85*SSIM (else L1 only)  loss_functions.py:111-112    */
  MDN_OPT_INST_MASK   = 1 << 5,  /* DS: post *= instance mask         loss_utils.py:127-138                  */
  MDN_OPT_CROSS_ENT   = 1 << 6,  /* DC: + w_d2_sim * cross entropy    loss_utils.py:72-78, loss_functions.py:132-133 */
  MDN_OPT_GRADS       = 1 << 7,  /* also write d(loss)/d(flow, mob, fmat) for an upstream gradient of 1      */
  MDN_OPT_CUDA_ARITH  = 1 << 8,  /* replay the rounding of the reference's CUDA-EAGER path where it differs from its
                                    CPU path: `tensor /= python_scalar` is a multiplication by the fp32-rounded
                                    reciprocal on CUDA (ATen BinaryDivTrueKernel.cu) but a true division on the CPU.
                                    Affects grid /= (w-1), (h-1) (loss_utils.py:29-30, utils.py:309-310) and
                                    post /= threshold (loss_utils.py:86).  Without the flag: CPU rounding.          */
  MDN_OPT_PAD_BORDER     = 1 << 9,  /* padding_mode of the flow warp's grid_sample (loss_utils.py:33; the `padding_mode`   */
  MDN_OPT_PAD_REFLECTION = 1 << 10  /* argument of Loss / LossModule, loss_functions.py:12,161): "border" / "reflection"
                                       instead of "zeros" (neither flag; what every caller upstream passes).  At most one. */
};

/* One pyramid level.  h = height, w = width of THIS level. */
typedef struct MdnScale {
  int32_t height, width;
  float flow_sx, flow_sy;   /* pixels = flow * (sx, sy): (w, h) for the nets' normalised flow (layers.py:101-103,
                               loss_functions.py:44), (1, 1) for a flow map already in pixels                   */
  float scale_div;          /* 2**scale: every term of this level is divided by it (loss_functions.py:40,55,59,147) */
  float pad_;
  const float* tgt;                    /* (B,3,h,w) target image ("color",0,s); PHOTO and SMOOTH              */
  const float* ref[MDN_MAX_PAIRS];     /* (B,3,h,w) source image ("color",i,s); PHOTO                          */
  const float* flow[MDN_MAX_PAIRS];    /* (B,2,h,w) optical flow target->source; EPIPOLAR and PHOTO            */
  const float* mob[MDN_MAX_PAIRS];     /* (B,1,h,w) mobile probability maps; EPIPOLAR, SMOOTH, CONSIS          */
  const float* fmat[MDN_MAX_PAIRS];    /* (B,3,3) fundamental matrix K^-T [t]x R K^-1 (loss_utils.py:50-62)    */
  const float* weight;                 /* (h,w) TG weight table (utils.py:355-379) or NULL                     */
  const uint8_t* inst;                 /* (B,h,w) {0,1} instance mask already resized to (h,w), or NULL        */
  /* gradient outputs for an upstream gradient of 1 (MDN_OPT_GRADS); each may be NULL to skip it */
  float* g_flow[MDN_MAX_PAIRS];        /* (B,2,h,w) w.r.t. `flow` as passed (flow_sx/sy chain rule applied)   */
  float* g_mob[MDN_MAX_PAIRS];         /* (B,1,h,w)                                                            */
  float* g_fmat[MDN_MAX_PAIRS];        /* (B,3,3)                                                              */
  /* optional per-pixel maps (the `outputs` dict / tuple returns of the reference); NULL to skip */
  float* post_map[MDN_MAX_PAIRS];      /* (B,1,h,w) post-processed epipolar map  ("epipolars")                */
  float* ori_map[MDN_MAX_PAIRS];       /* (B,1,h,w) |e|, or |e|/max in SN (upstream aliasing quirk) ("epipolar_ori") */
  float* warped[MDN_MAX_PAIRS];        /* (B,3,h,w) flow-warped source image ("warps")                        */
  float* diff[MDN_MAX_PAIRS];          /* (B,3,h,w) |tgt - warped| * valid ("diffs")                          */
  uint8_t* valid[MDN_MAX_PAIRS];       /* (B,1,h,w) validity mask, one channel ("valids" is its 3x repeat)    */
  float* ssim_map[MDN_MAX_PAIRS];      /* (B,3,h,w) SSIM distance map                                         */
  /* optional: the source image already in the layout the warp gather reads -- (B,h,w,4) fp32, (r, g, b, unused) per
   * pixel, as mdn_pack_rgb / mdn_image_pyramid_packed write it.  When given, ref[p] is not read (may be NULL) and the
   * call launches no repack kernel for that image (SURVEY.md 8f-N3). */
  const float* ref_packed[MDN_MAX_PAIRS];
} MdnScale;

typedef struct MdnLossDesc {
  int32_t batch, n_scales, n_pairs;
  int32_t post;        /* MdnPost     */
  int32_t mask_mode;   /* MdnMaskMode */
  int32_t flags;       /* MdnFlags    */
  double threshold;    /* T / TG divisor (opt.threshold, options.py:84-87); <= 0 means "None" (no division)  */
  float alpha;         /* weight of the non-trivial-solution term (opt.alpha)                                 */
  float w_d2_sim;      /* DC cross-entropy weight (opt.w_d2_sim)                                              */
  float w_e, w_s, w_c, w_p;  /* loss_functions.py:191-194                                                    */
  MdnScale scale[MDN_MAX_SCALES];
  /* Optional pose inputs (since ABI 2).  When cam[p] is given for every pair, the fundamental matrices are built INSIDE the
   * call -- F = K^-T ((t_x R) K^-1), loss_utils.py:50-62, with R = cam[:, :3, :3], t = cam[:, :3, 3]
   * (loss_functions.py:45-46) and K^-1 = inv_K[s][:, :3, :3] (:123), products accumulated like mdn_fundamental_fwd --
   * and scale[s].fmat[p] is ignored (may be NULL); inv_K[s] is then required for every scale.  With MDN_OPT_GRADS,
   * g_cam[p] (may be NULL) receives d(loss)/d(cam[p]): d/dR in [:3,:3], d/dt in [:3,3], zeros elsewhere -- what
   * mdn_fundamental_bwd would return for the call's d/dF, without the two extra launches. */
  const float* cam[MDN_MAX_PAIRS];     /* (B,4,4) relative pose target -> source frame p                          */
  float* g_cam[MDN_MAX_PAIRS];         /* (B,4,4)                                                                 */
  const float* inv_K[MDN_MAX_SCALES];  /* (B,4,4) inverse intrinsics of pyramid level s                           */
  /* Optional pose PARAMETERS instead of pose matrices (ABI 3): PoseNet's outputs as trainer.py:270 holds them, before
   * transformation_from_parameters (networks/layers.py:16-98, invert=False, trainer.py:272).  axisangle[p] and
   * translation[p] are (B,1,1,3) contiguous = 3 floats per sample; give them for every pair INSTEAD of cam[p] (inv_K as
   * above).  The kernels then build the pose themselves -- Rodrigues' formula with the reference's operation order
   * (angle = |v|, axis = v / (angle + 1e-7), R = cos I + (1 - cos) k k^T + sin [k]_x; M[:3,:3] = R, M[:3,3] = t) -- in the
   * threads that build F, and with MDN_OPT_GRADS g_axisangle[p] / g_translation[p] (B,1,1,3, each may be NULL) receive
   * d(loss)/d(axisangle[p]), d(loss)/d(translation[p]): the ~40 small ATen launches of layers.py:16-98 and their autograd
   * backward leave the step.  g_cam[p] may still be given (it receives d(loss)/d(built pose)). */
  const float* axisangle[MDN_MAX_PAIRS];
  const float* translation[MDN_MAX_PAIRS];
  float* g_axisangle[MDN_MAX_PAIRS];
  float* g_translation[MDN_MAX_PAIRS];
  /* Optional (ABI 3): a cudaEvent_t recorded, on ANOTHER stream, after the work that produces scale[s].inst (the DS / DC
   * instance masks: mdn_instance_mask_union / _resize).  The call launches its pre-pass (source repack, SN maxima) first
   * and makes `stream` wait for the event only in front of the kernels that read the masks, so the mask preparation
   * overlaps the pre-pass.  NULL: the masks are ready in stream order, as every other input. */
  void* inst_ready;
} MdnLossDesc;

/* loss_out layout (MDN_OUT_COUNT = 8 device floats) written by mdn_loss_fused.  MDN_OUT_APPLIED is the upstream
 * gradient the gradient buffers currently correspond to (1 after mdn_loss_fused); mdn_loss_scale_grads updates it. */
enum MdnLossOut { MDN_OUT_LOSS = 0, MDN_OUT_EPIP = 1, MDN_OUT_SMOOTH = 2, MDN_OUT_CONSIS = 3, MDN_OUT_PHOTO = 4,
                  MDN_OUT_APPLIED = 5, MDN_OUT_COUNT = 8 };

MDN_API int mdn_version(void);
MDN_API const char* mdn_last_error_string(void);

/* Bytes of device workspace mdn_loss_fused needs for this description (tile partial sums, per-sample
 * sums, SN max keys, a completion ticket, in-call fundamental matrices and -- with MDN_TERM_PHOTO -- the source
 * images repacked to one float4 per pixel for the warp gather: 16 bytes x pixels x pairs x scales).  The workspace
 * needs no initialisation and may be shared by calls with different descriptions on the same stream. */
MDN_API size_t mdn_loss_workspace_bytes(const MdnLossDesc* desc);

/*
 * The whole loss path in one call: replaces Loss.forward (loss_functions.py:170-205) and everything it
 * reaches -- LossModule.forward / single_mobile_mask_forward (:27-105), epipolar_loss (:117-138) with
 * get_epipolar_new (loss_utils.py:39-69) and the SN/T/TG/DS/DC post-processing (:72-138), photo_metric_loss
 * (:107-115) with inverse_warp (loss_utils.py:12-36) and SSIM (networks/layers.py:148-178), smooth_loss
 * (loss_utils.py:151-168), consistency_loss (:140-147 / loss_utils.py:171-177), the min mask (:176-178),
 * create_coords (:150-157) and get_scale_factor (layers.py:101-103) -- for all scales and both source
 * frames, forward AND (with MDN_OPT_GRADS) the gradients w.r.t. flow, mobile maps and fundamental matrices
 * for an upstream gradient of 1.  With a single scale / pair and a subset of the MDN_TERM_* flags it is
 * also what the individual reference functions map to.
 *
 *   loss_out[MDN_OUT_EPIP]   = sum_s sum_i (mean(bg*post) + alpha*mean|m log(bg+1e-5)| [+ w_d2_sim*mean(CE)]) / scale_div
 *   loss_out[MDN_OUT_SMOOTH] = sum_s sum_i smooth_loss / scale_div
 *   loss_out[MDN_OUT_CONSIS] = sum_s mean((sig(20(m0-.5)) - sig(20(m1-.5)))^2) / scale_div
 *   loss_out[MDN_OUT_PHOTO]  = sum_s sum_i (0.15*mean(diff) + 0.85*mean(SSIM)  |  mean(diff)) / scale_div
 *   loss_out[MDN_OUT_LOSS]   = w_e*EPIP + w_s*SMOOTH + w_c*CONSIS + w_p*PHOTO
 */
MDN_API int mdn_loss_fused(const MdnLossDesc* desc, float* loss_out, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Measurement aid (bench.py's roofline line): the same call, bracketed by CUDA events on `stream`; BLOCKS until the
 * work has finished and returns, in HOST memory, ms_out[0] = source-image repack kernel, ms_out[1] = the fused tile
 * kernel alone (the dominant kernel of the path), ms_out[2] = the finish kernel.  Not for use inside a training step.
 */
MDN_API int mdn_loss_fused_profile(const MdnLossDesc* desc, float* loss_out, void* workspace, size_t workspace_bytes, void* stream,
                                   float* ms_out);

/*
 * Backward of the call above for an arbitrary upstream gradient: multiplies every gradient buffer named in
 * `desc` by (*g / *applied) and stores *g into *applied (`applied` = loss_out + MDN_OUT_APPLIED of the forward
 * call: two floats, the value and a completion ticket).  When *g == *applied (the usual loss.backward(),
 * g == 1) the kernel exits without touching memory.  `g` and `applied` are device scalars.
 */
MDN_API int mdn_loss_scale_grads(const MdnLossDesc* desc, const float* g, float* applied, void* stream);

/*
 * Fundamental matrices for every (scale, source frame, sample) in one launch: F = K^-T ((t_x R) K^-1),
 * loss_utils.py:50-62, with R = cam[:, :3, :3], t = cam[:, :3, 3] (loss_functions.py:45-46) and
 * K^-1 = inv_K[:, :3, :3] (loss_functions.py:123).  `inv_K` is a HOST array of n_scales device pointers to (B,4,4)
 * matrices, `cam` a HOST array of n_pairs device pointers to (B,4,4) poses; fmat is (n_scales, n_pairs, B, 3, 3).
 * Each 3x3 product accumulates k = 0,1,2 with FMAs, the order of the batched SGEMM the reference runs.
 * The backward takes g_fmat (same shape) and writes g_cam[p] (B,4,4): d/dR in [:3,:3], d/dt in [:3,3], zeros elsewhere.
 */
MDN_API int mdn_fundamental_fwd(const float* const* inv_K, const float* const* cam, float* fmat, int32_t n_scales,
                                int32_t n_pairs, int32_t batch, void* stream);
MDN_API int mdn_fundamental_bwd(const float* const* inv_K, const float* const* cam, const float* g_fmat,
                                float* const* g_cam, int32_t n_scales, int32_t n_pairs, int32_t batch, void* stream);

/*
 * get_epipolar_new (loss_utils.py:39-69) for arbitrary homogeneous point sets: p1, p2 are (B,3,N), fmat
 * (B,3,3); out (B,1,N) is the SIGNED distance.  The backward takes the upstream gradient g_out (B,1,N)
 * and writes g_p1, g_p2 (B,3,N, either may be NULL) and g_fmat (B,3,3, may be NULL).
 */
MDN_API int mdn_epipolar_points_fwd(const float* p1, const float* p2, const float* fmat, float* out, int32_t batch,
                            int64_t n, void* stream);
MDN_API int mdn_epipolar_points_bwd(const float* p1, const float* p2, const float* fmat, const float* g_out, float* g_p1,
                            float* g_p2, float* g_fmat, int32_t batch, int64_t n, void* workspace,
                            size_t workspace_bytes, void* stream);
MDN_API size_t mdn_epipolar_points_workspace_bytes(int32_t batch, int64_t n);

/*
 * inverse_warp (loss_utils.py:12-36) / FlowWarp (utils.py:289-315): bilinear flow warp, align_corners=True,
 * zeros padding (bits 2-3 of `warp_flags`: 1 = border, 2 = reflection -- grid_sample's other padding modes).  flow is in pixels.  warped (B,C,h,w) may be NULL (FlowWarp: grid + validity only);
 * grid_out (B,h,w,2) normalised grid or NULL; valid (B,h,w) uint8 or NULL.  `warp_flags` bit 0 selects the
 * (g-0.5)*2 normalisation of utils.py:311 instead of 2*g-1 (loss_utils.py:31) -- same value, other rounding;
 * bit 1 selects the CUDA-eager rounding of `/= (w-1)` (see MDN_OPT_CUDA_ARITH).
 * The backward takes g_warped (B,C,h,w) and writes g_flow (B,2,h,w).
 */
MDN_API int mdn_flow_warp_fwd(const float* ref, const float* flow, float* warped, float* grid_out, uint8_t* valid,
                      int32_t batch, int32_t channels, int32_t height, int32_t width, int32_t warp_flags,
                      void* stream);
MDN_API int mdn_flow_warp_bwd(const float* ref, const float* flow, const float* g_warped, float* g_flow, int32_t batch,
                      int32_t channels, int32_t height, int32_t width, int32_t warp_flags, void* stream);

/*
 * SSIM module (networks/layers.py:148-178): out = clamp((1 - SSIM(x,y))/2, 0, 1), 3x3 reflect-padded.
 * x, y, out, g_out, g_x, g_y are (planes,h,w) with planes = B*C.  g_x / g_y may be NULL.
 */
MDN_API int mdn_ssim_fwd(const float* x, const float* y, float* out, int32_t planes, int32_t height, int32_t width,
                 void* stream);
MDN_API int mdn_ssim_bwd(const float* x, const float* y, const float* g_out, float* g_x, float* g_y, int32_t planes,
                 int32_t height, int32_t width, void* stream);

/*
 * Instance-mask preparation for the DS / DC modes, once per step for every pyramid level (SURVEY.md 8f-N2).
 *
 * mdn_instance_mask_union: get_batch_instance_mask (loss_utils.py:102-124) -- `masks` is a HOST array of `batch` device
 * pointers, masks[b] -> (counts[b], H, W) boolean (1 byte / element) instance masks of sample b (Detectron2
 * `pred_masks`); `counts` is a HOST array; out (B, H, W) uint8 = (sum over instances != 0).  One channel instead of
 * the reference's three identical int64 channels.
 *
 * mdn_instance_mask_resize: `Resize((h, w))(mask)` of loss_utils.py:73-75 / 135-137 for up to MDN_MAX_SCALES output
 * sizes in one launch -- torchvision's bilinear + antialias resize of the integer mask (ATen _upsample_bilinear2d_aa:
 * separable triangle filter of support in/out, fp32, horizontal then vertical) followed by round-half-to-even.
 * src (B, in_h, in_w) uint8 {0,1}; dst is a HOST array of n_out device pointers, dst[k] -> (B, out_h[k], out_w[k]) uint8
 * -- the `inst` tensors MdnScale wants.  Three launches (weight tables, horizontal pass into `workspace`, vertical pass).
 */
MDN_API int mdn_instance_mask_union(const uint8_t* const* masks, const int32_t* counts, uint8_t* out, int32_t batch,
                                    int64_t hw, void* stream);
/* The same union as mdn_instance_mask_union, but `masks` (batch device pointers) and `counts` (batch int32) are DEVICE
 * arrays, read by the kernel when it runs.  Captured into a CUDA graph, it follows whatever the tables hold at replay time.
 * The tables and the masks they point to must stay valid until the work has run.  counts[b] <= 0 gives an all-zero sample.
 * batch <= 65535; one launch. */
MDN_API int mdn_instance_mask_union_table(const uint8_t* const* masks, const int32_t* counts, uint8_t* out,
                                          int32_t batch, int64_t hw, void* stream);
MDN_API int mdn_instance_mask_resize(const uint8_t* src, int32_t batch, int32_t in_h, int32_t in_w, uint8_t* const* dst,
                                     const int32_t* out_h, const int32_t* out_w, int32_t n_out, void* workspace,
                                     size_t workspace_bytes, void* stream);
/* workspace of the call above: the horizontally resized fp32 rows, batch * in_h * sum(out_w) floats, plus the per-axis
 * weight tables (256-byte padded) */
MDN_API size_t mdn_instance_mask_resize_workspace_bytes(int32_t batch, int32_t in_h, int32_t in_w, const int32_t* out_h,
                                                        const int32_t* out_w, int32_t n_out);

/*
 * Image pyramid producer (SURVEY.md 8f-N3): the lower pyramid levels ("color", i, s), s >= 1, from the full-resolution
 * frame on the device -- torchvision `Resize((H / 2**s, W / 2**s))` of an fp32 tensor (bilinear + antialias, the
 * dataset-side resize of mono_dataset.py:106-125 applied to tensors), the same separable ATen filter as above without the
 * rounding.  src (planes, in_h, in_w) fp32 with planes = B * 3; dst is a HOST array of n_out device pointers,
 * dst[k] -> (planes, out_h[k], out_w[k]).  Workspace: mdn_instance_mask_resize_workspace_bytes(planes, ...).
 * Only the full-resolution frames then have to cross PCIe.
 */
MDN_API int mdn_image_pyramid(const float* src, int32_t planes, int32_t in_h, int32_t in_w, float* const* dst,
                              const int32_t* out_h, const int32_t* out_w, int32_t n_out, void* workspace,
                              size_t workspace_bytes, void* stream);

/* The same with every level written as (planes / 3, out_h, out_w, 4): one (r, g, b, unused) float4 per pixel -- the
 * `ref_packed` input of MdnScale.  planes must be a multiple of 3 (B x RGB).  Output sizes equal to the input size are
 * allowed (a pure repack of the full-resolution frame). */
MDN_API int mdn_image_pyramid_packed(const float* src, int32_t planes, int32_t in_h, int32_t in_w, float* const* dst,
                                     const int32_t* out_h, const int32_t* out_w, int32_t n_out, void* workspace,
                                     size_t workspace_bytes, void* stream);

/*
 * The dataset's ArrayToTensor + Normalize on the device (datasets/custom_transforms.py:72-80,103-112, mono_dataset.py:51-52,
 * 112): src (B,H,W,3) uint8 frames as the loader holds them, dst (B,3,H,W) fp32 = ((x / 255) - mean[c]) / std[c], every
 * operation rounded on its own like the CPU tensor ops of the reference.  `mean`, `std` are HOST arrays of 3 floats.
 * With it, frames cross PCIe as bytes (a quarter of the fp32 size).
 */
MDN_API int mdn_normalize_u8(const uint8_t* src, float* dst, int32_t batch, int32_t height, int32_t width,
                             const float* mean, const float* stdv, void* stream);

/* binary_image (utils.py:100-103): out = x >= threshold ? 1 : 0 */
MDN_API int mdn_binary_image(const float* x, float* out, int64_t n, float threshold, void* stream);

/*
 * Evaluation of mobile masks for a whole threshold sweep in one pass over the maps: the confusion counts of
 * binary_image(pred, thr) (utils.py:100-103) against moving-object masks, for every image and threshold.
 *
 * pred (batch, hw) fp32 mobile probabilities; gt (batch, hw) uint8, non-zero = moving (get_batch_instance_mask's != 0);
 * thresholds: n_thr fp32 values, 1 <= n_thr <= 1024.  A pixel is predicted moving at threshold t iff pred >= t in fp32:
 * a prediction equal to a threshold is moving at it, NaN is never moving, -0.0 >= 0.0.
 * counts (batch, n_thr, 4) int64 = [TP, FP, FN, TN] per image and threshold, exact; each row sums to hw.
 *
 * The thresholds must be strictly increasing and free of NaN (+-inf allowed): that is the CALLER's precondition, not
 * checked here.  Other thresholds give wrong counts, never an access outside the arrays.
 * workspace: mdn_mask_confusion_workspace_bytes(batch, n_thr) bytes (per-sample histograms; 0 on bad arguments).
 * Three operations on `stream`: a memset of the workspace, the counting kernel, the finish kernel.
 * Errors: NULL argument; batch outside 1..65535, hw outside 1..2^31-1 or n_thr outside 1..1024 (MDN_ERR_BAD_SHAPE);
 * a pointer that is not 16-byte aligned; a workspace that is too small.
 */
MDN_API size_t mdn_mask_confusion_workspace_bytes(int32_t batch, int32_t n_thr);
MDN_API int mdn_mask_confusion(const float* pred, const uint8_t* gt, const float* thresholds, int32_t n_thr,
                               int64_t* counts, int32_t batch, int64_t hw, void* workspace, size_t workspace_bytes,
                               void* stream);

/*
 * Evaluation of optical flow in one pass over the ground truth: end-point error (EPE) and KITTI Fl outliers per image and
 * region, from the network's flow at its own resolution.
 *
 * flow (batch, 2, h, w) fp32, the prediction at any resolution; gt_flow (batch, 2, H, W) fp32 in pixels of H x W;
 * gt_valid (batch, H, W) uint8, non-zero = valid; region (batch, H, W) uint8 labels, or NULL = every pixel in region 0
 * (then n_regions must be 1).  counts (batch, n_regions, 2) int64 = [valid, outliers]; epe_sum (batch, n_regions) fp64.
 *
 * Per ground-truth pixel (y, x) of sample b, every operation fp32 and rounded on its own (no contraction):
 *   1. source row (ATen upsample_bilinear2d, align_corners=False, no scale_factor): ry = float(h) / float(H),
 *      sy = ry * (float(y) + 0.5f) - 0.5f, 0 if below 0; y0 = (int)sy, dy = (y0 < h-1), ly1 = sy - y0, ly0 = 1 - ly1;
 *      the column likewise with w and W
 *   2. per channel c: f_c = ly0*(lx0*F[y0][x0] + lx1*F[y0][x0+dx]) + ly1*(lx0*F[y0+dy][x0] + lx1*F[y0+dy][x0+dx]) in
 *      that order (at h = H, w = W this is the input, except that 0 * a non-finite neighbour gives NaN as in ATen)
 *   3. u = f_0 * scale_x, v = f_1 * scale_y
 *   4. e = sqrt((u-gu)*(u-gu) + (v-gv)*(v-gv)), m = sqrt(gu*gu + gv*gv)
 *   5. outlier = e > abs_thr && e / m > rel_thr (the KITTI devkit's Fl test: abs_thr 3, rel_thr 0.05); m = 0 gives inf
 *      or NaN and the comparison treats it as IEEE does; a NaN e is never an outlier but does reach epe_sum
 *   6. the pixel counts iff gt_valid != 0 and its label r < n_regions (so 255 can mean "ignore"): it adds 1 to
 *      valid[b][r], outlier to outliers[b][r] and (double)e to epe_sum[b][r]
 *   7. an uncounted pixel's ground truth reaches no sum, whatever it holds (KITTI stores 0 there, other loaders NaN)
 * The fp64 sums are fixed trees over a grid that depends on the shapes only: bit-identical run to run and on any device.
 *
 * workspace: mdn_flow_errors_workspace_bytes(...) bytes (per-block partials; 0 on bad arguments).  Two kernels on
 * `stream`, no allocation, no synchronisation, no copy.
 * Errors: a NULL required pointer, or a NULL region with n_regions > 1 (MDN_ERR_NULL_POINTER); batch outside 1..65535,
 * a size < 1, h*w or H*W above 2^31-1, n_regions outside 1..8, a non-finite scale or threshold or a negative threshold
 * (MDN_ERR_BAD_SHAPE); a pointer that is not 16-byte aligned; a workspace that is too small.
 */
MDN_API size_t mdn_flow_errors_workspace_bytes(int32_t batch, int32_t height, int32_t width, int32_t gt_height,
                                               int32_t gt_width, int32_t n_regions);
MDN_API int mdn_flow_errors(const float* flow, int32_t height, int32_t width, float scale_x, float scale_y,
                            const float* gt_flow, const uint8_t* gt_valid, const uint8_t* region, int32_t n_regions,
                            int32_t gt_height, int32_t gt_width, int32_t batch, float abs_thr, float rel_thr,
                            int64_t* counts, double* epe_sum, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MDN_LOSS_H_ */
