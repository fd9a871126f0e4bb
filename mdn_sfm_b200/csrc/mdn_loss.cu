// mdn_loss.cu -- B200 (sm_100a) kernels + C ABI of the MDN_SfM loss path.  See include/mdn_loss.h.
//
// Kernel inventory
//   ref_pack_kernel      the pre-pass of a call, one launch: source images NCHW -> float4 per pixel for the warp gather
//                        (photometric term) and, in the same grid, the per-sample max / first arg-max of |e| (SN
//                        post-processing, loss_utils.py:96)
//   fused_tile_kernel    ONE launch over every (scale, sample, 64x16 tile): fundamental matrix from the pose, TMA-staged
//                        input tiles, epipolar map + post-processing + masked reductions, bilinear flow warp, SSIM + L1,
//                        smoothness, consistency, min mask, forward values AND gradients (upstream gradient 1),
//                        per-tile partial sums
//   finish_kernel        deterministic second stage, one block per sample: tile sums -> d/dF, SN arg-max fix-up, pose
//                        adjoint; last block -> loss scalars
//   scale_grads_kernel   backward for an upstream gradient != 1 (exits immediately when it is 1)
//   instance_union{,_table} / instance_resize_{weights,h,v}_kernel   DS / DC instance masks and fp32 image pyramids (torchvision
//                        antialiased Resize replayed)
//   mask_confusion{,_finish}_kernel   evaluation: [TP, FP, FN, TN] of binary_image(mobile, thr) for a threshold sweep
//   flow_errors{,_finish}_kernel   evaluation: end-point error and KITTI Fl outliers per image and region
//   small standalone kernels for the individually exported reference functions
//
// All of it is bandwidth/latency-bound stencil + gather work: no tensor cores by design.
#include "mdn_common.cuh"
#include "../../include/mdn_loss.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace mdn {

// ----------------------------------------------------------------------------------------------- geometry
constexpr int NTHREADS = 256;                         // block size of the small standalone kernels
constexpr int PACK_PX = 4;                            // pixels per thread of ref_pack_kernel
// fused kernel: TW x TH tile, one thread per 2-column x PR-row patch of pixels
constexpr int TW = 64, TH = 16;
// measured: 2 rows (256 threads / CTA) beats 4 rows (128 threads) at every shape tried
constexpr int PR = 2;                                        // rows of the per-thread pixel patch
static_assert(PR % 2 == 0 && TH % PR == 0, "patch rows (the SSIM adjoint gather takes them in pairs)");
constexpr int FT = (TW / 2) * (TH / PR), FWARPS = FT / 32;   // lane = column pair, warp = row group
static_assert(TW == 64, "one warp spans the tile width: 32 lanes x 2 columns");
// halo-2 planes (target / warped image / mobile maps): rows y0-2 .. y0+TH+1, columns x0-2 .. x0+TW+1 (W2 = TW + 4 of
// them).  Slot (r, j) lives at OFF2 + r * S2 + j.  The row pitch S2 = 72 and OFF2 = 2 are what lets ONE TMA box copy
// (72 x 20 x 1 floats at signed coordinates (x0 - 4, y0 - 2, plane), zero fill outside the tensor, dense rows) land a
// whole plane at its 128-byte aligned base; they also keep column x0 (j = 2) 16-byte aligned for the cp.async fallback
// and every even j 8-byte aligned for LDS.64.  R2P * 4 is a multiple of 128.
constexpr int W2 = TW + 4, S2 = TW + 8, R2H = TH + 4, OFF2 = 2, R2P = S2 * R2H;
static_assert((R2P * 4) % 128 == 0 && S2 >= OFF2 + W2, "TMA box geometry");
// halo-1 planes (SSIM adjoint coefficients): window rows y0-1 .. y0+TH, columns x0-1 .. x0+TW
constexpr int S1 = TW + 4, R1H = TH + 2, R1P = S1 * R1H;
constexpr int WPR = 3;                                      // window rows per SSIM patch (2 columns x WPR rows)
static_assert((TH + 2) % WPR == 0, "SSIM patches tile the halo-1 region exactly");
constexpr int NCP = (TW + 2) / 2, NPATCH = NCP * ((TH + 2) / WPR);
constexpr int RING = W2 * R2H - TW * TH;              // halo slots of the halo-2 region
constexpr int FUSED_MIN_CTAS = 2;  // 128 registers / thread, no spills; the larger L1 carve-out of 2 CTAs / SM helps the gather

// partial-sum slots per tile
constexpr int PAIR_SLOTS = 16;   // epi, nt, ce, l1, ssim, gF[9], pad, pad
constexpr int SL_EPI = 0, SL_NT = 1, SL_CE = 2, SL_L1 = 3, SL_SSIM = 4, SL_GF = 5;
constexpr int TAIL_BASE = 2 * PAIR_SLOTS;   // consis, smooth_x[0], smooth_y[0], smooth_x[1], smooth_y[1], pad x3
constexpr int SL_CONSIS = 0, SL_SMX = 1, SL_SMY = 2;
constexpr int TAIL_SLOTS = 8;
constexpr int NSLOT = TAIL_BASE + TAIL_SLOTS;   // 40

struct KScale {
  int h, w, tiles_x, tiles_y;
  int tile_begin;          // first tile index of this scale
  float sx, sy;            // flow -> pixels
  WarpGeom geom;
  float c_epi, c_nt, c_ce, c_l1, c_ssim, c_smx, c_smy, c_consis;   // gradient coefficients (upstream 1)
  const float* tgt; const float* ref[2]; const float* flow[2]; const float* mob[2]; const float* fmat[2];
  float4* refp[2];         // source images repacked to (r, g, b, -) per pixel (workspace; written by ref_pack_kernel)
  const float* weight; const uint8_t* inst;
  float* g_flow[2]; float* g_mob[2];
  float* post_map[2]; float* ori_map[2]; float* warped[2]; float* diff[2]; uint8_t* valid[2]; float* ssim_map[2];
};

struct KParams {
  int batch, n_scales, n_pairs, post, mask_mode, flags;
  int n_tiles;
  int prefetch_distance;             // tiles between a CTA and the tile whose inputs it prefetches into L2
  float threshold, inv_threshold;
  float* partials;                   // [n_tiles][NSLOT]
  const unsigned long long* snkey;   // [n_scales][n_pairs][batch] packed (bits(max)<<32 | ~argmax)
  // poses given instead of fundamental matrices (MdnLossDesc.cam / inv_K): F is built by the kernels that need it
  const float* cam[MDN_MAX_PAIRS];   // (B,4,4) or NULL
  const float* aa[MDN_MAX_PAIRS];    // or pose PARAMETERS: axis-angle (B,3) and translation (B,3); cam is then built in-kernel
  const float* tr[MDN_MAX_PAIRS];
  const float* inv_K[MDN_MAX_SCALES];
  float* fmat_ws;                    // [n_scales][n_pairs][batch][9] F as the fused kernel used it (written when cam is given)
  unsigned* ticket;                  // completion ticket of finish_kernel (zeroed by the fused kernel)
  int pack_begin[MDN_MAX_SCALES + 1], pack_blocks[MDN_MAX_SCALES];   // block ranges of ref_pack_kernel
  KScale sc[MDN_MAX_SCALES];
#ifndef MDN_EMU
  // TMA descriptors of the staged input planes, per scale: 0 target (w, h, 3 B), 1 / 2 the mobile maps (w, h, B); valid
  // where tma_ok[s] (row pitch a multiple of 16 bytes); otherwise the tile is staged with cp.async
  alignas(64) CUtensorMap tmap[MDN_MAX_SCALES][3];
#endif
  int tma_ok[MDN_MAX_SCALES];
};
static_assert(sizeof(KParams) <= 3800, "kernel parameter space");

// ----------------------------------------------------------------------------------------------- fundamental matrix
struct FundArgs {
  const float* inv_K[MDN_MAX_SCALES];
  const float* cam[MDN_MAX_PAIRS];
  const float* aa[MDN_MAX_PAIRS];      // pose parameters instead of cam (see pose_from_params)
  const float* tr[MDN_MAX_PAIRS];
  float* g_cam[MDN_MAX_PAIRS];
  float* g_aa[MDN_MAX_PAIRS];
  float* g_tr[MDN_MAX_PAIRS];
  int n_scales, n_pairs, batch;
};

// transformation_from_parameters (networks/layers.py:16-98, invert=False as trainer.py:272 calls it): Rodrigues' formula
// with the reference's operation order and separate roundings -- angle = |v| (:64), axis = v / (angle + 1e-7) (:65), cos /
// sin (:67-68), C = 1 - cos (:69), the nine entries (:87-95); M = T R (:38) leaves M[:3,:3] = R and M[:3,3] = t exactly
// (the products with T's zeros and ones add +0).  cam: 16 floats, row-major (4,4).
MDN_DEV void pose_from_params(const float* aa, const float* tr, float* cam) {
  const float vx = aa[0], vy = aa[1], vz = aa[2];
  const float angle = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(vx, vx), __fmul_rn(vy, vy)), __fmul_rn(vz, vz)));
  const float den = __fadd_rn(angle, 1e-7f);
  const float x = __fdiv_rn(vx, den), y = __fdiv_rn(vy, den), z = __fdiv_rn(vz, den);
  const float ca = cosf(angle), sa = sinf(angle);
  const float C = __fsub_rn(1.f, ca);
  const float xs = __fmul_rn(x, sa), ys = __fmul_rn(y, sa), zs = __fmul_rn(z, sa);
  const float xC = __fmul_rn(x, C), yC = __fmul_rn(y, C), zC = __fmul_rn(z, C);
  const float xyC = __fmul_rn(x, yC), yzC = __fmul_rn(y, zC), zxC = __fmul_rn(z, xC);
  cam[0] = __fadd_rn(__fmul_rn(x, xC), ca); cam[1] = __fsub_rn(xyC, zs); cam[2] = __fadd_rn(zxC, ys); cam[3] = tr[0];
  cam[4] = __fadd_rn(xyC, zs); cam[5] = __fadd_rn(__fmul_rn(y, yC), ca); cam[6] = __fsub_rn(yzC, xs); cam[7] = tr[1];
  cam[8] = __fsub_rn(zxC, ys); cam[9] = __fadd_rn(yzC, xs); cam[10] = __fadd_rn(__fmul_rn(z, zC), ca); cam[11] = tr[2];
  cam[12] = 0.f; cam[13] = 0.f; cam[14] = 0.f; cam[15] = 1.f;
}

// adjoint of the rotation part: gR = d(loss)/dR (3x3 row-major) -> g = d(loss)/d(axis-angle) (3)
MDN_DEV void pose_params_bwd(const float* aa, const float* gR, float* g) {
  const float vx = aa[0], vy = aa[1], vz = aa[2];
  const float angle = sqrtf(vx * vx + vy * vy + vz * vz);
  const float inv = 1.f / (angle + 1e-7f);
  const float x = vx * inv, y = vy * inv, z = vz * inv;
  const float ca = cosf(angle), sa = sinf(angle), C = 1.f - ca;
  const float s01 = gR[1] + gR[3], s02 = gR[2] + gR[6], s12 = gR[5] + gR[7];      // symmetric parts
  const float a01 = gR[3] - gR[1], a02 = gR[2] - gR[6], a12 = gR[7] - gR[5];      // antisymmetric parts
  const float dC = gR[0] * x * x + gR[4] * y * y + gR[8] * z * z + s01 * x * y + s02 * z * x + s12 * y * z;
  const float dsa = a01 * z + a02 * y + a12 * x;
  const float dca = gR[0] + gR[4] + gR[8] - dC;
  const float dx = 2.f * gR[0] * x * C + s01 * y * C + s02 * z * C + a12 * sa;
  const float dy = 2.f * gR[4] * y * C + s01 * x * C + s12 * z * C + a02 * sa;
  const float dz = 2.f * gR[8] * z * C + s02 * x * C + s12 * y * C + a01 * sa;
  // through cos / sin and through the normalisation of the axis; d|v|/dv = v / |v| (0 at the origin, like torch.norm)
  const float dangle = dsa * ca - dca * sa - (dx * vx + dy * vy + dz * vz) * inv * inv;
  const float k = angle > 0.f ? dangle / angle : 0.f;
  g[0] = dx * inv + k * vx; g[1] = dy * inv + k * vy; g[2] = dz * inv + k * vz;
}

// the (4,4) pose of (pair p, sample b): loaded, or built from the pose parameters
template <class A>
MDN_DEV void load_cam(const A& a, int p, int b, float* cam) {
  if (a.aa[p]) pose_from_params(a.aa[p] + b * 3, a.tr[p] + b * 3, cam);
  else {
    const float* src = a.cam[p] + b * 16;
#pragma unroll
    for (int k = 0; k < 16; ++k) cam[k] = src[k];
  }
}
template <class A>
MDN_DEV bool has_pose(const A& a, int p) { return a.cam[p] != nullptr || a.aa[p] != nullptr; }

MDN_DEV void mat3_mul(const float* A, const float* Bm, float* C) {   // C = A B, k-ordered FMA accumulation from 0
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float acc = __fmul_rn(A[i * 3], Bm[j]);
      acc = __fmaf_rn(A[i * 3 + 1], Bm[3 + j], acc);
      C[i * 3 + j] = __fmaf_rn(A[i * 3 + 2], Bm[6 + j], acc);
    }
}

MDN_DEV void load_pose(const float* cam, float* R, float* tx) {   // (4,4) row-major -> R (3x3), [t]_x (3x3)
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) R[i * 3 + j] = cam[i * 4 + j];
  const float t0 = cam[3], t1 = cam[7], t2 = cam[11];
  tx[0] = 0.f; tx[1] = -t2; tx[2] = t1; tx[3] = t2; tx[4] = 0.f; tx[5] = -t0; tx[6] = -t1; tx[7] = t0; tx[8] = 0.f;
}

// F = K^-T ((t_x R) K^-1) from M1 = t_x R and the (4,4) inverse intrinsics of one sample (loss_utils.py:61-62)
MDN_DEV void fundamental_from_m1(const float* M1, const float* kp, float* F) {
  float K[9], KT[9], M2[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) { K[r * 3 + c] = kp[r * 4 + c]; KT[c * 3 + r] = kp[r * 4 + c]; }
  mat3_mul(M1, K, M2);                                // loss_utils.py:62 (inner product first)
  mat3_mul(KT, M2, F);
}

MDN_DEV void fundamental_from_pose(const float* cam, const float* kp, float* F) {
  float R[9], tx[9], M1[9];
  load_pose(cam, R, tx);
  mat3_mul(tx, R, M1);                                // loss_utils.py:61
  fundamental_from_m1(M1, kp, F);
}

// One scale's term of dL/dM1 = sum_s K gF K^T (K = K^-1 of scale s, kp its (4,4) row-major matrix of the sample)
MDN_DEV void fundamental_bwd_scale_term(const float* kp, const float* gF, float* T2) {
  float K[9], KT[9], T1[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) { K[r * 3 + c] = kp[r * 4 + c]; KT[c * 3 + r] = kp[r * 4 + c]; }
  mat3_mul(K, gF, T1);
  mat3_mul(T1, KT, T2);
}

MDN_DEV void fundamental_bwd_finish(const FundArgs& A, const float* G1, int p, int b);

// d(loss)/d(cam[p][b]) from d(loss)/dF of every scale; g_fmat is [n_scales][n_pairs][batch][9]
MDN_DEV void fundamental_bwd_one(const FundArgs& A, const float* g_fmat, int p, int b) {
  float G1[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) G1[k] = 0.f;
  for (int s = 0; s < A.n_scales; ++s) {
    float T2[9], gF[9];
    const float* g = g_fmat + ((size_t)(s * A.n_pairs + p) * A.batch + b) * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) gF[k] = __ldcg(g + k);
    fundamental_bwd_scale_term(A.inv_K[s] + b * 16, gF, T2);
#pragma unroll
    for (int k = 0; k < 9; ++k) G1[k] += T2[k];
  }
  fundamental_bwd_finish(A, G1, p, b);
}

// ... from G1 = dL/dM1 (the scale terms added in scale order)
MDN_DEV void fundamental_bwd_finish(const FundArgs& A, const float* G1, int p, int b) {
  float R[9], tx[9], cam[16];
  load_cam(A, p, b, cam);
  load_pose(cam, R, tx);
  float txT[9], RT[9], gR[9], gTx[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) { txT[c * 3 + r] = tx[r * 3 + c]; RT[c * 3 + r] = R[r * 3 + c]; }
  mat3_mul(txT, G1, gR);                                // M1 = t_x R
  mat3_mul(G1, RT, gTx);
  const float gt0 = gTx[7] - gTx[5];                    // t0: t_x[2][1] = t0, t_x[1][2] = -t0
  const float gt1 = gTx[2] - gTx[6];                    // t1: t_x[0][2] = t1, t_x[2][0] = -t1
  const float gt2 = gTx[3] - gTx[1];                    // t2: t_x[1][0] = t2, t_x[0][1] = -t2
  if (A.g_cam[p]) {
    float* out = A.g_cam[p] + b * 16;
#pragma unroll
    for (int k = 0; k < 16; ++k) out[k] = 0.f;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) out[r * 4 + c] = gR[r * 3 + c];
    out[3] = gt0; out[7] = gt1; out[11] = gt2;
  }
  // pose parameters given: the adjoint of transformation_from_parameters too (M[:3,3] = t, M[:3,:3] = Rodrigues(axisangle))
  if (A.aa[p] && A.g_tr[p]) { float* o = A.g_tr[p] + b * 3; o[0] = gt0; o[1] = gt1; o[2] = gt2; }
  if (A.aa[p] && A.g_aa[p]) {
    float ga[3];
    pose_params_bwd(A.aa[p] + b * 3, gR, ga);
    float* o = A.g_aa[p] + b * 3;
    o[0] = ga[0]; o[1] = ga[1]; o[2] = ga[2];
  }
}

// the fundamental matrix of (scale s, pair, sample b): built from the pose when one was given, else loaded
MDN_DEV void tile_fmat(const KParams& P, int s, int pair, int b, float* F) {
  if (has_pose(P, pair)) {
    float cam[16];
    load_cam(P, pair, b, cam);
    fundamental_from_pose(cam, P.inv_K[s] + b * 16, F);
  } else {
    const float* src = P.sc[s].fmat[pair] + b * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) F[k] = __ldg(src + k);
  }
}

MDN_DEV float post_process(const KParams& P, float e, float snmax, float wgt, float& dpost_de) {
  // returns post (before the DS mask) and d(post)/d(e); wgt = Gaussian distance weight of the pixel (TG only)
  if (P.post == MDN_POST_SN) {
    float q = __fdiv_rn(e, snmax);            // loss_utils.py:98
    dpost_de = 2.f * q / snmax;
    return __fmul_rn(q, q);                   // :99
  }
  float r = e, dr = 1.f;
  if (P.threshold > 0.f) {                                                             // loss_utils.py:85-86
    r = (P.flags & MDN_OPT_CUDA_ARITH) ? __fmul_rn(r, P.inv_threshold) : __fdiv_rn(r, P.threshold);
    dr = dr * P.inv_threshold;
  }
  if (P.post == MDN_POST_TG) { r = __fdiv_rn(r, wgt); dr = dr / wgt; }   // :87-88
  dpost_de = 2.f * r * dr;
  return __fmul_rn(r, r);                     // :89
}

// ----------------------------------------------------------------------------------------------- SN pre-pass
MDN_DEV void sn_max_block(const KParams& P, unsigned long long* keys, const int chunks_per_img, const int chunk, const int job) {
  // chunk = chunk within image, job = (scale * n_pairs + pair) * batch + b
  int b = job % P.batch;
  int sp = job / P.batch;
  int pair = sp % P.n_pairs, s = sp / P.n_pairs;
  const KScale& S = P.sc[s];
  const int hw = S.h * S.w;
  float Fm[9];
  tile_fmat(P, s, pair, b, Fm);
  const float* fx = S.flow[pair] + (long long)b * 2 * hw;
  const float* fy = fx + hw;
  unsigned long long best = 0ull;
  auto consider = [&](int i, int x, int y, float fxv, float fyv) {
    float u = __fadd_rn((float)x, __fmul_rn(S.sx, fxv));
    float v = __fadd_rn((float)y, __fmul_rn(S.sy, fyv));
    Epi e = epipolar_distance(Fm, (float)x, (float)y, u, v);
    float ae = fabsf(e.d);
    if (ae == ae) {   // NaNs never win (torch.max would propagate; degenerate input)
      unsigned long long key = ((unsigned long long)__float_as_uint(ae) << 32) | (unsigned)(0xffffffffu - (unsigned)i);
      best = key > best ? key : best;
    }
  };
  if ((S.w & 3) == 0) {
    // four pixels of one row per trip (16-byte loads, one index division): the pass is bound by the bytes a thread keeps
    // in flight, not by its arithmetic
    const int quads = hw >> 2;
    const int per = (quads + chunks_per_img - 1) / chunks_per_img;
    const int beg = chunk * per, end = min(quads, beg + per);
    const float4* fx4 = reinterpret_cast<const float4*>(fx);
    const float4* fy4 = reinterpret_cast<const float4*>(fy);
#pragma unroll 2
    for (int q = beg + (int)threadIdx.x; q < end; q += blockDim.x) {
      const float4 a = __ldg(fx4 + q), c = __ldg(fy4 + q);
      const int i = q << 2, y = i / S.w, x = i - y * S.w;
      consider(i, x, y, a.x, c.x); consider(i + 1, x + 1, y, a.y, c.y);
      consider(i + 2, x + 2, y, a.z, c.z); consider(i + 3, x + 3, y, a.w, c.w);
    }
  } else {
    const int per = (hw + chunks_per_img - 1) / chunks_per_img;
    const int beg = chunk * per, end = min(hw, beg + per);
    for (int i = beg + (int)threadIdx.x; i < end; i += blockDim.x) {
      const int y = i / S.w, x = i - y * S.w;
      consider(i, x, y, __ldg(fx + i), __ldg(fy + i));
    }
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)(best & 0xffffffffu), m);
    unsigned hi = __shfl_xor_sync(0xffffffffu, (unsigned)(best >> 32), m);
    unsigned long long o = ((unsigned long long)hi << 32) | lo;
    best = o > best ? o : best;
  }
  if ((threadIdx.x & 31) == 0 && best) atomicMax(keys + job, best);
}

// ----------------------------------------------------------------------------------------------- source repack
// NCHW planes -> one float4 (r, g, b, 0) per pixel, so that the flow-warp gather of the fused kernel fetches the
// three channels of a bilinear corner with ONE 16-byte load (see gather_pair_packed).  Coalesced both ways: three
// 128-byte reads and one 512-byte write per warp.  grid.y = (scale * n_pairs + pair) * batch + b.
MDN_DEV void ref_pack_block(const KParams& P, const int bid) {
  // flat list of blocks: scale s owns blocks [pack_begin[s], pack_begin[s + 1]), pack_blocks[s] per (pair, sample) image
  int s = 0;
#pragma unroll
  for (int k = 1; k < MDN_MAX_SCALES; ++k)
    if (k < P.n_scales && bid >= P.pack_begin[k]) s = k;
  const KScale& S = P.sc[s];
  const int rem = bid - P.pack_begin[s];
  const int job = rem / P.pack_blocks[s], blk = rem - job * P.pack_blocks[s];
  const int pair = job / P.batch, b = job - pair * P.batch;
  const int hw = S.h * S.w;
  if (!S.ref[pair]) return;                       // this image came already packed (MdnScale.ref_packed)
  const float* src = S.ref[pair] + (size_t)b * 3 * hw;
  float4* dst = S.refp[pair] + (size_t)b * hw;
  // PACK_PX pixels per thread, one pixel per thread and instruction: every warp load is one 128-byte line of a plane,
  // every warp store 512 contiguous bytes
  const int i0 = blk * (NTHREADS * PACK_PX) + threadIdx.x;
  float r[PACK_PX], g[PACK_PX], bl[PACK_PX];
#pragma unroll
  for (int q = 0; q < PACK_PX; ++q) {
    const int i = i0 + q * NTHREADS;
    if (i < hw) { r[q] = __ldg(src + i); g[q] = __ldg(src + hw + i); bl[q] = __ldg(src + 2 * hw + i); }
  }
#pragma unroll
  for (int q = 0; q < PACK_PX; ++q) {
    const int i = i0 + q * NTHREADS;
    if (i < hw) dst[i] = make_float4(r[q], g[q], bl[q], 0.f);
  }
}

// The pre-pass of a call in ONE launch: blocks [0, n_pack) repack the source images, blocks [n_pack, n_pack + sn_chunks * n_keys)
// scan for the per-sample SN maxima.  The two jobs are independent (one streams the source images, the other the flows), so
// sharing a grid lets them overlap instead of running back to back (SN / DS / DC with the photometric term: -15 us per step).
__global__ void __launch_bounds__(NTHREADS) ref_pack_kernel(const __grid_constant__ KParams P, unsigned long long* keys, const int n_pack,
                                                            const int n_sn, const int ratio, const int sn_chunks) {
  const int bid = blockIdx.x;
  if (n_sn == 0) { ref_pack_block(P, bid); return; }
  // the two kinds of blocks INTERLEAVED (`ratio` repack blocks, then one SN block, ...): blocks are dispatched in index
  // order, so a grid that lists one job after the other would run them one after the other
  const int grp = bid / (ratio + 1), rem = bid - grp * (ratio + 1);
  if (rem < ratio) {
    const int k = grp * ratio + rem;
    if (k < n_pack) ref_pack_block(P, k);
  } else if (grp < n_sn) sn_max_block(P, keys, sn_chunks, grp % sn_chunks, grp / sn_chunks);
}

#include "mdn_fused.cuh"

// ----------------------------------------------------------------------------------------------- finish
struct FParams {
  KParams K;
  float* sample_sums;      // [n_scales][batch][NSLOT]
  float* loss_out;         // MDN_OUT_COUNT
  float* g_fmat[MDN_MAX_SCALES][2];
  float* gf_ws;            // [n_scales][n_pairs][batch][9] d(loss)/dF, for the pose adjoint of the last block
  float* g_cam[MDN_MAX_PAIRS];
  float* g_aa[MDN_MAX_PAIRS];
  float* g_tr[MDN_MAX_PAIRS];
  float alpha, w_d2, w_e, w_s, w_c, w_p, l1_coef, ssim_coef;
  float scale_div[MDN_MAX_SCALES];
  // reciprocals of the mean denominators, precomputed on the host in double: the single-thread epilogue multiplies
  // (a dependent chain of ~100 double DIVISIONS cost 14 us)
  double inv_N[MDN_MAX_SCALES], inv_div[MDN_MAX_SCALES], inv_cx[MDN_MAX_SCALES], inv_cy[MDN_MAX_SCALES];
};

constexpr int FIN_ROWS = 24;  // FIN_ROWS * NSLOT = 960 threads: at most ~5 tiles per thread at the headline shape

__global__ void __launch_bounds__(FIN_ROWS * NSLOT) finish_kernel(const __grid_constant__ FParams Q) {
  // One block per SAMPLE: it folds the sample's tiles of every scale, so it also holds every d/dF of the sample and runs
  // the pose adjoint itself; only the final fold into the loss scalars waits for the last block.
  const KParams& P = Q.K;
  __shared__ float part4[MDN_MAX_SCALES][FIN_ROWS][NSLOT];
  __shared__ float tots4[MDN_MAX_SCALES][NSLOT];
  __shared__ float pose_terms[MDN_MAX_SCALES][MDN_MAX_PAIRS][9];
  __shared__ bool is_last;
  const int b = blockIdx.x;
  const int slot = threadIdx.x % NSLOT, row = threadIdx.x / NSLOT;
  const bool grads = (P.flags & MDN_OPT_GRADS) != 0;
  // every scale in ONE round: the sample's tiles of all scales form one list walked with stride FIN_ROWS; a thread keeps
  // one accumulator per scale (fixed order per scale: deterministic)
  {
    int cum[MDN_MAX_SCALES + 1];
    cum[0] = 0;
#pragma unroll
    for (int s = 0; s < MDN_MAX_SCALES; ++s) cum[s + 1] = cum[s] + (s < P.n_scales ? P.sc[s].tiles_x * P.sc[s].tiles_y : 0);
    float t[MDN_MAX_SCALES];
#pragma unroll
    for (int s = 0; s < MDN_MAX_SCALES; ++s) t[s] = 0.f;
    // first tile of the sample at each scale, minus the scale's offset in the sample's list
    int first[MDN_MAX_SCALES];
#pragma unroll
    for (int s = 0; s < MDN_MAX_SCALES; ++s) first[s] = (s < P.n_scales ? P.sc[s].tile_begin + b * (cum[s + 1] - cum[s]) : 0) - cum[s];
    // four loads in flight per thread (the pass is a chain of L2 round trips otherwise); added in list order, as before
    constexpr int FU = 4;
    for (int item0 = row; item0 < cum[MDN_MAX_SCALES]; item0 += FU * FIN_ROWS) {
      float v[FU];
      int sc[FU];
#pragma unroll
      for (int u = 0; u < FU; ++u) {
        const int item = item0 + u * FIN_ROWS;
        int s = 0, f = first[0];
#pragma unroll
        for (int q = 1; q < MDN_MAX_SCALES; ++q)
          if (item >= cum[q]) { s = q; f = first[q]; }
        sc[u] = s;
        v[u] = (item < cum[MDN_MAX_SCALES]) ? __ldcg(P.partials + (unsigned)((f + item) * NSLOT + slot)) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < FU; ++u)
#pragma unroll
        for (int q = 0; q < MDN_MAX_SCALES; ++q) t[q] += (q == sc[u]) ? v[u] : 0.f;
    }
#pragma unroll
    for (int s = 0; s < MDN_MAX_SCALES; ++s) part4[s][row][slot] = t[s];
  }
  __syncthreads();
  if (threadIdx.x < (unsigned)(P.n_scales * NSLOT)) {
    const int s = threadIdx.x / NSLOT, k = threadIdx.x % NSLOT;
    float tot = 0.f;
    for (int r = 0; r < FIN_ROWS; ++r) tot += part4[s][r][k];
    tots4[s][k] = tot;
    Q.sample_sums[((long long)s * P.batch + b) * NSLOT + k] = tot;
  }
  __syncthreads();
  // d/dF of every (scale, pair) of the sample in parallel: thread = scale * n_pairs + pair
  if (grads && (P.flags & MDN_TERM_EPIPOLAR) && threadIdx.x < (unsigned)(P.n_scales * P.n_pairs)) {
    const int s = threadIdx.x / P.n_pairs, pair = threadIdx.x - s * P.n_pairs;
    const KScale& S = P.sc[s];
    const float (*part)[NSLOT] = &tots4[s];     // part[0][k] = this scale's sums

    float gF[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) gF[k] = part[0][pair * PAIR_SLOTS + SL_GF + k];
    if (P.post == MDN_POST_SN) {
      // d/d(max): -(2/M) * c_epi * sum(bg*post), routed to the first arg-max pixel (loss_utils.py:96-98 backward)
      unsigned long long key = P.snkey[(s * P.n_pairs + pair) * P.batch + b];
      float M = __uint_as_float((unsigned)(key >> 32));
      int idx = (int)(0xffffffffu - (unsigned)(key & 0xffffffffu));
      if (key != 0ull && M > 0.f) {
        const int hw = S.h * S.w;
        int y = idx / S.w, x = idx - y * S.w;
        const float* flx = S.flow[pair] + (long long)b * 2 * hw;
        float Fm[9];
        const float* Fsrc = has_pose(P, pair) ? P.fmat_ws + ((size_t)(s * P.n_pairs + pair) * P.batch + b) * 9 : S.fmat[pair] + b * 9;
#pragma unroll
        for (int k = 0; k < 9; ++k) Fm[k] = Fsrc[k];
        float u = __fadd_rn((float)x, __fmul_rn(S.sx, flx[idx]));
        float v = __fadd_rn((float)y, __fmul_rn(S.sy, flx[hw + idx]));
        Epi e = epipolar_distance(Fm, (float)x, (float)y, u, v);
        float ebar = -2.f * S.c_epi * part[0][pair * PAIR_SLOTS + SL_EPI] / M;
        float dbar = signf_(e.d) * ebar;
        float g2 = dbar / e.den, das = e.d / e.s;
        float g0 = g2 * (u - das * e.a), g1 = g2 * (v - das * e.b);
        if (S.g_flow[pair]) {
          S.g_flow[pair][(long long)b * 2 * hw + idx] += g2 * e.a * S.sx;
          S.g_flow[pair][(long long)b * 2 * hw + hw + idx] += g2 * e.b * S.sy;
        }
        float xf = (float)x, yf = (float)y;
        gF[0] += g0 * xf; gF[1] += g0 * yf; gF[2] += g0;
        gF[3] += g1 * xf; gF[4] += g1 * yf; gF[5] += g1;
        gF[6] += g2 * xf; gF[7] += g2 * yf; gF[8] += g2;
      }
    }
    if (Q.g_fmat[s][pair]) {
#pragma unroll
      for (int k = 0; k < 9; ++k) Q.g_fmat[s][pair][b * 9 + k] = gF[k];
    }
    if (Q.gf_ws) {
#pragma unroll
      for (int k = 0; k < 9; ++k) Q.gf_ws[((size_t)(s * P.n_pairs + pair) * P.batch + b) * 9 + k] = gF[k];
      // the pose adjoint's term of this (scale, pair), K gF K^T, while the matrix is in registers
      float T2[9];
      fundamental_bwd_scale_term(P.inv_K[s] + b * 16, gF, T2);
#pragma unroll
      for (int k = 0; k < 9; ++k) pose_terms[s][pair][k] = T2[k];
    }
  }
  __syncthreads();
  // pose adjoint of this sample (what mdn_fundamental_bwd computes): the scale terms added in scale order, then the
  // adjoint of M1 = [t]x R and of the pose parameters
  if (Q.gf_ws && threadIdx.x < (unsigned)P.n_pairs && (Q.g_cam[threadIdx.x] || Q.g_aa[threadIdx.x] || Q.g_tr[threadIdx.x])) {
    FundArgs A;
    for (int k = 0; k < MDN_MAX_SCALES; ++k) A.inv_K[k] = P.inv_K[k];
    for (int k = 0; k < MDN_MAX_PAIRS; ++k) {
      A.cam[k] = P.cam[k]; A.aa[k] = P.aa[k]; A.tr[k] = P.tr[k];
      A.g_cam[k] = Q.g_cam[k]; A.g_aa[k] = Q.g_aa[k]; A.g_tr[k] = Q.g_tr[k];
    }
    A.n_scales = P.n_scales; A.n_pairs = P.n_pairs; A.batch = P.batch;
    float G1[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) G1[k] = 0.f;
    for (int s = 0; s < P.n_scales; ++s) {
#pragma unroll
      for (int k = 0; k < 9; ++k) G1[k] += pose_terms[s][threadIdx.x][k];
    }
    fundamental_bwd_finish(A, G1, threadIdx.x, b);
  }
  // last block to arrive folds the per-sample sums into the loss scalars, in a fixed order
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned prev = atomicInc(P.ticket, gridDim.x - 1);   // (the fused kernel zeroed the ticket)
    is_last = (prev == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  __shared__ double tots[MDN_MAX_SCALES][NSLOT];
  if (threadIdx.x < (unsigned)(P.n_scales * NSLOT)) {
    const int ss = threadIdx.x / NSLOT, k = threadIdx.x % NSLOT;
    double t2 = 0;
    for (int bb = 0; bb < P.batch; ++bb) t2 += (double)Q.sample_sums[((long long)ss * P.batch + bb) * NSLOT + k];
    tots[ss][k] = t2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double epip = 0, smooth = 0, consis = 0, photo = 0;
    const bool own = P.mask_mode == MDN_MASK_OWN;
    for (int ss = 0; ss < P.n_scales; ++ss) {
      const KScale& Z = P.sc[ss];
      const double* tot = tots[ss];
      const double iN = Q.inv_N[ss], idiv = Q.inv_div[ss], icx = Q.inv_cx[ss], icy = Q.inv_cy[ss];
      for (int p = 0; p < P.n_pairs; ++p) {
        const double* tp = tot + p * PAIR_SLOTS;
        if (P.flags & MDN_TERM_EPIPOLAR) {
          double e = tp[SL_EPI] * iN + (double)Q.alpha * (tp[SL_NT] * iN);
          if (P.flags & MDN_OPT_CROSS_ENT) e += (double)Q.w_d2 * (tp[SL_CE] * iN);
          epip += e * idiv;
        }
        if (P.flags & MDN_TERM_PHOTO)
          photo += ((double)Q.l1_coef * (tp[SL_L1] * (iN * (1.0 / 3.0))) + (double)Q.ssim_coef * (tp[SL_SSIM] * (iN * (1.0 / 3.0)))) * idiv;
        if (P.flags & MDN_TERM_SMOOTH) {
          const int k = own ? p : 0;
          smooth += (tot[TAIL_BASE + SL_SMX + 2 * k] * icx + tot[TAIL_BASE + SL_SMY + 2 * k] * icy) * idiv;
        }
      }
      if (P.flags & MDN_TERM_CONSIS) consis += tot[TAIL_BASE + SL_CONSIS] * iN * idiv;
    }
    Q.loss_out[MDN_OUT_EPIP] = (float)epip;
    Q.loss_out[MDN_OUT_SMOOTH] = (float)smooth;
    Q.loss_out[MDN_OUT_CONSIS] = (float)consis;
    Q.loss_out[MDN_OUT_PHOTO] = (float)photo;
    Q.loss_out[MDN_OUT_APPLIED] = 1.f;
    Q.loss_out[MDN_OUT_APPLIED + 1] = 0.f;
    Q.loss_out[MDN_OUT_APPLIED + 2] = 0.f;
    Q.loss_out[MDN_OUT_LOSS] = (float)((double)Q.w_e * epip + (double)Q.w_s * smooth + (double)Q.w_c * consis + (double)Q.w_p * photo);
  }
}

// ----------------------------------------------------------------------------------------------- scale grads
struct GradList {
  int n;
  float* ptr[MDN_MAX_SCALES * 6 + 3 * MDN_MAX_PAIRS];
  long long count[MDN_MAX_SCALES * 6 + 3 * MDN_MAX_PAIRS];
};

__global__ void __launch_bounds__(NTHREADS) scale_grads_kernel(const __grid_constant__ GradList L, const float* g, float* applied,
                                                               unsigned* ticket) {
  __shared__ bool is_last;
  const float gv = __ldg(g), ap = *applied;
  if (gv == ap) return;                      // loss.backward() with the implicit upstream gradient of 1: nothing to do
  const float ratio = gv / ap;
  for (int k = 0; k < L.n; ++k) {
    float* p = L.ptr[k];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < L.count[k]; i += (long long)gridDim.x * blockDim.x)
      p[i] *= ratio;
  }
  // every block has read *applied before the last one to finish overwrites it
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicInc(ticket, gridDim.x - 1) == gridDim.x - 1);
  __syncthreads();
  if (is_last && threadIdx.x == 0) *applied = gv;
}

// ----------------------------------------------------------------------------------------------- standalone kernels
__global__ void __launch_bounds__(NTHREADS) epipolar_points_fwd_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                                                                       const float* __restrict__ fmat, float* __restrict__ out, long long n) {
  const int b = blockIdx.y;
  const float* F = fmat + b * 9;
  const float* a = p1 + (long long)b * 3 * n;
  const float* c = p2 + (long long)b * 3 * n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float x = a[i], y = a[n + i], z = a[2 * n + i];
    float fa = __fmaf_rn(F[2], z, __fmaf_rn(F[1], y, __fmul_rn(F[0], x)));
    float fb = __fmaf_rn(F[5], z, __fmaf_rn(F[4], y, __fmul_rn(F[3], x)));
    float fc = __fmaf_rn(F[8], z, __fmaf_rn(F[7], y, __fmul_rn(F[6], x)));
    float num = __fadd_rn(__fadd_rn(__fmul_rn(fa, c[i]), __fmul_rn(fb, c[n + i])), __fmul_rn(fc, c[2 * n + i]));
    float s = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(fa, fa), __fmul_rn(fb, fb)), 1e-10f));
    out[(long long)b * n + i] = __fdiv_rn(num, __fadd_rn(s, 1e-10f));
  }
}

constexpr int EPB_SLOTS = 16;
__global__ void __launch_bounds__(NTHREADS) epipolar_points_bwd_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                                                                       const float* __restrict__ fmat, const float* __restrict__ g_out,
                                                                       float* __restrict__ g_p1, float* __restrict__ g_p2,
                                                                       float* __restrict__ partials, long long n) {
  __shared__ float red[NTHREADS / 32][EPB_SLOTS];
  const int b = blockIdx.y;
  const float* F = fmat + b * 9;
  const float* a = p1 + (long long)b * 3 * n;
  const float* c = p2 + (long long)b * 3 * n;
  float acc[EPB_SLOTS];
#pragma unroll
  for (int k = 0; k < EPB_SLOTS; ++k) acc[k] = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float x = a[i], y = a[n + i], z = a[2 * n + i];
    float u = c[i], v = c[n + i], t = c[2 * n + i];
    float fa = __fmaf_rn(F[2], z, __fmaf_rn(F[1], y, __fmul_rn(F[0], x)));
    float fb = __fmaf_rn(F[5], z, __fmaf_rn(F[4], y, __fmul_rn(F[3], x)));
    float fc = __fmaf_rn(F[8], z, __fmaf_rn(F[7], y, __fmul_rn(F[6], x)));
    float num = fa * u + fb * v + fc * t;
    float s = sqrtf(fa * fa + fb * fb + 1e-10f);
    float den = s + 1e-10f;
    float d = num / den;
    float g = g_out[(long long)b * n + i];
    float g2 = g / den, das = d / s;
    float ga = g2 * (u - das * fa), gb = g2 * (v - das * fb), gc = g2 * t;   // d/d(Fp1)
    if (g_p2) {
      g_p2[(long long)b * 3 * n + i] = g2 * fa; g_p2[(long long)b * 3 * n + n + i] = g2 * fb; g_p2[(long long)b * 3 * n + 2 * n + i] = g2 * fc;
    }
    if (g_p1) {
      g_p1[(long long)b * 3 * n + i] = F[0] * ga + F[3] * gb + F[6] * gc;
      g_p1[(long long)b * 3 * n + n + i] = F[1] * ga + F[4] * gb + F[7] * gc;
      g_p1[(long long)b * 3 * n + 2 * n + i] = F[2] * ga + F[5] * gb + F[8] * gc;
    }
    acc[0] += ga * x; acc[1] += ga * y; acc[2] += ga * z;
    acc[3] += gb * x; acc[4] += gb * y; acc[5] += gb * z;
    acc[6] += gc * x; acc[7] += gc * y; acc[8] += gc * z;
  }
  warp_reduce_transpose<EPB_SLOTS>(acc);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane < EPB_SLOTS) red[warp][lane] = acc[0];
  __syncthreads();
  if (threadIdx.x < EPB_SLOTS) {
    float t = 0.f;
    for (int wq = 0; wq < (int)(blockDim.x >> 5); ++wq) t += red[wq][threadIdx.x];
    partials[((long long)b * gridDim.x + blockIdx.x) * EPB_SLOTS + threadIdx.x] = t;
  }
}

__global__ void epipolar_points_bwd_finish_kernel(const float* __restrict__ partials, float* __restrict__ g_fmat, int nblk) {
  const int b = blockIdx.x, k = threadIdx.x;
  if (k >= 9) return;
  float t = 0.f;
  for (int j = 0; j < nblk; ++j) t += partials[((long long)b * nblk + j) * EPB_SLOTS + k];
  g_fmat[b * 9 + k] = t;
}

__global__ void fundamental_fwd_kernel(const __grid_constant__ FundArgs A, float* __restrict__ fmat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.n_pairs * A.batch) return;
  const int p = i / A.batch, b = i - p * A.batch;
  float R[9], tx[9], M1[9], cam[16];
  load_cam(A, p, b, cam);
  load_pose(cam, R, tx);
  mat3_mul(tx, R, M1);                                  // loss_utils.py:61
  for (int s = 0; s < A.n_scales; ++s) {
    float F[9];
    fundamental_from_m1(M1, A.inv_K[s] + b * 16, F);
    float* out = fmat + ((size_t)(s * A.n_pairs + p) * A.batch + b) * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) out[k] = F[k];
  }
}

__global__ void fundamental_bwd_kernel(const __grid_constant__ FundArgs A, const float* __restrict__ g_fmat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.n_pairs * A.batch) return;
  const int p = i / A.batch;
  fundamental_bwd_one(A, g_fmat, p, i - p * A.batch);
}

__global__ void __launch_bounds__(NTHREADS) flow_warp_fwd_kernel(const float* __restrict__ ref, const float* __restrict__ flow,
                                                                 float* __restrict__ warped, float* __restrict__ grid_out,
                                                                 uint8_t* __restrict__ valid, int C, int h, int w, const WarpGeom G) {
  const int b = blockIdx.y;
  const int hw = h * w;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x) {
    int y = i / w, x = i - y * w;
    float fx = flow[(long long)b * 2 * hw + i], fy = flow[(long long)b * 2 * hw + hw + i];
    WarpCoord wc = warp_coord((float)x, (float)y, fx, fy, G);
    if (grid_out) { grid_out[((long long)b * hw + i) * 2] = wc.gx; grid_out[((long long)b * hw + i) * 2 + 1] = wc.gy; }
    if (valid) valid[(long long)b * hw + i] = wc.valid ? 1 : 0;
    if (warped) {
      Bilin bl = bilinear_setup(wc.ix, wc.iy, h, w);
      for (int c = 0; c < C; ++c) {
        float nw, ne, sw, se;
        bilinear_fetch(ref + ((long long)b * C + c) * hw, w, bl, nw, ne, sw, se);
        warped[((long long)b * C + c) * hw + i] = bilinear_value(bl, nw, ne, sw, se);
      }
    }
  }
}

__global__ void __launch_bounds__(NTHREADS) flow_warp_bwd_kernel(const float* __restrict__ ref, const float* __restrict__ flow,
                                                                 const float* __restrict__ g_warped, float* __restrict__ g_flow,
                                                                 int C, int h, int w, const WarpGeom G) {
  const int b = blockIdx.y;
  const int hw = h * w;
  const float wm1 = G.wm1, hm1 = G.hm1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x) {
    int y = i / w, x = i - y * w;
    float fx = flow[(long long)b * 2 * hw + i], fy = flow[(long long)b * 2 * hw + hw + i];
    WarpCoord wc = warp_coord((float)x, (float)y, fx, fy, G);
    Bilin bl = bilinear_setup(wc.ix, wc.iy, h, w);
    float gix = 0.f, giy = 0.f;
    for (int c = 0; c < C; ++c) {
      float nw, ne, sw, se, ddx, ddy;
      bilinear_fetch(ref + ((long long)b * C + c) * hw, w, bl, nw, ne, sw, se);
      bilinear_deriv(bl, nw, ne, sw, se, ddx, ddy);
      float g = g_warped[((long long)b * C + c) * hw + i];
      gix += g * ddx; giy += g * ddy;
    }
    gix *= wc.mx; giy *= wc.my;      // (1 with zeros padding)
    // grid_sample: * (size-1)/2 ; "2*g-1": * 2 ; "/= (size-1)": / (size-1)
    float tx = __fmul_rn(__fmul_rn(gix, __fmul_rn(wm1, 0.5f)), 2.f), ty = __fmul_rn(__fmul_rn(giy, __fmul_rn(hm1, 0.5f)), 2.f);
    g_flow[(long long)b * 2 * hw + i] = G.cuda_arith ? __fmul_rn(tx, G.inv_wm1) : __fdiv_rn(tx, wm1);
    g_flow[(long long)b * 2 * hw + hw + i] = G.cuda_arith ? __fmul_rn(ty, G.inv_hm1) : __fdiv_rn(ty, hm1);
  }
}

MDN_DEV void ssim_sums(const float* __restrict__ xp, const float* __restrict__ yp, int py, int px, int h, int w, float& sx,
                       float& sy, float& sxx, float& syy, float& sxy) {
  sx = sy = sxx = syy = sxy = 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    int ry = reflect1(py + dy, h);
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      int rx = reflect1(px + dx, w);
      float xv = __ldg(xp + (long long)ry * w + rx), yv = __ldg(yp + (long long)ry * w + rx);
      sx += xv; sy += yv; sxx += xv * xv; syy += yv * yv; sxy += xv * yv;
    }
  }
}

__global__ void __launch_bounds__(NTHREADS) ssim_fwd_kernel(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ out,
                                                            int h, int w) {
  const long long plane = (long long)blockIdx.y * h * w;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h * w; i += gridDim.x * blockDim.x) {
    int py = i / w, px = i - py * w;
    float sx, sy, sxx, syy, sxy;
    ssim_sums(x + plane, y + plane, py, px, h, w, sx, sy, sxx, syy, sxy);
    out[plane + i] = ssim_window(sx, sy, sxx, syy, sxy, false).J;
  }
}

// gather-form adjoint of (reflect pad -> 3x3 mean pools -> SSIM): every pixel q visits the <= 9 windows that touch it
__global__ void __launch_bounds__(NTHREADS) ssim_bwd_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                            const float* __restrict__ g_out, float* __restrict__ g_x, float* __restrict__ g_y,
                                                            int h, int w) {
  const long long plane = (long long)blockIdx.y * h * w;
  const float* xp = x + plane; const float* yp = y + plane;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h * w; i += gridDim.x * blockDim.x) {
    int qy = i / w, qx = i - qy * w;
    float xq = xp[i], yq = yp[i];
    float gx = 0.f, gy = 0.f;
    for (int dy = -1; dy <= 1; ++dy) {
      int py = qy + dy;
      if (py < 0 || py >= h) continue;
      int my = refl_mult(py, qy, h);
      for (int dx = -1; dx <= 1; ++dx) {
        int px = qx + dx;
        if (px < 0 || px >= w) continue;
        float mlt = (float)(my * refl_mult(px, qx, w));
        if (mlt == 0.f) continue;
        float sx, sy, sxx, syy, sxy;
        ssim_sums(xp, yp, py, px, h, w, sx, sy, sxx, syy, sxy);
        SsimOut so = ssim_window(sx, sy, sxx, syy, sxy, true);
        float g = mlt * g_out[plane + (long long)py * w + px] * (1.f / 9.f);
        gy += g * (so.dmu_y + 2.f * yq * so.dY2 + xq * so.dXY);
        gx += g * (so.dmu_x + 2.f * xq * so.dX2 + yq * so.dXY);
      }
    }
    if (g_x) g_x[plane + i] = gx;
    if (g_y) g_y[plane + i] = gy;
  }
}

// ----------------------------------------------------------------------------------------------- instance masks, pyramids
#include "mdn_resize.cuh"

// ----------------------------------------------------------------------------------------------- mask evaluation
#include "mdn_metrics.cuh"

// ----------------------------------------------------------------------------------------------- flow evaluation
#include "mdn_flow_eval.cuh"

__global__ void __launch_bounds__(NTHREADS) binary_image_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, float thr) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = (x[i] >= thr) ? 1.f : 0.f;
}

}  // namespace mdn

// =================================================================================================== C ABI
using namespace mdn;

static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, const char* what = "") {
  snprintf(g_err, sizeof(g_err), fmt, what);
  return code;
}
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" MDN_API int mdn_version(void) { return MDN_ABI_VERSION; }
extern "C" MDN_API const char* mdn_last_error_string(void) { return g_err; }

struct WsLayout { size_t partials, sample_sums, refpack, snkeys, ticket, fmat, gfmat, total; int n_tiles; };

// Tile numbering: the LAST scale's tiles come first (tile_begin decreases with the scale index).  In a pyramid those are
// the small levels, whose tiles are mostly ragged (the slower generic paths) -- they start first and the full tiles of
// level 0 fill the grid's tail (measured round 2: 214.1 vs 216.5 us per step).
static int plan_tiles(const MdnLossDesc* d, KParams& K) {
  int t = 0;
  for (int s = d->n_scales - 1; s >= 0; --s) {
    KScale& Z = K.sc[s];
    Z.h = d->scale[s].height; Z.w = d->scale[s].width;
    Z.tiles_x = (Z.w + TW - 1) / TW; Z.tiles_y = (Z.h + TH - 1) / TH;
    Z.tile_begin = t;
    t += Z.tiles_x * Z.tiles_y * d->batch;
  }
  K.n_tiles = t;
  return t;
}

static int check_desc(const MdnLossDesc* d) {
  if (!d) return fail(MDN_ERR_NULL_POINTER, "desc is NULL");
  if (d->batch < 1 || d->n_scales < 1 || d->n_scales > MDN_MAX_SCALES || d->n_pairs < 1 || d->n_pairs > MDN_MAX_PAIRS)
    return fail(MDN_ERR_BAD_SHAPE, "batch / n_scales / n_pairs out of range");
  if (d->post < MDN_POST_SN || d->post > MDN_POST_TG) return fail(MDN_ERR_UNSUPPORTED, "unknown post-processing mode");
  if (d->mask_mode < MDN_MASK_MIN || d->mask_mode > MDN_MASK_SHARED) return fail(MDN_ERR_UNSUPPORTED, "unknown mask mode");
  if ((d->flags & MDN_OPT_PAD_BORDER) && (d->flags & MDN_OPT_PAD_REFLECTION)) return fail(MDN_ERR_UNSUPPORTED, "two padding modes");
  if ((d->flags & MDN_TERM_CONSIS) && d->mask_mode == MDN_MASK_SHARED)
    return fail(MDN_ERR_UNSUPPORTED, "consistency term needs two mobile maps (not MDN_MASK_SHARED)");
  const int f = d->flags;
  // poses instead of fundamental matrices: all pairs or none, and the inverse intrinsics of every scale
  const bool params = d->axisangle[0] != nullptr;      // pose parameters instead of pose matrices (ABI 3)
  bool poses = d->cam[0] != nullptr || params;
  for (int p = 0; p < d->n_pairs; ++p) {
    if (params) {
      if (!d->axisangle[p] || !d->translation[p]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "axisangle[p] / translation[p] (give every pair's or none)");
      if (d->cam[p]) return fail(MDN_ERR_UNSUPPORTED, "give either cam[p] or axisangle[p] / translation[p], not both");
    } else {
      if ((d->cam[p] != nullptr) != poses) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "cam[p] (give every pair's pose or none)");
      if (d->axisangle[p] || d->translation[p] || d->g_axisangle[p] || d->g_translation[p])
        return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "axisangle[0] (pose parameters: all pairs or none)");
    }
  }
  if (poses)
    for (int s = 0; s < d->n_scales; ++s)
      if (!d->inv_K[s]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "inv_K[s] (required with cam)");
  for (int p = 0; p < d->n_pairs; ++p)
    if (d->g_cam[p] && !poses) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "cam[p] (g_cam needs the poses)");
  for (int s = 0; s < d->n_scales; ++s) {
    const MdnScale& S = d->scale[s];
    if (S.height < 2 || S.width < 2 || (long long)S.height * S.width > (1ll << 30)) return fail(MDN_ERR_BAD_SHAPE, "height/width must be >= 2");
#define NEED(p, what) do { if (!(p)) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", what); if (!aligned16(p)) return fail(MDN_ERR_MISALIGNED, "%s is not 16-byte aligned", what); } while (0)
#define OPT(p, what) do { if ((p) && !aligned16(p)) return fail(MDN_ERR_MISALIGNED, "%s is not 16-byte aligned", what); } while (0)
    if (f & (MDN_TERM_PHOTO | MDN_TERM_SMOOTH)) NEED(S.tgt, "tgt");
    if (f & (MDN_TERM_EPIPOLAR | MDN_TERM_SMOOTH | MDN_TERM_CONSIS)) {
      NEED(S.mob[0], "mob[0]");
      if (d->mask_mode != MDN_MASK_SHARED) NEED(S.mob[1], "mob[1]");   // MIN / OWN / consistency read both maps
    }
    for (int p = 0; p < d->n_pairs; ++p) {
      if (f & MDN_TERM_PHOTO) { if (S.ref_packed[p]) OPT(S.ref_packed[p], "ref_packed"); else NEED(S.ref[p], "ref"); }
      if (f & (MDN_TERM_PHOTO | MDN_TERM_EPIPOLAR)) NEED(S.flow[p], "flow");
      if ((f & MDN_TERM_EPIPOLAR) && !poses) { if (!S.fmat[p]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "fmat"); }
      OPT(S.g_flow[p], "g_flow"); OPT(S.g_mob[p], "g_mob"); OPT(S.post_map[p], "post_map"); OPT(S.ori_map[p], "ori_map");
      OPT(S.warped[p], "warped"); OPT(S.diff[p], "diff"); OPT(S.ssim_map[p], "ssim_map");
    }
    if ((f & MDN_TERM_EPIPOLAR) && d->post == MDN_POST_TG) NEED(S.weight, "weight");
    if ((f & MDN_TERM_EPIPOLAR) && (f & (MDN_OPT_INST_MASK | MDN_OPT_CROSS_ENT)) && !S.inst) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "inst");
#undef NEED
#undef OPT
  }
  return MDN_OK;
}

static WarpGeom make_geom(int h, int w, bool cuda_arith, bool flowwarp_norm, int pad = 0) {
  WarpGeom G;
  G.pad = pad;
  G.wm1 = (float)(w - 1); G.hm1 = (float)(h - 1);
  G.inv_wm1 = (float)(1.0 / (double)(w - 1)); G.inv_hm1 = (float)(1.0 / (double)(h - 1));
  G.cuda_arith = cuda_arith; G.flowwarp_norm = flowwarp_norm;
  return G;
}

static WsLayout ws_layout(const MdnLossDesc* d, int n_tiles) {
  WsLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
  L.partials = take((size_t)n_tiles * NSLOT * sizeof(float));
  L.sample_sums = take((size_t)d->n_scales * d->batch * NSLOT * sizeof(float));
  size_t packed = 0;   // repacked source images: 16 bytes per pixel, per pair, per scale (photometric term only)
  if (d->flags & MDN_TERM_PHOTO)
    for (int s = 0; s < d->n_scales; ++s)
      packed += (size_t)d->n_pairs * d->batch * d->scale[s].height * d->scale[s].width * sizeof(float4);
  L.refpack = take(packed);
  L.snkeys = take((size_t)d->n_scales * d->n_pairs * d->batch * sizeof(unsigned long long));
  L.ticket = take(256);
  const size_t nf = (size_t)d->n_scales * d->n_pairs * d->batch * 9 * sizeof(float);
  const bool poses = d->cam[0] != nullptr || d->axisangle[0] != nullptr;
  L.fmat = take(poses ? nf : 0);
  L.gfmat = take(poses ? nf : 0);
  L.total = off;
  L.n_tiles = n_tiles;
  return L;
}

extern "C" MDN_API size_t mdn_loss_workspace_bytes(const MdnLossDesc* d) {
  if (check_desc(d) != MDN_OK) return 0;
  KParams K;
  memset(&K, 0, sizeof(K));
  return ws_layout(d, plan_tiles(d, K)).total;
}

// ev (optional): four events recorded on `stream` before the source repack, before the fused kernel, after it and
// after the finish kernel (mdn_loss_fused_profile)
static int launch_fused(const MdnLossDesc* d, float* loss_out, void* workspace, size_t workspace_bytes, void* stream_, cudaEvent_t* ev) {
  int rc = check_desc(d);
  if (rc != MDN_OK) return rc;
  if (!loss_out) return fail(MDN_ERR_NULL_POINTER, "loss_out is NULL");
  cudaStream_t stream = (cudaStream_t)stream_;
  FParams Q;
  memset(&Q, 0, sizeof(Q));
  KParams& K = Q.K;
  WsLayout L = ws_layout(d, plan_tiles(d, K));
  if (!workspace || workspace_bytes < L.total) return fail(MDN_ERR_WORKSPACE, "workspace too small");
  if (!aligned16(workspace)) return fail(MDN_ERR_MISALIGNED, "%s is not 16-byte aligned", "workspace");
  char* ws = (char*)workspace;
  K.batch = d->batch; K.n_scales = d->n_scales; K.n_pairs = d->n_pairs; K.post = d->post; K.mask_mode = d->mask_mode;
  K.flags = d->flags; K.threshold = (float)d->threshold;
  K.inv_threshold = d->threshold > 0 ? (float)(1.0 / d->threshold) : 0.f;
  K.partials = (float*)(ws + L.partials);
  unsigned long long* keys = (unsigned long long*)(ws + L.snkeys);
  K.snkey = keys;
  Q.sample_sums = (float*)(ws + L.sample_sums);
  K.ticket = (unsigned*)(ws + L.ticket);
  Q.loss_out = loss_out;
  const bool poses = (d->cam[0] != nullptr || d->axisangle[0] != nullptr) && (d->flags & MDN_TERM_EPIPOLAR);
  if (poses) {
    K.fmat_ws = (float*)(ws + L.fmat);
    const bool gr = (d->flags & MDN_OPT_GRADS) != 0;
    for (int p = 0; p < d->n_pairs; ++p) {
      K.cam[p] = d->cam[p]; K.aa[p] = d->axisangle[p]; K.tr[p] = d->translation[p];
      Q.g_cam[p] = gr ? d->g_cam[p] : nullptr;
      Q.g_aa[p] = gr ? d->g_axisangle[p] : nullptr; Q.g_tr[p] = gr ? d->g_translation[p] : nullptr;
    }
    for (int s = 0; s < d->n_scales; ++s) K.inv_K[s] = d->inv_K[s];
    if (d->flags & MDN_OPT_GRADS) Q.gf_ws = (float*)(ws + L.gfmat);
  }
  const bool use_ssim = (d->flags & MDN_OPT_SSIM) != 0;
  Q.alpha = d->alpha; Q.w_d2 = d->w_d2_sim; Q.w_e = d->w_e; Q.w_s = d->w_s; Q.w_c = d->w_c; Q.w_p = d->w_p;
  Q.l1_coef = use_ssim ? 0.15f : 1.f; Q.ssim_coef = use_ssim ? 0.85f : 0.f;
  for (int s = 0; s < d->n_scales; ++s) {
    const MdnScale& S = d->scale[s];
    KScale& Z = K.sc[s];
    Z.sx = S.flow_sx; Z.sy = S.flow_sy;
    Z.geom = make_geom(Z.h, Z.w, (d->flags & MDN_OPT_CUDA_ARITH) != 0, false);
    const double div = S.scale_div > 0.f ? (double)S.scale_div : 1.0;
    Q.scale_div[s] = (float)div;
    Q.inv_N[s] = 1.0 / ((double)d->batch * Z.h * Z.w);
    Q.inv_div[s] = 1.0 / div;
    Q.inv_cx[s] = Z.w > 1 ? 1.0 / ((double)d->batch * Z.h * (Z.w - 1)) : 0.0;
    Q.inv_cy[s] = Z.h > 1 ? 1.0 / ((double)d->batch * (Z.h - 1) * Z.w) : 0.0;
    const double N = (double)d->batch * Z.h * Z.w;
    Z.c_epi = (float)(d->w_e / (div * N));
    Z.c_nt = (float)((double)d->w_e * d->alpha / (div * N));
    Z.c_ce = (float)((double)d->w_e * d->w_d2_sim / (div * N));
    Z.c_l1 = (float)((double)d->w_p * Q.l1_coef / (div * 3.0 * N));
    Z.c_ssim = (float)((double)d->w_p * Q.ssim_coef / (div * 3.0 * N));
    Z.c_smx = (float)(d->w_s / (div * (double)d->batch * Z.h * (Z.w - 1)));
    Z.c_smy = (float)(d->w_s / (div * (double)d->batch * (Z.h - 1) * Z.w));
    Z.c_consis = (float)(d->w_c / (div * N));
    Z.tgt = S.tgt; Z.weight = S.weight; Z.inst = S.inst;
    for (int p = 0; p < 2; ++p) {
      Z.ref[p] = S.ref[p]; Z.flow[p] = S.flow[p]; Z.mob[p] = S.mob[p]; Z.fmat[p] = S.fmat[p];
      Z.g_flow[p] = S.g_flow[p]; Z.g_mob[p] = S.g_mob[p]; Q.g_fmat[s][p] = S.g_fmat[p];
      Z.post_map[p] = S.post_map[p]; Z.ori_map[p] = S.ori_map[p]; Z.warped[p] = S.warped[p]; Z.diff[p] = S.diff[p];
      Z.valid[p] = S.valid[p]; Z.ssim_map[p] = S.ssim_map[p];
    }
  }
  bool any_repack = false;
  {   // carve the repacked source images out of the workspace
    float4* rp = (float4*)(ws + L.refpack);
    for (int s = 0; s < d->n_scales; ++s)
      for (int p = 0; p < d->n_pairs; ++p) {
        K.sc[s].refp[p] = (d->flags & MDN_TERM_PHOTO) ? rp : nullptr;
        if (d->flags & MDN_TERM_PHOTO) rp += (size_t)d->batch * K.sc[s].h * K.sc[s].w;
        if ((d->flags & MDN_TERM_PHOTO) && d->scale[s].ref_packed[p]) {     // the caller's packed image: no repack
          K.sc[s].refp[p] = reinterpret_cast<float4*>(const_cast<float*>(d->scale[s].ref_packed[p]));
          K.sc[s].ref[p] = nullptr;
        } else any_repack = true;
      }
  }
  // the completion ticket is zeroed by the fused kernel itself; only the SN pre-pass needs a cleared buffer
  const bool sn_pass = (d->flags & MDN_TERM_EPIPOLAR) && d->post == MDN_POST_SN;
  const int sn_chunks = 16;
  const size_t nkeys = (size_t)d->n_scales * d->n_pairs * d->batch;
  const bool photo = (d->flags & MDN_TERM_PHOTO) != 0;
  if (ev) cudaEventRecord(ev[0], stream);
  if (sn_pass && cudaMemsetAsync(keys, 0, nkeys * sizeof(unsigned long long), stream) != cudaSuccess) return fail(MDN_ERR_CUDA, "memset failed");
  int n_pack = 0;
  if (photo && any_repack) {
    for (int s = 0; s < d->n_scales; ++s) {
      K.pack_begin[s] = n_pack;
      K.pack_blocks[s] = (K.sc[s].h * K.sc[s].w + NTHREADS * PACK_PX - 1) / (NTHREADS * PACK_PX);
      n_pack += K.pack_blocks[s] * d->n_pairs * d->batch;
    }
    K.pack_begin[d->n_scales] = n_pack;
  }
  // one pre-pass launch: source repack blocks, then SN-maximum blocks (either part may be empty)
  const int n_sn = sn_pass ? sn_chunks * (int)nkeys : 0;
  const int ratio = n_sn ? (n_pack + n_sn - 1) / n_sn : 0;            // repack blocks per SN block (0: SN blocks only)
  const int n_pre = n_sn ? std::max(n_sn, ratio ? (n_pack + ratio - 1) / ratio : 0) * (ratio + 1) : n_pack;
  if (n_pre > 0) MDN_LAUNCH(ref_pack_kernel, dim3(n_pre), dim3(NTHREADS), 0, stream, K, keys, n_pack, n_sn, ratio, sn_chunks);
  // DS / DC: the instance masks may still be in flight on another stream (their preparation overlaps the pre-pass above);
  // the launches that read them wait for the caller's event here
  if (d->inst_ready && cudaStreamWaitEvent(stream, (cudaEvent_t)d->inst_ready, 0) != cudaSuccess) return fail(MDN_ERR_CUDA, "cudaStreamWaitEvent failed");
  const size_t smem = fused_smem_floats(photo) * sizeof(float);
  static_assert(fused_smem_floats(true) * sizeof(float) <= 113 * 1024, "two CTAs per SM");
  bool maps = false;
  for (int s = 0; s < d->n_scales; ++s)
    for (int p = 0; p < 2; ++p) {
      const MdnScale& S = d->scale[s];
      maps |= S.post_map[p] || S.ori_map[p] || S.warped[p] || S.diff[p] || S.valid[p] || S.ssim_map[p];
    }
  K.prefetch_distance = FUSED_MIN_CTAS * 148;   // one wave of resident CTAs (148 SMs on B200)
#ifndef MDN_EMU
  {
    // TMA descriptors for the input tiles (target image, mobile maps): one box copy per plane instead of ~400 cp.async
    // with their index arithmetic.  A scale keeps the cp.async staging where its row pitch is not a multiple of 16 bytes
    // or a descriptor could not be encoded (no cuTensorMapEncodeTiled from the driver).
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = [] {
      void* fn = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess) fn = nullptr;
      return (EncodeFn)fn;
    }();
    const bool need_tgt = (d->flags & (MDN_TERM_PHOTO | MDN_TERM_SMOOTH)) != 0;
    const bool need_mask = (d->flags & (MDN_TERM_EPIPOLAR | MDN_TERM_SMOOTH | MDN_TERM_CONSIS)) != 0;
    for (int s = 0; s < d->n_scales; ++s) {
      KScale& Z = K.sc[s];
      bool ok = encode != nullptr && (Z.w % 4) == 0;
      auto make = [&](CUtensorMap* m, const float* base, int planes) {
        if (!ok || !base) return;
        const cuuint64_t dims[3] = {(cuuint64_t)Z.w, (cuuint64_t)Z.h, (cuuint64_t)planes};
        const cuuint64_t strides[2] = {(cuuint64_t)Z.w * 4, (cuuint64_t)Z.w * Z.h * 4};
        const cuuint32_t box[3] = {(cuuint32_t)S2, (cuuint32_t)R2H, 1}, es[3] = {1, 1, 1};
        ok = encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
      };
      if (need_tgt) make(&K.tmap[s][0], Z.tgt, 3 * d->batch);
      if (need_mask) {
        make(&K.tmap[s][1], Z.mob[0], d->batch);
        if (d->mask_mode != MDN_MASK_SHARED) make(&K.tmap[s][2], Z.mob[1], d->batch);
      }
      K.tma_ok[s] = ok ? 1 : 0;
    }
    // every input tile arrives by TMA: the L2 prefetch of the next wave (flows only, then) no longer pays for its
    // instructions (measured round 2: 218.7 vs 219.5 / 201.1 vs 202.9 us per step without it); kept for cp.async staging
    bool all_tma = true;
    for (int s = 0; s < d->n_scales; ++s) all_tma = all_tma && K.tma_ok[s];
    if (all_tma) K.prefetch_distance = 1 << 30;
  }
#endif
  if (ev) cudaEventRecord(ev[1], stream);
  const dim3 grid(K.n_tiles), block(FT);
  // the instantiations, indexed [pad][photo][maps].  PAD is the padding_mode of the flow warp (0 zeros, 1 border,
  // 2 reflection); only the photometric term warps, so without it every pad index holds the zeros-padding kernels.
  using FusedFn = void (*)(KParams);
  static const FusedFn fused_kernels[3][2][2] = {
      {{fused_tile_kernel<false, false>, fused_tile_kernel<false, true>}, {fused_tile_kernel<true, false>, fused_tile_kernel<true, true>}},
      {{fused_tile_kernel<false, false>, fused_tile_kernel<false, true>}, {fused_tile_kernel<true, false, 1>, fused_tile_kernel<true, true, 1>}},
      {{fused_tile_kernel<false, false>, fused_tile_kernel<false, true>}, {fused_tile_kernel<true, false, 2>, fused_tile_kernel<true, true, 2>}}};
  // > 48 KB of dynamic shared memory needs the opt-in attribute, per device (idempotent; set once per device).  The bit is
  // published only after every attribute call succeeded, with an atomic OR: concurrent first calls from two host threads
  // may both set the attributes (harmless) but never see a half-initialised device.
  static std::atomic<unsigned long long> smem_opt_in_devices{0ull};
  int dev_index = 0;
#ifndef MDN_EMU
  cudaGetDevice(&dev_index);
#endif
  const unsigned long long dev_bit = 1ull << (dev_index & 63);
  if (!(smem_opt_in_devices.load(std::memory_order_acquire) & dev_bit)) {
    const int bytes = (int)(fused_smem_floats(true) * sizeof(float));
    cudaError_t a = cudaSuccess;
    for (const auto& by_photo : fused_kernels)
      for (const auto& by_maps : by_photo)
        for (const FusedFn kfn : by_maps)
          if (a == cudaSuccess) a = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (a != cudaSuccess) {
      cudaGetLastError();
      snprintf(g_err, sizeof(g_err), "the fused kernel needs %d bytes of opt-in shared memory per block on device %d: %s", bytes, dev_index,
               cudaGetErrorString(a));
      return MDN_ERR_CUDA;
    }
    smem_opt_in_devices.fetch_or(dev_bit, std::memory_order_release);
  }
  const int pad = (d->flags & MDN_OPT_PAD_BORDER) ? 1 : ((d->flags & MDN_OPT_PAD_REFLECTION) ? 2 : 0);
  const FusedFn kfn = fused_kernels[pad][photo][maps];
  MDN_LAUNCH(kfn, grid, block, smem, stream, K);
  if (ev) cudaEventRecord(ev[2], stream);
  MDN_LAUNCH(finish_kernel, dim3(d->batch), dim3(FIN_ROWS * NSLOT), 0, stream, Q);
  if (ev) cudaEventRecord(ev[3], stream);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return MDN_OK;
}

extern "C" MDN_API int mdn_loss_fused(const MdnLossDesc* d, float* loss_out, void* workspace, size_t workspace_bytes, void* stream) {
  return launch_fused(d, loss_out, workspace, workspace_bytes, stream, nullptr);
}

extern "C" MDN_API int mdn_loss_fused_profile(const MdnLossDesc* d, float* loss_out, void* workspace, size_t workspace_bytes, void* stream,
                                              float* ms_out) {
  if (!ms_out) return fail(MDN_ERR_NULL_POINTER, "ms_out is NULL");
  cudaEvent_t ev[4];
  for (int i = 0; i < 4; ++i)
    if (cudaEventCreate(&ev[i]) != cudaSuccess) return fail(MDN_ERR_CUDA, "cudaEventCreate failed");
  int rc = launch_fused(d, loss_out, workspace, workspace_bytes, stream, ev);
  if (rc == MDN_OK && cudaEventSynchronize(ev[3]) != cudaSuccess) rc = fail(MDN_ERR_CUDA, "cudaEventSynchronize failed");
  for (int i = 0; i < 3; ++i) {
    ms_out[i] = 0.f;
    if (rc == MDN_OK) cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
  }
  for (int i = 0; i < 4; ++i) cudaEventDestroy(ev[i]);
  return rc;
}

extern "C" MDN_API int mdn_loss_scale_grads(const MdnLossDesc* d, const float* g, float* applied, void* stream_) {
  if (!d || !g || !applied) return fail(MDN_ERR_NULL_POINTER, "desc / g / applied is NULL");
  if (d->batch < 1 || d->n_scales < 1 || d->n_scales > MDN_MAX_SCALES) return fail(MDN_ERR_BAD_SHAPE, "batch / n_scales out of range");
  cudaStream_t stream = (cudaStream_t)stream_;
  GradList L;
  memset(&L, 0, sizeof(L));
  for (int s = 0; s < d->n_scales; ++s) {
    const MdnScale& S = d->scale[s];
    const long long hw = (long long)S.height * S.width;
    for (int p = 0; p < MDN_MAX_PAIRS; ++p) {
      if (S.g_flow[p]) { L.ptr[L.n] = S.g_flow[p]; L.count[L.n++] = 2 * hw * d->batch; }
      if (S.g_mob[p]) { L.ptr[L.n] = S.g_mob[p]; L.count[L.n++] = hw * d->batch; }
      if (S.g_fmat[p]) { L.ptr[L.n] = S.g_fmat[p]; L.count[L.n++] = 9ll * d->batch; }
    }
  }
  for (int p = 0; p < MDN_MAX_PAIRS; ++p) {
    if (d->g_cam[p]) { L.ptr[L.n] = d->g_cam[p]; L.count[L.n++] = 16ll * d->batch; }
    if (d->g_axisangle[p]) { L.ptr[L.n] = d->g_axisangle[p]; L.count[L.n++] = 3ll * d->batch; }
    if (d->g_translation[p]) { L.ptr[L.n] = d->g_translation[p]; L.count[L.n++] = 3ll * d->batch; }
  }
  if (L.n == 0) return MDN_OK;
  // applied[1] (MDN_OUT_APPLIED + 1) is the completion ticket, zeroed by mdn_loss_fused
  MDN_LAUNCH(scale_grads_kernel, dim3(296), dim3(NTHREADS), 0, stream, L, g, applied, reinterpret_cast<unsigned*>(applied + 1));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return MDN_OK;
}

static int fund_args(FundArgs& A, const float* const* inv_K, const float* const* cam, float* const* g_cam, int n_scales,
                     int n_pairs, int batch) {
  if (!inv_K || !cam) return fail(MDN_ERR_NULL_POINTER, "inv_K / cam pointer array is NULL");
  if (n_scales < 1 || n_scales > MDN_MAX_SCALES || n_pairs < 1 || n_pairs > MDN_MAX_PAIRS || batch < 1)
    return fail(MDN_ERR_BAD_SHAPE, "n_scales / n_pairs / batch out of range");
  memset(&A, 0, sizeof(A));
  A.n_scales = n_scales; A.n_pairs = n_pairs; A.batch = batch;
  for (int s = 0; s < n_scales; ++s) { if (!inv_K[s]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "inv_K[s]"); A.inv_K[s] = inv_K[s]; }
  for (int p = 0; p < n_pairs; ++p) {
    if (!cam[p]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "cam[p]");
    A.cam[p] = cam[p];
    if (g_cam) { if (!g_cam[p]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "g_cam[p]"); A.g_cam[p] = g_cam[p]; }
  }
  return MDN_OK;
}

extern "C" MDN_API int mdn_fundamental_fwd(const float* const* inv_K, const float* const* cam, float* fmat, int32_t n_scales,
                                           int32_t n_pairs, int32_t batch, void* stream) {
  FundArgs A;
  int rc = fund_args(A, inv_K, cam, nullptr, n_scales, n_pairs, batch);
  if (rc != MDN_OK) return rc;
  if (!fmat) return fail(MDN_ERR_NULL_POINTER, "fmat is NULL");
  const int n = n_pairs * batch;
  MDN_LAUNCH(fundamental_fwd_kernel, dim3((n + 63) / 64), dim3(64), 0, (cudaStream_t)stream, A, fmat);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_fundamental_bwd(const float* const* inv_K, const float* const* cam, const float* g_fmat,
                                           float* const* g_cam, int32_t n_scales, int32_t n_pairs, int32_t batch, void* stream) {
  FundArgs A;
  if (!g_cam) return fail(MDN_ERR_NULL_POINTER, "g_cam pointer array is NULL");
  int rc = fund_args(A, inv_K, cam, g_cam, n_scales, n_pairs, batch);
  if (rc != MDN_OK) return rc;
  if (!g_fmat) return fail(MDN_ERR_NULL_POINTER, "g_fmat is NULL");
  const int n = n_pairs * batch;
  MDN_LAUNCH(fundamental_bwd_kernel, dim3((n + 63) / 64), dim3(64), 0, (cudaStream_t)stream, A, g_fmat);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

static inline unsigned blocks_for(long long n, int cap = 148 * 8) {
  long long b = (n + NTHREADS - 1) / NTHREADS;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

extern "C" MDN_API int mdn_epipolar_points_fwd(const float* p1, const float* p2, const float* fmat, float* out, int32_t batch,
                                       int64_t n, void* stream) {
  if (!p1 || !p2 || !fmat || !out) return fail(MDN_ERR_NULL_POINTER, "p1 / p2 / fmat / out is NULL");
  if (batch < 1 || n < 1) return fail(MDN_ERR_BAD_SHAPE, "batch and n must be >= 1");
  MDN_LAUNCH(epipolar_points_fwd_kernel, dim3(blocks_for(n), batch), dim3(NTHREADS), 0, (cudaStream_t)stream, p1, p2, fmat, out, (long long)n);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

static const int EPB_BLOCKS = 64;
extern "C" MDN_API size_t mdn_epipolar_points_workspace_bytes(int32_t batch, int64_t) {
  return (size_t)(batch < 1 ? 0 : batch) * EPB_BLOCKS * EPB_SLOTS * sizeof(float);
}

extern "C" MDN_API int mdn_epipolar_points_bwd(const float* p1, const float* p2, const float* fmat, const float* g_out, float* g_p1,
                                       float* g_p2, float* g_fmat, int32_t batch, int64_t n, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  if (!p1 || !p2 || !fmat || !g_out) return fail(MDN_ERR_NULL_POINTER, "p1 / p2 / fmat / g_out is NULL");
  if (batch < 1 || n < 1) return fail(MDN_ERR_BAD_SHAPE, "batch and n must be >= 1");
  if (!workspace || workspace_bytes < mdn_epipolar_points_workspace_bytes(batch, n)) return fail(MDN_ERR_WORKSPACE, "workspace too small");
  MDN_LAUNCH(epipolar_points_bwd_kernel, dim3(EPB_BLOCKS, batch), dim3(NTHREADS), 0, (cudaStream_t)stream, p1, p2, fmat, g_out, g_p1, g_p2,
             (float*)workspace, (long long)n);
  if (g_fmat) MDN_LAUNCH(epipolar_points_bwd_finish_kernel, dim3(batch), dim3(32), 0, (cudaStream_t)stream, (const float*)workspace, g_fmat, EPB_BLOCKS);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_flow_warp_fwd(const float* ref, const float* flow, float* warped, float* grid_out, uint8_t* valid,
                                 int32_t batch, int32_t channels, int32_t height, int32_t width, int32_t warp_flags, void* stream) {
  if (!flow || (warped && !ref)) return fail(MDN_ERR_NULL_POINTER, "flow / ref is NULL");
  if (batch < 1 || channels < 0 || height < 2 || width < 2) return fail(MDN_ERR_BAD_SHAPE, "bad warp shape (h,w >= 2)");
  MDN_LAUNCH(flow_warp_fwd_kernel, dim3(blocks_for((long long)height * width), batch), dim3(NTHREADS), 0, (cudaStream_t)stream, ref, flow, warped,
             grid_out, valid, (int)channels, (int)height, (int)width, make_geom(height, width, (warp_flags & 2) != 0, (warp_flags & 1) != 0, (warp_flags >> 2) & 3));
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_flow_warp_bwd(const float* ref, const float* flow, const float* g_warped, float* g_flow, int32_t batch,
                                 int32_t channels, int32_t height, int32_t width, int32_t warp_flags, void* stream) {
  if (!ref || !flow || !g_warped || !g_flow) return fail(MDN_ERR_NULL_POINTER, "ref / flow / g_warped / g_flow is NULL");
  if (batch < 1 || channels < 1 || height < 2 || width < 2) return fail(MDN_ERR_BAD_SHAPE, "bad warp shape (h,w >= 2)");
  MDN_LAUNCH(flow_warp_bwd_kernel, dim3(blocks_for((long long)height * width), batch), dim3(NTHREADS), 0, (cudaStream_t)stream, ref, flow, g_warped,
             g_flow, (int)channels, (int)height, (int)width, make_geom(height, width, (warp_flags & 2) != 0, false, (warp_flags >> 2) & 3));
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_ssim_fwd(const float* x, const float* y, float* out, int32_t planes, int32_t height, int32_t width, void* stream) {
  if (!x || !y || !out) return fail(MDN_ERR_NULL_POINTER, "x / y / out is NULL");
  if (planes < 1 || height < 2 || width < 2) return fail(MDN_ERR_BAD_SHAPE, "bad SSIM shape (h,w >= 2)");
  MDN_LAUNCH(ssim_fwd_kernel, dim3(blocks_for((long long)height * width), planes), dim3(NTHREADS), 0, (cudaStream_t)stream, x, y, out, (int)height, (int)width);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_ssim_bwd(const float* x, const float* y, const float* g_out, float* g_x, float* g_y, int32_t planes,
                            int32_t height, int32_t width, void* stream) {
  if (!x || !y || !g_out) return fail(MDN_ERR_NULL_POINTER, "x / y / g_out is NULL");
  if (planes < 1 || height < 2 || width < 2) return fail(MDN_ERR_BAD_SHAPE, "bad SSIM shape (h,w >= 2)");
  MDN_LAUNCH(ssim_bwd_kernel, dim3(blocks_for((long long)height * width), planes), dim3(NTHREADS), 0, (cudaStream_t)stream, x, y, g_out, g_x, g_y,
             (int)height, (int)width);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_instance_mask_union(const uint8_t* const* masks, const int32_t* counts, uint8_t* out, int32_t batch,
                                               int64_t hw, void* stream) {
  if (!masks || !counts || !out) return fail(MDN_ERR_NULL_POINTER, "masks / counts / out is NULL");
  if (batch < 1 || hw < 1) return fail(MDN_ERR_BAD_SHAPE, "batch / hw out of range");
  for (int b0 = 0; b0 < batch; b0 += UNION_CHUNK) {
    UnionArgs A;
    memset(&A, 0, sizeof(A));
    const int nb = std::min(UNION_CHUNK, batch - b0);
    for (int b = 0; b < nb; ++b) {
      if (counts[b0 + b] < 0 || (counts[b0 + b] > 0 && !masks[b0 + b])) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "masks[b]");
      A.masks[b] = masks[b0 + b]; A.count[b] = counts[b0 + b];
    }
    MDN_LAUNCH(instance_union_kernel, dim3(blocks_for(hw, 296), nb), dim3(NTHREADS), 0, (cudaStream_t)stream, A, out + (long long)b0 * hw, (long long)hw);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_instance_mask_union_table(const uint8_t* const* masks, const int32_t* counts, uint8_t* out,
                                                     int32_t batch, int64_t hw, void* stream) {
  if (!masks || !counts || !out) return fail(MDN_ERR_NULL_POINTER, "masks / counts / out is NULL");
  if (batch < 1 || batch > 65535 || hw < 1) return fail(MDN_ERR_BAD_SHAPE, "batch / hw out of range");
  MDN_LAUNCH(instance_union_table_kernel, dim3(blocks_for(hw, 296), batch), dim3(NTHREADS), 0, (cudaStream_t)stream, masks,
             (const int*)counts, out, (long long)hw);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

static inline int aa_taps(int in_size, int out_size) {   // ceil(support) * 2 + 1 with support = max(in / out, 1)
  const float sc = (float)in_size / (float)out_size;
  return (int)ceilf(sc >= 1.f ? sc : 1.f) * 2 + 1;
}

struct ResizeWs { size_t tmp[MDN_MAX_SCALES], wxt[MDN_MAX_SCALES], wyt[MDN_MAX_SCALES], xspan[MDN_MAX_SCALES], yspan[MDN_MAX_SCALES], total; };

static ResizeWs resize_ws_layout(int batch, int in_h, int in_w, const int32_t* out_h, const int32_t* out_w, int n_out) {
  ResizeWs L;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
  for (int k = 0; k < n_out; ++k) {
    L.tmp[k] = take((size_t)batch * in_h * out_w[k] * sizeof(float));
    L.wxt[k] = take((size_t)aa_taps(in_w, out_w[k]) * out_w[k] * sizeof(float));
    L.wyt[k] = take((size_t)aa_taps(in_h, out_h[k]) * out_h[k] * sizeof(float));
    L.xspan[k] = take((size_t)out_w[k] * sizeof(int2));
    L.yspan[k] = take((size_t)out_h[k] * sizeof(int2));
  }
  L.total = off;
  return L;
}

static int check_resize_sizes(int32_t batch, int32_t in_h, int32_t in_w, const int32_t* out_h, const int32_t* out_w, int32_t n_out) {
  if (!out_h || !out_w) return fail(MDN_ERR_NULL_POINTER, "out_h / out_w is NULL");
  if (batch < 1 || in_h < 1 || in_w < 1 || n_out < 1 || n_out > MDN_MAX_SCALES) return fail(MDN_ERR_BAD_SHAPE, "batch / size / n_out out of range");
  for (int k = 0; k < n_out; ++k)
    if (out_h[k] < 1 || out_w[k] < 1) return fail(MDN_ERR_BAD_SHAPE, "output size out of range");
  return MDN_OK;
}

extern "C" MDN_API size_t mdn_instance_mask_resize_workspace_bytes(int32_t batch, int32_t in_h, int32_t in_w, const int32_t* out_h,
                                                                   const int32_t* out_w, int32_t n_out) {
  if (check_resize_sizes(batch, in_h, in_w, out_h, out_w, n_out) != MDN_OK) return 0;
  return resize_ws_layout(batch, in_h, in_w, out_h, out_w, n_out).total;
}

template <typename TIn, typename TOut>
static int launch_resize(const TIn* src, int32_t batch, int32_t in_h, int32_t in_w, TOut* const* dst, const int32_t* out_h,
                         const int32_t* out_w, int32_t n_out, void* workspace, size_t workspace_bytes, void* stream,
                         bool packed = false) {
  if (!src || !dst) return fail(MDN_ERR_NULL_POINTER, "src / dst is NULL");
  int rc = check_resize_sizes(batch, in_h, in_w, out_h, out_w, n_out);
  if (rc != MDN_OK) return rc;
  ResizeArgs A;
  memset(&A, 0, sizeof(A));
  A.n_out = n_out; A.batch = batch; A.ih = in_h; A.iw = in_w; A.packed = packed ? 1 : 0;
  const ResizeWs L = resize_ws_layout(batch, in_h, in_w, out_h, out_w, n_out);
  if (!workspace || workspace_bytes < L.total) return fail(MDN_ERR_WORKSPACE, "workspace too small");
  if (!aligned16(workspace)) return fail(MDN_ERR_MISALIGNED, "%s is not 16-byte aligned", "workspace");
  char* ws = (char*)workspace;
  int hrows = 0, vrows = 0, max_w = 0, n_idx = 0;
  const int hgroups = (in_h + AA_HROWS - 1) / AA_HROWS;
  for (int k = 0; k < n_out; ++k) {
    if (!dst[k]) return fail(MDN_ERR_NULL_POINTER, "%s is NULL", "dst[k]");
    A.dst[k] = dst[k]; A.oh[k] = out_h[k]; A.ow[k] = out_w[k];
    A.tmp[k] = (float*)(ws + L.tmp[k]); A.wxt[k] = (float*)(ws + L.wxt[k]); A.wyt[k] = (float*)(ws + L.wyt[k]);
    A.xspan[k] = (int2*)(ws + L.xspan[k]); A.yspan[k] = (int2*)(ws + L.yspan[k]);
    A.ty[k] = aa_taps(in_h, out_h[k]);
    A.row_begin[k] = hrows; A.vrow_begin[k] = vrows;
    if (aa_taps(in_h, out_h[k]) > AA_MAXTAPS || aa_taps(in_w, out_w[k]) > AA_MAXTAPS)
      return fail(MDN_ERR_UNSUPPORTED, "down-scaling factor above 500 is not supported");
    const int chunks = (out_w[k] + 127) / 128;
    hrows += batch * hgroups * chunks;
    vrows += batch * ((out_h[k] + AA_VROWS - 1) / AA_VROWS) * chunks;
    max_w = std::max(max_w, (int)out_w[k]);
    n_idx += out_w[k] + out_h[k];
  }
  A.row_begin[n_out] = hrows; A.vrow_begin[n_out] = vrows;
  cudaStream_t st = (cudaStream_t)stream;
  MDN_LAUNCH(instance_resize_weights_kernel, dim3((n_idx + NTHREADS / 32 - 1) / (NTHREADS / 32)), dim3(NTHREADS), 0, st, A, n_idx);
  // {0,1} masks: one fused pass out of bit-packed rows when every level's source window fits a block's shared memory
  // (down-scaling factors up to ~15 at these widths); otherwise, and for fp32 images, the two separable passes
  bool fused = sizeof(TIn) == 1 && sizeof(TOut) == 1 && !getenv("MDN_RESIZE_TWO_PASS");
  int frows = 0;
  for (int k = 0; k < n_out && fused; ++k) {
    const double sy = std::max(1.0, (double)in_h / out_h[k]), sx = std::max(1.0, (double)in_w / out_w[k]);
    const int ty = aa_taps(in_h, out_h[k]), tx = aa_taps(in_w, out_w[k]);
    const int cols = std::min(128, (int)out_w[k]);
    // source columns a 128-column chunk can span (+ alignment to a 32-pixel word + the funnel shift's slack word)
    const int words = (int)std::ceil((cols * sx + tx + 2) / 32.0) + 2;
    // R output rows need at most (R - 1) sy + 1 + ty source rows
    if (words > AF_W || ty + 1 > AF_NR) { fused = false; break; }
    const int R = std::min((int)std::floor((AF_NR - ty - 1) / sy) + 1, 16);
    A.frows[k] = R;
    A.frow_begin[k] = frows;
    frows += batch * ((out_h[k] + R - 1) / R) * ((out_w[k] + 127) / 128);
  }
  A.frow_begin[n_out] = frows;
  const int nwg = (in_w + 31) / 32 + 1;      // packed row pitch in words (one zero word of slack)
  if (fused && (size_t)batch * in_h * nwg * sizeof(unsigned) > (size_t)batch * in_h * out_w[0] * sizeof(float)) fused = false;
  if (fused) {
    unsigned* gbits = reinterpret_cast<unsigned*>(A.tmp[0]);     // (the two-pass temporary of level 0 is free on this path)
    const long long n_words = (long long)batch * in_h * nwg;
    (void)n_words;
    MDN_LAUNCH(mask_bitpack_kernel, dim3(std::min(batch * in_h, 148 * 16)), dim3(NTHREADS), 0, st,
               reinterpret_cast<const uint8_t*>(src), gbits, batch * in_h, (int)in_w, nwg);
    MDN_LAUNCH(instance_mask_resize_fused_kernel, dim3(frows), dim3(128), 0, st, A, (const unsigned*)gbits, nwg);
  } else {
    { auto kfn = instance_resize_h_kernel<TIn>; MDN_LAUNCH(kfn, dim3(hrows), dim3(128), 0, st, A, src); }
    { auto kfn = instance_resize_v_kernel<TOut>; MDN_LAUNCH(kfn, dim3(vrows), dim3(128), 0, st, A); }
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_instance_mask_resize(const uint8_t* src, int32_t batch, int32_t in_h, int32_t in_w, uint8_t* const* dst,
                                                const int32_t* out_h, const int32_t* out_w, int32_t n_out, void* workspace,
                                                size_t workspace_bytes, void* stream) {
  return launch_resize<uint8_t, uint8_t>(src, batch, in_h, in_w, dst, out_h, out_w, n_out, workspace, workspace_bytes, stream);
}

extern "C" MDN_API int mdn_image_pyramid(const float* src, int32_t planes, int32_t in_h, int32_t in_w, float* const* dst,
                                         const int32_t* out_h, const int32_t* out_w, int32_t n_out, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  return launch_resize<float, float>(src, planes, in_h, in_w, dst, out_h, out_w, n_out, workspace, workspace_bytes, stream);
}

extern "C" MDN_API int mdn_image_pyramid_packed(const float* src, int32_t planes, int32_t in_h, int32_t in_w, float* const* dst,
                                                const int32_t* out_h, const int32_t* out_w, int32_t n_out, void* workspace,
                                                size_t workspace_bytes, void* stream) {
  if (planes % 3) return fail(MDN_ERR_BAD_SHAPE, "planes must be a multiple of 3 (B x RGB)");
  return launch_resize<float, float>(src, planes, in_h, in_w, dst, out_h, out_w, n_out, workspace, workspace_bytes, stream, true);
}

extern "C" MDN_API int mdn_normalize_u8(const uint8_t* src, float* dst, int32_t batch, int32_t height, int32_t width,
                                        const float* mean, const float* stdv, void* stream) {
  if (!src || !dst || !mean || !stdv) return fail(MDN_ERR_NULL_POINTER, "src / dst / mean / std is NULL");
  if (batch < 1 || height < 1 || width < 1) return fail(MDN_ERR_BAD_SHAPE, "batch / height / width out of range");
  NormArgs A;
  for (int c = 0; c < 3; ++c) { A.mean[c] = mean[c]; A.stdv[c] = stdv[c]; }
  const long long hw = (long long)height * width;
  MDN_LAUNCH(normalize_u8_kernel, dim3(blocks_for(hw, 148 * 4), batch), dim3(NTHREADS), 0, (cudaStream_t)stream, src, dst, hw, A);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API int mdn_binary_image(const float* x, float* out, int64_t n, float threshold, void* stream) {
  if (!x || !out) return fail(MDN_ERR_NULL_POINTER, "x / out is NULL");
  if (n < 1) return MDN_OK;
  MDN_LAUNCH(binary_image_kernel, dim3(blocks_for(n)), dim3(NTHREADS), 0, (cudaStream_t)stream, x, out, (long long)n, threshold);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" MDN_API size_t mdn_mask_confusion_workspace_bytes(int32_t batch, int32_t n_thr) {
  if (batch < 1 || batch > 65535 || n_thr < 1 || n_thr > CONF_MAX_THR) {
    fail(MDN_ERR_BAD_SHAPE, "batch / n_thr out of range");
    return 0;
  }
  return (size_t)batch * 2 * (size_t)(n_thr + 1) * sizeof(unsigned);
}

extern "C" MDN_API int mdn_mask_confusion(const float* pred, const uint8_t* gt, const float* thresholds, int32_t n_thr,
                                          int64_t* counts, int32_t batch, int64_t hw, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  if (!pred || !gt || !thresholds || !counts || !workspace)
    return fail(MDN_ERR_NULL_POINTER, "pred / gt / thresholds / counts / workspace is NULL");
  if (batch < 1 || batch > 65535 || hw < 1 || hw > 2147483647ll || n_thr < 1 || n_thr > CONF_MAX_THR)
    return fail(MDN_ERR_BAD_SHAPE, "batch / hw / n_thr out of range");
  if (!aligned16(pred) || !aligned16(gt) || !aligned16(thresholds) || !aligned16(counts) || !aligned16(workspace))
    return fail(MDN_ERR_MISALIGNED, "%s is not 16-byte aligned", "pred / gt / thresholds / counts / workspace");
  const size_t need = mdn_mask_confusion_workspace_bytes(batch, n_thr);
  if (workspace_bytes < need) return fail(MDN_ERR_WORKSPACE, "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(workspace, 0, need, st);
  if (e != cudaSuccess) return fail(MDN_ERR_CUDA, "cudaMemsetAsync failed: %s", cudaGetErrorString(e));
  int top = 1;
  while (2 * top <= n_thr) top *= 2;
  // enough pixels per block that the flush of its 2 (K + 1) bins stays small next to its counting; at most about
  // 8 blocks per SM over the batch
  const long long per_block = std::max<long long>(CONF_THREADS * 16, 8ll * 2 * (n_thr + 1));
  const long long bx = std::max<long long>(1, std::min<long long>((hw + per_block - 1) / per_block, (148 * 8 + batch - 1) / batch));
  MDN_LAUNCH(mask_confusion_kernel, dim3((unsigned)bx, batch), dim3(CONF_THREADS), 0, st, pred, gt, thresholds, (int)n_thr,
             top, (unsigned*)workspace, (long long)hw);
  MDN_LAUNCH(mask_confusion_finish_kernel, dim3(batch), dim3(CONF_THREADS), 0, st, (const unsigned*)workspace, (int)n_thr,
             (long long*)counts);
  e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

// Blocks per sample of flow_errors_kernel: a function of the ground-truth size alone, never of the device.
static int flow_errors_blocks(long long gt_hw) {
  const long long quads = (gt_hw + 3) / 4, per_block = (long long)FE_THREADS * FE_QUADS_PER_THREAD;
  return (int)std::max<long long>(1, std::min<long long>((quads + per_block - 1) / per_block, FE_MAX_BLOCKS));
}

static bool flow_errors_shape_ok(int32_t batch, int32_t height, int32_t width, int32_t gt_height, int32_t gt_width,
                                 int32_t n_regions) {
  return batch >= 1 && batch <= 65535 && height >= 1 && width >= 1 && gt_height >= 1 && gt_width >= 1 &&
         (long long)height * width <= 2147483647ll && (long long)gt_height * gt_width <= 2147483647ll &&
         n_regions >= 1 && n_regions <= FE_MAX_REGIONS;
}

extern "C" MDN_API size_t mdn_flow_errors_workspace_bytes(int32_t batch, int32_t height, int32_t width,
                                                          int32_t gt_height, int32_t gt_width, int32_t n_regions) {
  if (!flow_errors_shape_ok(batch, height, width, gt_height, gt_width, n_regions)) {
    fail(MDN_ERR_BAD_SHAPE, "batch / sizes / n_regions out of range");
    return 0;
  }
  const size_t parts = (size_t)batch * flow_errors_blocks((long long)gt_height * gt_width) * n_regions;
  return parts * (sizeof(double) + 2 * sizeof(long long));
}

template <int RT>
static void flow_errors_launch(const FlowArgs& a, int batch, long long* counts, double* epe_sum, cudaStream_t st) {
  MDN_LAUNCH(flow_errors_kernel<RT>, dim3(a.nblk, batch), dim3(FE_THREADS), 0, st, a);
  MDN_LAUNCH(flow_errors_finish_kernel<RT>, dim3(batch), dim3(FE_THREADS), 0, st, (const double*)a.part_sum,
             (const long long*)a.part_cnt, a.nblk, a.R, counts, epe_sum);
}

extern "C" MDN_API int mdn_flow_errors(const float* flow, int32_t height, int32_t width, float scale_x, float scale_y,
                                       const float* gt_flow, const uint8_t* gt_valid, const uint8_t* region,
                                       int32_t n_regions, int32_t gt_height, int32_t gt_width, int32_t batch,
                                       float abs_thr, float rel_thr, int64_t* counts, double* epe_sum, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  if (!flow || !gt_flow || !gt_valid || !counts || !epe_sum || !workspace)
    return fail(MDN_ERR_NULL_POINTER, "flow / gt_flow / gt_valid / counts / epe_sum / workspace is NULL");
  if (!region && n_regions > 1) return fail(MDN_ERR_NULL_POINTER, "region is NULL with n_regions > 1");
  if (!flow_errors_shape_ok(batch, height, width, gt_height, gt_width, n_regions))
    return fail(MDN_ERR_BAD_SHAPE, "batch / sizes / n_regions out of range");
  if (!std::isfinite(scale_x) || !std::isfinite(scale_y) || !std::isfinite(abs_thr) || !std::isfinite(rel_thr) ||
      abs_thr < 0.f || rel_thr < 0.f)
    return fail(MDN_ERR_BAD_SHAPE, "scale / threshold out of range (non-finite or a negative threshold)");
  if (!aligned16(flow) || !aligned16(gt_flow) || !aligned16(gt_valid) || (region && !aligned16(region)) ||
      !aligned16(counts) || !aligned16(epe_sum) || !aligned16(workspace))
    return fail(MDN_ERR_MISALIGNED, "%s is not 16-byte aligned",
                "flow / gt_flow / gt_valid / region / counts / epe_sum / workspace");
  const size_t need = mdn_flow_errors_workspace_bytes(batch, height, width, gt_height, gt_width, n_regions);
  if (workspace_bytes < need) return fail(MDN_ERR_WORKSPACE, "workspace too small");
  FlowArgs a;
  a.flow = flow; a.gt = gt_flow; a.valid = gt_valid; a.region = region;
  a.nblk = flow_errors_blocks((long long)gt_height * gt_width);
  a.part_sum = (double*)workspace;
  a.part_cnt = (long long*)(a.part_sum + (size_t)batch * a.nblk * n_regions);
  a.h = height; a.w = width; a.H = gt_height; a.W = gt_width; a.R = n_regions;
  a.ry = (float)height / (float)gt_height;     // ATen's area_pixel_compute_scale: input / output in fp32
  a.rx = (float)width / (float)gt_width;
  a.scale_x = scale_x; a.scale_y = scale_y; a.abs_thr = abs_thr; a.rel_thr = rel_thr;
  cudaStream_t st = (cudaStream_t)stream;
  long long* c = (long long*)counts;
  if (n_regions == 1) flow_errors_launch<1>(a, batch, c, epe_sum, st);
  else if (n_regions == 2) flow_errors_launch<2>(a, batch, c, epe_sum, st);
  else if (n_regions <= 4) flow_errors_launch<4>(a, batch, c, epe_sum, st);
  else flow_errors_launch<8>(a, batch, c, epe_sum, st);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MDN_OK : fail(MDN_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}
