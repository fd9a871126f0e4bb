// mdn_common.cuh -- per-pixel math of the MDN_SfM loss path, written once and shared by every kernel.
//
// Each helper replays the fp32 operation ORDER of the upstream ATen composition it cites (separate
// roundings via __f*_rn where the reference rounds separately and a contraction would change a floor(),
// a validity bit or a cancellation), because parity (fwd 1e-5, grads 1e-4, masks bit exact) is only
// reachable that way (SURVEY.md section 7 "hard parts").
#pragma once

#ifdef MDN_EMU
#include "cuda_emu.h"
#include "cuda_emu_match.h"   // __match_any_sync, __popc, __ffs (tests/emu)
#else
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda/ptx>
#define MDN_DYN_SMEM(name) extern __shared__ __align__(128) float name[]
#define MDN_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
#endif

#include <stdint.h>

#define MDN_DEV __device__ __forceinline__

namespace mdn {

// ---------------------------------------------------------------------------------------------------
// Epipolar distance, loss_utils.py:64-67 with p1 = (x, y, 1), p2 = (u, v, 1) (loss_functions.py:120-122).
// Fully intrinsic so that the SN max pre-pass and the main pass produce bit-identical values.
struct Epi {
  float a, b, c;   // F p1
  float s, den;    // sqrt(a^2+b^2+1e-10), s + 1e-10
  float d;         // signed distance
};

MDN_DEV Epi epipolar_distance(const float* F, float x, float y, float u, float v) {
  Epi e;
  // bmm row . (x, y, 1): k-ordered FMA chain
  e.a = __fmaf_rn(F[2], 1.f, __fmaf_rn(F[1], y, __fmul_rn(F[0], x)));
  e.b = __fmaf_rn(F[5], 1.f, __fmaf_rn(F[4], y, __fmul_rn(F[3], x)));
  e.c = __fmaf_rn(F[8], 1.f, __fmaf_rn(F[7], y, __fmul_rn(F[6], x)));
  // (Fp1 * p2).sum(1): three separately rounded products, summed in order
  float num = __fadd_rn(__fadd_rn(__fmul_rn(e.a, u), __fmul_rn(e.b, v)), e.c);
  float ss = __fadd_rn(__fadd_rn(__fmul_rn(e.a, e.a), __fmul_rn(e.b, e.b)), 1e-10f);
  e.s = __fsqrt_rn(ss);
  e.den = __fadd_rn(e.s, 1e-10f);
  e.d = __fdiv_rn(num, e.den);
  return e;
}

// ---------------------------------------------------------------------------------------------------
// Flow -> sampling coordinates, loss_utils.py:27-34 followed by grid_sample's un-normalisation
// (align_corners=True): every op rounded on its own, exactly as the separate ATen kernels do.
struct WarpCoord {
  float gx, gy;    // normalised grid in [-1,1]
  float ix, iy;    // un-normalised source coordinates (after the padding mode's clip / reflection)
  float mx, my;    // d(ix) / d(un-padded ix), likewise y: 1 for zeros padding
  bool valid;      // max(|gx|,|gy|) <= 1
};

struct WarpGeom {
  float wm1, hm1;          // w-1, h-1
  float inv_wm1, inv_hm1;  // (float)(1.0 / (double)(w-1)): what ATen's CUDA `tensor /= scalar` multiplies by
  bool cuda_arith;         // MDN_OPT_CUDA_ARITH
  bool flowwarp_norm;      // utils.py:311 normalisation
  int pad;                 // grid_sample padding_mode: 0 zeros, 1 border, 2 reflection (standalone warp kernels)
};

// grid_sample's padding modes on the un-normalised coordinate (ATen GridSampler.h / GridSampler.cuh, align_corners=True:
// clip_coordinates_set_grad, reflect_coordinates_set_grad with twice_low = 0, twice_high = 2 (size - 1)).  size_m1 = size - 1
// >= 1.  mult = d(out) / d(in): 0 where the coordinate was clipped, -1 on a reflected branch.
constexpr int PAD_ZEROS = 0, PAD_BORDER = 1, PAD_REFLECTION = 2;
MDN_DEV float pad_clip(float in, float size_m1, float& mult) {
  if (in <= 0.f) { mult = 0.f; return 0.f; }
  if (in >= size_m1) { mult = 0.f; return size_m1; }
  mult = 1.f;
  return in;
}
MDN_DEV float pad_coordinate(float in, float size_m1, int pad, float& mult) {
  mult = 1.f;
  if (pad == PAD_ZEROS) return in;
  float m_refl = 1.f;
  if (pad == PAD_REFLECTION) {
    if (in < 0.f) { m_refl = -1.f; in = -in; }
    const float extra = fmodf(in, size_m1);
    const int flips = (int)floorf(__fdiv_rn(in, size_m1));
    if (flips % 2 == 0) in = extra;
    else { m_refl = -m_refl; in = __fsub_rn(size_m1, extra); }
  }
  float m_clip;
  in = pad_clip(in, size_m1, m_clip);
  mult = m_refl * m_clip;
  return in;
}

MDN_DEV WarpCoord warp_coord(float x, float y, float fx, float fy, const WarpGeom& G) {
  WarpCoord c;
  const float wm1 = G.wm1, hm1 = G.hm1;
  const bool flowwarp_norm = G.flowwarp_norm;
  float px = __fadd_rn(x, fx), py = __fadd_rn(y, fy);
  float gx, gy;
  if (G.cuda_arith) { gx = __fmul_rn(px, G.inv_wm1); gy = __fmul_rn(py, G.inv_hm1); }
  else { gx = __fdiv_rn(px, wm1); gy = __fdiv_rn(py, hm1); }
  if (flowwarp_norm) {  // utils.py:311  (g - 0.5) * 2
    gx = __fmul_rn(__fsub_rn(gx, 0.5f), 2.f);
    gy = __fmul_rn(__fsub_rn(gy, 0.5f), 2.f);
  } else {              // loss_utils.py:31  2 * g - 1
    gx = __fsub_rn(__fmul_rn(2.f, gx), 1.f);
    gy = __fsub_rn(__fmul_rn(2.f, gy), 1.f);
  }
  c.gx = gx; c.gy = gy;
  c.valid = (fabsf(gx) <= 1.f) && (fabsf(gy) <= 1.f);
  c.ix = pad_coordinate(__fmul_rn(__fmul_rn(__fadd_rn(gx, 1.f), 0.5f), wm1), wm1, G.pad, c.mx);
  c.iy = pad_coordinate(__fmul_rn(__fmul_rn(__fadd_rn(gy, 1.f), 0.5f), hm1), hm1, G.pad, c.my);
  return c;
}

// Bilinear footprint (grid_sample, bilinear, zeros padding): corner offsets + weights + in-bounds bits.
struct Bilin {
  int x0, y0;
  float ax0, ax1, ay0, ay1;   // (x0+1-ix), (ix-x0), (y0+1-iy), (iy-y0)
  bool xl, xr, yt, yb;        // corner column / row inside the image
};

MDN_DEV Bilin bilinear_setup(float ix, float iy, int h, int w) {
  Bilin b;
  float x0f = floorf(ix), y0f = floorf(iy);
  b.ax0 = (x0f + 1.f) - ix; b.ax1 = ix - x0f;
  b.ay0 = (y0f + 1.f) - iy; b.ay1 = iy - y0f;
  b.x0 = __float2int_rd(ix); b.y0 = __float2int_rd(iy);
  b.xl = (b.x0 >= 0) & (b.x0 < w);
  b.xr = (b.x0 >= -1) & (b.x0 < w - 1);
  b.yt = (b.y0 >= 0) & (b.y0 < h);
  b.yb = (b.y0 >= -1) & (b.y0 < h - 1);
  return b;
}

// One channel: value and d(value)/d(ix), d(value)/d(iy) (GridSampler.cu backward formulas).
MDN_DEV void bilinear_fetch(const float* __restrict__ plane, int w, const Bilin& b, float& nw, float& ne, float& sw,
                            float& se) {
  const float* r0 = plane + (long long)b.y0 * w + b.x0;
  nw = (b.yt && b.xl) ? __ldg(r0) : 0.f;
  ne = (b.yt && b.xr) ? __ldg(r0 + 1) : 0.f;
  sw = (b.yb && b.xl) ? __ldg(r0 + w) : 0.f;
  se = (b.yb && b.xr) ? __ldg(r0 + w + 1) : 0.f;
}

MDN_DEV float bilinear_value(const Bilin& b, float nw, float ne, float sw, float se) {
  float o = nw * (b.ax0 * b.ay0);
  o += ne * (b.ax1 * b.ay0);
  o += sw * (b.ax0 * b.ay1);
  o += se * (b.ax1 * b.ay1);
  return o;
}

MDN_DEV void bilinear_deriv(const Bilin& b, float nw, float ne, float sw, float se, float& ddx, float& ddy) {
  ddx = b.ay0 * (ne - nw) + b.ay1 * (se - sw);
  ddy = b.ax0 * (sw - nw) + b.ax1 * (se - ne);
}

// ---------------------------------------------------------------------------------------------------
// Packed fp32x2 arithmetic (Blackwell FADD2 / FMUL2 / FFMA2: two IEEE-rn results per issue slot).  The FP32 pipe
// does the same lane-operations per clock either way; what the packed forms save is ISSUE slots, which is what
// bounds the fused kernel (DESIGN.md section 4).  Every op is rn per half, never contracted, so results are
// identical to the scalar __f*_rn forms.
#ifdef MDN_EMU
MDN_DEV float2 add2(float2 a, float2 b) { return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)); }
MDN_DEV float2 mul2(float2 a, float2 b) { return make_float2(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)); }
MDN_DEV float2 fma2(float2 a, float2 b, float2 c) { return make_float2(__fmaf_rn(a.x, b.x, c.x), __fmaf_rn(a.y, b.y, c.y)); }
MDN_DEV float rcp_fast(float x) { return 1.0f / x; }
MDN_DEV float ex2_fast(float x) { return exp2f(x); }
MDN_DEV float lg2_fast(float x) { return log2f(x); }
MDN_DEV float sqrt_fast(float x) { return sqrtf(x); }
#else
MDN_DEV float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
MDN_DEV float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
MDN_DEV float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
MDN_DEV float rcp_fast(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
MDN_DEV float ex2_fast(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
MDN_DEV float lg2_fast(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
MDN_DEV float sqrt_fast(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
#endif
MDN_DEV float2 splat2(float a) { return make_float2(a, a); }
// Makes a pointer opaque to the optimiser, so that it is kept as ONE 64-bit register pair and `p + u32_offset` is a
// single IMAD.WIDE.U32.  Without it nvcc keeps "constant-bank base + 64-bit element index" and re-derives every
// address with a 4-instruction IADD3 / IADD3.X / LEA / LEA.HI.X sequence.
template <class T>
MDN_DEV T* opaque_ptr(T* p) {
#ifndef MDN_EMU
  asm volatile("" : "+l"(p));
#endif
  return p;
}
MDN_DEV float2 ld2s(const float* p) { return *reinterpret_cast<const float2*>(p); }     // 8-byte aligned
MDN_DEV void st2s(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }

// ---------------------------------------------------------------------------------------------------
// Two horizontally adjacent output pixels of the flow warp at once, from a source image REPACKED to one float4
// (r, g, b, -) per pixel (ref_pack_kernel).  The coordinate chain is warp_coord()'s with the same roundings (2 g - 1
// and (g + 1) / 2 * (n - 1) need one rounding each because the doubling / halving is exact).  Zero padding is folded
// into the bilinear FRACTIONS: a masked fraction zeroes both the value weight and the derivative coefficient of its
// corners.  Corner addresses are clamped into the image, so every load is legal and the loads of a pixel pair are in
// flight together.  The four corners of a pixel are four 16-byte loads that bring all three channels at once -- a
// third of the load instructions and of the L1 wavefronts / L2 sector requests of a planar gather, which is what
// bounds the gather when neighbouring pixels sample unrelated places.  Coordinates, fractions and masks are packed
// over the two PIXELS; the interpolation is packed over the (r, g) CHANNELS of one pixel with the weight as the
// broadcast scalar operand, b is scalar.  Output: per pixel e (0 / 1) value and derivatives of the three channels.
struct GatherPx {
  float v[3], dx[3], dy[3];
};

MDN_DEV float4 ldg4(const float4* p) { return __ldg(p); }

template <bool DERIV, int PAD = PAD_ZEROS>
MDN_DEV void gather_pair_packed(const float4* __restrict__ pk, int h, int w, float2 xs, float2 ys, float2 fx, float2 fy,
                                const WarpGeom& G, GatherPx* out, bool& valid_a, bool& valid_b) {
  const float2 one = splat2(1.f), neg1 = splat2(-1.f), two = splat2(2.f);
  // NOTE: fx / fy must come from SCALAR multiplies: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (it
  // honours .rn only for scalar ops), which would move x + sx * f by an ulp and flip bilinear cells
  const float2 px = add2(xs, fx), py = add2(ys, fy);
  float2 gx, gy;
  if (G.cuda_arith) { gx = mul2(px, splat2(G.inv_wm1)); gy = mul2(py, splat2(G.inv_hm1)); }
  else {
    gx = make_float2(__fdiv_rn(px.x, G.wm1), __fdiv_rn(px.y, G.wm1));
    gy = make_float2(__fdiv_rn(py.x, G.hm1), __fdiv_rn(py.y, G.hm1));
  }
  gx = fma2(two, gx, neg1);                     // loss_utils.py:31
  gy = fma2(two, gy, neg1);
  valid_a = (fabsf(gx.x) <= 1.f) & (fabsf(gy.x) <= 1.f);
  valid_b = (fabsf(gx.y) <= 1.f) & (fabsf(gy.y) <= 1.f);
  float2 ix = mul2(add2(gx, one), splat2(0.5f * G.wm1));   // grid_sample un-normalisation, align_corners=True
  float2 iy = mul2(add2(gy, one), splat2(0.5f * G.hm1));
  float2 gmx = one, gmy = one;     // border / reflection padding: the coordinate is clipped / folded back, its gradient scaled
  if (PAD != PAD_ZEROS) {
    ix.x = pad_coordinate(ix.x, G.wm1, PAD, gmx.x); ix.y = pad_coordinate(ix.y, G.wm1, PAD, gmx.y);
    iy.x = pad_coordinate(iy.x, G.hm1, PAD, gmy.x); iy.y = pad_coordinate(iy.y, G.hm1, PAD, gmy.y);
  }
  const float2 x0f = make_float2(floorf(ix.x), floorf(ix.y)), y0f = make_float2(floorf(iy.x), floorf(iy.y));
  float2 ax1 = fma2(x0f, neg1, ix), ax0 = fma2(ix, neg1, add2(x0f, one));
  float2 ay1 = fma2(y0f, neg1, iy), ay0 = fma2(iy, neg1, add2(y0f, one));
  unsigned o00[2], o01[2], o10[2], o11[2];
  float mx0[2], mx1[2], my0[2], my1[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int x0 = min(max(__float2int_rd(e ? ix.y : ix.x), -2), w), y0 = min(max(__float2int_rd(e ? iy.y : iy.x), -2), h);
    const int x1 = x0 + 1, y1 = y0 + 1;
    const bool bx0 = (unsigned)x0 < (unsigned)w, bx1 = (unsigned)x1 < (unsigned)w;
    const bool by0 = (unsigned)y0 < (unsigned)h, by1 = (unsigned)y1 < (unsigned)h;
    const unsigned cx0 = bx0 ? x0 : 0, cx1 = bx1 ? x1 : 0;
    const unsigned r0 = (by0 ? y0 : 0) * w, r1 = (by1 ? y1 : 0) * w;
    o00[e] = r0 + cx0; o01[e] = r0 + cx1; o10[e] = r1 + cx0; o11[e] = r1 + cx1;
    mx0[e] = bx0 ? 1.f : 0.f; mx1[e] = bx1 ? 1.f : 0.f; my0[e] = by0 ? 1.f : 0.f; my1[e] = by1 ? 1.f : 0.f;
  }
  const float2 fx0 = make_float2(mx0[0], mx0[1]), fx1 = make_float2(mx1[0], mx1[1]);
  const float2 fy0 = make_float2(my0[0], my0[1]), fy1 = make_float2(my1[0], my1[1]);
  ax0 = mul2(ax0, fx0); ax1 = mul2(ax1, fx1); ay0 = mul2(ay0, fy0); ay1 = mul2(ay1, fy1);
  const float2 w00 = mul2(ax0, ay0), w01 = mul2(ax1, ay0), w10 = mul2(ax0, ay1), w11 = mul2(ax1, ay1);
  float2 cx00, cx01, cx10, cx11, cy00, cy01, cy10, cy11;
  if (DERIV) {
    const float2 nfx0 = mul2(fx0, neg1), nfy0 = mul2(fy0, neg1);
    cx00 = mul2(ay0, nfx0); cx01 = mul2(ay0, fx1); cx10 = mul2(ay1, nfx0); cx11 = mul2(ay1, fx1);
    cy00 = mul2(ax0, nfy0); cy01 = mul2(ax1, nfy0); cy10 = mul2(ax0, fy1); cy11 = mul2(ax1, fy1);
  }
  float4 v00[2], v01[2], v10[2], v11[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    v00[e] = ldg4(pk + o00[e]); v01[e] = ldg4(pk + o01[e]); v10[e] = ldg4(pk + o10[e]); v11[e] = ldg4(pk + o11[e]);
  }
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const float a00 = e ? w00.y : w00.x, a01 = e ? w01.y : w01.x, a10 = e ? w10.y : w10.x, a11 = e ? w11.y : w11.x;
    const float2 rg = fma2(make_float2(v11[e].x, v11[e].y), splat2(a11), fma2(make_float2(v10[e].x, v10[e].y), splat2(a10),
                      fma2(make_float2(v01[e].x, v01[e].y), splat2(a01), mul2(make_float2(v00[e].x, v00[e].y), splat2(a00)))));
    out[e].v[0] = rg.x; out[e].v[1] = rg.y;
    out[e].v[2] = fmaf(v11[e].z, a11, fmaf(v10[e].z, a10, fmaf(v01[e].z, a01, v00[e].z * a00)));
    if (DERIV) {
      const float b00 = e ? cx00.y : cx00.x, b01 = e ? cx01.y : cx01.x, b10 = e ? cx10.y : cx10.x, b11 = e ? cx11.y : cx11.x;
      const float2 dxrg = fma2(make_float2(v11[e].x, v11[e].y), splat2(b11), fma2(make_float2(v10[e].x, v10[e].y), splat2(b10),
                          fma2(make_float2(v01[e].x, v01[e].y), splat2(b01), mul2(make_float2(v00[e].x, v00[e].y), splat2(b00)))));
      out[e].dx[0] = dxrg.x; out[e].dx[1] = dxrg.y;
      out[e].dx[2] = fmaf(v11[e].z, b11, fmaf(v10[e].z, b10, fmaf(v01[e].z, b01, v00[e].z * b00)));
      const float c00 = e ? cy00.y : cy00.x, c01 = e ? cy01.y : cy01.x, c10 = e ? cy10.y : cy10.x, c11 = e ? cy11.y : cy11.x;
      const float2 dyrg = fma2(make_float2(v11[e].x, v11[e].y), splat2(c11), fma2(make_float2(v10[e].x, v10[e].y), splat2(c10),
                          fma2(make_float2(v01[e].x, v01[e].y), splat2(c01), mul2(make_float2(v00[e].x, v00[e].y), splat2(c00)))));
      out[e].dy[0] = dyrg.x; out[e].dy[1] = dyrg.y;
      out[e].dy[2] = fmaf(v11[e].z, c11, fmaf(v10[e].z, c10, fmaf(v01[e].z, c01, v00[e].z * c00)));
      if (PAD != PAD_ZEROS) {
        const float mxe = e ? gmx.y : gmx.x, mye = e ? gmy.y : gmy.x;
#pragma unroll
        for (int c = 0; c < 3; ++c) { out[e].dx[c] *= mxe; out[e].dy[c] *= mye; }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// SSIM, networks/layers.py:164-178, from the five 3x3 window SUMS (reflect padding applied by the caller).
struct SsimOut {
  float J;            // clamp((1 - n/d)/2, 0, 1)
  float dmu_y, dY2, dXY;   // dz/d(mu_y) (total, incl. through sigma_y, sigma_xy), dz/dE[y^2], dz/dE[xy]; 0 outside the clamp gate
  float dmu_x, dX2;        // same for x (used by the standalone SSIM backward)
};

MDN_DEV SsimOut ssim_window(float sx, float sy, float sxx, float syy, float sxy, bool want_grad) {
  const float C1 = 0.0001f, C2 = 0.0009f;
  // avg_pool2d divides the window sum by 9.  The sums already differ from the reference's in the last ulp (separable
  // order), so a correctly rounded quotient buys nothing: multiply by rn(1/9).  sigma = E[x^2] - mu^2 keeps the
  // reference's separate roundings (no FMA contraction of the cancelling difference).
  const float r9 = 0.111111111f;
  float mu_x = __fmul_rn(sx, r9), mu_y = __fmul_rn(sy, r9);
  float mxx = __fmul_rn(mu_x, mu_x), myy = __fmul_rn(mu_y, mu_y), mxy = __fmul_rn(mu_x, mu_y);
  float sig_x = __fsub_rn(__fmul_rn(sxx, r9), mxx);
  float sig_y = __fsub_rn(__fmul_rn(syy, r9), myy);
  float sig_xy = __fsub_rn(__fmul_rn(sxy, r9), mxy);
  float n1 = __fmaf_rn(2.f, mxy, C1);          // == (2 mu_x) mu_y + C1: doubling is exact
  float n2 = __fmaf_rn(2.f, sig_xy, C2);
  float d1 = __fadd_rn(__fadd_rn(mxx, myy), C1);
  float d2 = __fadd_rn(__fadd_rn(sig_x, sig_y), C2);
  float n = __fmul_rn(n1, n2), D = __fmul_rn(d1, d2);
  float invD = __fdividef(1.f, D);        // D >= C1*C2 > 0; 2-ulp reciprocal is far inside the 1e-5 budget
  float z = __fmul_rn(__fsub_rn(1.f, n * invD), 0.5f);
  SsimOut o;
  o.J = fminf(fmaxf(z, 0.f), 1.f);
  o.dmu_y = o.dY2 = o.dXY = o.dmu_x = o.dX2 = 0.f;
  if (want_grad) {
    const float gate = (z >= 0.f && z <= 1.f) ? 0.5f : 0.f;   // clamp backward gate is inclusive; 0.5 = d z / d(1 - n/D)
    float nbar = -gate * invD;            // dz/dn
    float Dbar = gate * n * invD * invD;  // dz/dD
    float dn1 = nbar * n2, dn2 = nbar * n1, dd1 = Dbar * d2, dd2 = Dbar * d1;
    float t1 = 2.f * (dn1 - dn2), t2 = 2.f * (dd1 - dd2);
    o.dmu_y = mu_x * t1 + mu_y * t2;
    o.dmu_x = mu_y * t1 + mu_x * t2;
    o.dY2 = dd2;
    o.dX2 = dd2;
    o.dXY = 2.f * dn2;
  }
  return o;
}

// Two windows at once (packed fp32x2), used by the fused kernel.  kk = c_ssim / 9 per window, or 0 for a window
// outside the image.  Returns J = clamp((1 - n/D) / 2, 0, 1) and the adjoint coefficients of
//   d(sum_w k_w J_w) / d(warped tap y) = A + B * y + C * x        (x = target tap)
// i.e. A = kk dJ/dmu_y, B = 2 kk dJ/dE[y^2], C = kk dJ/dE[xy].  sigma = E[.^2] - mu^2 keeps the reference's two
// roundings (fma(-1, m, t) rounds t - m once, t already rounded).
struct Ssim2 { float2 J, A, B, C; };

MDN_DEV Ssim2 ssim_window2(float2 sx, float2 sy, float2 sxx, float2 syy, float2 sxy, float2 kk) {
  const float2 r9 = splat2(0.111111111f), neg1 = splat2(-1.f), two = splat2(2.f);
  const float2 C1 = splat2(0.0001f), C2 = splat2(0.0009f);
  const float2 mx = mul2(sx, r9), my = mul2(sy, r9);
  const float2 mxx = mul2(mx, mx), myy = mul2(my, my), mxy = mul2(mx, my);
  const float2 vx = fma2(mxx, neg1, mul2(sxx, r9));
  const float2 vy = fma2(myy, neg1, mul2(syy, r9));
  const float2 cxy = fma2(mxy, neg1, mul2(sxy, r9));
  const float2 n1 = fma2(two, mxy, C1), n2 = fma2(two, cxy, C2);
  const float2 d1 = add2(add2(mxx, myy), C1), d2 = add2(add2(vx, vy), C2);
  const float2 n = mul2(n1, n2), D = mul2(d1, d2);           // D >= C1 * C2 > 0
  const float2 r = make_float2(rcp_fast(D.x), rcp_fast(D.y));
  const float2 S = mul2(n, r);
  Ssim2 o;
  o.J.x = __saturatef(fmaf(S.x, -0.5f, 0.5f));               // (1 - S) / 2: the halving is exact
  o.J.y = __saturatef(fmaf(S.y, -0.5f, 0.5f));
  // clamp gate (inclusive, like clamp's backward): 0 <= (1 - S)/2 <= 1  <=>  |S| <= 1
  const float2 kg = make_float2(fabsf(S.x) <= 1.f ? kk.x : 0.f, fabsf(S.y) <= 1.f ? kk.y : 0.f);
  const float2 a = mul2(kg, r);                              // -2 kk dJ/dn
  const float2 e = mul2(a, S);                               //  2 kk dJ/dD * (-1) ... e d2 = 2 kk dJ/dd1, e d1 = 2 kk dJ/dd2
  const float2 t1 = mul2(a, fma2(n2, neg1, n1));             // 2 kk (dJ/dn1 - dJ/dn2) = a (n1 - n2)
  const float2 t2 = mul2(e, fma2(d1, neg1, d2));             // 2 kk (dJ/dd1 - dJ/dd2)
  o.A = fma2(my, t2, mul2(mx, t1));
  o.B = mul2(e, d1);
  o.C = mul2(a, mul2(n1, neg1));
  return o;
}

MDN_DEV int reflect1(int t, int n) {   // ReflectionPad2d(1): -1 -> 1, n -> n-2
  t = t < 0 ? -t : t;
  return t >= n ? 2 * n - 2 - t : t;
}

// multiplicity with which window centre p (in image) touches pixel q along one axis of length n
MDN_DEV int refl_mult(int p, int q, int n) {
  int c = 0;
#pragma unroll
  for (int d = -1; d <= 1; ++d) c += (reflect1(p + d, n) == q);
  return c;
}

// 4-byte asynchronous global -> shared copy (LDGSTS); zero-fills when `pred` is false.  Completion: cp_async_wait_all().
MDN_DEV void cp_async_f32(float* smem_dst, const float* gsrc, bool pred) {
#ifdef MDN_EMU
  *smem_dst = pred ? *gsrc : 0.f;
#else
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = pred ? 4 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
#endif
}
// 16-byte variant (both addresses 16-byte aligned); zero-fills when `pred` is false
MDN_DEV void cp_async_f32x4(float* smem_dst, const float* gsrc, bool pred) {
#ifdef MDN_EMU
  for (int i = 0; i < 4; ++i) smem_dst[i] = pred ? gsrc[i] : 0.f;
#else
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = pred ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
#endif
}
// 8-byte variant (both addresses 8-byte aligned): even image widths that are not a multiple of four (1242)
MDN_DEV void cp_async_f32x2(float* smem_dst, const float* gsrc, bool pred) {
#ifdef MDN_EMU
  for (int i = 0; i < 2; ++i) smem_dst[i] = pred ? gsrc[i] : 0.f;
#else
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = pred ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
#endif
}
// Pulls a 128-byte line into L2 (no register, no stall): used to fetch the NEXT wave's inputs from HBM ahead of time
MDN_DEV void prefetch_l2(const void* p) {
#ifndef MDN_EMU
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#endif
}
MDN_DEV void cp_async_wait_all() {
#ifndef MDN_EMU
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
#endif
}

MDN_DEV float signf_(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }
// signf_(x) * v, bit for bit (v finite), in three instructions instead of five: the sign bit of x flips v; zero / NaN x give 0
MDN_DEV float signmul(float x, float v) {
  const float r = __uint_as_float(__float_as_uint(v) ^ (__float_as_uint(x) & 0x80000000u));
  return (x < 0.f || x > 0.f) ? r : 0.f;
}

// ---------------------------------------------------------------------------------------------------
// Transposing butterfly: reduces NV per-lane values over the 32 lanes of a warp with NV-ish shuffles
// instead of 5*NV.  On return lane l holds, in v[0], the warp total of value (l % NV).
template <int NV>
MDN_DEV void warp_reduce_transpose(float* v) {
  const int lane = threadIdx.x & 31;
  // the halving (transposing) steps first: they leave ONE value per lane, so the full-width steps that fold the 32 / NV
  // groups of lanes cost one shuffle each instead of NV
#pragma unroll
  for (int half = NV / 2; half >= 1; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      float send = up ? v[i] : v[i + half];
      float keep = up ? v[i + half] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
#pragma unroll
  for (int m = NV; m <= 16; m <<= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], m);
}

}  // namespace mdn
