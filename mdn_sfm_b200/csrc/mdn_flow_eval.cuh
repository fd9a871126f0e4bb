// mdn_flow_eval.cuh -- evaluation of optical flow: end-point error and KITTI Fl outliers per image and region, from the
// network's flow at its own resolution against ground truth at another, in one read of the ground truth.  Included by
// mdn_loss.cu INSIDE namespace mdn.  Entry points: mdn_flow_errors / _workspace_bytes (include/mdn_loss.h, where the
// per-pixel arithmetic is stated; flow_tap / flow_bilinear / flow_pixel below are that statement in code).
//
// flow_errors_kernel<RT>: grid (blocks per sample, B).  A thread takes 4 consecutive ground-truth pixels of one sample
// per step -- 4-byte loads of gt_valid and region, 16- / 8-byte / scalar loads of the two gt_flow planes, whichever the
// plane's offset allows -- up-samples the prediction there by bilinear gathers (served from L1 / L2: the prediction is
// small), and adds e, 1 and the outlier bit to per-region accumulators in registers.  Each block writes its per-region
// partials to the workspace; flow_errors_finish_kernel<RT> (one block per sample) adds them.  Both reductions are fixed
// trees and the grid depends on the shapes only, so the fp64 sums are bit-identical run to run and on any device.

constexpr int FE_THREADS = 256;
constexpr int FE_MAX_REGIONS = 8;
constexpr int FE_QUADS_PER_THREAD = 4;    // a block covers about FE_THREADS * 4 * 4 = 4096 pixels of a sample
constexpr int FE_MAX_BLOCKS = 1024;       // per sample; a larger image is strided over

// One source row (or column) of ATen's upsample_bilinear2d, align_corners=False, no scale_factor: r = in / out in fp32,
// s = max(r * (i + 0.5) - 0.5, 0), i0 = (int)s, i1 = i0 + (i0 < n - 1), l1 = s - i0, l0 = 1 - l1.  i0 is also clamped to
// n - 1, which only matters where fp32 rounding of a size near 2^24 would take ATen past the last row.
struct FlowTap { int i0, i1; float l0, l1; };

MDN_DEV FlowTap flow_tap(int i, float r, int n) {
  float s = __fsub_rn(__fmul_rn(r, __fadd_rn((float)i, 0.5f)), 0.5f);
  s = s < 0.f ? 0.f : s;
  FlowTap t;
  t.i0 = min((int)s, n - 1);
  t.i1 = t.i0 + (t.i0 < n - 1 ? 1 : 0);
  t.l1 = __fsub_rn(s, (float)t.i0);
  t.l0 = __fsub_rn(1.f, t.l1);
  return t;
}

// l0y * (l0x * F[y0][x0] + l1x * F[y0][x1]) + l1y * (l0x * F[y1][x0] + l1x * F[y1][x1]), every operation rounded on its
// own; ty.i0 / ty.i1 are already row offsets (row * w).
MDN_DEV float flow_bilinear(const float* __restrict__ F, const FlowTap& ty, const FlowTap& tx) {
  const float a = __fadd_rn(__fmul_rn(tx.l0, __ldg(F + ty.i0 + tx.i0)), __fmul_rn(tx.l1, __ldg(F + ty.i0 + tx.i1)));
  const float b = __fadd_rn(__fmul_rn(tx.l0, __ldg(F + ty.i1 + tx.i0)), __fmul_rn(tx.l1, __ldg(F + ty.i1 + tx.i1)));
  return __fadd_rn(__fmul_rn(ty.l0, a), __fmul_rn(ty.l1, b));
}

struct FlowArgs {
  const float* flow;       // (B, 2, h, w)
  const float* gt;         // (B, 2, H, W)
  const uint8_t* valid;    // (B, H, W)
  const uint8_t* region;   // (B, H, W) or NULL (every pixel in region 0)
  double* part_sum;        // (B, nblk, R) per-block sums of e
  long long* part_cnt;     // (B, nblk, R, 2) per-block [valid, outliers]
  int h, w, H, W, R, nblk;
  float rx, ry, scale_x, scale_y, abs_thr, rel_thr;
};

template <int RT>
struct FlowAcc {
  double s[RT];
  unsigned n[RT], o[RT];
};

// One ground-truth pixel at column x of the row `ty` (row offsets into the prediction).  The pixel counts iff valid != 0
// and lab < R; an uncounted pixel's e is selected away, so whatever its ground truth holds (NaN, inf) reaches no sum.
template <int RT>
MDN_DEV void flow_pixel(FlowAcc<RT>& acc, const FlowArgs& a, const float* __restrict__ F0, const float* __restrict__ F1,
                        const FlowTap& ty, int x, float gu, float gv, unsigned valid, unsigned lab) {
  const FlowTap tx = flow_tap(x, a.rx, a.w);
  const float u = __fmul_rn(flow_bilinear(F0, ty, tx), a.scale_x);
  const float v = __fmul_rn(flow_bilinear(F1, ty, tx), a.scale_y);
  const float du = __fsub_rn(u, gu), dv = __fsub_rn(v, gv);
  const float e = __fsqrt_rn(__fadd_rn(__fmul_rn(du, du), __fmul_rn(dv, dv)));
  const float m = __fsqrt_rn(__fadd_rn(__fmul_rn(gu, gu), __fmul_rn(gv, gv)));
  const bool out = e > a.abs_thr && __fdiv_rn(e, m) > a.rel_thr;    // NaN e: false
  const bool counted = valid != 0u && lab < (unsigned)a.R;
  const double ed = (double)e;
#pragma unroll
  for (int r = 0; r < RT; ++r) {
    const bool hit = counted && lab == (unsigned)r;
    acc.s[r] += hit ? ed : 0.0;
    acc.n[r] += hit ? 1u : 0u;
    acc.o[r] += (hit && out) ? 1u : 0u;
  }
}

// The row taps of ground-truth row y as offsets into a prediction plane.
MDN_DEV FlowTap flow_row(int y, const FlowArgs& a) {
  FlowTap t = flow_tap(y, a.ry, a.h);
  t.i0 *= a.w;
  t.i1 *= a.w;
  return t;
}

// 4 consecutive floats at p + 4 i, where p + 4 i is `mis` elements past a 16-byte boundary (a per-sample constant).
MDN_DEV void flow_load4(const float* __restrict__ p, long long i, int mis, float (&out)[4]) {
  const float* q = p + 4 * i;
  if (mis == 0) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(q));
    out[0] = t.x; out[1] = t.y; out[2] = t.z; out[3] = t.w;
  } else if (mis == 2) {
    const float2 t0 = __ldg(reinterpret_cast<const float2*>(q)), t1 = __ldg(reinterpret_cast<const float2*>(q + 2));
    out[0] = t0.x; out[1] = t0.y; out[2] = t1.x; out[3] = t1.y;
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) out[k] = __ldg(q + k);
  }
}

// v[r] summed over the block by a fixed tree; the result is in every thread's v.  s: RT * FE_THREADS elements of T.
template <int RT, class T>
MDN_DEV void flow_block_sum(T (&v)[RT], T* s) {
  const int t = threadIdx.x;
#pragma unroll
  for (int r = 0; r < RT; ++r) s[r * FE_THREADS + t] = v[r];
  __syncthreads();
  for (int d = FE_THREADS / 2; d > 0; d >>= 1) {
    if (t < d) {
#pragma unroll
      for (int r = 0; r < RT; ++r) s[r * FE_THREADS + t] += s[r * FE_THREADS + t + d];
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < RT; ++r) v[r] = s[r * FE_THREADS];
  __syncthreads();    // s is reused by the next call
}

// grid (a.nblk, B).  RT = R rounded up to 1, 2, 4 or 8.
template <int RT>
__global__ void __launch_bounds__(FE_THREADS) flow_errors_kernel(const FlowArgs a) {
  __shared__ double s_red[RT * FE_THREADS];
  const int b = blockIdx.y;
  const long long HW = (long long)a.H * a.W, hw = (long long)a.h * a.w;
  const float* F0 = a.flow + (long long)b * 2 * hw;
  const float* F1 = F0 + hw;
  // valid and region have 16-byte aligned bases and the sample's element offset sb, so the scalar head makes both 4-byte
  // aligned; the gt_flow planes start at 2 sb and 2 sb + HW, so after the head they sit `mu` / `mv` floats past a 16-byte
  // boundary (for 375 x 1242 one is 0 and the other 2).
  const long long sb = (long long)b * HW;
  const long long head = min((long long)((-sb) & 3), HW);
  const long long n4 = (HW - head) >> 2;
  const float* gu = a.gt + 2 * sb + head;
  const float* gv = gu + HW;
  const int mu = (int)((2 * sb + head) & 3), mv = (int)((2 * sb + HW + head) & 3);
  const unsigned* v4 = reinterpret_cast<const unsigned*>(a.valid + sb + head);
  const unsigned* r4 = a.region ? reinterpret_cast<const unsigned*>(a.region + sb + head) : nullptr;

  FlowAcc<RT> acc;
#pragma unroll
  for (int r = 0; r < RT; ++r) { acc.s[r] = 0.0; acc.n[r] = 0u; acc.o[r] = 0u; }

  // the scalar head (< 4 pixels) and tail (< 4 pixels) of the sample, before the body: nothing of them stays live across
  // the loop
  if (blockIdx.x == 0 && threadIdx.x < 8) {
    const long long tail0 = head + 4 * n4, t = threadIdx.x;
    const long long e = t < 4 ? (t < head ? t : -1) : (tail0 + (t - 4) < HW ? tail0 + (t - 4) : -1);
    if (e >= 0) {
      const int y = (int)(e / a.W), x = (int)(e - (long long)y * a.W);
      const float* g = a.gt + 2 * sb + e;
      flow_pixel<RT>(acc, a, F0, F1, flow_row(y, a), x, g[0], g[HW], a.valid[sb + e], a.region ? a.region[sb + e] : 0u);
    }
  }
  for (long long i = (long long)blockIdx.x * FE_THREADS + threadIdx.x; i < n4; i += (long long)gridDim.x * FE_THREADS) {
    const unsigned vq = __ldg(v4 + i);
    const unsigned lq = r4 ? __ldg(r4 + i) : 0u;
    float U[4], V[4];
    flow_load4(gu, i, mu, U);
    flow_load4(gv, i, mv, V);
    if (vq == 0u) continue;          // four invalid pixels add nothing
    // the row taps once per quad, and again where the quad runs into the next row
    int p = (int)(head + 4 * i), y = p / a.W, x = p - y * a.W;
    FlowTap ty = flow_row(y, a);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (q > 0 && ++x == a.W) {
        x = 0;
        ty = flow_row(++y, a);
      }
      flow_pixel<RT>(acc, a, F0, F1, ty, x, U[q], V[q], (vq >> (8 * q)) & 0xffu, (lq >> (8 * q)) & 0xffu);
    }
  }

  flow_block_sum<RT, double>(acc.s, s_red);
  flow_block_sum<RT, unsigned>(acc.n, reinterpret_cast<unsigned*>(s_red));
  flow_block_sum<RT, unsigned>(acc.o, reinterpret_cast<unsigned*>(s_red));
  if (threadIdx.x == 0) {
    const long long k = ((long long)b * a.nblk + blockIdx.x) * a.R;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      if (r < a.R) {
        a.part_sum[k + r] = acc.s[r];
        a.part_cnt[2 * (k + r) + 0] = acc.n[r];
        a.part_cnt[2 * (k + r) + 1] = acc.o[r];
      }
    }
  }
}

// One block per sample: thread t adds the partials of blocks t, t + FE_THREADS, ... in that order, then a fixed tree.
template <int RT>
__global__ void __launch_bounds__(FE_THREADS) flow_errors_finish_kernel(const double* __restrict__ part_sum,
                                                                        const long long* __restrict__ part_cnt, int nblk,
                                                                        int R, long long* __restrict__ counts,
                                                                        double* __restrict__ epe_sum) {
  __shared__ double s_red[RT * FE_THREADS];
  const int b = blockIdx.x;
  double s[RT];
  long long n[RT], o[RT];
#pragma unroll
  for (int r = 0; r < RT; ++r) { s[r] = 0.0; n[r] = 0; o[r] = 0; }
  for (int j = threadIdx.x; j < nblk; j += FE_THREADS) {
    const long long k = ((long long)b * nblk + j) * R;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      if (r < R) {
        s[r] += part_sum[k + r];
        n[r] += part_cnt[2 * (k + r) + 0];
        o[r] += part_cnt[2 * (k + r) + 1];
      }
    }
  }
  flow_block_sum<RT, double>(s, s_red);
  flow_block_sum<RT, long long>(n, reinterpret_cast<long long*>(s_red));
  flow_block_sum<RT, long long>(o, reinterpret_cast<long long*>(s_red));
  if (threadIdx.x == 0) {
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      if (r < R) {
        epe_sum[(long long)b * R + r] = s[r];
        counts[2 * ((long long)b * R + r) + 0] = n[r];
        counts[2 * ((long long)b * R + r) + 1] = o[r];
      }
    }
  }
}
