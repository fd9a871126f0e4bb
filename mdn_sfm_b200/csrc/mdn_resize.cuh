// mdn_resize.cuh -- instance-mask union and the antialiased-bilinear resize (torchvision Resize / ATen
// _upsample_bilinear2d_aa replayed) for {0,1} masks and fp32 image pyramids.  Included by mdn_loss.cu INSIDE namespace mdn.
// Entry points: mdn_instance_mask_union / _union_table / _resize, mdn_image_pyramid / _packed (include/mdn_loss.h).

// get_batch_instance_mask (loss_utils.py:102-124): union of the N boolean instance masks of a sample.
constexpr int UNION_CHUNK = 32;   // samples per launch (pointer table passed by value)
struct UnionArgs {
  const uint8_t* masks[UNION_CHUNK];
  int count[UNION_CHUNK];
};

// One sample's union, spread over the blocks of grid.x: `n` planes of `hw` bytes at `src` -> `hw` bytes {0,1} at `dst`
// (n <= 0: all zero).  Four, two or one pixel per thread, as `hw` and the alignment of `src` / `dst` allow.
MDN_DEV void instance_union_sample(const uint8_t* src, int n, uint8_t* dst, long long hw) {
  const bool wide = (hw & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 3) == 0;
  if (wide) {   // four pixels per thread
    const long long n4 = hw >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
      unsigned v = 0;
      for (int k = 0; k < n; ++k) v |= __ldg(reinterpret_cast<const unsigned*>(src + (long long)k * hw) + i);
      const unsigned nz = ((v & 0x7f7f7f7fu) + 0x7f7f7f7fu | v) & 0x80808080u;    // 0x80 in every non-zero byte
      reinterpret_cast<unsigned*>(dst)[i] = nz >> 7;
    }
    return;
  }
  const bool pair = (hw & 1) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 1) == 0;
  if (pair) {   // two pixels per thread (375 x 1242 is even, not a multiple of 4)
    const long long n2 = hw >> 1;
    const long long step = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // four independent pixel pairs in flight per thread (the pass waits on load latency, not on arithmetic)
    for (; i + 3 * step < n2; i += 4 * step) {
      unsigned v[4] = {0, 0, 0, 0};
      for (int k = 0; k < n; ++k) {
        const unsigned short* p = reinterpret_cast<const unsigned short*>(src + (long long)k * hw);
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] |= __ldg(p + i + q * step);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        reinterpret_cast<unsigned short*>(dst)[i + q * step] = (unsigned short)(((v[q] & 0xffu) ? 1u : 0u) | ((v[q] & 0xff00u) ? 0x100u : 0u));
    }
    for (; i < n2; i += step) {
      unsigned v = 0;
      for (int k = 0; k < n; ++k) v |= __ldg(reinterpret_cast<const unsigned short*>(src + (long long)k * hw) + i);
      reinterpret_cast<unsigned short*>(dst)[i] = (unsigned short)(((v & 0xffu) ? 1u : 0u) | ((v & 0xff00u) ? 0x100u : 0u));
    }
    return;
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += (long long)gridDim.x * blockDim.x) {
    unsigned v = 0;
    for (int k = 0; k < n; ++k) v |= __ldg(src + (long long)k * hw + i);   // sum(pred_masks, 0) != 0
    dst[i] = v ? 1 : 0;
  }
}

__global__ void __launch_bounds__(NTHREADS) instance_union_kernel(const __grid_constant__ UnionArgs A, uint8_t* __restrict__ out, long long hw) {
  const int b = blockIdx.y;
  instance_union_sample(A.masks[b], A.count[b], out + (long long)b * hw, hw);
}

// The same union with the (pointer, count) table in device memory, read when the kernel runs: a CUDA graph that
// captured this launch follows whatever the table holds at replay time.  One launch, grid.y = batch.
__global__ void __launch_bounds__(NTHREADS) instance_union_table_kernel(const uint8_t* const* __restrict__ masks,
                                                                        const int* __restrict__ counts,
                                                                        uint8_t* __restrict__ out, long long hw) {
  const int b = blockIdx.y;
  instance_union_sample(masks[b], counts[b], out + (long long)b * hw, hw);
}

// torchvision Resize (bilinear, antialias, align_corners=False) of a {0,1} mask followed by round-to-nearest-even, as
// `Resize(size)(int64 mask)` does (loss_utils.py:73-75, 135-137): ATen's separable triangle filter
// (_upsample_bilinear2d_aa: _compute_weights_span / _compute_weights / interpolate_aa_single_dim) in fp32 with the same
// operation order -- weights w_j = f((j + xmin - center + 0.5) / scale) / sum, horizontal pass, then vertical.
struct ResizeArgs {
  void* dst[MDN_MAX_SCALES];           // uint8 masks or fp32 planes
  float* tmp[MDN_MAX_SCALES];          // (B, in_h, out_w[k]) horizontally resized rows (workspace)
  float* wxt[MDN_MAX_SCALES];          // [taps_x][out_w[k]] normalised x weights (workspace)
  float* wyt[MDN_MAX_SCALES];          // [out_h[k]][ty[k]] normalised y weights (workspace)
  int2* xspan[MDN_MAX_SCALES];         // [out_w[k]] (first source column, taps)
  int2* yspan[MDN_MAX_SCALES];         // [out_h[k]]
  int ty[MDN_MAX_SCALES];              // row stride of wyt = taps per output row (upper bound)
  int oh[MDN_MAX_SCALES], ow[MDN_MAX_SCALES];
  int row_begin[MDN_MAX_SCALES + 1];   // first blockIdx.y of each output size, horizontal pass (row groups)
  int vrow_begin[MDN_MAX_SCALES + 1];  // ... vertical pass (output rows)
  int n_out, batch, ih, iw;
  int packed;                          // fp32 outputs as one (r, g, b, 0) float4 per pixel (planes = images x 3)
  int frows[MDN_MAX_SCALES];           // fused mask pass: output rows per block
  int frow_begin[MDN_MAX_SCALES + 1];  // ... first blockIdx.x of each output size
};

MDN_DEV float aa_tri(float x) { x = x < 0.f ? -x : x; return x < 1.f ? __fsub_rn(1.f, x) : 0.f; }

// Span and weights of output index i along one axis, with the operation order and precisions of ATen's CPU helper
// (_compute_indices_min_size_weights_aa, the oracle's path): the `+ 0.5` literals are double there, so those sums --
// and the product with 1/scale -- are formed in double and rounded to fp32 once.  (ATen's CUDA helper adds j to a
// pre-rounded xmin - center in fp32: it can differ in the last bit of a weight, which shows only where a resized
// value is an exact 0.5 tie.)
struct AaSpan {
  int xmin, xsize;
  float center, invscale, total;
  MDN_DEV float raw(int j) const {      // un-normalised triangle weight of tap j
    return aa_tri((float)(((double)__fsub_rn((float)(j + xmin), center) + 0.5) * (double)invscale));
  }
  MDN_DEV float weight(int j) const { return total != 0.f ? __fdiv_rn(raw(j), total) : raw(j); }
};

MDN_DEV AaSpan aa_span_no_total(int i, int in_size, float scale) {
  AaSpan sp;
  const float support = (scale >= 1.f) ? scale : 1.f;                     // (interp_size * 0.5) * scale, interp_size = 2
  sp.center = (float)((double)scale * ((double)i + 0.5));
  sp.xmin = max((int)(long long)((double)__fsub_rn(sp.center, support) + 0.5), 0);
  sp.xsize = min((int)(long long)((double)__fadd_rn(sp.center, support) + 0.5), in_size) - sp.xmin;
  sp.xsize = min(max(sp.xsize, 0), (int)ceilf(support) * 2 + 1);
  sp.invscale = (scale >= 1.f) ? (float)(1.0 / (double)scale) : 1.f;
  sp.total = 0.f;
  return sp;
}

// Three launches: the per-axis spans / normalised weights of every output index (a few thousand floats, the only place
// that needs the double-precision steps of aa_span_no_total), then two separable passes as the library does them (the
// intermediate is rounded to fp32 exactly like ATen's temporary tensor):
//   H: tmp_k[b][y][ox] = sum_j src[b][y][xmin + j] * wx[j]   for every source row y and every output size k
//   V: dst_k[b][oy][ox] = round(sum_y tmp_k[b][ymin + y][ox] * wy[y])
// `output = src[0] * w[0]; output += src[j] * w[j]` (basic_loop_aa_horizontal / _vertical): the library builds contract
// the update into an FMA (GCC -ffp-contract=fast with FMA targets on the CPU, nvcc -fmad on CUDA).
constexpr int AA_HROWS = 8;      // source rows per block of the horizontal pass
constexpr int AA_VROWS = 4;      // output rows per block of the vertical pass

// one WARP per (output size k, axis, output index): the lanes evaluate the taps in parallel, lane 0 adds them up in tap
// order (the library's sequential `total_w += w`), the lanes divide.  span -> A.xspan / A.yspan, weights ->
// A.wxt[k][tap][ox] / A.wyt[k][oy][tap]
constexpr int AA_MAXTAPS = 1024;   // per-warp staging of the raw taps (down-scaling factors up to ~500)
__global__ void __launch_bounds__(NTHREADS) instance_resize_weights_kernel(const __grid_constant__ ResizeArgs A, const int n_idx) {
  __shared__ float raw_s[NTHREADS / 32][AA_MAXTAPS];
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  int i = blockIdx.x * (NTHREADS / 32) + wrp;
  const bool live = i < n_idx;        // (whole warps; idle ones still walk the warp-level synchronisation below)
  int k = 0, axis = 0;
  if (live)
    for (; k < A.n_out; ++k) {
      if (i < A.ow[k]) { axis = 0; break; }
      i -= A.ow[k];
      if (i < A.oh[k]) { axis = 1; break; }
      i -= A.oh[k];
    }
  const int in_size = axis ? A.ih : A.iw, out_size = axis ? A.oh[k] : A.ow[k];
  AaSpan sp = aa_span_no_total(live ? i : 0, in_size, __fdiv_rn((float)in_size, (float)out_size));   // area_pixel_compute_scale
  if (!live) sp.xsize = 0;
  float* raw = raw_s[wrp];
  for (int j = lane; j < sp.xsize; j += 32) raw[j] = sp.raw(j);
  __syncwarp();
  float total = 0.f;
  if (lane == 0)
    for (int j = 0; j < sp.xsize; ++j) total = __fadd_rn(total, raw[j]);
  total = __shfl_sync(0xffffffffu, total, 0);
  if (lane == 0 && live) (axis ? A.yspan[k] : A.xspan[k])[i] = make_int2(sp.xmin, sp.xsize);
  for (int j = lane; j < sp.xsize; j += 32) {
    const float wj = total != 0.f ? __fdiv_rn(raw[j], total) : raw[j];
    if (axis) A.wyt[k][(long long)i * A.ty[k] + j] = wj;
    else A.wxt[k][(long long)j * A.ow[k] + i] = wj;
  }
}

// flat grid: output size k owns blocks [row_begin[k], row_begin[k + 1]) = (b, group of AA_HROWS source rows, 128-column chunk)
template <typename TIn>
__global__ void __launch_bounds__(128) instance_resize_h_kernel(const __grid_constant__ ResizeArgs A, const TIn* __restrict__ src) {
  int k = 0;
#pragma unroll
  for (int q = 1; q < MDN_MAX_SCALES; ++q)
    if (q < A.n_out && (int)blockIdx.x >= A.row_begin[q]) k = q;
  const int ow = A.ow[k];
  const int chunks = (ow + 127) / 128;
  int rem = blockIdx.x - A.row_begin[k];
  const int cx = rem % chunks;
  rem /= chunks;
  const int ox = cx * 128 + threadIdx.x;
  if (ox >= ow) return;
  const int groups = (A.ih + AA_HROWS - 1) / AA_HROWS;
  const int b = rem / groups, y0 = (rem - b * groups) * AA_HROWS;
  const int2 sp = __ldg(A.xspan[k] + ox);
  const float* wcol = A.wxt[k] + ox;
  const int ny = min(AA_HROWS, A.ih - y0);
  // row pointers once (rows past the image re-read the last valid row; their sums are not stored): the tap loop is
  // load + accumulate only.  A {0,1} byte times w is w or 0 and fma(1, w, t) == t + w exactly, so the mask path needs no
  // integer->float conversion: t += byte ? w : 0.
  const TIn* rp[AA_HROWS];
#pragma unroll
  for (int y = 0; y < AA_HROWS; ++y) rp[y] = src + ((long long)b * A.ih + y0 + min(y, ny - 1)) * A.iw + sp.x;
  auto term = [](TIn v, float wj) -> float { return sizeof(TIn) == 1 ? (v ? wj : 0.f) : __fmul_rn((float)v, wj); };
  float t[AA_HROWS];
  {
    const float w0 = __ldg(wcol);
#pragma unroll
    for (int y = 0; y < AA_HROWS; ++y) t[y] = term(__ldg(rp[y]), w0);
  }
  // four taps per trip: the byte loads use immediate offsets from row pointers bumped once per trip (address arithmetic
  // was 2/3 of this kernel); the AA_HROWS rows are independent chains sharing the weights
  auto acc = [](float tt, TIn v, float wj) -> float { return sizeof(TIn) == 1 ? __fadd_rn(tt, v ? wj : 0.f) : __fmaf_rn((float)v, wj, tt); };
  int j = 1;
#pragma unroll
  for (int y = 0; y < AA_HROWS; ++y) rp[y] += 1;
  const float* wp = wcol + ow;
  for (; j + 4 <= sp.y; j += 4, wp += 4 * (size_t)ow) {
    const float w0 = __ldg(wp), w1 = __ldg(wp + ow), w2 = __ldg(wp + 2 * (size_t)ow), w3 = __ldg(wp + 3 * (size_t)ow);
#pragma unroll
    for (int y = 0; y < AA_HROWS; ++y) {
      const TIn v0 = __ldg(rp[y]), v1 = __ldg(rp[y] + 1), v2 = __ldg(rp[y] + 2), v3 = __ldg(rp[y] + 3);
      t[y] = acc(acc(acc(acc(t[y], v0, w0), v1, w1), v2, w2), v3, w3);
      rp[y] += 4;
    }
  }
  for (; j < sp.y; ++j, wp += ow) {
    const float wj = __ldg(wp);
#pragma unroll
    for (int y = 0; y < AA_HROWS; ++y) { t[y] = acc(t[y], __ldg(rp[y]), wj); rp[y] += 1; }
  }
  float* tmp = A.tmp[k] + ((long long)b * A.ih + y0) * ow + ox;
#pragma unroll
  for (int y = 0; y < AA_HROWS; ++y)
    if (y < ny) tmp[(size_t)y * ow] = t[y];
}

// flat grid: (k, b, group of AA_VROWS output rows, 128-column chunk).  TOut = uint8_t: round to nearest even and
// store the integer mask; TOut = float: store the resized value (image pyramids, mdn_image_pyramid)
template <typename TOut>
__global__ void __launch_bounds__(128) instance_resize_v_kernel(const __grid_constant__ ResizeArgs A) {
  int k = 0;
#pragma unroll
  for (int q = 1; q < MDN_MAX_SCALES; ++q)
    if (q < A.n_out && (int)blockIdx.x >= A.vrow_begin[q]) k = q;
  const int oh = A.oh[k], ow = A.ow[k];
  const int chunks = (ow + 127) / 128;
  int rem = blockIdx.x - A.vrow_begin[k];
  const int cx = rem % chunks;
  rem /= chunks;
  const int ox = cx * 128 + threadIdx.x;
  if (ox >= ow) return;
  const int groups = (oh + AA_VROWS - 1) / AA_VROWS;
  const int b = rem / groups, oy0 = (rem - b * groups) * AA_VROWS;
  // the AA_VROWS output rows advance together, tap by tap: their loads are independent, so AA_VROWS (x2 by unrolling)
  // are in flight per thread instead of one (this pass waits on L2 / HBM latency, not on arithmetic)
  int2 sp[AA_VROWS];
  const float* col[AA_VROWS];
  const float* wrow[AA_VROWS];
  float out[AA_VROWS];
  int maxn = 0;
#pragma unroll
  for (int r = 0; r < AA_VROWS; ++r) {
    const int oy = min(oy0 + r, oh - 1);
    sp[r] = __ldg(A.yspan[k] + oy);
    if (oy0 + r >= oh) sp[r].y = 0;
    wrow[r] = A.wyt[k] + (long long)oy * A.ty[k];
    col[r] = A.tmp[k] + ((long long)b * A.ih + sp[r].x) * ow + ox;
    maxn = max(maxn, sp[r].y);
    out[r] = 0.f;
  }
#pragma unroll 2
  for (int y = 0; y < maxn; ++y) {
    float v[AA_VROWS], wv[AA_VROWS];
#pragma unroll
    for (int r = 0; r < AA_VROWS; ++r)
      if (y < sp[r].y) { v[r] = *col[r]; wv[r] = __ldg(wrow[r] + y); col[r] += ow; }
#pragma unroll
    for (int r = 0; r < AA_VROWS; ++r)
      if (y < sp[r].y) out[r] = (y == 0) ? __fmul_rn(v[r], wv[r]) : __fmaf_rn(v[r], wv[r], out[r]);
  }
#pragma unroll
  for (int r = 0; r < AA_VROWS; ++r) {
    if (oy0 + r >= oh) continue;
    if (A.packed) {      // plane b = image * 3 + channel -> component `channel` of the pixel's float4
      float* dst = reinterpret_cast<float*>(A.dst[k]) + (((long long)(b / 3) * oh + oy0 + r) * ow + ox) * 4 + (b % 3);
      *dst = out[r];
      if (b % 3 == 2) dst[1] = 0.f;
      continue;
    }
    TOut* dst = reinterpret_cast<TOut*>(A.dst[k]) + ((long long)b * oh + oy0 + r) * ow + ox;
    if (sizeof(TOut) == 1) *dst = (TOut)rintf(out[r]);      // torch.round, then the cast back to integers
    else *dst = (TOut)out[r];
  }
}

// The {0,1} MASK path: the mask is bit-packed once (mask_bitpack_kernel, 1 bit per pixel), then ONE launch does both
// passes: a block owns 128 output columns x frows[k] output rows of one (size k, sample).  It (1) fetches the packed
// source rows its outputs need, (2) runs the horizontal pass out of those bits -- a tap is `if (bit) t += w`, exactly the
// library's `t += byte * w` for a {0,1} byte, in tap order -- keeping the fp32 intermediate in shared memory instead
// of the (B, in_h, out_w) global temporary, and (3) the vertical pass + round-half-even.  Same arithmetic, same order,
// bit-identical to the two-pass kernels above; a source row is read as 1 bit per tap instead of 1 byte load per tap, and
// the 2 x 21 MB round trip of the temporary (B = 12, 375 x 1242 -> 4 levels) is gone.
constexpr int AF_NR = 48;      // source rows a block can hold
constexpr int AF_W = 56;       // 32-pixel words per packed row (incl. one word of slack for the funnel shift)
static_assert(AF_W <= 64, "the fill loop maps 64 threads to a packed row");

// {0,1} bytes -> bits: word j of row r holds pixels 32 j .. 32 j + 31 (a warp reads 32 consecutive bytes, __ballot_sync
// makes them one word); rows are `nwg` words apart, zero past the image
__global__ void __launch_bounds__(NTHREADS) mask_bitpack_kernel(const uint8_t* __restrict__ src, unsigned* __restrict__ bits, const int rows,
                                                                const int iw, const int nwg) {
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {          // a block packs whole rows: uniform trip counts
    const uint8_t* sr = src + (long long)r * iw;
    unsigned* br = bits + (long long)r * nwg;
#pragma unroll 2
    for (int j0 = 0; j0 < nwg; j0 += NTHREADS / 32) {
      const int j = j0 + wrp, x = 32 * j + lane;
      const unsigned v = (j < nwg && x < iw) ? (unsigned)__ldg(sr + x) : 0u;
      const unsigned m = __ballot_sync(0xffffffffu, v != 0u);
      if (j < nwg && lane == 0) br[j] = m;
    }
  }
}

__global__ void __launch_bounds__(128) instance_mask_resize_fused_kernel(const __grid_constant__ ResizeArgs A, const unsigned* __restrict__ gbits, const int nwg) {
  __shared__ unsigned bits[AF_NR][AF_W];
  __shared__ float tmpS[AF_NR][128];
  // blocks are numbered from the LAST output size backwards: in a pyramid that is the smallest level, whose blocks walk the
  // most source rows per output row -- the longest blocks start first
  const int bid = (int)(gridDim.x - 1 - blockIdx.x);
  int k = 0;
#pragma unroll
  for (int q = 1; q < MDN_MAX_SCALES; ++q)
    if (q < A.n_out && bid >= A.frow_begin[q]) k = q;
  const int oh = A.oh[k], ow = A.ow[k], R = A.frows[k];
  const int chunks = (ow + 127) / 128;
  int rem = bid - A.frow_begin[k];
  const int cx = rem % chunks;
  rem /= chunks;
  const int groups = (oh + R - 1) / R;
  const int b = rem / groups, oy0 = (rem - b * groups) * R;
  const int tid = threadIdx.x;
  const int ox = cx * 128 + tid;
  const bool live = ox < ow;
  // source window of the block: spans are monotone in the output index
  const int2 xf = __ldg(A.xspan[k] + cx * 128), xl = __ldg(A.xspan[k] + min(ow, cx * 128 + 128) - 1);
  const int w_lo = xf.x & ~31;
  const int nw = min(((xl.x + xl.y - w_lo + 31) >> 5) + 1, AF_W);
  const int oy1 = min(oy0 + R, oh) - 1;
  const int2 yf = __ldg(A.yspan[k] + oy0), yl = __ldg(A.yspan[k] + oy1);
  const int y_lo = yf.x, nr = min(yl.x + yl.y - yf.x, AF_NR);
  // (1) the packed rows [y_lo, y_lo + nr) x words [w_lo / 32, w_lo / 32 + nw) of the sample
  {
    const unsigned* gb = gbits + ((long long)b * A.ih + y_lo) * nwg + (w_lo >> 5);
    const int jmax = nwg - (w_lo >> 5);
    const int j = tid & 63;               // (AF_W <= 64: two rows per trip, no division)
    if (j < nw)
      for (int r = tid >> 6; r < nr; r += 2) bits[r][j] = (j < jmax) ? __ldg(gb + (unsigned)(r * nwg + j)) : 0u;
  }
  __syncthreads();
  // (2) horizontal pass: column ox of every packed row, eight rows share a weight load
  if (live) {
    const int2 sp = __ldg(A.xspan[k] + ox);
    const int o = sp.x - w_lo;
    const float* wcol = A.wxt[k] + ox;
    for (int r0 = 0; r0 < nr; r0 += 8) {
      float t[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) t[q] = 0.f;       // (0 + w == w: the library's `t = src[0] * w[0]` start)
      for (int jc = 0; jc < sp.y; jc += 32) {
        const int idx = (o + jc) >> 5, sh = (o + jc) & 31;
        unsigned win[8];
#pragma unroll
        for (int q = 0; q < 8; ++q)
          win[q] = (r0 + q < nr) ? __funnelshift_r(bits[r0 + q][idx], bits[r0 + q][min(idx + 1, AF_W - 1)], sh) : 0u;
        const int nj = min(32, sp.y - jc);
        const float* wp = wcol + (size_t)jc * ow;
        for (int j = 0; j < nj; ++j, wp += ow) {
          const float wj = __ldg(wp);
          const unsigned m = 1u << j;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (win[q] & m) t[q] = __fadd_rn(t[q], wj);
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (r0 + q < nr) tmpS[r0 + q][tid] = t[q];
    }
  }
  __syncthreads();
  // (3) vertical pass, round half to even, store.  The y weights of the block's rows are the same for every column:
  // staged in shared memory (over the packed bits, which are dead now), read back as broadcasts
  float* wyS = reinterpret_cast<float*>(&bits[0][0]);
  const int ty = A.ty[k], nrow = oy1 - oy0 + 1;
  const bool w_fit = nrow * ty <= AF_NR * AF_W;
  if (w_fit) {
    const float* wsrc = A.wyt[k] + (unsigned)(oy0 * ty);
    for (int i = tid; i < nrow * ty; i += 128) wyS[i] = __ldg(wsrc + i);
  }
  __syncthreads();
  if (live) {
    uint8_t* dcol = reinterpret_cast<uint8_t*>(A.dst[k]) + ((long long)b * oh + oy0) * ow + ox;
    for (int r = 0; r < nrow; ++r) {
      const int2 sp = __ldg(A.yspan[k] + oy0 + r);
      const float* col = &tmpS[sp.x - y_lo][tid];
      float out = 0.f;
      if (w_fit) {
        const float* wrow = wyS + r * ty;
        if (sp.y > 0) out = __fmul_rn(col[0], wrow[0]);
        int y = 1;
        for (; y + 4 <= sp.y; y += 4) {
          const float v0 = col[y * 128], v1 = col[(y + 1) * 128], v2 = col[(y + 2) * 128], v3 = col[(y + 3) * 128];
          out = __fmaf_rn(v3, wrow[y + 3], __fmaf_rn(v2, wrow[y + 2], __fmaf_rn(v1, wrow[y + 1], __fmaf_rn(v0, wrow[y], out))));
        }
        for (; y < sp.y; ++y) out = __fmaf_rn(col[y * 128], wrow[y], out);
      } else {
        const float* wrow = A.wyt[k] + (long long)(oy0 + r) * ty;
        if (sp.y > 0) out = __fmul_rn(col[0], __ldg(wrow));
        for (int y = 1; y < sp.y; ++y) out = __fmaf_rn(col[y * 128], __ldg(wrow + y), out);
      }
      dcol[(unsigned)(r * ow)] = (uint8_t)rintf(out);
    }
  }
}


// ----------------------------------------------------------------------------------------------- uint8 frames -> fp32 NCHW
// ArrayToTensor + Normalize of the dataset (datasets/custom_transforms.py:72-80, 103-112): HWC uint8 -> CHW,
// x.float() / 255, then (t - mean) / std per channel, each op rounded on its own like the CPU tensor ops the dataset runs.
struct NormArgs { float mean[3], stdv[3]; };

__global__ void __launch_bounds__(NTHREADS) normalize_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, long long hw,
                                                                const NormArgs A) {
  const int b = blockIdx.y;
  const uint8_t* s = src + (long long)b * hw * 3;
  float* d = dst + (long long)b * hw * 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float t = __fdiv_rn((float)__ldg(s + i * 3 + c), 255.f);
      d[(long long)c * hw + i] = __fdiv_rn(__fsub_rn(t, A.mean[c]), A.stdv[c]);
    }
  }
}
