// mdn_fused.cuh -- the fused tile kernel.  Included by mdn_loss.cu INSIDE namespace mdn (after KParams).
//
// One CTA (FT threads) = one TW x TH = 64x16 tile of one sample at one scale; both (target, source) pairs are
// processed by the same CTA so that d(loss)/d(mobile) is written exactly once.  A thread owns a 2-column x PR-row
// patch of pixels (lane = column pair, warp = row group): every global access is an 8-byte vector, every shared
// memory access an LDS.64 / STS.64, and the arithmetic of the two columns is packed fp32x2 (FFMA2 / FADD2 / FMUL2).
// The channel / patch loops are ROLLED: the kernel is issue- and instruction-fetch-bound, so code size is kept near 5 k
// instructions; state that must survive a rolled loop lives in thread-private shared memory (sm.D, sm.FL).
//
// Shared memory (95 KB; two CTAs per SM inside the 196 KB carve-out):
//   sT [3][R2P]      target image, tile + 2-pixel halo, reflection padded (slot -1 holds pixel 1, slot n holds n-2)
//   sM [2][R2P]      the two mobile maps, same layout, zero outside the image
//                    (sT and sM arrive by TMA: one 72 x 20 box per plane on an mbarrier; cp.async where the row pitch
//                    is not a multiple of 16 bytes)
//   sW [3][R2P]      warped source image of the current pair, same layout
//   sQ [3][R1P]      SSIM adjoint coefficient planes (A, B, C) of the current pair AND channel, tile + 1-pixel halo
//   sD [6][PR][FT]   thread-private float2 slots: d(warped_c)/d(ix), d(warped_c)/d(iy) of the own pixels
//   sFL [PR][2][FT]  thread-private float2 slots: the flow of the own pixels (P1 -> P4)
// Per pair (with the poses given, nine threads first rebuild F = K^-T [t]x R K^-1 of the (pair, sample)):
//   P1  one rolled loop over pixel PAIRS: the thread's PR own pairs, then its share of the halo ring.  flow ->
//       sampling coordinates -> bilinear gather of the 3 source channels (gather_pair_packed) -> sW; derivatives -> sD
//   per channel c (rolled):
//     P2  SSIM windows over the tile + 1-pixel halo in 2x3 patches: 3-tap row sums of (x, y, x^2, y^2, xy) for two
//         columns from two LDS.64 per image row, a sliding column sum, two windows per packed evaluation
//         (ssim_window2); writes the adjoint planes of channel c
//     P3  the thread's own pixels: separable 3x3 adjoint gather of the three planes (packed), L1 term, chain rule
//         to d(loss)/d(ix, iy)
//   P4  both rows of the patch: epipolar distance, post-processing, masked sums and their adjoints; d(loss)/d(flow)
// then the tail: smoothness + consistency + routing of d/dmask through the min; block reduction.  P4 and the tail read
// nothing from global memory.

struct FusedSmem {
  float* T;      // [3][R2P]
  float* W;      // [3][R2P]
  float* Q;      // [3][R1P]
  float* D;      // [6][PR][FT] float2
  float* M;      // [2][R2P] the two mobile maps, tile + halo, ZERO outside the image (halo-2 layout, 1 pixel used)
  float* FL;     // [PR][2][FT] float2: flow (x, y planes) of the own pixels, stashed by P1 for P4
  float* red;    // [FWARPS][NSLOT]
  float* fm;     // [2][16] fundamental matrix + SN maximum of the (pair, sample); then the TMA mbarrier (8 bytes)
};

__host__ __device__ constexpr size_t fused_smem_floats(bool photo) {
  return 3 * R2P + (size_t)FWARPS * NSLOT + 32 + 32 + 2 * R2P + (photo ? 3 * R2P + 3 * R1P + 6 * PR * FT * 2 + PR * 2 * FT * 2 : 0);
}

template <int NV>
MDN_DEV void flush_acc(float* v, float* red, int slot_base) {
  warp_reduce_transpose<NV>(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane < NV) red[warp * NSLOT + slot_base + lane] += v[0];
}

// image coordinate whose value a shared-memory slot at coordinate t holds (ReflectionPad2d(1)); -1 = none
MDN_DEV int stage_index(int t, int n) {
  if (t < 0) return (t == -1) ? 1 : -1;
  if (t >= n) return (t == n) ? n - 2 : -1;
  return t;
}

// (r, j) of the first pixel of the i-th PAIR of the halo ring of the halo-2 region: two top rows, two bottom rows
// (S2 / 2 pairs each), then the two side pairs of every interior row
constexpr int RINGP = 2 * W2 + 2 * TH;
MDN_DEV void ring_pair(int i, int& r, int& j) {
  constexpr int HP = W2 / 2;
  if (i < 2 * HP) { r = i / HP; j = 2 * (i - r * HP); }
  else if (i < 4 * HP) { i -= 2 * HP; r = i / HP; j = 2 * (i - r * HP); r += TH + 2; }
  else { i -= 4 * HP; r = 2 + (i >> 1); j = (i & 1) ? TW + 2 : 0; }
}

MDN_DEV float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }

template <bool B> struct BoolTag { static constexpr bool value = B; };

// PAD: grid_sample padding mode of the flow warp (0 zeros = what the reference's callers pass, 1 border, 2 reflection)
template <bool PHOTO, bool MAPS, int PAD = 0>
__global__ void __launch_bounds__(FT, FUSED_MIN_CTAS) fused_tile_kernel(const __grid_constant__ KParams P) {
  MDN_DYN_SMEM(smem_raw);
  const int tid = threadIdx.x;
  const int t = tid & 31, g = tid >> 5;    // column pair, row group (= warp)
  if (blockIdx.x == 0 && tid == 0) *P.ticket = 0u;   // finish_kernel's completion ticket (it runs after this grid)
  const bool use_ssim = PHOTO && (P.flags & MDN_OPT_SSIM);
  const bool epi_on = (P.flags & MDN_TERM_EPIPOLAR) != 0;
  const bool smooth_on = (P.flags & MDN_TERM_SMOOTH) != 0;
  const bool consis_on = (P.flags & MDN_TERM_CONSIS) != 0;
  const bool grads = (P.flags & MDN_OPT_GRADS) != 0;
  const bool own = P.mask_mode == MDN_MASK_OWN;
  const bool shared_mask = P.mask_mode == MDN_MASK_SHARED;
  const bool minmode = !own && !shared_mask;
  const bool need_tgt = PHOTO || smooth_on;
  const bool need_mask = epi_on || smooth_on || consis_on;

  FusedSmem sm;
  sm.T = smem_raw;
  sm.red = sm.T + 3 * R2P;
  sm.fm = sm.red + FWARPS * NSLOT;
  sm.M = sm.fm + 64;     // (fm + 32 .. fm + 63: the mbarrier and padding that keeps the planes 128-byte aligned)
  sm.W = sm.M + 2 * R2P;
  sm.Q = sm.W + 3 * R2P;
  sm.D = sm.Q + 3 * R1P;
  sm.FL = sm.D + 6 * PR * FT * 2;

  // ---- which tile
  int s = 0;      // (tile_begin decreases with the scale index: the last scale owns the first tiles, see plan_tiles)
#pragma unroll
  for (int k = 1; k < MDN_MAX_SCALES; ++k)
    if (k < P.n_scales && (int)blockIdx.x < P.sc[k - 1].tile_begin) s = k;
  const KScale& S = P.sc[s];
  int rem = blockIdx.x - S.tile_begin;
  const int tiles_per_img = S.tiles_x * S.tiles_y;
  const int b = rem / tiles_per_img;
  rem -= b * tiles_per_img;
  const int ty = rem / S.tiles_x, tx = rem - ty * S.tiles_x;
  const int x0 = tx * TW, y0 = ty * TH;
  const int h = S.h, w = S.w, hw = h * w;
  const float sx = S.sx, sy = S.sy;      // per-scale constants live in registers, not in indexed constant-bank loads
  const WarpGeom geom = S.geom;
  // tile holds a pixel whose 3x3 adjoint gather sees a reflected tap (rows 1, h-2 / columns 1, w-2)
  const bool border = (y0 == 0) | (h - 2 >= y0 && h - 2 < y0 + TH) | (x0 == 0) | (w - 2 >= x0 && w - 2 < x0 + TW);

  // the 2 x PR pixels this thread owns
  const int px0 = x0 + 2 * t, px1 = px0 + 1;
  const int py0 = y0 + PR * g;
  const bool in0 = px0 < w, in1 = px1 < w;
  const bool weven = (w & 1) == 0;
  const bool vec = weven & in1;             // 8-byte accesses at (row, px0): aligned and both columns inside
  const int o2own = OFF2 + (PR * g + 2) * S2 + 2 * t + 2;   // halo-2 slot of the patch's first pixel

  for (int i = tid; i < FWARPS * NSLOT; i += FT) sm.red[i] = 0.f;

  // ---- L2 prefetch of the inputs of the tile that will run in this CTA slot one wave from now: every input byte is
  // read from HBM exactly once, so without this each tile's first touches (target staging, flow, mobile maps) pay
  // the full DRAM latency in front of dependent work.  One 128-byte line per thread and plane row segment.
  {
    const int nt = (int)blockIdx.x + P.prefetch_distance;
    if (nt < P.n_tiles) {
      int s2 = 0;
#pragma unroll
      for (int k = 1; k < MDN_MAX_SCALES; ++k)
        if (k < P.n_scales && nt < P.sc[k - 1].tile_begin) s2 = k;
      const KScale& Z = P.sc[s2];
      int r2 = nt - Z.tile_begin;
      const int tpi = Z.tiles_x * Z.tiles_y;
      const int b2 = r2 / tpi;
      r2 -= b2 * tpi;
      const int ty2 = r2 / Z.tiles_x, tx2 = r2 - ty2 * Z.tiles_x;
      const int hw2 = Z.h * Z.w;
      // rows of the tile x (3 target + 2 x 2 flow + 2 mobile planes) x two 128-byte lines per 64-pixel row
      constexpr int NPL = 9;
      for (int i = tid; i < NPL * TH * 2; i += FT) {
        const int pl = i / (TH * 2), rr = i - pl * (TH * 2);
        const int y = ty2 * TH + (rr >> 1), x = tx2 * TW + (rr & 1) * 32;
        if (y < Z.h && x < Z.w) {
          const float* base;
          if (pl < 3) base = need_tgt ? Z.tgt + ((size_t)b2 * 3 + pl) * hw2 : nullptr;
          else if (pl < 7) { const int q = pl - 3; base = Z.flow[q >> 1] ? Z.flow[q >> 1] + ((size_t)b2 * 2 + (q & 1)) * hw2 : nullptr; }
          else base = (need_mask && Z.mob[pl - 7]) ? Z.mob[pl - 7] + (size_t)b2 * hw2 : nullptr;
          // planes that arrive by TMA are asynchronous anyway: only the flows (loaded by the gather phase) are worth it
          if (P.tma_ok[s2] && (pl < 3 || pl >= 7)) base = nullptr;
          if (base) prefetch_l2(base + (size_t)y * Z.w + x);
        }
      }
    }
  }

  // ---- TMA staging needs an mbarrier in shared memory, initialised before anybody polls it
  uint64_t* tma_bar = reinterpret_cast<uint64_t*>(sm.fm + 32);
  const bool use_tma = P.tma_ok[s] != 0;
#ifndef MDN_EMU
  if (use_tma) {
    if (tid == 0) {
      cuda::ptx::mbarrier_init(tma_bar, 1);
      cuda::ptx::fence_proxy_async(cuda::ptx::space_shared);
    }
    __syncthreads();
  }
#endif
  // waits for the staged planes (both mechanisms), then patches the reflection ring a TMA copy cannot produce
  auto staging_done = [&]() {
    cp_async_wait_all();
#ifndef MDN_EMU
    if (use_tma) {
      while (!cuda::ptx::mbarrier_try_wait_parity(tma_bar, 0u)) {}
      // ReflectionPad2d(1) of the image planes: slots at x = -1 / w and y = -1 / h take the mirrored pixel, which the box
      // delivered (it lies inside the image and inside this tile).  Block-uniform: interior tiles skip it.
      const int jw = w - x0 + 2, rh = h - y0 + 2;        // slot column of x = w, slot row of y = h
      const bool bx = (x0 == 0) | (jw < W2), by = (y0 == 0) | (rh < R2H);
      if (need_tgt && (bx | by)) {
        __syncthreads();
        for (int i = tid; i < 3 * (2 * R2H + 2 * W2); i += FT) {
          const int c = i / (2 * R2H + 2 * W2);
          int q = i - c * (2 * R2H + 2 * W2), r, j;
          if (q < 2 * R2H) { r = q >> 1; j = (q & 1) ? jw : 1; }          // the two ring columns
          else { q -= 2 * R2H; j = q >> 1; r = (q & 1) ? rh : 1; }        // the two ring rows
          if ((unsigned)j >= (unsigned)W2 || (unsigned)r >= (unsigned)R2H) continue;
          const int x = x0 - 2 + j, y = y0 - 2 + r;
          if ((unsigned)x < (unsigned)w && (unsigned)y < (unsigned)h) continue;      // a real pixel
          const int xx = stage_index(x, w), yy = stage_index(y, h);
          if ((xx | yy) < 0) continue;                                               // beyond the reflected ring: stays 0
          float* pl = sm.T + c * R2P + OFF2;
          pl[r * S2 + j] = pl[(yy - (y0 - 2)) * S2 + (xx - (x0 - 2))];
        }
      }
    }
#endif
  };

  // ---- P0: stage the target image (planes 0-2: halo 2, reflection padded) and the two mobile maps (planes 3-4: zero
  // outside the image) with cp.async; the copies land while P1 runs.  Nothing after this reads them from global memory.
  const float* mob0 = opaque_ptr(need_mask ? S.mob[0] + (size_t)b * hw : nullptr);
  const float* mob1 = opaque_ptr(need_mask ? (shared_mask ? mob0 : S.mob[1] + (size_t)b * hw) : nullptr);
  {
    const int pl0 = need_tgt ? 0 : 3, pl1 = need_mask ? (shared_mask ? 4 : 5) : 3;
    const float* tg = need_tgt ? S.tgt + (size_t)b * 3 * hw : nullptr;
    auto plane_src = [&](int pl) -> const float* { return pl < 3 ? tg + (size_t)pl * hw : (pl == 3 ? mob0 : mob1); };
    auto plane_dst = [&](int pl) -> float* { return pl < 3 ? sm.T + pl * R2P : sm.M + (pl - 3) * R2P; };
    // source coordinate of slot coordinate t: reflected for the image planes, none (-1 -> zero fill) for the maps
    auto src_index = [&](int pl, int tt, int n) { return pl < 3 ? stage_index(tt, n) : ((unsigned)tt < (unsigned)n ? tt : -1); };
#ifndef MDN_EMU
    if (use_tma) {
      // one TMA box per plane: 72 x 20 floats at (x0 - 4, y0 - 2, plane), zeros outside the tensor, arriving on the mbarrier
      // initialised above; the reflected ring of the image planes is patched after the wait (border tiles only)
      if (tid == 0) {
        namespace ptx = cuda::ptx;
        ptx::mbarrier_arrive_expect_tx(ptx::sem_release, ptx::scope_cta, ptx::space_shared, tma_bar, (unsigned)((pl1 - pl0) * R2P * 4));
        for (int pl = pl0; pl < pl1; ++pl) {
          const int32_t coord[3] = {x0 - 4, y0 - 2, pl < 3 ? b * 3 + pl : b};
          ptx::cp_async_bulk_tensor(ptx::space_cluster, ptx::space_global, plane_dst(pl), &P.tmap[s][pl < 3 ? 0 : pl - 2], coord, tma_bar);
        }
      }
    } else
#endif
    if (((w & 1) == 0) & (x0 + TW <= w)) {
      if ((w & 3) == 0) {
        // interior columns as 16-byte copies (global x0 + 4q and slot OFF2 + 2 + 4q are both 16-byte aligned)
        for (int i = tid + pl0 * R2H * (TW / 4); i < pl1 * R2H * (TW / 4); i += FT) {
          const int c = i / (R2H * (TW / 4)), rr = i - c * (R2H * (TW / 4));
          const int r = rr / (TW / 4), q = rr - r * (TW / 4);
          const int yy = src_index(c, y0 - 2 + r, h);
          const bool ok = yy >= 0;
          cp_async_f32x4(plane_dst(c) + OFF2 + r * S2 + 2 + 4 * q, plane_src(c) + (ok ? yy * w : 0) + x0 + 4 * q, ok);
        }
      } else {
        // even width, rows 8-byte aligned only (375 x 1242): 8-byte copies
        for (int i = tid + pl0 * R2H * (TW / 2); i < pl1 * R2H * (TW / 2); i += FT) {
          const int c = i / (R2H * (TW / 2)), rr = i - c * (R2H * (TW / 2));
          const int r = rr / (TW / 2), q = rr - r * (TW / 2);
          const int yy = src_index(c, y0 - 2 + r, h);
          const bool ok = yy >= 0;
          cp_async_f32x2(plane_dst(c) + OFF2 + r * S2 + 2 + 2 * q, plane_src(c) + (ok ? yy * w : 0) + x0 + 2 * q, ok);
        }
      }
      for (int i = tid + pl0 * R2H * 4; i < pl1 * R2H * 4; i += FT) {
        const int c = i / (R2H * 4), rr = i - c * (R2H * 4);
        const int r = rr >> 2, k = rr & 3;
        const int j = (k < 2) ? k : TW + k;
        const int yy = src_index(c, y0 - 2 + r, h), xx = src_index(c, x0 - 2 + j, w);
        const bool ok = (yy | xx) >= 0;
        cp_async_f32(plane_dst(c) + OFF2 + r * S2 + j, plane_src(c) + (ok ? yy * w + xx : 0), ok);
      }
    } else {
      for (int i = tid + pl0 * R2H * W2; i < pl1 * R2H * W2; i += FT) {
        const int c = i / (R2H * W2), rr = i - c * (R2H * W2);
        const int r = rr / W2, j = rr - r * W2;
        const int yy = src_index(c, y0 - 2 + r, h), xx = src_index(c, x0 - 2 + j, w);
        const bool ok = (yy | xx) >= 0;
        cp_async_f32(plane_dst(c) + OFF2 + r * S2 + j, plane_src(c) + (ok ? yy * w + xx : 0), ok);
      }
    }
  }
  const float* sM0 = sm.M;
  const float* sM1 = shared_mask ? sm.M : sm.M + R2P;
  bool staged = false;   // cp.async copies completed and the block synchronised

  // accumulated d(loss)/d(mask used by the pairs) of the own pixels; the rolled row loops rotate this ring
  float2 mbar[PR];
#pragma unroll
  for (int k = 0; k < PR; ++k) mbar[k] = make_float2(0.f, 0.f);

  // the two horizontally adjacent values at (y, px0), (y, px1) of a plane; 0 outside the image.  Offsets are unsigned
  // 32-bit (one IMAD.WIDE.U32 per address).
  auto load_pair = [&](const float* plane, int y) -> float2 {
    if (!(((unsigned)y < (unsigned)h) & in0)) return make_float2(0.f, 0.f);
    const float* p = plane + (unsigned)(y * w + px0);
    if (vec) return ldg2(p);
    return make_float2(__ldg(p), in1 ? __ldg(p + 1) : 0.f);
  };
  auto store_pair = [&](float* plane, int y, float2 v) {   // caller guarantees y < h and in0
    float* p = plane + (unsigned)(y * w + px0);
    if (vec) *reinterpret_cast<float2*>(p) = v;
    else { p[0] = v.x; if (in1) p[1] = v.y; }
  };
  auto load_one = [&](const float* plane, int y, int x) -> float {
    return (((unsigned)y < (unsigned)h) & ((unsigned)x < (unsigned)w)) ? __ldg(plane + (unsigned)(y * w + x)) : 0.f;
  };

  // ---- tail (per mask q): smoothness + consistency + routing of d/dmask to the mobile maps, rolled over the rows
  // of the patch.  OWN mode calls it once per pair with that pair's own map, MIN / SHARED once after both pairs.
  auto tail = [&](const int q) {
    float acc[TAIL_SLOTS];
#pragma unroll
    for (int k = 0; k < TAIL_SLOTS; ++k) acc[k] = 0.f;
    // in MIN / SHARED mode the reference evaluates smooth_loss once per source frame with the SAME mask
    const float rep = own ? 1.f : (float)P.n_pairs;
    const float cx = rep * S.c_smx, cy = rep * S.c_smy, cc40 = S.c_consis * 40.f;
    const float third_l2e = (1.f / 3.f) * 1.4426950408889634f;
    const float* mq = ((own && q) ? sM1 : sM0) + o2own;     // first raw map the stencil reads (staged, 0 outside the image)
    const float* m0s = sM0 + o2own;
    const float* m1s = sM1 + o2own;
    // Straight-line over the PR rows of the patch: raw maps of rows py0-1 .. py0+PR and the stencil mask left / right
    // of the patch (shared memory, staged in P0), the target rows, the PR+1 vertical and 3 PR horizontal edge weights,
    // the stencil.
    float2 a0[PR + 2], a1[PR + 2], mm[PR + 2];
#pragma unroll
    for (int r = 0; r < PR + 2; ++r) {
      a0[r] = ld2s(mq + (r - 1) * S2);
      a1[r] = minmode ? ld2s(m1s + (r - 1) * S2) : a0[r];
    }
    float ml[PR], mr[PR];
#pragma unroll
    for (int k = 0; k < PR; ++k) {
      ml[k] = mr[k] = 0.f;
      if (smooth_on) {
        ml[k] = mq[k * S2 - 1]; mr[k] = mq[k * S2 + 2];
        if (minmode) {
          const float l1 = m1s[k * S2 - 1], r1 = m1s[k * S2 + 2];
          ml[k] = (ml[k] <= l1) ? ml[k] : l1; mr[k] = (mr[k] <= r1) ? mr[k] : r1;
        }
      }
    }
    // raw maps of the own rows for the consistency term: (a0, a1) are (first map read, second) = (map q, -) in OWN mode
    float2 v0[PR], v1[PR];
#pragma unroll
    for (int k = 0; k < PR; ++k) {
      v0[k] = (own && q) ? (consis_on ? ld2s(m0s + k * S2) : a0[k + 1]) : a0[k + 1];
      v1[k] = own ? (q ? a0[k + 1] : (consis_on ? ld2s(m1s + k * S2) : a0[k + 1])) : a1[k + 1];
    }
#pragma unroll
    for (int r = 0; r < PR + 2; ++r)
      mm[r] = minmode ? make_float2((a0[r].x <= a1[r].x) ? a0[r].x : a1[r].x, (a0[r].y <= a1[r].y) ? a0[r].y : a1[r].y) : a0[r];
    float2 ev[PR + 1];      // vertical edge weights: ev[r] between rows py0-1+r and py0+r, both columns
    float eh[PR][3];        // horizontal edge weights of row k: (x-1|x), (x|x+1), (x+1|x+2)
#pragma unroll
    for (int r = 0; r < PR + 1; ++r) ev[r] = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < PR; ++k) eh[k][0] = eh[k][1] = eh[k][2] = 0.f;
    if (smooth_on) {
      float2 sv[PR + 1];
      float sl[PR], smid[PR], sr[PR];
#pragma unroll
      for (int r = 0; r < PR + 1; ++r) sv[r] = make_float2(0.f, 0.f);
#pragma unroll
      for (int k = 0; k < PR; ++k) sl[k] = smid[k] = sr[k] = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float2 tr[PR + 2];
#pragma unroll
        for (int r = 0; r < PR + 2; ++r) tr[r] = ld2s(sm.T + c * R2P + o2own + (r - 1) * S2);
#pragma unroll
        for (int r = 0; r < PR + 1; ++r) {
          const float2 d = fma2(tr[r + 1], splat2(-1.f), tr[r]);
          sv[r].x += fabsf(d.x); sv[r].y += fabsf(d.y);
        }
#pragma unroll
        for (int k = 0; k < PR; ++k) {
          const float* Tr = sm.T + c * R2P + o2own + k * S2;
          sl[k] += fabsf(Tr[-1] - tr[k + 1].x); smid[k] += fabsf(tr[k + 1].x - tr[k + 1].y); sr[k] += fabsf(tr[k + 1].y - Tr[2]);
        }
      }
#pragma unroll
      for (int r = 0; r < PR + 1; ++r) {
        const int ya = py0 - 1 + r;      // edge between rows ya and ya + 1
        const bool ok = (ya >= 0) & (ya + 1 < h);
        ev[r].x = (ok & in0) ? ex2_fast(-sv[r].x * third_l2e) : 0.f;
        ev[r].y = (ok & in1) ? ex2_fast(-sv[r].y * third_l2e) : 0.f;
      }
#pragma unroll
      for (int k = 0; k < PR; ++k) {
        const bool rowin = (py0 + k < h) & in0;
        eh[k][0] = (rowin & (px0 > 0)) ? ex2_fast(-sl[k] * third_l2e) : 0.f;
        eh[k][1] = (rowin & in1) ? ex2_fast(-smid[k] * third_l2e) : 0.f;
        eh[k][2] = (rowin & (px1 + 1 < w)) ? ex2_fast(-sr[k] * third_l2e) : 0.f;
      }
    }
#pragma unroll
    for (int k = 0; k < PR; ++k) {
      const int y = py0 + k;
      if (!((y < h) & in0)) continue;
      float2 gm = mbar[k];
      if (smooth_on) {
        const float2 mc = mm[k + 1], mu = mm[k], mn = mm[k + 2];
        // d0 = m(x-1) - m(x), d1 = m(x) - m(x+1), d2 = m(x+1) - m(x+2); each pixel counts its right / lower edge
        const float d0 = ml[k] - mc.x, d1 = mc.x - mc.y, d2 = mc.y - mr[k];
        acc[SL_SMX + 2 * q] += fabsf(d1) * eh[k][1] + fabsf(d2) * eh[k][2];
        const float s0 = signmul(d0, eh[k][0]), s1 = signmul(d1, eh[k][1]), s2 = signmul(d2, eh[k][2]);
        const float2 du = fma2(mc, splat2(-1.f), mu), dn = fma2(mn, splat2(-1.f), mc);   // m(y-1) - m(y), m(y) - m(y+1)
        acc[SL_SMY + 2 * q] += fabsf(dn.x) * ev[k + 1].x + fabsf(dn.y) * ev[k + 1].y;
        gm.x += cx * (s1 - s0) + cy * (signmul(dn.x, ev[k + 1].x) - signmul(du.x, ev[k].x));
        gm.y += cx * (s2 - s1) + cy * (signmul(dn.y, ev[k + 1].y) - signmul(du.y, ev[k].y));
      }
      float2 g0, g1;
      if (own) { g0 = q ? make_float2(0.f, 0.f) : gm; g1 = q ? gm : make_float2(0.f, 0.f); }
      else if (shared_mask) { g0 = gm; g1 = make_float2(0.f, 0.f); }
      else {
        const bool f0 = a0[k + 1].x <= a1[k + 1].x, f1 = a0[k + 1].y <= a1[k + 1].y;
        g0 = make_float2(f0 ? gm.x : 0.f, f1 ? gm.y : 0.f);
        g1 = make_float2(f0 ? 0.f : gm.x, f1 ? 0.f : gm.y);
      }
      if (consis_on) {
        // sigmoid(20 (m - 0.5)) = 1 / (1 + 2^(-20 log2(e) (m - 0.5)))
        const float kk = -20.f * 1.4426950408889634f;
        const float2 t0 = fma2(v0[k], splat2(kk), splat2(-0.5f * kk)), t1 = fma2(v1[k], splat2(kk), splat2(-0.5f * kk));
        const float2 p = make_float2(rcp_fast(1.f + ex2_fast(t0.x)), rcp_fast(1.f + ex2_fast(t0.y)));
        const float2 r = make_float2(rcp_fast(1.f + ex2_fast(t1.x)), rcp_fast(1.f + ex2_fast(t1.y)));
        float2 df = fma2(r, splat2(-1.f), p);
        if (!in1) df.y = 0.f;
        // OWN mode visits every pixel once per map: count the value once, and give each map its own gradient
        if (!own || q == 0) {
          acc[SL_CONSIS] += df.x * df.x + df.y * df.y;
          g0 = fma2(mul2(mul2(df, splat2(cc40)), p), fma2(p, splat2(-1.f), splat2(1.f)), g0);
        }
        if (!own || q == 1 || P.n_pairs == 1)
          g1 = fma2(mul2(mul2(df, splat2(-cc40)), r), fma2(r, splat2(-1.f), splat2(1.f)), g1);
      }
      if (grads) {
        if (S.g_mob[0] && (!own || q == 0)) store_pair(S.g_mob[0] + (size_t)b * hw, y, g0);
        if (S.g_mob[1] && !shared_mask && (!own || q == 1 || P.n_pairs == 1)) store_pair(S.g_mob[1] + (size_t)b * hw, y, g1);
      }
    }
#pragma unroll
    for (int k = 0; k < PR; ++k) mbar[k] = make_float2(0.f, 0.f);
    flush_acc<TAIL_SLOTS>(acc, sm.red, TAIL_BASE);
  };

  // ---- per (target, source) pair
#pragma unroll 1
  for (int pair = 0; pair < P.n_pairs; ++pair) {
    float acc[PAIR_SLOTS];
#pragma unroll
    for (int k = 0; k < PAIR_SLOTS; ++k) acc[k] = 0.f;
    const float* flx = opaque_ptr(S.flow[pair] + (size_t)b * 2 * hw);
    const float* fly = opaque_ptr(flx + hw);
    float2 gix[PR], giy[PR];         // d(loss)/d(ix), d(loss)/d(iy) of the own pixels
#pragma unroll
    for (int k = 0; k < PR; ++k) { gix[k] = giy[k] = make_float2(0.f, 0.f); }

    if (epi_on && tid < 10) {   // fundamental matrix + SN maximum of this (pair, sample): staged now, read in P4
      float v = 1.f;
      if (tid < 9) {
        if (has_pose(P, pair)) {
          // poses given: every one of the nine threads builds F (81 FMAs) and keeps its own entry; the sample's first
          // tile publishes it for finish_kernel's SN fix-up
          float Fp[9];
          tile_fmat(P, s, pair, b, Fp);
#pragma unroll
          for (int k = 0; k < 9; ++k) if (k == tid) v = Fp[k];
          if ((x0 | y0) == 0) P.fmat_ws[((size_t)(s * P.n_pairs + pair) * P.batch + b) * 9 + tid] = v;
        } else v = __ldg(S.fmat[pair] + b * 9 + tid);
      }
      else if (P.post == MDN_POST_SN) v = __uint_as_float((unsigned)(P.snkey[(s * P.n_pairs + pair) * P.batch + b] >> 32));
      sm.fm[(pair & 1) * 16 + tid] = v;   // double-buffered by pair: a fast warp may start pair 1 while others read pair 0's
    }
    if (PHOTO) {
      const float4* rfp = opaque_ptr(S.refp[pair] + (size_t)b * hw);   // source image, (r, g, b, -) per pixel
      unsigned vbits = 0;            // validity of own pixel (k, e): bit 2k + e
      // -- P1: own pairs (it < PR), then this thread's share of the halo ring.  The flow of the NEXT slot is loaded
      // before the gather of the current one, so the dependent load chain flow -> coordinates -> gather overlaps.
      constexpr int N_IT = PR + (RINGP + FT - 1) / FT;
      struct Slot { int r, j, ya, xa, xb; float2 fx, fy; bool live; };
      auto prep = [&](int it, Slot& q) {
        q.live = it < N_IT;
        q.r = PR * g + 2 + it; q.j = 2 * t + 2;
        if (it >= PR) {
          const int i = tid + (it - PR) * FT;
          q.live = q.live & (i < RINGP);
          ring_pair(q.live ? i : 0, q.r, q.j);
        }
        // source pixels of the two slots: real pixels inside the image, reflected copies on the padding ring
        q.ya = stage_index(y0 - 2 + q.r, h);
        q.xa = stage_index(x0 - 2 + q.j, w); q.xb = stage_index(x0 - 1 + q.j, w);
        q.fx = q.fy = make_float2(0.f, 0.f);
        if (q.live) {
          const bool oka = (q.ya | q.xa) >= 0, okb = (q.ya | q.xb) >= 0;
          if (oka & okb & weven & (q.xb == q.xa + 1)) {
            const unsigned o = q.ya * w + q.xa;
            q.fx = ldg2(flx + o); q.fy = ldg2(fly + o);
          } else {
            const unsigned oa = oka ? q.ya * w + q.xa : 0, ob = okb ? q.ya * w + q.xb : 0;
            q.fx = make_float2(__ldg(flx + oa), __ldg(flx + ob)); q.fy = make_float2(__ldg(fly + oa), __ldg(fly + ob));
          }
        }
      };
      // stores one gathered pair: warped values -> sW, and for an own pair (k >= 0) derivatives -> sD, validity bits
      auto put = [&](const GatherPx* G2, bool valid_a, bool valid_b, int r, int j, bool oka, bool okb, int k, float2 fx, float2 fy) {
        float* Wd = sm.W + OFF2 + r * S2 + j;
#pragma unroll
        for (int c = 0; c < 3; ++c) st2s(Wd + c * R2P, make_float2(oka ? G2[0].v[c] : 0.f, okb ? G2[1].v[c] : 0.f));
        if (k >= 0) {
          const int y = y0 - 2 + r;
          const bool ra = (y < h) & in0, rb = (y < h) & in1;     // real pixels (not padding)
          vbits |= ((valid_a & ra) ? 1u : 0u) << (2 * k);
          vbits |= ((valid_b & rb) ? 2u : 0u) << (2 * k);
          float* Dd = sm.D + (k * FT + tid) * 2;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            st2s(Dd + (2 * c) * PR * FT * 2, make_float2(G2[0].dx[c], G2[1].dx[c]));
            st2s(Dd + (2 * c + 1) * PR * FT * 2, make_float2(G2[0].dy[c], G2[1].dy[c]));
          }
          // the flow of the own pixels, for P4 (0 for padding slots, like a masked global load)
          st2s(sm.FL + ((2 * k) * FT + tid) * 2, make_float2(oka ? fx.x : 0.f, okb ? fx.y : 0.f));
          st2s(sm.FL + ((2 * k + 1) * FT + tid) * 2, make_float2(oka ? fy.x : 0.f, okb ? fy.y : 0.f));
          if (MAPS && ra) {
            const size_t o = (size_t)y * w + px0;
            if (S.valid[pair]) { S.valid[pair][(size_t)b * hw + o] = valid_a ? 1 : 0; if (rb) S.valid[pair][(size_t)b * hw + o + 1] = valid_b ? 1 : 0; }
            if (S.warped[pair]) {
#pragma unroll
              for (int c = 0; c < 3; ++c) {
                S.warped[pair][((size_t)b * 3 + c) * hw + o] = G2[0].v[c];
                if (rb) S.warped[pair][((size_t)b * 3 + c) * hw + o + 1] = G2[1].v[c];
              }
            }
          }
        }
      };
      // tiles that lie fully inside an even-width image (the common case): the own pairs are real, 8-byte aligned
      // pixels -- no reflection / slot arithmetic, one LDG.64 per flow plane, next row's flow loaded a row ahead
      const bool tile_full = weven & (x0 + TW <= w) & (y0 + TH <= h);
      const int it0 = tile_full ? PR : 0;
      Slot cur;
      // the first slot of the rolled loop (on a full tile: this thread's halo-ring slot) is prepared BEFORE the own rows, so that its
      // flow loads fly while the own rows are gathered (-1 % per step; the slot's geometry costs ten registers across the own rows)
      prep(it0, cur);
      if (tile_full) {
        unsigned o = (unsigned)(py0 * w + px0);
        float2 fxn = ldg2(flx + o), fyn = ldg2(fly + o);
        const float2 xs = make_float2((float)px0, (float)px1);
#pragma unroll      // (unrolled: the corner loads of row k + 1 are scheduled above the interpolation of row k)
        for (int k = 0; k < PR; ++k) {
          const float2 fxc = fxn, fyc = fyn;
          o += w;
          if (k + 1 < PR) { fxn = ldg2(flx + o); fyn = ldg2(fly + o); }
          const float2 fxp = make_float2(__fmul_rn(sx, fxc.x), __fmul_rn(sx, fxc.y));
          const float2 fyp = make_float2(__fmul_rn(sy, fyc.x), __fmul_rn(sy, fyc.y));
          GatherPx G2[2];
          bool va, vb;
          gather_pair_packed<true, PAD>(rfp, h, w, xs, splat2((float)(py0 + k)), fxp, fyp, geom, G2, va, vb);
          put(G2, va, vb, PR * g + 2 + k, 2 * t + 2, true, true, k, fxc, fyc);
        }
      }
#pragma unroll 1
      for (int it = it0; it < N_IT; ++it) {
        Slot nxt;
        if (it + 1 < N_IT) prep(it + 1, nxt);      // (block-uniform: nothing to prepare behind the last slot)
        else { nxt = cur; nxt.live = false; }
        if (!cur.live) break;
        const bool oka = (cur.ya | cur.xa) >= 0, okb = (cur.ya | cur.xb) >= 0;
        // flow -> pixels with SCALAR multiplies (see gather_pair_packed)
        const float2 fxp = make_float2(__fmul_rn(sx, cur.fx.x), __fmul_rn(sx, cur.fx.y));
        const float2 fyp = make_float2(__fmul_rn(sy, cur.fy.x), __fmul_rn(sy, cur.fy.y));
        GatherPx G2[2];
        bool va, vb;
        gather_pair_packed<true, PAD>(rfp, h, w, make_float2((float)cur.xa, (float)cur.xb), splat2((float)cur.ya), fxp, fyp, geom, G2, va, vb);
        put(G2, va, vb, cur.r, cur.j, oka, okb, it < PR ? it : -1, cur.fx, cur.fy);
        cur = nxt;
      }
      if (!staged) { staging_done(); staged = true; }
      __syncthreads();

      float2 vmask[PR];   // validity of the own pixels as 0 / 1
#pragma unroll
      for (int k = 0; k < PR; ++k) vmask[k] = make_float2((vbits >> (2 * k)) & 1u ? 1.f : 0.f, (vbits >> (2 * k + 1)) & 1u ? 1.f : 0.f);

      const float kq = S.c_ssim * (1.f / 9.f), c_l1 = S.c_l1;

      // -- P3: the own pixels of channel c.  BORDER adds the reflection multiplicities of the adjoint gather: pixel
      // column 1 / w-2 and pixel row 1 / h-2 collect the out-of-image tap of the windows in column 0 / w-1 and row
      // 0 / h-1 a second time.  Two instantiations, selected by a block-uniform branch.
      auto p3 = [&](const int c, auto border_tag) {
        constexpr bool BORDER = decltype(border_tag)::value;
        float2 tv[PR], wv[PR];
#pragma unroll
        for (int k = 0; k < PR; ++k) {
          tv[k] = ld2s(sm.T + c * R2P + o2own + k * S2);
          wv[k] = ld2s(sm.W + c * R2P + o2own + k * S2);
        }
        float2 wbar[PR];
#pragma unroll
        for (int k = 0; k < PR; ++k) wbar[k] = make_float2(0.f, 0.f);
        if (use_ssim & grads) {
          float2 fl = make_float2(0.f, 0.f), fr = fl;
          if (BORDER) {
            fl = make_float2(px0 == 1 ? 1.f : 0.f, px1 == 1 ? 1.f : 0.f);
            fr = make_float2(px0 == w - 2 ? 1.f : 0.f, px1 == w - 2 ? 1.f : 0.f);
          }
          float2 Sg[3][PR];
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            const float* Qa = sm.Q + a * R1P + (PR * g) * S1 + 2 * t;
            float2 Hq[PR + 2];
#pragma unroll
            for (int rr = 0; rr < PR + 2; ++rr) {
              const float2 qa = ld2s(Qa + rr * S1), qb = ld2s(Qa + rr * S1 + 2);
              const float m = qa.y + qb.x;
              Hq[rr] = make_float2(qa.x + m, m + qb.y);
              if (BORDER) Hq[rr] = fma2(fr, qb, fma2(fl, qa, Hq[rr]));
            }
#pragma unroll
            for (int k = 0; k < PR; k += 2) {       // rows k, k+1 share Hq[k+1] + Hq[k+2]
              const float2 m12 = add2(Hq[k + 1], Hq[k + 2]);
              Sg[a][k] = add2(Hq[k], m12); Sg[a][k + 1] = add2(m12, Hq[k + 3]);
            }
            if (BORDER) {
#pragma unroll
              for (int k = 0; k < PR; ++k) {
                const float ftk = (py0 + k == 1) ? 1.f : 0.f, fbk = (py0 + k == h - 2) ? 1.f : 0.f;
                Sg[a][k] = fma2(splat2(fbk), Hq[k + 2], fma2(splat2(ftk), Hq[k], Sg[a][k]));
              }
            }
          }
#pragma unroll
          for (int k = 0; k < PR; ++k) wbar[k] = fma2(tv[k], Sg[2][k], fma2(wv[k], Sg[1][k], Sg[0][k]));
        }
        // L1 term: |tgt - warped| * valid  (loss_functions.py:109-110)
#pragma unroll
        for (int k = 0; k < PR; ++k) {
          const float d0 = tv[k].x - wv[k].x, d1 = tv[k].y - wv[k].y;
          const float a0 = fabsf(d0) * vmask[k].x, a1 = fabsf(d1) * vmask[k].y;
          acc[SL_L1] += a0 + a1;
          if (MAPS && S.diff[pair]) {
            const int y = py0 + k;
            if ((y < h) & in0) S.diff[pair][((size_t)b * 3 + c) * hw + (size_t)y * w + px0] = a0;
            if ((y < h) & in1) S.diff[pair][((size_t)b * 3 + c) * hw + (size_t)y * w + px1] = a1;
          }
          if (grads) {
            wbar[k].x -= signmul(d0, c_l1 * vmask[k].x);      // == c_l1 * sign(d0) * valid: every factor but one is 0 / +-1
            wbar[k].y -= signmul(d1, c_l1 * vmask[k].y);
            const float* Dd = sm.D + (k * FT + tid) * 2 + (2 * c) * PR * FT * 2;
            gix[k] = fma2(wbar[k], ld2s(Dd), gix[k]);
            giy[k] = fma2(wbar[k], ld2s(Dd + PR * FT * 2), giy[k]);
          }
        }
      };

#pragma unroll 1
      for (int c = 0; c < 3; ++c) {
        // -- P2: SSIM windows of channel c, 2 columns x WPR rows per patch
        if (use_ssim) {
#pragma unroll 1
          for (int patch = tid; patch < NPATCH; patch += FT) {
            const int rg = patch / NCP, cp = patch - rg * NCP;
            const int o2 = c * R2P + OFF2 + (WPR * rg) * S2 + 2 * cp;
            const float* Tp = sm.T + o2;
            const float* Wp = sm.W + o2;
            const int wx0 = x0 - 1 + 2 * cp, wy0 = y0 - 1 + WPR * rg;
            const bool ci0 = (unsigned)wx0 < (unsigned)w, ci1 = (unsigned)(wx0 + 1) < (unsigned)w;
            // windows that belong to this tile's own pixels (the SSIM loss sum counts every window once)
            const float it0 = (ci0 & (cp >= 1)) ? 1.f : 0.f, it1 = (ci1 & (cp < NCP - 1)) ? 1.f : 0.f;
            const float2 kcol = make_float2(ci0 ? kq : 0.f, ci1 ? kq : 0.f);
            float2 H[3][5];   // 3-tap row sums of (x, y, xx, yy, xy) of the last three image rows, for both columns
#pragma unroll
            for (int rr = 0; rr < WPR + 2; ++rr) {
              const float2 ta = ld2s(Tp + rr * S2), tb = ld2s(Tp + rr * S2 + 2);
              const float2 wa = ld2s(Wp + rr * S2), wb = ld2s(Wp + rr * S2 + 2);
              float2* Hc = H[rr % 3];
              const float mt = ta.y + tb.x, mw = wa.y + wb.x;
              Hc[0] = make_float2(ta.x + mt, mt + tb.y);
              Hc[1] = make_float2(wa.x + mw, mw + wb.y);
              const float mtt = fmaf(tb.x, tb.x, ta.y * ta.y), mww = fmaf(wb.x, wb.x, wa.y * wa.y), mtw = fmaf(tb.x, wb.x, ta.y * wa.y);
              Hc[2] = make_float2(fmaf(ta.x, ta.x, mtt), fmaf(tb.y, tb.y, mtt));
              Hc[3] = make_float2(fmaf(wa.x, wa.x, mww), fmaf(wb.y, wb.y, mww));
              Hc[4] = make_float2(fmaf(ta.x, wa.x, mtw), fmaf(tb.y, wb.y, mtw));
              if (rr >= 2) {
                const int q = rr - 2;                       // window row inside the patch
                const int r1 = WPR * rg + q, wy = wy0 + q;  // halo-1 row, image row
                const bool ri = (unsigned)wy < (unsigned)h;
                float2 V[5];
#pragma unroll
                for (int m = 0; m < 5; ++m) V[m] = add2(add2(H[0][m], H[1][m]), H[2][m]);
                const Ssim2 so = ssim_window2(V[0], V[1], V[2], V[3], V[4], ri ? kcol : make_float2(0.f, 0.f));
                const bool rit = ri & (r1 >= 1) & (r1 <= TH);
                acc[SL_SSIM] += rit ? fmaf(so.J.x, it0, so.J.y * it1) : 0.f;
                if (MAPS && S.ssim_map[pair] && rit) {
                  float* dst = S.ssim_map[pair] + ((size_t)b * 3 + c) * hw + (size_t)wy * w + wx0;
                  if (it0 != 0.f) dst[0] = so.J.x;
                  if (it1 != 0.f) dst[1] = so.J.y;
                }
                float* Qd = sm.Q + r1 * S1 + 2 * cp;
                st2s(Qd, so.A); st2s(Qd + R1P, so.B); st2s(Qd + 2 * R1P, so.C);
              }
            }
          }
          __syncthreads();
        }
        if (border) p3(c, BoolTag<true>()); else p3(c, BoolTag<false>());
        if (use_ssim) __syncthreads();   // Q (and, after the last channel, W) is rewritten next
      }
    }

    if (!PHOTO && !staged) { staging_done(); staged = true; __syncthreads(); }

    // -- P4: epipolar forward + adjoint, d(loss)/d(flow)
    {
      float Fm[9];
      float snmax = 1.f;
      if (epi_on) {
        if (!PHOTO) __syncthreads();     // (the photometric path has synchronised since sm.fm was written)
#pragma unroll
        for (int k = 0; k < 9; ++k) Fm[k] = sm.fm[(pair & 1) * 16 + k];
        snmax = sm.fm[(pair & 1) * 16 + 9];
      }
      const float c_epi = S.c_epi, c_nt = S.c_nt, c_ce = S.c_ce;
      float* gflx = opaque_ptr(S.g_flow[pair] ? S.g_flow[pair] + (size_t)b * 2 * hw : nullptr);
      float* gfly = opaque_ptr(gflx ? gflx + hw : nullptr);
      const float* mq0 = ((own && pair) ? sM1 : sM0) + o2own;
      const bool use_inst = (P.flags & (MDN_OPT_INST_MASK | MDN_OPT_CROSS_ENT)) != 0, use_wgt = P.post == MDN_POST_TG;
      struct Row { float2 fx, fy, m0, m1, kin, wgt; };
      auto fetch = [&](int k, Row& R) {
        const int y = py0 + k;
        R.kin = R.wgt = make_float2(1.f, 1.f);
        R.fx = R.fy = R.m0 = R.m1 = make_float2(0.f, 0.f);
        if (epi_on & (k < PR)) {
          if (PHOTO) {   // stashed by P1
            R.fx = ld2s(sm.FL + ((2 * k) * FT + tid) * 2); R.fy = ld2s(sm.FL + ((2 * k + 1) * FT + tid) * 2);
          } else { R.fx = load_pair(flx, y); R.fy = load_pair(fly, y); }
          R.m0 = ld2s(mq0 + k * S2);
          R.m1 = minmode ? ld2s(sM1 + o2own + k * S2) : R.m0;
          if (use_wgt) {
            R.wgt = load_pair(S.weight, y);
            if (!in1) R.wgt.y = 1.f;     // (odd widths: the column past the image must not turn 1 / weight into inf, inf * 0 = NaN)
          }
          if (use_inst & (y < h) & in0) {
            const uint8_t* ip = S.inst + (size_t)b * hw + (unsigned)(y * w + px0);
            R.kin = make_float2((float)__ldg(ip), in1 ? (float)__ldg(ip + 1) : 0.f);
          }
        }
      };
      // Both pixels of a row at once (packed).  Exactness is kept where the reference cancels: u, v and the
      // numerator p2^T F p1 replay the reference's separate roundings with SCALAR ops (ptxas would contract packed
      // mul + add); a^2 + b^2, the square root, the division and the post-processing are a few ulp off the reference
      // (fast reciprocal / sqrt), far inside the 1e-5 budget.  post = (d k)^2 with k = 1/max (SN), 1/thr (T),
      // 1/(thr w) (TG): no |d| / sign(d) needed, d(post)/dd = 2 (d k) k.
      float2 accp[PAIR_SLOTS];     // packed partial sums of this phase (slot layout of acc[])
#pragma unroll
      for (int k = 0; k < PAIR_SLOTS; ++k) accp[k] = make_float2(0.f, 0.f);
      const float2 xf2 = make_float2((float)px0, (float)px1);
      const float kbase = (P.post == MDN_POST_SN) ? rcp_fast(snmax) : ((P.threshold > 0.f) ? P.inv_threshold : 1.f);
      const float2 live = make_float2(1.f, in1 ? 1.f : 0.f);   // the second column may lie outside a ragged image
      // straight-line over the PR rows: all global loads of the patch are issued first (one round of latency instead
      // of one per row), and the rows' dependent chains (sqrt -> rcp -> ... -> adjoint) interleave
      Row rows[PR];
#pragma unroll
      for (int k = 0; k < PR; ++k) fetch(k, rows[k]);
#pragma unroll
      for (int k = 0; k < PR; ++k) {
        const Row& cur = rows[k];
        const int y = py0 + k;
        // (w-1)/2 [grid_sample] * 2 [2g-1] / (w-1) [/= w-1] * sx [scale factor]
        float2 gfx = mul2(gix[k], splat2(sx)), gfy = mul2(giy[k], splat2(sy));
        float2 mb = make_float2(0.f, 0.f);
        if ((y < h) & in0) {
          if (epi_on) {
            const float yf = (float)y;
            const float2 m = make_float2((cur.m0.x <= cur.m1.x) ? cur.m0.x : cur.m1.x, (cur.m0.y <= cur.m1.y) ? cur.m0.y : cur.m1.y);
            const float2 u = add2(xf2, make_float2(__fmul_rn(sx, cur.fx.x), __fmul_rn(sx, cur.fx.y)));
            const float2 v = add2(splat2(yf), make_float2(__fmul_rn(sy, cur.fy.x), __fmul_rn(sy, cur.fy.y)));
            // F p1 (loss_utils.py:64): k-ordered FMA chains, exactly as epipolar_distance()
            const float2 ea = add2(fma2(splat2(Fm[1]), splat2(yf), mul2(splat2(Fm[0]), xf2)), splat2(Fm[2]));
            const float2 eb = add2(fma2(splat2(Fm[4]), splat2(yf), mul2(splat2(Fm[3]), xf2)), splat2(Fm[5]));
            const float2 ec = add2(fma2(splat2(Fm[7]), splat2(yf), mul2(splat2(Fm[6]), xf2)), splat2(Fm[8]));
            const float2 num = make_float2(__fadd_rn(__fadd_rn(__fmul_rn(ea.x, u.x), __fmul_rn(eb.x, v.x)), ec.x),
                                           __fadd_rn(__fadd_rn(__fmul_rn(ea.y, u.y), __fmul_rn(eb.y, v.y)), ec.y));
            const float2 ss = add2(fma2(ea, ea, mul2(eb, eb)), splat2(1e-10f));
            const float2 den = add2(make_float2(sqrt_fast(ss.x), sqrt_fast(ss.y)), splat2(1e-10f));
            const float2 rden = make_float2(rcp_fast(den.x), rcp_fast(den.y));
            const float2 dd = mul2(num, rden);                                 // signed epipolar distance
            float2 kw = splat2(kbase);
            if (use_wgt) kw = make_float2(kbase * rcp_fast(cur.wgt.x), kbase * rcp_fast(cur.wgt.y));
            const float2 rs = mul2(dd, kw);
            float2 post = mul2(rs, rs);
            float2 kmask = cur.kin;
            if (P.flags & MDN_OPT_INST_MASK) post = mul2(post, kmask); else kmask = make_float2(1.f, 1.f);
            const float2 bg = add2(splat2(1.f), mul2(m, splat2(-1.f)));
            const float2 bge = add2(bg, splat2(1e-5f));
            const float2 lg = mul2(make_float2(lg2_fast(bge.x), lg2_fast(bge.y)), splat2(0.6931471805599453f));
            const float2 ml = mul2(m, lg);
            accp[SL_EPI] = fma2(mul2(bg, post), live, accp[SL_EPI]);
            acc[SL_NT] += fabsf(ml.x) + (in1 ? fabsf(ml.y) : 0.f);
            if (P.flags & MDN_OPT_CROSS_ENT) {
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                if (e && !in1) continue;
                const float me = e ? m.y : m.x, bge0 = e ? bg.y : bg.x, ke = e ? cur.kin.y : cur.kin.x;
                const float l1 = __logf(me + 1e-10f), l0 = __logf(bge0 + 1e-10f);
                acc[SL_CE] += -(ke * l1 + (1.f - ke) * l0);
                const float t = c_ce * (__fdividef(1.f - ke, bge0 + 1e-10f) - __fdividef(ke, me + 1e-10f));
                if (e) mb.y += t; else mb.x += t;
              }
            }
            if (MAPS) {
              const size_t o = (size_t)b * hw + (size_t)y * w + px0;
              if (S.post_map[pair]) { S.post_map[pair][o] = post.x; if (in1) S.post_map[pair][o + 1] = post.y; }
              if (S.ori_map[pair]) {
                const float s0 = (P.post == MDN_POST_SN) ? kbase : 1.f;
                S.ori_map[pair][o] = fabsf(dd.x) * s0; if (in1) S.ori_map[pair][o + 1] = fabsf(dd.y) * s0;
              }
            }
            if (grads) {
              const float2 rb = make_float2(rcp_fast(bge.x), rcp_fast(bge.y));
              const float2 tnt = fma2(mul2(m, rb), splat2(-1.f), lg);            // lg - m / (bg + 1e-5)
              mb = fma2(post, splat2(-c_epi), mb);
              mb.x += signmul(ml.x, c_nt * tnt.x); mb.y += signmul(ml.y, c_nt * tnt.y);
              // d(loss)/dd = c_epi bg kmask 2 (d k) k
              const float2 dbar = mul2(mul2(mul2(bg, kmask), splat2(2.f * c_epi)), mul2(rs, kw));
              const float2 g2 = mul2(mul2(dbar, rden), live);
              const float2 das = mul2(dd, rden);                                 // d / s (s and s + 1e-10 agree to 1e-5)
              gfx = fma2(mul2(g2, ea), splat2(sx), gfx);
              gfy = fma2(mul2(g2, eb), splat2(sy), gfy);
              const float2 g0 = mul2(g2, fma2(mul2(das, ea), splat2(-1.f), u)), g1 = mul2(g2, fma2(mul2(das, eb), splat2(-1.f), v));
              accp[SL_GF + 0] = fma2(g0, xf2, accp[SL_GF + 0]); accp[SL_GF + 1] = fma2(g0, splat2(yf), accp[SL_GF + 1]); accp[SL_GF + 2] = add2(accp[SL_GF + 2], g0);
              accp[SL_GF + 3] = fma2(g1, xf2, accp[SL_GF + 3]); accp[SL_GF + 4] = fma2(g1, splat2(yf), accp[SL_GF + 4]); accp[SL_GF + 5] = add2(accp[SL_GF + 5], g1);
              accp[SL_GF + 6] = fma2(g2, xf2, accp[SL_GF + 6]); accp[SL_GF + 7] = fma2(g2, splat2(yf), accp[SL_GF + 7]); accp[SL_GF + 8] = add2(accp[SL_GF + 8], g2);
            }
          }
          if (grads && gflx) {
            store_pair(gflx, y, gfx);
            store_pair(gfly, y, gfy);
          }
        }
        mbar[k] = add2(mbar[k], mb);
      }
#pragma unroll
      for (int k = 0; k < PAIR_SLOTS; ++k) acc[k] += accp[k].x + accp[k].y;
    }
    flush_acc<PAIR_SLOTS>(acc, sm.red, pair * PAIR_SLOTS);
    if (need_mask && own) tail(pair);
  }
  if (need_mask && !own) tail(0);

  __syncthreads();
  for (int k = tid; k < NSLOT; k += FT) {
    float tsum = 0.f;
#pragma unroll
    for (int wq = 0; wq < FWARPS; ++wq) tsum += sm.red[wq * NSLOT + k];
    P.partials[(size_t)blockIdx.x * NSLOT + k] = tsum;
  }
}
