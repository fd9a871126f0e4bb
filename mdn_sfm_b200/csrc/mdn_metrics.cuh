// mdn_metrics.cuh -- evaluation of mobile masks: confusion counts of binary_image(pred, thr) (utils.py:100-103) against
// moving-object masks, for a whole threshold sweep in one read of the maps.  Included by mdn_loss.cu INSIDE namespace mdn.
// Entry points: mdn_mask_confusion / _workspace_bytes (include/mdn_loss.h).
//
// mask_confusion_kernel bins every pixel by j = #{k : pred >= thr[k]} (0..K) and its label (gt != 0) into a shared
// histogram of 2 x (K + 1) counters, then adds the block's non-zero bins to the sample's global histogram; the finish
// kernel turns each histogram into per-threshold [TP, FP, FN, TN] by suffix sums.  Integer counts throughout, so the
// result does not depend on the order in which blocks run.

constexpr int CONF_MAX_THR = 1024;   // K <= 1024: 4 KB of thresholds + 8.2 KB of bins, static shared memory
constexpr int CONF_THREADS = 256;

// One pixel into the block histogram.  Lanes with the same key are counted by one shared atomic (mobile maps are mostly
// near 0, so most lanes of a warp land in one bin).  Every lane of the warp calls it; key < 0 adds nothing.
MDN_DEV void conf_add(unsigned* s_hist, int key) {
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  if (key >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(s_hist + key, (unsigned)__popc(peers));
}

// j[q] = #{k : x[q] >= thr[k]} for ascending thresholds, by binary lifting over powers of two from `top` (the largest
// power of two <= K) down to 1; the N searches interleave, so their shared loads are independent.  NaN compares false
// everywhere and gets 0.  The probe index is clamped into 0..K-1, so unsorted thresholds give some j in 0..K but never a
// read outside thr[0..K-1].
template <int N>
MDN_DEV void conf_bins(const float* s_thr, int K, int top, const float (&x)[N], int (&j)[N]) {
#pragma unroll
  for (int q = 0; q < N; ++q) j[q] = 0;
  for (int step = top; step > 0; step >>= 1) {
#pragma unroll
    for (int q = 0; q < N; ++q) {
      const int t = j[q] + step;
      const float th = s_thr[min(t, K) - 1];
      if (t <= K && x[q] >= th) j[q] = t;
    }
  }
}

// grid (blocks per sample, B).  hist: B x [neg_0 .. neg_K, pos_0 .. pos_K] uint32, zeroed before the launch.
__global__ void __launch_bounds__(CONF_THREADS) mask_confusion_kernel(const float* __restrict__ pred,
                                                                      const uint8_t* __restrict__ gt,
                                                                      const float* __restrict__ thr, int K, int top,
                                                                      unsigned* __restrict__ hist, long long hw) {
  __shared__ float s_thr[CONF_MAX_THR];
  __shared__ unsigned s_hist[2 * (CONF_MAX_THR + 1)];
  const int nbins = 2 * (K + 1);
  for (int i = threadIdx.x; i < K; i += blockDim.x) s_thr[i] = thr[i];
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) s_hist[i] = 0u;
  __syncthreads();

  // pred and gt have 16-byte aligned bases and the same element offset, so a sample that starts misaligned (h*w % 4 != 0)
  // has the same scalar head in both; the body is float4 + 4-byte loads.
  const long long base = (long long)blockIdx.y * hw;
  const long long head = min((long long)((-base) & 3), hw);
  const long long n4 = (hw - head) >> 2;
  const float4* p4 = reinterpret_cast<const float4*>(pred + base + head);
  const unsigned* g4 = reinterpret_cast<const unsigned*>(gt + base + head);
  const long long stride = (long long)gridDim.x * blockDim.x;
  // the trip count is uniform over the block: every lane reaches every conf_add
  for (long long i0 = (long long)blockIdx.x * blockDim.x; i0 < n4; i0 += stride) {
    const long long i = i0 + threadIdx.x;
    const bool ok = i < n4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    unsigned lab = 0;
    if (ok) {
      v = __ldg(p4 + i);
      lab = __ldg(g4 + i);
    }
    const float x[4] = {v.x, v.y, v.z, v.w};
    int j[4];
    conf_bins<4>(s_thr, K, top, x, j);
#pragma unroll
    for (int q = 0; q < 4; ++q)
      conf_add(s_hist, ok ? (((lab >> (8 * q)) & 0xffu) ? K + 1 : 0) + j[q] : -1);
  }
  if (blockIdx.x == 0) {   // the scalar head (< 4 pixels) and tail (< 4 pixels) of the sample
    const long long tail0 = head + 4 * n4, t = threadIdx.x;
    const long long e = t < head ? t : (t >= 4 && tail0 + (t - 4) < hw ? tail0 + (t - 4) : -1);
    const float x[1] = {e >= 0 ? pred[base + e] : 0.f};
    int j[1];
    conf_bins<1>(s_thr, K, top, x, j);
    conf_add(s_hist, e >= 0 ? (gt[base + e] ? K + 1 : 0) + j[0] : -1);
  }
  __syncthreads();
  unsigned* h = hist + (long long)blockIdx.y * nbins;
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) {
    const unsigned c = s_hist[i];
    if (c) atomicAdd(h + i, c);
  }
}

// One block per sample: TP_k = sum_{j > k} pos_j, FP_k = sum_{j > k} neg_j, FN_k = P - TP_k, TN_k = N - FP_k.
// Thread t owns a contiguous run of bins; a suffix scan over the threads' sums gives each run what lies above it.
__global__ void __launch_bounds__(CONF_THREADS) mask_confusion_finish_kernel(const unsigned* __restrict__ hist, int K,
                                                                             long long* __restrict__ counts) {
  __shared__ unsigned s_neg[CONF_THREADS], s_pos[CONF_THREADS];
  const int t = threadIdx.x, nb = K + 1;
  const unsigned* neg = hist + (long long)blockIdx.x * 2 * nb;
  const unsigned* pos = neg + nb;
  const int per = (nb + CONF_THREADS - 1) / CONF_THREADS;
  const int lo = min(t * per, nb), hi = min(lo + per, nb);
  unsigned sn = 0, sp = 0;
  for (int j = lo; j < hi; ++j) { sn += neg[j]; sp += pos[j]; }
  s_neg[t] = sn; s_pos[t] = sp;
  __syncthreads();
  for (int d = 1; d < CONF_THREADS; d <<= 1) {   // inclusive suffix sums over the threads
    const unsigned an = t + d < CONF_THREADS ? s_neg[t + d] : 0u, ap = t + d < CONF_THREADS ? s_pos[t + d] : 0u;
    __syncthreads();
    s_neg[t] += an; s_pos[t] += ap;
    __syncthreads();
  }
  const long long N = s_neg[0], P = s_pos[0];
  long long fp = t + 1 < CONF_THREADS ? s_neg[t + 1] : 0u, tp = t + 1 < CONF_THREADS ? s_pos[t + 1] : 0u;
  long long* out = counts + (long long)blockIdx.x * K * 4;
  for (int j = hi - 1; j >= lo; --j) {
    if (j < K) {
      out[4 * j + 0] = tp;
      out[4 * j + 1] = fp;
      out[4 * j + 2] = P - tp;
      out[4 * j + 3] = N - fp;
    }
    tp += pos[j]; fp += neg[j];
  }
}
