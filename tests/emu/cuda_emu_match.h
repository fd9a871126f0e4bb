// cuda_emu_match.h -- warp match and bit intrinsics for the SIMT emulator (cuda_emu.h), used ONLY by the CPU-side tests.
//
// TEST INFRASTRUCTURE, NOT A FALLBACK: included after cuda_emu.h when the kernel source is compiled with -DMDN_EMU
// (mdn_common.cuh).  The mask-evaluation kernel (mdn_metrics.cuh) aggregates its shared-memory histogram updates with
// __match_any_sync and counts a group with __popc / __ffs.
#pragma once

// lanes of the caller's warp holding the same value (all 32 lanes call it): one rendezvous, then each lane reads the
// values of its warp
static inline unsigned __match_any_sync(unsigned, int v) {
  mdn_emu::State& s = mdn_emu::st();
  s.xchg[s.cur] = (uint32_t)v;
  mdn_emu::yield_to_scheduler();
  const int w0 = s.cur & ~31;
  unsigned m = 0;
  for (int l = 0; l < 32; ++l) m |= (s.xchg[w0 + l] == (uint32_t)v) ? (1u << l) : 0u;
  mdn_emu::yield_to_scheduler();
  return m;
}
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __ffs(unsigned v) { return __builtin_ffs((int)v); }
