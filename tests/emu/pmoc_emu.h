// Warp-synchronous CPU emulator -- TEST INFRASTRUCTURE ONLY (never loaded by pymoc_b200).
//
// It lets the unit tests execute the *product kernel sources* (pymoc_b200/csrc/*.cu,
// compiled with g++ -DPMOC_EMU) on the build container, which has no GPU: every CUDA
// thread is a ucontext fiber, a block's fibers run round-robin on one OS thread, and the
// warp collectives (shuffles, ballot, reductions, barriers) rendezvous through a
// per-warp exchange buffer.  Blocks are distributed over OS threads.  It shares no
// code with the oracle and is not a fallback: the package raises if the CUDA library or a
// GPU is missing.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <functional>

namespace pmemu {

struct Ctx {  // what a fiber sees
  int tid, nthreads;
  long long bid, nblocks;
  char* smem;
};
Ctx* cur();
// Rendezvous of the calling fiber's warp: publishes `bytes` (<= 16) of `val`, waits for all 32
// lanes, returns a pointer to the 32 published slots (16-byte stride), valid until the next one.
const unsigned char* exchange(const void* val, int bytes);
void block_barrier();
// Aborts when smem_bytes exceeds what one block of the device may use: the device would refuse that launch, so the
// library must have refused it before.
void launch(long long grid, int block, size_t smem_bytes, const std::function<void()>& body);

}  // namespace pmemu

namespace rt {
inline int lane() { return pmemu::cur()->tid & 31; }
inline int warp_in_block() { return pmemu::cur()->tid >> 5; }
inline int warps_per_block() { return pmemu::cur()->nthreads >> 5; }
inline long long block_idx() { return pmemu::cur()->bid; }
inline double* smem() { return reinterpret_cast<double*>(pmemu::cur()->smem); }

template <class T>
inline T xchg(T v, int src) {
  const unsigned char* all = pmemu::exchange(&v, sizeof(T));
  T out;
  std::memcpy(&out, all + 16 * (src & 31), sizeof(T));
  return out;
}
inline double shfl(double v, int src) { return xchg(v, src); }
inline double shfl_up(double v, int d) { int l = lane(); return xchg(v, l >= d ? l - d : l); }
inline double shfl_down(double v, int d) { int l = lane(); return xchg(v, l + d < 32 ? l + d : l); }
inline double shfl_xor(double v, int m) { return xchg(v, lane() ^ m); }
inline int shfl_i(int v, int src) { return xchg(v, src); }
inline double shfl_w(double v, int src, int w) { int l = lane(); return xchg(v, (l & ~(w - 1)) + (src & (w - 1))); }
inline double shfl_up_w(double v, int d, int w) { int l = lane(), s = l & (w - 1); return xchg(v, s >= d ? l - d : l); }
inline double shfl_down_w(double v, int d, int w) { int l = lane(), s = l & (w - 1); return xchg(v, s + d < w ? l + d : l); }
inline unsigned ballot(bool p) {
  int v = p ? 1 : 0;
  const unsigned char* all = pmemu::exchange(&v, sizeof(int));
  unsigned m = 0;
  for (int l = 0; l < 32; ++l) {
    int x;
    std::memcpy(&x, all + 16 * l, sizeof(int));
    if (x) m |= 1u << l;
  }
  return m;
}
inline int max_i(int v) {
  const unsigned char* all = pmemu::exchange(&v, sizeof(int));
  int m = v;
  for (int l = 0; l < 32; ++l) {
    int x;
    std::memcpy(&x, all + 16 * l, sizeof(int));
    if (x > m) m = x;
  }
  return m;
}
inline int min_i(int v) { return -max_i(-v); }
inline unsigned min_u(unsigned v) {
  const unsigned char* all = pmemu::exchange(&v, sizeof(unsigned));
  unsigned m = v;
  for (int l = 0; l < 32; ++l) {
    unsigned x;
    std::memcpy(&x, all + 16 * l, sizeof(unsigned));
    if (x < m) m = x;
  }
  return m;
}
inline void syncwarp() { int z = 0; (void)pmemu::exchange(&z, sizeof(int)); }
inline void syncblock() { pmemu::block_barrier(); }
}  // namespace rt
