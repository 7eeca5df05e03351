// Fiber scheduler behind pmoc_emu.h -- TEST INFRASTRUCTURE ONLY.
#include "pmoc_emu.h"

#include <ucontext.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

namespace pmemu {
namespace {

constexpr size_t kStack = 256 * 1024;
constexpr size_t kMaxSmem = 227 * 1024;  // dynamic shared memory one block of sm_100 may opt in to
constexpr size_t kGuard = 8 * 1024;      // checked after every block: catches writes past the kernel's plan

struct Warp {
  alignas(16) unsigned char slot[2][32][16];
  int arrived = 0;
  unsigned gen = 0;
};

struct Fiber {
  ucontext_t uc;
  Ctx ctx;
  bool done = false;
  char* stack = nullptr;
};

struct Block {
  std::vector<Fiber> fibers;
  std::vector<Warp> warps;
  ucontext_t sched;
  int running = -1;
  int bar_arrived = 0;
  unsigned bar_gen = 0;
  const std::function<void()>* body = nullptr;
};

thread_local Block* t_blk = nullptr;

void yield_to_scheduler() { swapcontext(&t_blk->fibers[t_blk->running].uc, &t_blk->sched); }

void trampoline() {
  Block* b = t_blk;
  (*b->body)();
  b->fibers[b->running].done = true;
  yield_to_scheduler();
}

void run_block(Block& blk, long long bid, long long nblocks, int nthreads, char* smem,
               const std::function<void()>& body) {
  t_blk = &blk;
  blk.body = &body;
  blk.bar_arrived = 0;
  for (auto& w : blk.warps) { w.arrived = 0; w.gen = 0; }
  for (int t = 0; t < nthreads; ++t) {
    Fiber& f = blk.fibers[t];
    f.done = false;
    f.ctx = Ctx{t, nthreads, bid, nblocks, smem};
    getcontext(&f.uc);
    f.uc.uc_stack.ss_sp = f.stack;
    f.uc.uc_stack.ss_size = kStack;
    f.uc.uc_link = nullptr;
    makecontext(&f.uc, trampoline, 0);
  }
  int remaining = nthreads;
  while (remaining > 0) {
    for (int t = 0; t < nthreads; ++t) {
      Fiber& f = blk.fibers[t];
      if (f.done) continue;
      blk.running = t;
      swapcontext(&blk.sched, &f.uc);
      if (f.done) --remaining;
    }
  }
  t_blk = nullptr;
}

}  // namespace

Ctx* cur() { return &t_blk->fibers[t_blk->running].ctx; }

const unsigned char* exchange(const void* val, int bytes) {
  Block* b = t_blk;
  const int tid = b->fibers[b->running].ctx.tid;
  Warp& w = b->warps[tid >> 5];
  const unsigned g = w.gen;
  std::memcpy(w.slot[g & 1][tid & 31], val, bytes);
  if (++w.arrived == 32) {
    w.arrived = 0;
    w.gen = g + 1;
  } else {
    while (w.gen == g) yield_to_scheduler();
  }
  return &w.slot[g & 1][0][0];
}

void block_barrier() {
  Block* b = t_blk;
  const unsigned g = b->bar_gen;
  if (++b->bar_arrived == (int)b->fibers.size()) {
    b->bar_arrived = 0;
    b->bar_gen = g + 1;
  } else {
    while (b->bar_gen == g) yield_to_scheduler();
  }
}

void launch(long long grid, int block, size_t smem_bytes, const std::function<void()>& body) {
  if (smem_bytes > kMaxSmem) {
    std::fprintf(stderr, "pmemu: launch with %zu bytes of dynamic shared memory, more than one block can use\n", smem_bytes);
    std::abort();
  }
  if (block % 32 != 0) {
    std::fprintf(stderr, "pmemu: block size must be a multiple of 32\n");
    std::abort();
  }
  unsigned hw = std::thread::hardware_concurrency();
  const char* env = std::getenv("PMOC_EMU_THREADS");
  int nthr = env ? std::atoi(env) : (int)(hw ? hw : 1);
  if (nthr > grid) nthr = (int)grid;
  if (nthr < 1) nthr = 1;
  std::atomic<long long> next{0};
  auto worker = [&]() {
    Block blk;
    blk.fibers.resize(block);
    blk.warps.resize(block / 32);
    for (auto& f : blk.fibers) f.stack = (char*)std::malloc(kStack);
    // The device does not clear shared memory: NaN bytes make a read of a value nobody wrote show in the results.
    std::vector<unsigned char> smem(smem_bytes + kGuard);
    for (;;) {
      long long bid = next.fetch_add(1);
      if (bid >= grid) break;
      std::memset(smem.data(), 0xFF, smem.size());
      run_block(blk, bid, grid, block, reinterpret_cast<char*>(smem.data()), body);
      for (size_t i = smem_bytes; i < smem.size(); ++i)
        if (smem[i] != 0xFF) {
          std::fprintf(stderr, "pmemu: block %lld wrote shared memory byte %zu, past the %zu bytes launched with\n", bid,
                       i, smem_bytes);
          std::abort();
        }
    }
    for (auto& f : blk.fibers) std::free(f.stack);
  };
  if (nthr == 1) {
    worker();
  } else {
    std::vector<std::thread> pool;
    for (int i = 0; i < nthr; ++i) pool.emplace_back(worker);
    for (auto& t : pool) t.join();
  }
}

}  // namespace pmemu
