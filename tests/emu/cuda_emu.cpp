// cuda_emu.cpp -- fiber scheduler of the SIMT emulator (TEST INFRASTRUCTURE ONLY, see cuda_emu.h)
#include "cuda_emu.h"

namespace emu {
Block* g_block = nullptr;
uint3_emu threadIdx_, blockIdx_, blockDim_, gridDim_;
long long g_event_serial = 0, g_live_events = 0;
static const size_t kStack = 256 * 1024;

static void switch_to(int next) {
  Block* B = g_block;
  const int prev = B->cur;
  B->cur = next;
  threadIdx_.x = (unsigned)next;
  if (prev == next) return;
  swapcontext(&B->fibers[prev].ctx, &B->fibers[next].ctx);
  threadIdx_.x = (unsigned)B->cur;
}

void yield() {
  Block* B = g_block;
  int n = B->cur;
  for (int k = 0; k < B->nthreads; ++k) {
    n = (n + 1) % B->nthreads;
    if (!B->fibers[n].done) break;
  }
  const int me = B->cur;
  if (n == me) return;
  switch_to(n);
  threadIdx_.x = (unsigned)me;
}

void warp_barrier() {
  Block* B = g_block;
  const int me = B->cur;
  const int w = me / 32;
  const int gen = B->warp_gen[w];
  if (++B->warp_arrived[w] == warp_nthreads(w)) {
    B->warp_arrived[w] = 0;
    B->warp_gen[w]++;
    return;
  }
  while (B->warp_gen[w] == gen) yield();
  threadIdx_.x = (unsigned)me;
}

void block_barrier() {
  Block* B = g_block;
  const int me = B->cur;
  const int gen = B->block_gen;
  if (++B->block_arrived == B->nthreads) {
    B->block_arrived = 0;
    B->block_gen++;
    return;
  }
  while (B->block_gen == gen) yield();
  threadIdx_.x = (unsigned)me;
}

static void fiber_entry() {
  Block* B = g_block;
  B->body();
  B->fibers[B->cur].done = true;
  // hand control to any unfinished fiber, else back to main
  for (;;) {
    int n = -1;
    for (int k = 1; k <= B->nthreads; ++k) {
      const int c = (B->cur + k) % B->nthreads;
      if (!B->fibers[c].done) { n = c; break; }
    }
    if (n < 0) {
      setcontext(&B->main);
    } else {
      B->cur = n;
      threadIdx_.x = (unsigned)n;
      setcontext(&B->fibers[n].ctx);
    }
  }
}

void launch(dim3 grid, dim3 block, size_t smem_bytes, const std::function<void()>& body) {
  Block B;
  B.nthreads = (int)block.x;
  B.body = body;
  B.smem.assign(smem_bytes + 64, 0);
  B.fibers.resize(B.nthreads);
  for (auto& f : B.fibers) f.stack = (char*)std::malloc(kStack);
  g_block = &B;
  blockDim_.x = block.x; blockDim_.y = blockDim_.z = 1;
  gridDim_.x = grid.x; gridDim_.y = gridDim_.z = 1;
  threadIdx_.y = threadIdx_.z = 0;
  blockIdx_.y = blockIdx_.z = 0;
  for (unsigned b = 0; b < grid.x; ++b) {
    blockIdx_.x = b;
    B.block_arrived = 0;
    for (int w = 0; w < 64; ++w) B.warp_arrived[w] = 0;
    for (int t = 0; t < B.nthreads; ++t) {
      Fiber& f = B.fibers[t];
      f.done = false;
      getcontext(&f.ctx);
      f.ctx.uc_stack.ss_sp = f.stack;
      f.ctx.uc_stack.ss_size = kStack;
      f.ctx.uc_link = nullptr;
      makecontext(&f.ctx, (void (*)())fiber_entry, 0);
    }
    B.cur = 0;
    threadIdx_.x = 0;
    swapcontext(&B.main, &B.fibers[0].ctx);
  }
  for (auto& f : B.fibers) std::free(f.stack);
  g_block = nullptr;
}
}  // namespace emu

// emulator build only (not part of include/idocp_b200.h): lets the tests check that destroying a handle releases its events
extern "C" int idocp_b200_emu_live_events(void) { return static_cast<int>(emu::g_live_events); }
