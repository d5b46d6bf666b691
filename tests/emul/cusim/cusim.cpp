// cusim.cpp -- TEST INFRASTRUCTURE.  The scheduler behind tests/emul/cusim/cuda_runtime.h: the
// threads of a block as fibers, barriers and warp collectives as rendezvous.
#include <ucontext.h>

#include <algorithm>
#include <vector>

#include "cuda_runtime.h"

// AddressSanitizer builds (CUSIM_ASAN=1, tests/emul/cusim_build.py): tell it about the stack switches
#if defined(__SANITIZE_ADDRESS__)
#include <sanitizer/common_interface_defs.h>
#define CUSIM_ASAN_START(save, bottom, size) __sanitizer_start_switch_fiber(save, bottom, size)
#define CUSIM_ASAN_FINISH(save, bottom, size) __sanitizer_finish_switch_fiber(save, bottom, size)
#else
#define CUSIM_ASAN_START(save, bottom, size) ((void) 0)
#define CUSIM_ASAN_FINISH(save, bottom, size) ((void) 0)
#endif

namespace cusim {

thread_local ThreadCtx *T = nullptr;
thread_local BlockCtx *B = nullptr;

namespace {

constexpr size_t STACK_BYTES = 256 * 1024;

struct Warp {
  uint64_t vals[32];       // deposits of the collective being formed
  uint64_t snap[32];       // values of the last completed collective, while its lanes read them
  uint32_t arrived = 0;    // lanes that have deposited
  uint32_t mask = 0;       // mask the first depositor named
  uint32_t snap_arrived = 0;
  uint32_t readers = 0;    // lanes that have not yet released the snapshot
  uint32_t exited = 0;     // lanes whose thread has left the kernel
  uint64_t gen = 0;        // completed collectives
};

struct Block {             // a block that is alive: one at a time, or the whole grid of a cooperative launch
  BlockCtx ctx;
  std::vector<Warp> warps;
  uint32_t bar_arrived = 0, live = 0;
  uint64_t bar_gen = 0;
};

struct Fiber {
  ucontext_t ctx;
  ThreadCtx t;
  uint32_t block = 0, rank = 0;   // index into blocks, thread rank inside the block
  bool done = true;
  void *asan_fake = nullptr;      // the sanitizer's bookkeeping while this fiber is switched out
};

thread_local std::vector<Fiber> fibers;
struct Stacks : std::vector<char *> {      // fiber stacks of this host thread, freed when it ends
  ~Stacks() {
    for (char *p : *this) free(p);
  }
};
thread_local Stacks stacks;
thread_local std::vector<Block> blocks;
thread_local ucontext_t sched_ctx;
thread_local const std::function<void()> *body = nullptr;
thread_local uint32_t cur = 0, total_live = 0;
thread_local uint64_t progress = 0;        // bumped whenever any thread changes the state of a wait
thread_local uint32_t grid_arrived = 0;
thread_local uint64_t grid_gen = 0;
thread_local void *sched_asan_fake = nullptr;
thread_local const void *sched_stack_bottom = nullptr;
thread_local size_t sched_stack_size = 0;

void yield() {
  Fiber &f = fibers[cur];
  CUSIM_ASAN_START(&f.asan_fake, sched_stack_bottom, sched_stack_size);
  swapcontext(&f.ctx, &sched_ctx);
  CUSIM_ASAN_FINISH(fibers[cur].asan_fake, &sched_stack_bottom, &sched_stack_size);
}

void fiber_main() {
  CUSIM_ASAN_FINISH(nullptr, &sched_stack_bottom, &sched_stack_size);
  (*body)();
  Fiber &f = fibers[cur];
  f.done = true;
  Block &b = blocks[f.block];
  b.live--;
  total_live--;
  b.warps[f.rank >> 5].exited |= 1u << (f.rank & 31u);
  progress++;
  CUSIM_ASAN_START(nullptr, sched_stack_bottom, sched_stack_size);     // this fiber does not come back
  swapcontext(&f.ctx, &sched_ctx);
}

[[noreturn]] void die(const char *what) {
  const Fiber &f = fibers[cur];
  const BlockCtx &c = blocks[f.block].ctx;
  fprintf(stderr, "cusim: %s (block %u,%u thread %u)\n", what, c.bid.x, c.bid.y, f.rank);
  abort();
}

// Order in which the threads get their turns.  CUSIM_ORDER = 0 (default): ascending; 1: descending;
// any other number: a pseudo-random order per pass, seeded by it.  Results must not depend on it:
// between two rendezvous a thread may only touch what no other thread touches.
uint64_t order_mode = [] {
  const char *e = getenv("CUSIM_ORDER");
  return e != nullptr ? (uint64_t) strtoull(e, nullptr, 10) : 0ull;
}();
uint64_t order_seed() { return order_mode; }
thread_local uint64_t rng_state = 0;
uint32_t next_rand() {
  rng_state = rng_state * 6364136223846793005ull + 1442695040888963407ull;
  return (uint32_t) (rng_state >> 33);
}

// fibers [0, n) are set up; give them turns until all have left the kernel
void schedule(uint32_t n) {
  const uint64_t mode = order_seed();
  std::vector<uint32_t> perm(n);
  for (uint32_t i = 0; i < n; i++) perm[i] = mode == 1 ? n - 1 - i : i;
  if (mode > 1 && rng_state == 0) rng_state = mode;
  while (total_live) {
    const uint64_t before = progress;
    if (mode > 1)
      for (uint32_t i = n; i > 1; i--) std::swap(perm[i - 1], perm[next_rand() % i]);
    for (uint32_t k = 0; k < n; k++) {
      const uint32_t t = perm[k];
      if (fibers[t].done) continue;
      cur = t;
      T = &fibers[t].t;
      B = &blocks[fibers[t].block].ctx;
      CUSIM_ASAN_START(&sched_asan_fake, stacks[t], STACK_BYTES);
      swapcontext(&sched_ctx, &fibers[t].ctx);
      CUSIM_ASAN_FINISH(sched_asan_fake, nullptr, nullptr);
      T = nullptr;
    }
    if (total_live && progress == before)
      die("deadlock: every thread waits at a barrier or collective that cannot complete");
  }
}

void prepare(uint32_t n) {
  if (fibers.size() < n) fibers.resize(n);
  while (stacks.size() < n) stacks.push_back((char *) malloc(STACK_BYTES));
}

void start_fiber(uint32_t idx, uint32_t block, uint32_t rank, dim3 blk) {
  Fiber &f = fibers[idx];
  f.done = false;
  f.block = block;
  f.rank = rank;
  f.t.tid = uint3{rank % blk.x, (rank / blk.x) % blk.y, rank / (blk.x * blk.y)};
  getcontext(&f.ctx);
  f.ctx.uc_stack.ss_sp = stacks[idx];
  f.ctx.uc_stack.ss_size = STACK_BYTES;
  f.ctx.uc_link = &sched_ctx;
  makecontext(&f.ctx, fiber_main, 0);
}

void init_block(Block &b, uint3 bid, dim3 blk, dim3 grid, void *dyn, uint32_t nthreads) {
  b.ctx.bid = bid;
  b.ctx.bdim = blk;
  b.ctx.gdim = grid;
  b.ctx.dyn_smem = dyn;
  b.warps.assign((nthreads + 31) / 32, Warp());
  if (nthreads & 31u) b.warps.back().exited = ~0u << (nthreads & 31u);   // lanes that do not exist
  b.bar_arrived = 0;
  b.bar_gen = 0;
  b.live = nthreads;
}

}  // namespace

void set_order(uint64_t mode) {
  order_mode = mode;
  rng_state = 0;
}

void block_barrier() {
  Block &b = blocks[fibers[cur].block];
  const uint64_t gen = b.bar_gen;
  b.bar_arrived++;
  progress++;
  for (;;) {
    if (b.bar_gen != gen) break;
    if (b.bar_arrived >= b.live) {        // threads that left the kernel do not hold the barrier up
      b.bar_arrived = 0;
      b.bar_gen++;
      progress++;
      break;
    }
    yield();
  }
}

void grid_barrier() {
  const uint64_t gen = grid_gen;
  grid_arrived++;
  progress++;
  for (;;) {
    if (grid_gen != gen) break;
    if (grid_arrived >= total_live) {
      grid_arrived = 0;
      grid_gen++;
      progress++;
      break;
    }
    yield();
  }
}

const uint64_t *warp_collect(uint32_t mask, uint64_t v, uint32_t *arrived_out) {
  const Fiber &f = fibers[cur];
  Warp &w = blocks[f.block].warps[f.rank >> 5];
  const uint32_t bit = 1u << (f.rank & 31u);
  if (!(mask & bit)) die("a lane calls a warp collective with a mask that does not name it");
  while (w.readers) yield();              // the previous collective is still being read
  if (w.arrived == 0) w.mask = mask;
  else if (w.mask != mask) die("lanes of one warp meet in a collective with different masks");
  w.vals[f.rank & 31u] = v;
  w.arrived |= bit;
  progress++;
  const uint64_t gen = w.gen;
  for (;;) {
    if (w.gen != gen) break;
    if (((w.arrived | w.exited) & mask) == mask) {
      memcpy(w.snap, w.vals, sizeof(w.snap));
      w.snap_arrived = w.arrived;
      w.readers = w.arrived;
      w.arrived = 0;
      w.gen++;
      progress++;
      break;
    }
    yield();
  }
  *arrived_out = w.snap_arrived;
  return w.snap;
}

void warp_release() {
  const Fiber &f = fibers[cur];
  Warp &w = blocks[f.block].warps[f.rank >> 5];
  w.readers &= ~(1u << (f.rank & 31u));
  progress++;
}

void run_grid(dim3 grid, dim3 blk, size_t smem, const std::function<void()> &kernel_body) {
  if (T != nullptr) die("a kernel launch from inside a kernel");
  const uint32_t nthreads = blk.x * blk.y * blk.z;
  if (nthreads == 0 || nthreads > 1024) {
    fprintf(stderr, "cusim: block of %u threads\n", nthreads);
    abort();
  }
  prepare(nthreads);
  std::vector<uint64_t> dyn((smem + 15) / 8 + 2);
  void *dyn_p = (void *) (((uintptr_t) dyn.data() + 15) & ~(uintptr_t) 15);
  body = &kernel_body;
  blocks.resize(1);
  for (uint32_t bz = 0; bz < grid.z; bz++)
    for (uint32_t by = 0; by < grid.y; by++)
      for (uint32_t bx = 0; bx < grid.x; bx++) {
        init_block(blocks[0], uint3{bx, by, bz}, blk, grid, dyn_p, nthreads);
        total_live = nthreads;
        for (uint32_t t = 0; t < nthreads; t++) start_fiber(t, 0, t, blk);
        schedule(nthreads);
      }
  B = nullptr;
  body = nullptr;
}

// every block of the grid alive at once (grid-wide barriers).  __shared__ is `static` in this model,
// i.e. shared by ALL blocks here: only kernels without static shared memory may be launched this way
// (true of the product's one cooperative kernel, k_fire_rounds_all).
void run_grid_coop(dim3 grid, dim3 blk, size_t smem, const std::function<void()> &kernel_body) {
  if (T != nullptr) die("a kernel launch from inside a kernel");
  const uint32_t nthreads = blk.x * blk.y * blk.z, nblocks = grid.x * grid.y * grid.z;
  if (nthreads == 0 || nthreads > 1024 || nblocks == 0 || (uint64_t) nblocks * nthreads > 16384) {
    fprintf(stderr, "cusim: cooperative grid of %u x %u threads\n", nblocks, nthreads);
    abort();
  }
  prepare(nblocks * nthreads);
  std::vector<std::vector<uint64_t>> dyn(nblocks, std::vector<uint64_t>((smem + 15) / 8 + 2));
  body = &kernel_body;
  blocks.resize(nblocks);
  total_live = nblocks * nthreads;
  grid_arrived = 0;
  for (uint32_t b = 0; b < nblocks; b++) {
    const uint3 bid{b % grid.x, (b / grid.x) % grid.y, b / (grid.x * grid.y)};
    init_block(blocks[b], bid, blk, grid, (void *) (((uintptr_t) dyn[b].data() + 15) & ~(uintptr_t) 15), nthreads);
    for (uint32_t t = 0; t < nthreads; t++) start_fiber(b * nthreads + t, b, t, blk);
  }
  schedule(nblocks * nthreads);
  B = nullptr;
  body = nullptr;
}

long long live_allocs = 0;
unsigned long long stream_syncs = 0;

}  // namespace cusim

// device and pinned allocations not yet freed, and host synchronisations (cudaStreamSynchronize) so
// far, of all contexts
extern "C" long long cusim_live_allocs() {
  return __atomic_load_n(&cusim::live_allocs, __ATOMIC_RELAXED);
}
extern "C" unsigned long long cusim_stream_syncs() {
  return __atomic_load_n(&cusim::stream_syncs, __ATOMIC_RELAXED);
}

// the order of the threads' turns from now on (see CUSIM_ORDER)
extern "C" void cusim_set_order(uint64_t mode) {
  cusim::set_order(mode);
}
