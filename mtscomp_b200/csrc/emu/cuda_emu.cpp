// cuda_emu.cpp — fiber scheduler for cuda_emu.h (development tool, see the header's banner).
#include "cuda_emu.h"

#include <mutex>
#include <unordered_map>

thread_local uint3 threadIdx, blockIdx;
thread_local dim3 blockDim, gridDim;

namespace emu {

thread_local Block* g_blk = nullptr;
thread_local unsigned char* g_dyn_smem = nullptr;
thread_local int g_last_error = 0;

static std::mutex g_attr_mu;
static std::unordered_map<const void*, size_t> g_max_dyn_smem;   // kernel -> its MaxDynamicSharedMemorySize

int set_max_dyn_smem(const void* fn, int bytes) {
  if (bytes < 0 || (size_t)bytes > kDynSmemOptin) return cudaErrorInvalidValue;
  std::lock_guard<std::mutex> g(g_attr_mu);
  g_max_dyn_smem[fn] = (size_t)bytes;
  return 0;
}

static size_t max_dyn_smem(const void* fn) {
  std::lock_guard<std::mutex> g(g_attr_mu);
  auto it = g_max_dyn_smem.find(fn);
  return it == g_max_dyn_smem.end() ? kDynSmemDefault : it->second;
}

asm(R"(
.text
.globl emu_switch
.type emu_switch,@function
emu_switch:
  pushq %rbp
  pushq %rbx
  pushq %r12
  pushq %r13
  pushq %r14
  pushq %r15
  movq %rsp, (%rdi)
  movq %rsi, %rsp
  popq %r15
  popq %r14
  popq %r13
  popq %r12
  popq %rbx
  popq %rbp
  ret
.size emu_switch,.-emu_switch
)");

static const size_t kStack = 96 * 1024;

static void fiber_entry() {
  Block* b = g_blk;
  (*b->body)();
  b->done[b->cur] = 1;
  b->alive--;
  if (b->bar_count > 0 && b->bar_count == (int)b->alive) __emu_release_block(b);
  yield();
  abort();  // a finished fiber is never resumed
}

static void set_tid(unsigned t, dim3 bd) {
  threadIdx.x = t % bd.x;
  threadIdx.y = (t / bd.x) % bd.y;
  threadIdx.z = t / (bd.x * bd.y);
}

static void run_block(Block& b, dim3 bd, const std::function<void()>& body) {
  unsigned n = bd.x * bd.y * bd.z;
  b.nthreads = b.alive = n;
  b.body = &body;
  b.bar_count = 0; b.bar_acc = 0; b.bar_and = 1;
  for (int i = 0; i < 16; i++) b.nb_count[i] = 0;
  if (b.stacks.size() < n) {
    size_t old = b.stacks.size();
    b.stacks.resize(n);
    for (size_t i = old; i < n; i++) b.stacks[i] = (char*)aligned_alloc(64, kStack);
  }
  b.sp.assign(n, nullptr);
  b.done.assign(n, 0);
  b.warps.assign((n + 31) / 32, Warp());
  for (unsigned t = 0; t < n; t++) {
    uintptr_t top = ((uintptr_t)b.stacks[t] + kStack) & ~(uintptr_t)15;
    void** s = (void**)top;
    s[-1] = nullptr;
    s[-2] = (void*)&fiber_entry;
    for (int i = 3; i <= 8; i++) s[-i] = nullptr;
    b.sp[t] = (void*)(s - 8);
  }
  g_blk = &b;
  unsigned remaining = n;
  unsigned long spins = 0;
  while (remaining) {
    unsigned progressed = 0;
    for (unsigned t = 0; t < n; t++) {
      if (b.done[t] == 2) continue;
      b.cur = (int)t;
      set_tid(t, bd);
      emu_switch(&b.sched_sp, b.sp[t]);
      if (b.done[t] == 1) { b.done[t] = 2; remaining--; progressed++; }
    }
    if (!progressed && ++spins > 50000000ul) { fprintf(stderr, "emu: deadlock suspected\n"); abort(); }
    if (progressed) spins = 0;
  }
  g_blk = nullptr;
}

void launch(const void* fn, dim3 grid, dim3 block, size_t smem, const std::function<void()>& body) {
  if (smem > kDynSmemOptin || smem > max_dyn_smem(fn)) { g_last_error = cudaErrorInvalidValue; return; }
  size_t nblocks = (size_t)grid.x * grid.y * grid.z;
  if (nblocks == 0) return;
  unsigned nthr = std::thread::hardware_concurrency();
  const char* e = getenv("MTS_EMU_THREADS");
  if (e) nthr = (unsigned)atoi(e);
  if (nthr < 1) nthr = 1;
  if (nthr > nblocks) nthr = (unsigned)nblocks;
  std::atomic<size_t> next(0);
  auto worker = [&]() {
    Block b;
    std::vector<unsigned char> dyn(smem + 64);
    g_dyn_smem = (unsigned char*)(((uintptr_t)dyn.data() + 15) & ~(uintptr_t)15);
    gridDim = grid;
    blockDim = block;
    for (;;) {
      size_t i = next.fetch_add(1);
      if (i >= nblocks) break;
      blockIdx.x = (unsigned)(i % grid.x);
      blockIdx.y = (unsigned)((i / grid.x) % grid.y);
      blockIdx.z = (unsigned)(i / ((size_t)grid.x * grid.y));
      run_block(b, block, body);
    }
    for (char* s : b.stacks) free(s);
    g_dyn_smem = nullptr;
  };
  if (nthr == 1) { worker(); return; }
  std::vector<std::thread> th;
  for (unsigned i = 0; i < nthr; i++) th.emplace_back(worker);
  for (auto& t : th) t.join();
}

}  // namespace emu
