// capi.cu — the C-ABI shim (include/mtscomp_b200.h) over the sm_100a kernels.  Host-side orchestration only: table
// building, scratch management, launches on one stream, copies.  No codec arithmetic happens on the host.
#include "../../include/mtscomp_b200.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "deflate.cuh"
#include "inflate.cuh"
#include "inflate_par.cuh"
#include "inflate_seg.cuh"
#include "transform.cuh"

using namespace mts;

namespace {

thread_local std::string g_err;

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  bool host = false;
  int ensure(size_t n) {
    if (n <= cap) return 0;
    release();
    size_t want = n + n / 8 + 4096;
    cudaError_t e = host ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
    if (e != cudaSuccess) { p = nullptr; cap = 0; cudaGetLastError(); return -1; }
    cap = want;
    return 0;
  }
  void release() {
    if (p) { if (host) cudaFreeHost(p); else cudaFree(p); }
    p = nullptr; cap = 0;
  }
};

static const int INDEX_TAIL = 16;                  // {segment bytes, k, magic, sum}: the end of both index formats (deflate.cuh)
static const int INDEX_TAIL_V2 = 24;               // the second format has {sub-block bytes, step bytes} before it

}  // namespace

struct mtsb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  std::string err;
  // params
  long long par_inflate = 1;   // decode index-less zlib streams block-parallel (inflate_par.cuh)
  long long par_indexed = 1;    // indexed segments of GPU-written chunks also go through the block kernels
  long long par_cells = -1;     // index-less streams: -1 by stream count, 1 = blocks resolved in parallel into cells, 0 = chain of tiles
  long long par_lz_wide = -1;   // LZ resolve kernel shape: -1 by stream count, 1 = 1024-thread CTAs, 0 = 256-thread CTAs
  long long par_batch_bytes = 2ll << 30;   // host-buffer sub-batch of index-less chunks (output bytes): large enough to amortise the block search
  long long par_stats[4] = {0, 0, 0, 0};   // last call: survivors, candidates, chained blocks, streams resumed
  long long seg_bytes = 262144, batch_bytes = 2ll << 30, host_batch_bytes = 512ll << 20, write_index = 1;
  cudaStream_t copy_in = nullptr, copy_out = nullptr;   // H2D / D2H streams of the host-buffer paths
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr}, ev_done = nullptr;
  int lz_ctas_per_sm = 2;
  // device scratch
  Buf d_pstreams, d_surv, d_cand, d_pcount, d_tokens, d_cells, d_ptab, d_plist, d_pbad;   // block-parallel inflate scratch
  std::vector<uint32_t> lz_adler;   // per segment of the current sub-batch: adler32 left by par_lz_kernel ...
  std::vector<char> lz_adler_have;  // ... where it produced the whole stream
  Buf d_pieces;
  long long par_single_pass = 1;   // par_block_kernel keeps the tokens of its counting pass (see par_decode)
  Buf d_segv2, d_btab, d_subout;                                                          // indexed (second format) segments
  long long seg_v2 = 1;         // indexed segments of the second format go through seg_tokens / seg_resolve
  bool ignore_index = false;    // (internal) decode every chunk as a plain zlib stream: the retry of chunks whose index misled
  Buf d_raw, d_raw2, d_out2, d_comp2, d_T, d_tok, d_hist, d_codes, d_hdrs, d_tab, d_so, d_seg_adler, d_chunk_adler, d_chunk_off, d_out,
      d_partial, d_comp, d_status, d_tadler, d_gather, d_subabs, d_subtok, d_invstate, d_invcells;
  int inv_cells_isz = 0;           // element size of the launch that last wrote the look-back cells
  unsigned inv_epoch = 0;          // epoch of the last inv_tile_kernel launch (tags its look-back cells)
  long long inv_order_block = 2;   // inv_tile_kernel: consecutive tiles of a chunk that get consecutive tickets
  long long inv_single_pass = 1;   // channel-major inverse transform in one pass (inv_tile_kernel); 0: tile sums + apply
  Buf h_tab, h_small;
  // timings
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  struct Span { int stage; cudaEvent_t a, b; };
  std::vector<Span> spans;
  float last_ms[8] = {0};
  long long launches = 0;
  bool attr_set = false;

  mtsb_ctx() { h_tab.host = true; h_small.host = true; }
  cudaEvent_t ev() {
    if (ev_used == ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e); }
    return ev_pool[ev_used++];
  }
  void begin(int stage) { Span s{stage, ev(), nullptr}; cudaEventRecord(s.a, stream); spans.push_back(s); }
  void end() { spans.back().b = ev(); cudaEventRecord(spans.back().b, stream); }
  void reset_timing() { ev_used = 0; spans.clear(); launches = 0; for (float& f : last_ms) f = 0; }
  void collect_timing() {
    for (auto& s : spans) {
      float ms = 0;
      if (s.b && cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) last_ms[s.stage] += ms;
    }
    float tot = 0;
    for (int i = 0; i < 7; i++) tot += last_ms[i];
    last_ms[7] = tot;
  }
};

namespace {

int fail(mtsb_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  g_err = buf;
  return code;
}

#define CK(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e__ = (call);                                                                        \
    if (e__ != cudaSuccess) return fail(c, MTSB_E_CUDA, "%s: %s", #call, cudaGetErrorString(e__)); \
  } while (0)
#define CKL()                                                                                                  \
  do {                                                                                                         \
    cudaError_t e__ = cudaGetLastError();                                                                      \
    if (e__ != cudaSuccess) return fail(c, MTSB_E_CUDA, "kernel launch (%s:%d): %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
  } while (0)
#define NEED(buf, n)                                                                       \
  do {                                                                                     \
    if ((buf).ensure(n)) return fail(c, MTSB_E_NOMEM, "cannot allocate %zu bytes for " #buf, (size_t)(n)); \
  } while (0)

int tile_rows(int nc, int isz, int extra_rows) {
  long long P = isz == 1 ? tile_pitch<uint8_t>(nc) : isz == 2 ? tile_pitch<uint16_t>(nc) : (nc | 1);
  long long tt = 98304 / (P * isz) - extra_rows;
  return (int)std::min<long long>(64, tt);
}
size_t tile_smem(int nc, int isz, int rows) {
  long long P = isz == 1 ? tile_pitch<uint8_t>(nc) : isz == 2 ? tile_pitch<uint16_t>(nc) : (nc | 1);
  return (size_t)(P * isz * rows);
}

#ifndef MTS_LZ_NT
#define MTS_LZ_NT 512
#endif
static const int LZ_NT = MTS_LZ_NT;   // threads (= units per step) of an lz77 CTA
#ifndef MTS_NO_SMEM_ASSERT
static_assert(2 * (LzSmem<1, LZ_NT>::total + 1024) <= 233472 && 2 * (LzSmem<2, LZ_NT>::total + 1024) <= 233472,
              "two lz77 CTAs must fit the 228 KB shared memory of an sm_100 SM");
#endif

int set_attrs(mtsb_ctx* c) {
  if (c->attr_set) return 0;
  CK(cudaFuncSetAttribute(fwd_transform_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(fwd_transform_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(fwd_transform_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(fwd_transform_kernel<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(fwd_transform_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(fwd_transform_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute((par_lz_kernel<1024, 16384>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PAR_LZ_MIRROR));
  CK(cudaFuncSetAttribute((par_lz_kernel<256, 4096>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PAR_LZ_MIRROR));
#define MTS_INV_ATTR(T) \
  CK(cudaFuncSetAttribute((inv_tile_kernel<T, 4, 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, 73728)); \
  CK(cudaFuncSetAttribute((inv_tile_kernel<T, 2, 2>), cudaFuncAttributeMaxDynamicSharedMemorySize, 73728)); \
  CK(cudaFuncSetAttribute((inv_tile_kernel<T, 1, 4>), cudaFuncAttributeMaxDynamicSharedMemorySize, 73728));
  MTS_INV_ATTR(uint8_t) MTS_INV_ATTR(uint16_t) MTS_INV_ATTR(uint32_t) MTS_INV_ATTR(uint64_t)
#undef MTS_INV_ATTR
#define MTS_FWD_ATTR(T) \
  CK(cudaFuncSetAttribute((fwd_tile_kernel<T, 4, 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, 73728)); \
  CK(cudaFuncSetAttribute((fwd_tile_kernel<T, 2, 2>), cudaFuncAttributeMaxDynamicSharedMemorySize, 73728)); \
  CK(cudaFuncSetAttribute((fwd_tile_kernel<T, 1, 4>), cudaFuncAttributeMaxDynamicSharedMemorySize, 73728));
  MTS_FWD_ATTR(uint8_t) MTS_FWD_ATTR(uint16_t) MTS_FWD_ATTR(uint32_t) MTS_FWD_ATTR(uint64_t)
  MTS_FWD_ATTR(float) MTS_FWD_ATTR(double)
#undef MTS_FWD_ATTR
  CK(cudaFuncSetAttribute(inv_apply_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(inv_apply_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(inv_apply_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(inv_apply_kernel<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
  CK(cudaFuncSetAttribute(lz77_kernel<1, LZ_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LzSmem<1, LZ_NT>::total));
  CK(cudaFuncSetAttribute(lz77_kernel<2, LZ_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LzSmem<2, LZ_NT>::total));
  CK(cudaFuncSetAttribute(lz77_kernel<1, LZ_NT>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  CK(cudaFuncSetAttribute(lz77_kernel<2, LZ_NT>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  CK(cudaFuncSetAttribute(par_block_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  CK(cudaFuncSetAttribute(seg_resolve_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  c->attr_set = true;
  return 0;
}

// Small host<->device table transfers on the compute stream are done by kernels over mapped pinned memory: a
// cudaMemcpyAsync would queue on the copy engines behind the large sub-batch transfers of the copy streams and stall
// the kernels (measured: the table upload only ran after the NEXT sub-batch's 256 MB upload).
__global__ void table_copy_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src, size_t n16) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}
int small_copy(mtsb_ctx* c, void* dst, const void* src, size_t bytes) {
  size_t n16 = (bytes + 15) / 16;
  if (!n16) return 0;
  unsigned grid = (unsigned)std::min<size_t>((n16 + 255) / 256, 64);
  MTS_LAUNCH(table_copy_kernel, dim3(grid), dim3(256), 0, c->stream, (uint4*)dst, (const uint4*)src, n16);
  c->launches++;
  CKL();
  return 0;
}

// ---------------------------------------------------------------- launches shared by several entry points
template <class T>
int launch_fwd_t(mtsb_ctx* c, const void* raw, void* tbuf, const ChunkDesc* d_cd, int n_chunks, int max_ns, int nc,
                 int flags) {
  if (!(flags & FLAG_ORDER_C) && nc <= 4 * INV_TILE_MAXT) {
    // channel-major output: TMA-staged tile of G runs of R rows (+ the row above), a thread owns J channels; at most
    // 70 KB of shared memory
    const int R = ColRun<T>::R;
    const int J = nc <= INV_TILE_MAXT ? 1 : nc <= 2 * INV_TILE_MAXT ? 2 : 4, G = 4 / J;
    const int TT = G * R;
    const int threads = (((nc + J - 1) / J) + 31) / 32 * 32;
    const size_t smem = 16 + (size_t)(TT + 1) * nc * sizeof(T) + 32;
    dim3 grid((max_ns + TT - 1) / TT, n_chunks);
    auto k = J == 1 ? fwd_tile_kernel<T, 4, 1> : J == 2 ? fwd_tile_kernel<T, 2, 2> : fwd_tile_kernel<T, 1, 4>;
    MTS_LAUNCH(k, grid, dim3(threads), smem, c->stream, (const T*)raw, (T*)tbuf, d_cd, nc, flags);
    c->launches++;
    CKL();
    return 0;
  }
  int TT = tile_rows(nc, sizeof(T), 1);
  if (TT < 1) return fail(c, MTSB_E_ARG, "n_channels=%d too large for the transform tile", nc);
  dim3 grid((max_ns + TT - 1) / TT, n_chunks);
  auto k = fwd_transform_kernel<T>;
  MTS_LAUNCH(k, grid, dim3(512), tile_smem(nc, sizeof(T), TT + 1), c->stream, (const T*)raw, (T*)tbuf, d_cd, nc, TT, flags);
  c->launches++;
  CKL();
  return 0;
}
int launch_fwd(mtsb_ctx* c, int isz, const void* raw, void* tbuf, const ChunkDesc* d_cd, int n_chunks, int max_ns,
               int nc, int flags) {
  if (flags & FLAG_FLOAT) {
    if (isz == 4) return launch_fwd_t<float>(c, raw, tbuf, d_cd, n_chunks, max_ns, nc, flags);
    if (isz == 8) return launch_fwd_t<double>(c, raw, tbuf, d_cd, n_chunks, max_ns, nc, flags);
    return fail(c, MTSB_E_ARG, "floating point itemsize %d not supported (4, 8)", isz);
  }
  switch (isz) {
    case 1: return launch_fwd_t<uint8_t>(c, raw, tbuf, d_cd, n_chunks, max_ns, nc, flags);
    case 2: return launch_fwd_t<uint16_t>(c, raw, tbuf, d_cd, n_chunks, max_ns, nc, flags);
    case 4: return launch_fwd_t<uint32_t>(c, raw, tbuf, d_cd, n_chunks, max_ns, nc, flags);
    case 8: return launch_fwd_t<uint64_t>(c, raw, tbuf, d_cd, n_chunks, max_ns, nc, flags);
  }
  return fail(c, MTSB_E_ARG, "itemsize %d not supported (1, 2, 4, 8)", isz);
}

template <class T>
int launch_inv_t(mtsb_ctx* c, const void* tbuf, void* out, const ChunkDesc* d_cd, int n_chunks, int max_ns, int nc,
                 int flags) {
  if (!(flags & FLAG_ORDER_C) && c->inv_single_pass && nc <= 4 * INV_TILE_MAXT) {
    // channel-major input: one pass, carries by decoupled look-back; a tile is G runs of R rows, a thread owns J
    // channels (G * J = 4 runs of 32 bytes in its registers), at most 64 KB of shared memory per tile
    const int R = ColRun<T>::R;
    const int J = nc <= INV_TILE_MAXT ? 1 : nc <= 2 * INV_TILE_MAXT ? 2 : 4, G = 4 / J;
    const int ob = (int)std::max<long long>(1, c->inv_order_block);
    const int TT = G * R, max_tiles = ((max_ns + TT - 1) / TT + ob - 1) / ob * ob;
    const int threads = (((nc + J - 1) / J) + 31) / 32 * 32;
    const size_t smem = 16 + 16 + (((size_t)TT * nc * sizeof(T) + 15) & ~(size_t)15) + 16;
    const size_t n_tiles = (size_t)n_chunks * max_tiles;
    const bool td = (flags & FLAG_TIME_DIFF) != 0;
    // look-back cells: tagged with the launch's epoch, so they are only cleared when the buffer is new or the epochs
    // are used up
    const size_t cells_bytes = td ? n_tiles * nc * inv_state_bytes<T>() + 256 : 256;
    const void* before = c->d_invcells.p;
    NEED(c->d_invcells, cells_bytes);
    // (a word of one element size can read as a valid one of another, and the 64-bit layout depends on the cell count)
    if (c->d_invcells.p != before || c->inv_epoch >= INV_EPOCH_MAX || c->inv_cells_isz != (int)sizeof(T) || sizeof(T) == 8) {
      CK(cudaMemsetAsync(c->d_invcells.p, 0, c->d_invcells.cap, c->stream));
      c->inv_epoch = 0;
      c->inv_cells_isz = (int)sizeof(T);
    }
    const unsigned epoch = ++c->inv_epoch;
    NEED(c->d_invstate, 64);
    CK(cudaMemsetAsync(c->d_invstate.p, 0, 64, c->stream));
    auto k = J == 1 ? inv_tile_kernel<T, 4, 1> : J == 2 ? inv_tile_kernel<T, 2, 2> : inv_tile_kernel<T, 1, 4>;
    MTS_LAUNCH(k, dim3((unsigned)n_tiles), dim3(threads), smem, c->stream, (const T*)tbuf, (T*)out, d_cd, n_chunks, nc,
               max_tiles, flags, ob, c->d_invcells.p, epoch, (unsigned*)c->d_invstate.p);
    c->launches++;
    CKL();
    return 0;
  }
  const bool fast = !(flags & (FLAG_ORDER_C | FLAG_SPATIAL_DIFF));
  int TT = fast ? 256 : tile_rows(nc, sizeof(T), 0);
  if (TT < 1) return fail(c, MTSB_E_ARG, "n_channels=%d too large for the transform tile", nc);
  int max_tiles = (max_ns + TT - 1) / TT;
  dim3 grid(max_tiles, n_chunks);
  T* partial = nullptr;
  if (flags & FLAG_TIME_DIFF) {
    NEED(c->d_partial, (size_t)n_chunks * max_tiles * nc * sizeof(T));
    partial = (T*)c->d_partial.p;
    auto k1 = inv_tile_sums_kernel<T>;
    MTS_LAUNCH(k1, grid, dim3(512), 0, c->stream, (const T*)tbuf, partial, d_cd, nc, TT, max_tiles, flags);
    CKL();
    auto k2 = inv_tile_scan_kernel<T>;
    MTS_LAUNCH(k2, dim3((nc + 255) / 256, n_chunks), dim3(256), 0, c->stream, partial, d_cd, nc, TT, max_tiles);
    CKL();
    c->launches += 2;
  }
  if (fast) {
    auto k3 = inv_cols_kernel<T>;
    MTS_LAUNCH(k3, dim3(max_tiles, (nc + 127) / 128, n_chunks), dim3(128), 0, c->stream, (const T*)tbuf, (T*)out, (const T*)partial, d_cd, nc, TT, max_tiles, flags);
  } else {
    auto k3 = inv_apply_kernel<T>;
    MTS_LAUNCH(k3, grid, dim3(512), tile_smem(nc, sizeof(T), TT), c->stream, (const T*)tbuf, (T*)out, (const T*)partial, d_cd, nc, TT, max_tiles, flags);
  }
  c->launches++;
  CKL();
  return 0;
}
// float32 / float64: sequential sums in the reference's order (transform.cuh); the spatial pass works on a scratch copy
template <class T>
int launch_inv_float(mtsb_ctx* c, const void* tbuf, void* out, const ChunkDesc* d_cd, int n_chunks, int max_ns, int nc,
                     int flags, size_t span_elems) {
  const T* in = (const T*)tbuf;
  if (flags & FLAG_SPATIAL_DIFF) {
    NEED(c->d_partial, span_elems * sizeof(T) + 256);
    auto k1 = inv_float_space_kernel<T>;
    MTS_LAUNCH(k1, dim3((max_ns + 127) / 128, n_chunks), dim3(128), 0, c->stream, in, (T*)c->d_partial.p, d_cd, nc, flags);
    CKL();
    c->launches++;
    in = (const T*)c->d_partial.p;
  }
  auto k2 = inv_float_time_kernel<T>;
  MTS_LAUNCH(k2, dim3((nc + 127) / 128, n_chunks), dim3(128), 0, c->stream, in, (T*)out, d_cd, nc, flags);
  CKL();
  c->launches++;
  return 0;
}

int launch_inv(mtsb_ctx* c, int isz, const void* tbuf, void* out, const ChunkDesc* d_cd, int n_chunks, int max_ns,
               int nc, int flags, size_t span_elems) {
  if (flags & FLAG_FLOAT) {
    if (isz == 4) return launch_inv_float<float>(c, tbuf, out, d_cd, n_chunks, max_ns, nc, flags, span_elems);
    if (isz == 8) return launch_inv_float<double>(c, tbuf, out, d_cd, n_chunks, max_ns, nc, flags, span_elems);
    return fail(c, MTSB_E_ARG, "floating point itemsize %d not supported (4, 8)", isz);
  }
  switch (isz) {
    case 1: return launch_inv_t<uint8_t>(c, tbuf, out, d_cd, n_chunks, max_ns, nc, flags);
    case 2: return launch_inv_t<uint16_t>(c, tbuf, out, d_cd, n_chunks, max_ns, nc, flags);
    case 4: return launch_inv_t<uint32_t>(c, tbuf, out, d_cd, n_chunks, max_ns, nc, flags);
    case 8: return launch_inv_t<uint64_t>(c, tbuf, out, d_cd, n_chunks, max_ns, nc, flags);
  }
  return fail(c, MTSB_E_ARG, "itemsize %d not supported (1, 2, 4, 8)", isz);
}

long long seg_size_for(const mtsb_ctx* c, long long ns, int itemsize, int flags) {
  // prefer whole channel runs ('F' order) so that segment boundaries coincide with the rows' seeds
  long long target = std::max<long long>(c->seg_bytes, 4096);
  long long run = ns * itemsize;
  long long s = target;
  if (!(flags & FLAG_ORDER_C) && run > 0 && run <= target) s = std::max<long long>(1, target / run) * run;
  s = std::min<long long>(s, 1ll << 30);
  return std::max<long long>(itemsize, s / itemsize * itemsize);   // whole elements: int16 units stay 2-byte aligned
}
long long stored_bound(long long m) { return m + 5 * ((m + 65534) / 65535); }
long long chunk_bound(const mtsb_ctx* c, long long raw, long long seg) {
  long long k = (raw + seg - 1) / seg, full = raw / seg, rem = raw - full * seg;
  long long b = 2 + full * stored_bound(seg) + (rem ? stored_bound(rem) : 0) + 6;
  if (c->write_index) b += 4 * (full * idx_n_sub(seg) + (rem ? idx_n_sub(rem) : 0)) + 4 * k + INDEX_TAIL_V2;
  return b;
}

bool valid_common(mtsb_ctx* c, int n_chunks, const long long* rows, int nc, int isz) {
  if (!c || n_chunks < 1 || !rows || nc < 1 || rows[0] != 0) return false;
  if (isz != 1 && isz != 2 && isz != 4 && isz != 8) return false;
  for (int i = 0; i < n_chunks; i++) {
    long long ns = rows[i + 1] - rows[i];
    if (ns < 1 || ns * nc * isz > 0x7fffffffll || ns > 0x7fffffffll) return false;
  }
  return true;
}

}  // namespace

// =============================================================================================== basic API
extern "C" {

int mtsb_version(void) { return 100; }

int mtsb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

mtsb_ctx* mtsb_create(int device_id, void* stream) {
  int n = mtsb_device_count();
  if (device_id < 0 || device_id >= n) { fail(nullptr, MTSB_E_CUDA, "no CUDA device %d (found %d)", device_id, n); return nullptr; }
  if (cudaSetDevice(device_id) != cudaSuccess) { fail(nullptr, MTSB_E_CUDA, "cudaSetDevice(%d) failed", device_id); return nullptr; }
  mtsb_ctx* c = new mtsb_ctx();
  c->device = device_id;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device_id) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
  if (stream) { c->stream = (cudaStream_t)stream; c->own_stream = false; }
  else {
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
      fail(nullptr, MTSB_E_CUDA, "cudaStreamCreate failed"); delete c; return nullptr;
    }
    c->own_stream = true;
  }
  if (cudaStreamCreateWithFlags(&c->copy_in, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->copy_out, cudaStreamNonBlocking) != cudaSuccess) {
    fail(nullptr, MTSB_E_CUDA, "cudaStreamCreate failed"); mtsb_destroy(c); return nullptr;
  }
  for (int i = 0; i < 2; i++) {
    cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming);
  }
  cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming);
  if (set_attrs(c)) { g_err = c->err; mtsb_destroy(c); return nullptr; }
  return c;
}

void mtsb_destroy(mtsb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  Buf* bufs[] = {&c->d_pstreams, &c->d_surv, &c->d_cand, &c->d_pcount, &c->d_tokens, &c->d_cells, &c->d_ptab, &c->d_plist, &c->d_pbad,
                 &c->d_segv2, &c->d_btab, &c->d_subout, &c->d_pieces,
                 &c->d_raw, &c->d_raw2, &c->d_out2, &c->d_comp2, &c->d_T, &c->d_tok, &c->d_hist, &c->d_codes, &c->d_hdrs, &c->d_tab, &c->d_so,
                 &c->d_seg_adler, &c->d_chunk_adler, &c->d_chunk_off, &c->d_out, &c->d_partial, &c->d_comp,
                 &c->d_status, &c->d_tadler, &c->d_gather, &c->d_subabs, &c->d_subtok, &c->d_invstate, &c->d_invcells, &c->h_tab, &c->h_small};
  for (Buf* b : bufs) b->release();
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  for (int i = 0; i < 2; i++) { if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]); if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]); }
  if (c->ev_done) cudaEventDestroy(c->ev_done);
  if (c->copy_in) cudaStreamDestroy(c->copy_in);
  if (c->copy_out) cudaStreamDestroy(c->copy_out);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

const char* mtsb_last_error(mtsb_ctx* c) { return c ? c->err.c_str() : g_err.c_str(); }

int mtsb_sync(mtsb_ctx* c) {
  if (!c) return MTSB_E_ARG;
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int mtsb_set_param(mtsb_ctx* c, const char* name, long long v) {
  if (!c || !name) return MTSB_E_ARG;
  std::string s(name);
  if (s == "seg_bytes") { if (v < 4096 || v > (1ll << 30)) return fail(c, MTSB_E_ARG, "seg_bytes out of range"); c->seg_bytes = v; }
  else if (s == "batch_bytes") { if (v < (1 << 20)) return fail(c, MTSB_E_ARG, "batch_bytes too small"); c->batch_bytes = v; }
  else if (s == "host_batch_bytes") { if (v < (1 << 20)) return fail(c, MTSB_E_ARG, "host_batch_bytes too small"); c->host_batch_bytes = v; }
  else if (s == "write_index") c->write_index = v ? 1 : 0;
  else if (s == "par_inflate") c->par_inflate = v ? 1 : 0;
  else if (s == "par_indexed") c->par_indexed = v ? 1 : 0;
  else if (s == "par_single_pass") c->par_single_pass = v ? 1 : 0;
  else if (s == "seg_v2") c->seg_v2 = v ? 1 : 0;
  else if (s == "inv_single_pass") c->inv_single_pass = v ? 1 : 0;
  else if (s == "inv_epoch") c->inv_epoch = (unsigned)v;          // (tests: the wrap of the look-back epochs)
  else if (s == "inv_order_block") c->inv_order_block = std::min<long long>(std::max<long long>(v, 1), 64);
  else if (s == "par_cells") c->par_cells = v < 0 ? -1 : (v ? 1 : 0);
  else if (s == "par_lz_wide") c->par_lz_wide = v < 0 ? -1 : (v ? 1 : 0);
  else if (s == "par_batch_bytes") { if (v < (1 << 20)) return fail(c, MTSB_E_ARG, "par_batch_bytes too small"); c->par_batch_bytes = v; }
  else if (s == "lz_ctas_per_sm") c->lz_ctas_per_sm = (int)std::min<long long>(8, std::max<long long>(1, v));
  else return fail(c, MTSB_E_ARG, "unknown parameter %s", name);
  return 0;
}

long long mtsb_get_param(mtsb_ctx* c, const char* name) {
  if (!c || !name) return MTSB_E_ARG;
  std::string s(name);
  if (s == "seg_bytes") return c->seg_bytes;
  if (s == "batch_bytes") return c->batch_bytes;
  if (s == "host_batch_bytes") return c->host_batch_bytes;
  if (s == "write_index") return c->write_index;
  if (s == "par_inflate") return c->par_inflate;
  if (s == "par_lz_wide") return c->par_lz_wide;
  if (s == "par_cells") return c->par_cells;
  if (s == "par_indexed") return c->par_indexed;
  if (s == "par_single_pass") return c->par_single_pass;
  if (s == "seg_v2") return c->seg_v2;
  if (s == "inv_single_pass") return c->inv_single_pass;
  if (s == "inv_order_block") return c->inv_order_block;
  if (s == "inv_epoch") return c->inv_epoch;
  if (s == "par_batch_bytes") return c->par_batch_bytes;
  if (s == "par_survivors") return c->par_stats[0];
  if (s == "par_candidates") return c->par_stats[1];
  if (s == "par_chained") return c->par_stats[2];
  if (s == "par_resumed") return c->par_stats[3];
  if (s == "lz_ctas_per_sm") return c->lz_ctas_per_sm;
  if (s == "sm_count") return c->sm_count;
  return MTSB_E_ARG;
}

long long mtsb_compress_bound(mtsb_ctx* c, long long raw_bytes, long long ns, int nc, int itemsize, int flags) {
  if (!c || raw_bytes < 0) return MTSB_E_ARG;
  (void)nc;
  return chunk_bound(c, raw_bytes, seg_size_for(c, ns, itemsize, flags));
}

#if defined(MTS_LZ_PROFILE) && !defined(MTSCOMP_EMU)
// development only (not in the public header): read and reset the lz77 phase counters
int mtsb_debug_lz_profile(unsigned long long* out16) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out16, g_lz_prof, sizeof(unsigned long long) * 16) != cudaSuccess) return -1;
  unsigned long long z[16] = {0};
  cudaMemcpyToSymbol(g_lz_prof, z, sizeof z);
  return 0;
}
#endif

int mtsb_last_timings(mtsb_ctx* c, float* out, int n) {
  if (!c || !out) return 0;
  int k = std::min(n, 8);
  for (int i = 0; i < k; i++) out[i] = c->last_ms[i];
  return k;
}
long long mtsb_last_launches(mtsb_ctx* c) { return c ? c->launches : 0; }

void* mtsb_host_alloc(long long bytes) {
  void* p = nullptr;
  if (bytes <= 0 || cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void mtsb_host_free(void* p) { if (p) cudaFreeHost(p); }
void* mtsb_device_alloc(mtsb_ctx* c, long long bytes) {
  void* p = nullptr;
  if (!c || bytes <= 0) return nullptr;
  cudaSetDevice(c->device);
  if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void mtsb_device_free(mtsb_ctx* c, void* p) { if (c && p) { cudaSetDevice(c->device); cudaFree(p); } }
int mtsb_memcpy(mtsb_ctx* c, void* dst, const void* src, long long bytes, int kind) {
  if (!c || !dst || !src || bytes < 0) return MTSB_E_ARG;
  cudaMemcpyKind k = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  CK(cudaMemcpyAsync(dst, src, (size_t)bytes, k, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

// =============================================================================================== transforms
static int single_chunk_desc(mtsb_ctx* c, long long ns) {
  NEED(c->h_tab, 4096);
  NEED(c->d_tab, 4096);
  ChunkDesc cd{0, (int)ns, 0, 0, 0};
  memcpy(c->h_tab.p, &cd, sizeof cd);
  CK(cudaMemcpyAsync(c->d_tab.p, c->h_tab.p, sizeof cd, cudaMemcpyHostToDevice, c->stream));
  return 0;
}

int mtsb_delta_transform(mtsb_ctx* c, const void* src, int src_is_device, long long ns, int nc, int itemsize,
                         int flags, void* dst, int dst_is_device) {
  long long rows[2] = {0, ns};
  if (!valid_common(c, 1, rows, nc, itemsize) || !src || !dst) return fail(c, MTSB_E_ARG, "delta_transform: bad arguments");
  cudaSetDevice(c->device);
  c->reset_timing();
  size_t bytes = (size_t)ns * nc * itemsize;
  int r = single_chunk_desc(c, ns);
  if (r) return r;
  const void* raw = src;
  if (!src_is_device) { NEED(c->d_raw, bytes + 256); CK(cudaMemcpyAsync(c->d_raw.p, src, bytes, cudaMemcpyHostToDevice, c->stream)); raw = c->d_raw.p; }
  void* t = dst;
  if (!dst_is_device) { NEED(c->d_T, bytes + 8192); t = c->d_T.p; }
  r = launch_fwd(c, itemsize, raw, t, (const ChunkDesc*)c->d_tab.p, 1, (int)ns, nc, flags);
  if (r) return r;
  if (!dst_is_device) CK(cudaMemcpyAsync(dst, t, bytes, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int mtsb_inverse_transform(mtsb_ctx* c, const void* src, int src_is_device, long long ns, int nc, int itemsize,
                           int flags, void* dst, int dst_is_device, uint32_t* adler32_out) {
  long long rows[2] = {0, ns};
  if (!valid_common(c, 1, rows, nc, itemsize) || !src || !dst) return fail(c, MTSB_E_ARG, "inverse_transform: bad arguments");
  cudaSetDevice(c->device);
  c->reset_timing();
  size_t bytes = (size_t)ns * nc * itemsize;
  const int ASEG = 1 << 16;
  int nas = (int)((bytes + ASEG - 1) / ASEG);
  size_t tab_bytes = 256 + (size_t)nas * sizeof(AdlerSeg) + 64;
  NEED(c->h_tab, tab_bytes);
  NEED(c->d_tab, tab_bytes);
  char* h = (char*)c->h_tab.p;
  ChunkDesc cd{0, (int)ns, 0, 0, 0};
  memcpy(h, &cd, sizeof cd);
  int firsts[2] = {0, nas};
  memcpy(h + 64, firsts, sizeof firsts);
  AdlerSeg* as = (AdlerSeg*)(h + 256);
  for (int i = 0; i < nas; i++) { as[i].off = (long long)i * ASEG; as[i].len = (int)std::min<size_t>(ASEG, bytes - (size_t)i * ASEG); as[i].pad_ = 0; }
  { int rc_ = small_copy(c, c->d_tab.p, h, tab_bytes); if (rc_) return rc_; }
  const void* t = src;
  if (!src_is_device) { NEED(c->d_T, bytes + 8192); CK(cudaMemcpyAsync(c->d_T.p, src, bytes, cudaMemcpyHostToDevice, c->stream)); t = c->d_T.p; }
  void* o = dst;
  if (!dst_is_device) { NEED(c->d_out, bytes + 256); o = c->d_out.p; }
  char* d = (char*)c->d_tab.p;
  if (adler32_out) {
    NEED(c->d_seg_adler, (size_t)nas * 4);
    NEED(c->d_chunk_adler, 64);
    MTS_LAUNCH(adler_partial_kernel, dim3(nas), dim3(256), 0, c->stream, (const uint8_t*)t, (const AdlerSeg*)(d + 256), (uint32_t*)c->d_seg_adler.p);
    CKL();
    MTS_LAUNCH(adler_combine_kernel, dim3(1), dim3(32), 0, c->stream, (const AdlerSeg*)(d + 256), (const uint32_t*)c->d_seg_adler.p, (const int*)(d + 64), 1, (uint32_t*)c->d_chunk_adler.p);
    CKL();
    c->launches += 2;
    CK(cudaMemcpyAsync(adler32_out, c->d_chunk_adler.p, 4, cudaMemcpyDeviceToHost, c->stream));
  }
  int r = launch_inv(c, itemsize, t, o, (const ChunkDesc*)d, 1, (int)ns, nc, flags, (size_t)ns * nc);
  if (r) return r;
  if (!dst_is_device) CK(cudaMemcpyAsync(dst, o, bytes, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

// =============================================================================================== compress
int mtsb_compress_chunks(mtsb_ctx* c, const void* src, int src_is_device, int n_chunks, const long long* chunk_rows,
                         int nc, int itemsize, int flags, void* dst, int dst_is_device, long long dst_capacity,
                         long long* out_offsets) {
  if (!valid_common(c, n_chunks, chunk_rows, nc, itemsize) || !src || !dst || !out_offsets)
    return fail(c, MTSB_E_ARG, "compress_chunks: bad arguments");
  cudaSetDevice(c->device);
  c->reset_timing();
  const long long row_bytes = (long long)nc * itemsize;
  // capacity check against the worst case
  long long need = 0;
  for (int i = 0; i < n_chunks; i++) {
    long long ns = chunk_rows[i + 1] - chunk_rows[i];
    need += chunk_bound(c, ns * row_bytes, seg_size_for(c, ns, itemsize, flags));
  }
  if (dst_capacity < need) return fail(c, MTSB_E_CAPACITY, "dst_capacity %lld < bound %lld", dst_capacity, need);

  out_offsets[0] = 0;
  long long total_out = 0;
  // sub-batches: bounded by batch_bytes; smaller when a host buffer is involved so that copies pipeline with kernels
  const bool host_io = !src_is_device || !dst_is_device;
  // device-resident calls have nothing to overlap with: one large sub-batch keeps the persistent match-finder CTAs
  // busy to the end (measured on 600 chunks: 2 GiB 99.9, 4 GiB 100.6, one 13.9 GB batch 101.7 GB/s)
  const long long sb_limit = host_io ? std::min(c->batch_bytes, c->host_batch_bytes) : std::max<long long>(c->batch_bytes, 16ll << 30);
  std::vector<int> sb_first;
  long long max_sb_bytes = 0, max_sb_bound = 0;
  for (int a = 0; a < n_chunks;) {
    sb_first.push_back(a);
    int b = a;
    long long bb = 0, bd = 0;
    while (b < n_chunks && b - a < 60000) {
      long long ns = chunk_rows[b + 1] - chunk_rows[b], cb = ns * row_bytes;
      if (b > a && bb + cb > sb_limit) break;
      bb += cb; bd += chunk_bound(c, cb, seg_size_for(c, ns, itemsize, flags)); b++;
    }
    max_sb_bytes = std::max(max_sb_bytes, bb);
    max_sb_bound = std::max(max_sb_bound, bd);
    a = b;
  }
  sb_first.push_back(n_chunks);
  const int n_sb = (int)sb_first.size() - 1;
  Buf* raw_buf[2] = {&c->d_raw, &c->d_raw2};
  Buf* out_buf[2] = {&c->d_out, &c->d_out2};
  if (!src_is_device) { NEED(c->d_raw, (size_t)max_sb_bytes + 256); if (n_sb > 1) NEED(c->d_raw2, (size_t)max_sb_bytes + 256); }
  if (!dst_is_device) { NEED(c->d_out, (size_t)max_sb_bound + 256); if (n_sb > 1) NEED(c->d_out2, (size_t)max_sb_bound + 256); }
  auto sb_bytes = [&](int k) { return (chunk_rows[sb_first[k + 1]] - chunk_rows[sb_first[k]]) * row_bytes; };
  if (!src_is_device) {
    // the copy-in stream must not start before work already queued on the caller's stream (e.g. producing `src`)
    CK(cudaEventRecord(c->ev_done, c->stream));
    CK(cudaStreamWaitEvent(c->copy_in, c->ev_done, 0));
    CK(cudaMemcpyAsync(raw_buf[0]->p, (const char*)src, (size_t)sb_bytes(0), cudaMemcpyHostToDevice, c->copy_in));
    CK(cudaEventRecord(c->ev_in[0], c->copy_in));
  }
  for (int k = 0; k < n_sb; k++) {
    const int c0 = sb_first[k], c1 = sb_first[k + 1];
    const long long bbytes = sb_bytes(k);
    const int nb = c1 - c0;
    const long long row0 = chunk_rows[c0];
    // tables
    std::vector<ChunkDesc> cds(nb);
    std::vector<DeflateSeg> segs;
    std::vector<int> first(nb + 1);
    int max_ns = 0, n_subs = 0;
    long long bound = 0;
    for (int i = 0; i < nb; i++) {
      long long ns = chunk_rows[c0 + i + 1] - chunk_rows[c0 + i];
      long long raw = ns * row_bytes;
      long long seg = seg_size_for(c, ns, itemsize, flags);
      int k = (int)((raw + seg - 1) / seg);
      cds[i].elem_off = (chunk_rows[c0 + i] - row0) * nc;
      cds[i].ns = (int)ns;
      cds[i].first_seg = (int)segs.size();
      cds[i].n_seg = k;
      cds[i].pad_ = (int)seg;
      first[i] = (int)segs.size();
      max_ns = std::max(max_ns, (int)ns);
      long long base = cds[i].elem_off * itemsize;
      for (int j = 0; j < k; j++) {
        DeflateSeg s;
        s.in_off = base + (long long)j * seg;
        s.tok_off = s.in_off;
        s.in_len = (int)std::min<long long>(seg, raw - (long long)j * seg);
        s.chunk = i;
        s.flags = (j == 0 ? SEG_FIRST : 0) | (j == k - 1 ? SEG_LAST : 0);
        s.sub_first = n_subs;
        n_subs += idx_n_sub(s.in_len);
        segs.push_back(s);
      }
      bound += chunk_bound(c, raw, seg);
    }
    first[nb] = (int)segs.size();
    const int n_segs = (int)segs.size();
    // table blob: [ChunkDesc nb][DeflateSeg n_segs][AdlerSeg n_segs][first nb+1]
    size_t o_cd = 0, o_seg = (o_cd + nb * sizeof(ChunkDesc) + 255) & ~(size_t)255;
    size_t o_as = (o_seg + n_segs * sizeof(DeflateSeg) + 255) & ~(size_t)255;
    size_t o_first = (o_as + n_segs * sizeof(AdlerSeg) + 255) & ~(size_t)255;
    size_t tab_bytes = o_first + (nb + 1) * sizeof(int);
    NEED(c->h_tab, tab_bytes);
    NEED(c->d_tab, tab_bytes);
    char* h = (char*)c->h_tab.p;
    memcpy(h + o_cd, cds.data(), nb * sizeof(ChunkDesc));
    memcpy(h + o_seg, segs.data(), n_segs * sizeof(DeflateSeg));
    AdlerSeg* as = (AdlerSeg*)(h + o_as);
    for (int i = 0; i < n_segs; i++) { as[i].off = segs[i].in_off; as[i].len = segs[i].in_len; as[i].pad_ = 0; }
    memcpy(h + o_first, first.data(), (nb + 1) * sizeof(int));
    // scratch
    NEED(c->d_T, (size_t)bbytes + 16384);
    NEED(c->d_tok, (size_t)bbytes * 2 + 4096);
    NEED(c->d_hist, (size_t)n_segs * HIST_STRIDE * 4);
    NEED(c->d_codes, (size_t)n_segs * CODE_STRIDE * 4);
    NEED(c->d_hdrs, (size_t)n_segs * HDR_WORDS * 4);
    NEED(c->d_so, (size_t)n_segs * sizeof(DeflateSegOut));
    NEED(c->d_seg_adler, (size_t)n_segs * 4);
    NEED(c->d_chunk_adler, (size_t)nb * 4);
    NEED(c->d_chunk_off, (size_t)(nb + 1) * 8);
    NEED(c->d_subabs, (size_t)n_subs * 8 + 64);
    NEED(c->d_subtok, (size_t)n_subs * 8 + 64);
    NEED(c->h_small, (size_t)(nb + 1) * 8);
    const char* d = (const char*)c->d_tab.p;
    const ChunkDesc* d_cd = (const ChunkDesc*)(d + o_cd);
    const DeflateSeg* d_seg = (const DeflateSeg*)(d + o_seg);
    const AdlerSeg* d_as = (const AdlerSeg*)(d + o_as);
    const int* d_first = (const int*)(d + o_first);

    c->begin(0);
    { int rc_ = small_copy(c, c->d_tab.p, h, tab_bytes); if (rc_) return rc_; }
    // only now queue the next sub-batch's upload: the copy engine serves transfers in submission order, so the small
    // table upload above must not sit behind it
    if (!src_is_device && k + 1 < n_sb) {
      CK(cudaMemcpyAsync(raw_buf[(k + 1) & 1]->p, (const char*)src + chunk_rows[sb_first[k + 1]] * row_bytes,
                         (size_t)sb_bytes(k + 1), cudaMemcpyHostToDevice, c->copy_in));
      CK(cudaEventRecord(c->ev_in[(k + 1) & 1], c->copy_in));
    }
    const void* raw = (const char*)src + row0 * row_bytes;
    if (!src_is_device) {
      CK(cudaStreamWaitEvent(c->stream, c->ev_in[k & 1], 0));
      raw = raw_buf[k & 1]->p;
    }
    c->end();
    unsigned char* outp;
    if (dst_is_device) outp = (unsigned char*)dst + total_out;
    else {
      if (k >= 2) CK(cudaStreamWaitEvent(c->stream, c->ev_out[k & 1], 0));   // D2H of sub-batch k-2 has drained it
      outp = (unsigned char*)out_buf[k & 1]->p;
    }

    c->begin(1);
    int r = launch_fwd(c, itemsize, raw, c->d_T.p, d_cd, nb, max_ns, nc, flags);
    if (r) return r;
    c->end();
    c->begin(3);
    {
      NEED(c->d_invstate, 256);
      CK(cudaMemsetAsync(c->d_invstate.p, 0, 64, c->stream));    // the match finder's segment counter
      int grid = std::min(n_segs, c->sm_count * c->lz_ctas_per_sm);
      if (itemsize == 2) {
        auto k = lz77_kernel<2, LZ_NT>;
        MTS_LAUNCH(k, dim3(grid), dim3(LZ_NT + 32), (LzSmem<2, LZ_NT>::total), c->stream, (const unsigned char*)c->d_T.p, d_seg, n_segs, (unsigned short*)c->d_tok.p, (unsigned*)c->d_hist.p, (DeflateSegOut*)c->d_so.p, (unsigned*)c->d_seg_adler.p, c->write_index ? (unsigned long long*)c->d_subtok.p : (unsigned long long*)nullptr, (unsigned*)c->d_invstate.p);
      } else {
        auto k = lz77_kernel<1, LZ_NT>;
        MTS_LAUNCH(k, dim3(grid), dim3(LZ_NT + 32), (LzSmem<1, LZ_NT>::total), c->stream, (const unsigned char*)c->d_T.p, d_seg, n_segs, (unsigned short*)c->d_tok.p, (unsigned*)c->d_hist.p, (DeflateSegOut*)c->d_so.p, (unsigned*)c->d_seg_adler.p, c->write_index ? (unsigned long long*)c->d_subtok.p : (unsigned long long*)nullptr, (unsigned*)c->d_invstate.p);
      }
      CKL();
      c->launches++;
    }
    c->end();
    c->begin(4);
    // the match finder left each segment's adler32 (it streams every byte of T anyway): fold them per chunk
    MTS_LAUNCH(adler_combine_kernel, dim3((nb + 127) / 128), dim3(128), 0, c->stream, d_as, (const uint32_t*)c->d_seg_adler.p, d_first, nb, (uint32_t*)c->d_chunk_adler.p);
    CKL();
    c->launches++;
    MTS_LAUNCH(huff_kernel, dim3(n_segs), dim3(32), 0, c->stream, d_seg, n_segs, (unsigned*)c->d_hist.p, (unsigned*)c->d_codes.p, (unsigned*)c->d_hdrs.p, (DeflateSegOut*)c->d_so.p);
    CKL();
    MTS_LAUNCH(scan_kernel, dim3(1), dim3(1024), 0, c->stream, d_seg, n_segs, (DeflateSegOut*)c->d_so.p, (long long*)c->d_chunk_off.p, nb, d_cd, (int)c->write_index);
    CKL();
    c->launches += 2;
    c->end();
    c->begin(5);
    auto ek = itemsize == 2 ? encode_kernel<true> : encode_kernel<false>;
    MTS_LAUNCH(ek, dim3(n_segs), dim3(ENC_THREADS), 0, c->stream, (const unsigned char*)c->d_T.p, d_seg, n_segs, (const unsigned short*)c->d_tok.p, (const unsigned*)c->d_codes.p, (const unsigned*)c->d_hdrs.p, (const DeflateSegOut*)c->d_so.p, (const unsigned*)c->d_chunk_adler.p, outp, (const unsigned long long*)c->d_subtok.p, c->write_index ? (unsigned long long*)c->d_subabs.p : (unsigned long long*)nullptr);
    CKL();
    c->launches++;
    if (c->write_index) {
      MTS_LAUNCH(trailer_kernel, dim3(nb), dim3(128), 0, c->stream, d_seg, (const DeflateSegOut*)c->d_so.p, d_cd,
                 (const long long*)c->d_chunk_off.p, (const unsigned long long*)c->d_subabs.p, outp,
                 (unsigned)(LZ_NT * (itemsize == 2 ? 2 : 1)));
      CKL();
      c->launches++;
    }
    c->end();
    { int rc_ = small_copy(c, c->h_small.p, c->d_chunk_off.p, (size_t)(nb + 1) * 8); if (rc_) return rc_; }
    CK(cudaStreamSynchronize(c->stream));
    const long long* co = (const long long*)c->h_small.p;
    if (co[nb] > bound) return fail(c, MTSB_E_CAPACITY, "internal: sub-batch output %lld exceeds bound %lld", co[nb], bound);
    for (int i = 0; i < nb; i++) out_offsets[c0 + i + 1] = total_out + co[i + 1];
    if (!dst_is_device) {
      // the kernels of this sub-batch are complete (synchronised above): drain it on the copy-out stream
      CK(cudaMemcpyAsync((char*)dst + total_out, outp, (size_t)co[nb], cudaMemcpyDeviceToHost, c->copy_out));
      CK(cudaEventRecord(c->ev_out[k & 1], c->copy_out));
    }
    total_out += co[nb];
  }
  if (!dst_is_device) CK(cudaStreamSynchronize(c->copy_out));
  c->collect_timing();
  return 0;
}

// =============================================================================================== decompress
__global__ void gather_bytes_kernel(const unsigned char* __restrict__ base, const long long* __restrict__ src_off,
                                    const int* __restrict__ len, const long long* __restrict__ dst_off,
                                    unsigned char* __restrict__ dst) {
  const long long so = src_off[blockIdx.x], dof = dst_off[blockIdx.x];
  const int n = len[blockIdx.x];
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[dof + i] = base[so + i];
}

// Fetch `n` ranges of the compressed buffer to host memory (direct reads for host buffers, one gather kernel + one
// copy for device buffers).
static int fetch_ranges(mtsb_ctx* c, const unsigned char* comp, int comp_is_device, const std::vector<long long>& off,
                        const std::vector<int>& len, std::vector<unsigned char>& out, std::vector<long long>& dpos) {
  size_t n = off.size(), total = 0;
  dpos.resize(n);
  for (size_t i = 0; i < n; i++) { dpos[i] = (long long)total; total += (size_t)len[i]; }
  out.resize(total);
  if (!total) return 0;
  if (!comp_is_device) {
    for (size_t i = 0; i < n; i++) memcpy(out.data() + dpos[i], comp + off[i], (size_t)len[i]);
    return 0;
  }
  size_t tb = n * 20 + 64;
  NEED(c->h_tab, tb + total);
  NEED(c->d_tab, tb);
  NEED(c->d_gather, total);
  char* h = (char*)c->h_tab.p;
  size_t o1 = n * 8, o2 = n * 16;
  memcpy(h, off.data(), n * 8);
  memcpy(h + o1, dpos.data(), n * 8);
  memcpy(h + o2, len.data(), n * 4);
  CK(cudaMemcpyAsync(c->d_tab.p, h, tb, cudaMemcpyHostToDevice, c->stream));
  const char* d = (const char*)c->d_tab.p;
  MTS_LAUNCH(gather_bytes_kernel, dim3((unsigned)n), dim3(128), 0, c->stream, comp, (const long long*)d, (const int*)(d + o2), (const long long*)(d + o1), (unsigned char*)c->d_gather.p);
  CKL();
  c->launches++;
  CK(cudaMemcpyAsync(h + tb, c->d_gather.p, total, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  memcpy(out.data(), h + tb, total);
  return 0;
}

static uint32_t rd32(const unsigned char* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }

// The block-parallel decoder for the streams `ps` (segs[ids[i]] each).  blks == nullptr: plain zlib streams, the
// blocks are searched for on the device (find -> validate into per-stream buckets -> sort).  Otherwise blks holds one
// known block per stream (the indexed segments of GPU-written chunks).  No host round trip between the kernels: one
// synchronisation at the end fetches the per-stream results.  The streams whose chain of blocks was resolved are
// rewritten as INF_RESUME tails; the others are left untouched (full serial decode).
static int par_decode(mtsb_ctx* c, const unsigned char* dcomp, std::vector<InflateSeg>& segs, const std::vector<int>& ids,
                      const std::vector<ParStream>& ps, const std::vector<ParBlk>* blks, long long in_total, int max_in,
                      unsigned char* dT, int zflag) {
  const int ns = (int)ps.size();
  if (ns == 0) return 0;
  // bucket of candidate blocks per stream: zlib level 6 closes a block about every 29 KB of output here; streams with
  // denser candidates overflow their bucket and are decoded serially
  const unsigned bcap = blks ? 1u : (unsigned)(max_in / 8192 + 64);
  const size_t n_slots = (size_t)ns * bcap;
  if (n_slots > 0x7fffffffull) return 0;
  const size_t surv_cap = (size_t)std::max<long long>(1 << 20, in_total * 8 / 300);
  // token slots: one per 6 bits of input (typical streams spend 9..15 bits per token); if that is not enough the blocks
  // that do not fit end the chain of their stream (serial decode of the rest)
  const long long tok_total = in_total * 8 / 6 + 4096;
  const size_t o_keys = ((size_t)ns * 4 + 255) & ~(size_t)255;      // d_cand: [bucket fill counts | bucket keys]
  NEED(c->d_pstreams, (size_t)ns * sizeof(ParStream));
  NEED(c->d_pcount, 256);
  NEED(c->d_pbad, (size_t)ns * sizeof(ParRes) + 64);
  NEED(c->d_plist, n_slots * sizeof(ParBlk));
  NEED(c->d_tokens, (size_t)tok_total * 4 + 64);
  // plain streams: the counting pass of par_block_kernel leaves its tokens in a scratch area with one slot per
  // PAR_PIECE_BITS input bits (addressed by the bit's offset in the buffer), from where they are copied instead of decoded again
  unsigned* d_pieces = nullptr;
  if (!blks && c->par_single_pass) {
    long long span = 0;
    for (int i = 0; i < ns; i++) span = std::max(span, ps[i].in_off + ps[i].in_len);
    NEED(c->d_pieces, ((size_t)span * 8 / PAR_PIECE_BITS + 64) * 4);
    d_pieces = (unsigned*)c->d_pieces.p;
  }
  const size_t o_blk = ((size_t)ns * sizeof(ParStream) + 255) & ~(size_t)255;   // host staging: [streams | blocks]
  NEED(c->h_tab, o_blk + (blks ? n_slots * sizeof(ParBlk) : 0) + 64);
  NEED(c->h_small, 4096 + (size_t)ns * (sizeof(ParRes) + 4) + 64);
  memcpy(c->h_tab.p, ps.data(), (size_t)ns * sizeof(ParStream));
  { int r = small_copy(c, c->d_pstreams.p, c->h_tab.p, (size_t)ns * sizeof(ParStream)); if (r) return r; }
  CK(cudaMemsetAsync(c->d_pcount.p, 0, 256, c->stream));           // [0] survivors, [4..5] token cursor
  const ParStream* d_ps = (const ParStream*)c->d_pstreams.p;
  unsigned* d_cnt = (unsigned*)c->d_pcount.p;
  if (blks) {
    memcpy((char*)c->h_tab.p + o_blk, blks->data(), n_slots * sizeof(ParBlk));
    { int r = small_copy(c, c->d_plist.p, (char*)c->h_tab.p + o_blk, n_slots * sizeof(ParBlk)); if (r) return r; }
  } else {
    NEED(c->d_surv, surv_cap * 8);
    NEED(c->d_cand, o_keys + n_slots * 4);
    unsigned* d_bcount = (unsigned*)c->d_cand.p;
    unsigned* d_keys = (unsigned*)((char*)c->d_cand.p + o_keys);
    CK(cudaMemsetAsync(d_bcount, 0, (size_t)ns * 4, c->stream));
    MTS_LAUNCH(par_find_kernel, dim3((max_in / 4 + 2 + 256 * PAR_FIND_WORDS - 1) / (256 * PAR_FIND_WORDS), ns), dim3(256), 0,
               c->stream, dcomp, d_ps, (unsigned long long*)c->d_surv.p, (unsigned)surv_cap, d_cnt);
    CKL();
    MTS_LAUNCH(par_validate_kernel, dim3(c->sm_count * 16), dim3(128), 0, c->stream, dcomp, d_ps,
               (const unsigned long long*)c->d_surv.p, (unsigned)surv_cap, d_keys, bcap, d_bcount, (const unsigned*)d_cnt);
    CKL();
    MTS_LAUNCH(par_sort_kernel, dim3(ns), dim3(32), 0, c->stream, d_ps, (const unsigned*)d_keys, bcap, (const unsigned*)d_bcount,
               (const unsigned*)d_cnt, (unsigned)surv_cap, (ParBlk*)c->d_plist.p);
    CKL();
    c->launches += 3;
  }
  MTS_LAUNCH(par_block_kernel, dim3((unsigned)((n_slots + PAR_BLK_WARPS - 1) / PAR_BLK_WARPS)), dim3(PAR_BLK_WARPS * 32), 0, c->stream,
             dcomp, d_ps, (ParBlk*)c->d_plist.p, (unsigned)n_slots, (unsigned*)c->d_tokens.p,
             (unsigned long long*)((char*)c->d_pcount.p + 16), (unsigned long long)tok_total, d_pieces);
  CKL();
  // measured (ms of inflate, chain of tiles / cells): 1 stream 23.4 / 4.1, 8 streams 25.4 / 9.6, 64 streams 35 / 48,
  // 600 streams 180 / 415 -> the cells path is the low-latency path for a handful of streams only
  const bool use_cells = !blks && (c->par_cells < 0 ? ns <= 16 : c->par_cells == 1);
  if (use_cells) {
    // few streams: resolve the blocks of a stream in parallel (cells + markers), then cells -> bytes per stream
    long long lo = ps[0].out_off, hi = ps[0].out_off + ps[0].out_len;
    for (int i = 1; i < ns; i++) { lo = std::min(lo, ps[i].out_off); hi = std::max(hi, ps[i].out_off + ps[i].out_len); }
    NEED(c->d_cells, (size_t)(hi - lo) * 2 + 64);
    MTS_LAUNCH(par_chain_kernel, dim3((ns + 63) / 64), dim3(64), 0, c->stream, d_ps, (ParBlk*)c->d_plist.p, bcap, (unsigned)ns,
               (ParRes*)c->d_pbad.p);
    CKL();
    auto k = par_lzc_kernel<256, 4096>;
    MTS_LAUNCH(k, dim3((unsigned)n_slots), dim3(256), 0, c->stream, d_ps, (ParBlk*)c->d_plist.p, (const unsigned*)c->d_tokens.p,
               (unsigned short*)c->d_cells.p, lo);
    CKL();
    MTS_LAUNCH(par_cells_kernel, dim3((unsigned)n_slots), dim3(256), 0, c->stream, d_ps, (const ParBlk*)c->d_plist.p, bcap,
               (const unsigned short*)c->d_cells.p, lo, dT, (ParRes*)c->d_pbad.p);
    CKL();
    c->launches += 3;
  } else if (c->par_lz_wide < 0 ? ns <= 2 * c->sm_count : c->par_lz_wide == 1) {
    auto k = par_lz_kernel<1024, 16384>;
    MTS_LAUNCH(k, dim3(ns), dim3(1024), PAR_LZ_MIRROR, c->stream, d_ps, (const ParBlk*)c->d_plist.p, bcap, (const unsigned*)c->d_tokens.p, dT,
               (ParRes*)c->d_pbad.p);
    CKL();
    c->launches++;
  } else {
    auto k = par_lz_kernel<256, 4096>;
    MTS_LAUNCH(k, dim3(ns), dim3(256), PAR_LZ_MIRROR, c->stream, d_ps, (const ParBlk*)c->d_plist.p, bcap, (const unsigned*)c->d_tokens.p, dT,
               (ParRes*)c->d_pbad.p);
    CKL();
    c->launches++;
  }
  c->launches++;
  char* hs = (char*)c->h_small.p;
  { int r = small_copy(c, hs, c->d_pcount.p, 64); if (r) return r; }
  { int r = small_copy(c, hs + 4096, c->d_pbad.p, (size_t)ns * sizeof(ParRes)); if (r) return r; }
  const size_t o_bc = 4096 + (((size_t)ns * sizeof(ParRes) + 15) & ~(size_t)15);
  if (!blks) { int r = small_copy(c, hs + o_bc, c->d_cand.p, (size_t)ns * 4); if (r) return r; }
  CK(cudaStreamSynchronize(c->stream));
  if (!blks) {
    c->par_stats[0] += ((const unsigned*)hs)[0];
    for (int i = 0; i < ns; i++) c->par_stats[1] += ((const unsigned*)(hs + o_bc))[i];
  }
  const ParRes* res = (const ParRes*)(hs + 4096);
  for (int sidx = 0; sidx < ns; sidx++) {
    const ParRes& r = res[sidx];
    c->par_stats[2] += r.n_done;
    if (r.n_done == 0 || (r.flags & 2)) continue;              // full serial decode of this stream
    InflateSeg& s = segs[ids[sidx]];
    s.flags = zflag | INF_RESUME | ((r.flags & 1) ? INF_NO_BLOCKS : 0);
    s.start_bit = r.tail_bit;
    s.opos0 = r.tail_out;
    c->par_stats[3]++;
    if ((r.flags & 4) && zflag && r.tail_out == (unsigned)s.out_len && (size_t)ids[sidx] < c->lz_adler.size()) {
      c->lz_adler[ids[sidx]] = r.adler;          // the whole stream went through par_lz_kernel: its adler32 is known
      c->lz_adler_have[ids[sidx]] = 1;
    }
  }
  return 0;
}

// The indexed segments of GPU-written chunks (`ids`: indices into segs): every segment is one dynamic block at bit 0
// followed by the empty stored block that byte-aligns the next segment (deflate.cuh), so the blocks are known without
// any search; a segment stored uncompressed simply fails the header parse and stays serial.
static int par_phase_indexed(mtsb_ctx* c, const unsigned char* dcomp, std::vector<InflateSeg>& segs, const std::vector<int>& ids,
                             unsigned char* dT) {
  const int ns = (int)ids.size();
  std::vector<ParStream> ps(ns);
  std::vector<ParBlk> blks(ns);
  long long in_total = 0;
  int max_in = 0;
  for (int i = 0; i < ns; i++) {
    const InflateSeg& s = segs[ids[i]];
    ps[i].in_off = s.in_off; ps[i].out_off = s.out_off; ps[i].in_len = s.in_len; ps[i].out_len = s.out_len;
    ps[i].first_bit = 0; ps[i].pad_ = 0;
    ParBlk& b = blks[i];
    b.stream = (unsigned)i; b.bit = 0; b.limit = (unsigned)s.in_len * 8u;
    b.end_bit = 0; b.n_tok = 0; b.out_len = 0; b.flags = 0; b.pad_ = 0; b.tok_off = 0;
    in_total += s.in_len;
    max_in = std::max(max_in, s.in_len);
  }
  return par_decode(c, dcomp, segs, ids, ps, &blks, in_total, max_in, dT, 0);
}

// The indexed segments of chunks with the second index format: `ids` index into segs, v2[i] describes segs[ids[i]].
// seg_tokens_kernel (lane per indexed sub-block) + seg_resolve_kernel (all tokens of a step at once); segments that
// pass become INF_RESUME tails (the serial kernel then only checks the empty stored block behind them), the others
// are decoded serially from their start.
static int par_phase_v2(mtsb_ctx* c, const unsigned char* dcomp, std::vector<InflateSeg>& segs, const std::vector<int>& ids,
                        std::vector<SegV2>& v2, unsigned char* dT, std::vector<uint32_t>& seg_ad, std::vector<char>& seg_ok) {
  seg_ad.assign(ids.size(), 0);
  seg_ok.assign(ids.size(), 0);
  const size_t SMEM = SEG_RING + (SEG_MAX_STEPS + 1) * 4;
  const long long GROUP_SUBS = (4ll << 30) / IDX_SUB_BYTES;     // sub-blocks per launch pair: bounds the token scratch (~9 GB)
  size_t a = 0;
  while (a < ids.size()) {
    size_t b = a;
    long long subs = 0;
    while (b < ids.size() && (b == a || subs + idx_n_sub(v2[b].out_len) <= GROUP_SUBS)) { v2[b].sub_first = (int)subs; subs += idx_n_sub(v2[b].out_len); b++; }
    const int ns = (int)(b - a);
    NEED(c->d_segv2, (size_t)ns * sizeof(SegV2));
    NEED(c->d_tokens, (size_t)subs * SEG_TOK_STRIDE * 4 + 64);
    NEED(c->d_btab, (size_t)subs * SEG_BATCHES * sizeof(uint2) + 64);
    NEED(c->d_subout, (size_t)subs * sizeof(SubOut) + 64);
    NEED(c->d_pbad, (size_t)ns * sizeof(ParRes) + 64);
    NEED(c->d_tadler, (size_t)ns * 4 + 64);
    NEED(c->h_tab, (size_t)ns * sizeof(SegV2) + 64);
    NEED(c->h_small, 4096 + (size_t)ns * (sizeof(ParRes) + 4) + 128);
    memcpy(c->h_tab.p, v2.data() + a, (size_t)ns * sizeof(SegV2));
    { int r = small_copy(c, c->d_segv2.p, c->h_tab.p, (size_t)ns * sizeof(SegV2)); if (r) return r; }
    MTS_LAUNCH(seg_tokens_kernel, dim3(ns), dim3(32), 0, c->stream, dcomp, (const SegV2*)c->d_segv2.p, (unsigned*)c->d_tokens.p,
               (uint2*)c->d_btab.p, (SubOut*)c->d_subout.p, (ParRes*)c->d_pbad.p);
    CKL();
    MTS_LAUNCH(seg_resolve_kernel, dim3(ns), dim3(SEG_RES_WARPS * 32), SMEM, c->stream, (const SegV2*)c->d_segv2.p,
               (const unsigned*)c->d_tokens.p, (const uint2*)c->d_btab.p, (const SubOut*)c->d_subout.p, dT, (ParRes*)c->d_pbad.p,
               (unsigned*)c->d_tadler.p);
    CKL();
    c->launches += 2;
    char* hs = (char*)c->h_small.p;
    const size_t o_ad = 4096 + (((size_t)ns * sizeof(ParRes) + 15) & ~(size_t)15);
    { int r = small_copy(c, hs + 4096, c->d_pbad.p, (size_t)ns * sizeof(ParRes)); if (r) return r; }
    { int r = small_copy(c, hs + o_ad, c->d_tadler.p, (size_t)ns * 4); if (r) return r; }
    CK(cudaStreamSynchronize(c->stream));
    const ParRes* res = (const ParRes*)(hs + 4096);
    for (int i = 0; i < ns; i++) {
      const ParRes& r = res[i];
      c->par_stats[2] += r.n_done;
      if (r.n_done == 0 || (r.flags & 2)) continue;             // full serial decode of this segment
      seg_ok[a + i] = 1;
      seg_ad[a + i] = ((const uint32_t*)(hs + o_ad))[i];
      InflateSeg& sg = segs[ids[a + i]];
      sg.flags = INF_RESUME;
      sg.start_bit = r.tail_bit;
      sg.opos0 = r.tail_out;
      c->par_stats[3]++;
    }
    a = b;
  }
  return 0;
}

// Block-parallel decode of the whole-stream segments `whole` (indices into segs): plain zlib streams.
static int par_phase(mtsb_ctx* c, const unsigned char* dcomp, std::vector<InflateSeg>& segs, const std::vector<int>& whole,
                     unsigned char* dT) {
  const int ns = (int)whole.size();
  std::vector<ParStream> ps(ns);
  long long in_total = 0;
  int max_in = 0;
  for (int i = 0; i < ns; i++) {
    const InflateSeg& s = segs[whole[i]];
    ps[i].in_off = s.in_off; ps[i].out_off = s.out_off; ps[i].in_len = s.in_len; ps[i].out_len = s.out_len;
    ps[i].first_bit = 16; ps[i].pad_ = 0;
    in_total += s.in_len;
    max_in = std::max(max_in, s.in_len);
  }
  return par_decode(c, dcomp, segs, whole, ps, nullptr, in_total, max_in, dT, INF_ZLIB);
}

int mtsb_decompress_chunks(mtsb_ctx* c, const void* comp_, int comp_is_device, const long long* comp_offsets,
                           int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags, void* dst,
                           int dst_is_device, int* chunk_status) {
  if (!valid_common(c, n_chunks, chunk_rows, nc, itemsize) || !comp_ || !comp_offsets || !dst)
    return fail(c, MTSB_E_ARG, "decompress_chunks: bad arguments");
  for (int i = 0; i < n_chunks; i++) {
    long long l = comp_offsets[i + 1] - comp_offsets[i];
    if (l < 1 || l > 0x7fffffffll) return fail(c, MTSB_E_ARG, "decompress_chunks: bad compressed length of chunk %d", i);
  }
  cudaSetDevice(c->device);
  c->reset_timing();
  for (long long& v : c->par_stats) v = 0;
  const unsigned char* comp = (const unsigned char*)comp_;
  const long long row_bytes = (long long)nc * itemsize;

  // ---- plan: look for the segment index after each chunk's zlib stream
  c->begin(1);
  std::vector<int> nseg(n_chunks, 0);
  std::vector<long long> segb(n_chunks, 0), idx_extra(n_chunks, 0);
  std::vector<char> idx_v2(n_chunks, 0);
  std::vector<unsigned> idx_step(n_chunks, 0);
  std::vector<unsigned char> tails, idx;
  std::vector<long long> tpos, ipos;
  {
    std::vector<long long> off;
    std::vector<int> len;
    std::vector<int> who;
    for (int i = 0; i < n_chunks; i++) {
      long long l = comp_offsets[i + 1] - comp_offsets[i];
      if (l >= 2 + 6 + 4 + INDEX_TAIL && !c->ignore_index) { off.push_back(comp_offsets[i + 1] - INDEX_TAIL); len.push_back(INDEX_TAIL); who.push_back(i); }
    }
    int r = fetch_ranges(c, comp, comp_is_device, off, len, tails, tpos);
    if (r) return r;
    std::vector<long long> off2, tail_by_chunk(n_chunks, -1);
    std::vector<int> len2;
    std::vector<int> who2;
    for (size_t j = 0; j < who.size(); j++) {
      const unsigned char* t = tails.data() + tpos[j];
      int i = who[j];
      tail_by_chunk[i] = tpos[j];
      long long l = comp_offsets[i + 1] - comp_offsets[i];
      long long raw = (chunk_rows[i + 1] - chunk_rows[i]) * row_bytes;
      uint32_t sb = rd32(t), k = rd32(t + 4), magic = rd32(t + 8);
      if ((magic != IDX_MAGIC_V1 && magic != IDX_MAGIC_V2) || sb == 0 || k == 0) continue;
      if ((long long)k != (raw + sb - 1) / sb) continue;
      // second format: {sub-block bytes, step bytes} and the sub-block table lie before the k lengths
      long long extra = 0;
      if (magic == IDX_MAGIC_V2) {
        long long full = raw / sb, rem = raw - full * sb;
        extra = 8 + 4 * (full * idx_n_sub(sb) + (rem ? idx_n_sub(rem) : 0));
      }
      if (8 + 4ll * k + INDEX_TAIL + extra >= l) continue;
      nseg[i] = (int)k; segb[i] = sb; idx_extra[i] = extra; idx_v2[i] = magic == IDX_MAGIC_V2;
      off2.push_back(comp_offsets[i + 1] - INDEX_TAIL - 4ll * k - extra - 4);   // adler32 | [sub table] | k lengths | [2 words]
      len2.push_back((int)(4 * k + 4 + extra));
      who2.push_back(i);
    }
    r = fetch_ranges(c, comp, comp_is_device, off2, len2, idx, ipos);
    if (r) return r;
    // validate: lengths must tile the stream body exactly, and match the checksum word
    std::vector<long long> ipos_by_chunk(n_chunks, -1);
    for (size_t j = 0; j < who2.size(); j++) {
      int i = who2[j];
      const unsigned char* p = idx.data() + ipos[j];
      const unsigned char* t = tails.data() + tail_by_chunk[i];
      long long l = comp_offsets[i + 1] - comp_offsets[i];
      unsigned long long sum = 0;
      bool ok = true;
      const unsigned char* lens = p + 4 + (idx_v2[i] ? idx_extra[i] - 8 : 0);    // after the adler32 and the sub-block table
      for (int q = 0; q < nseg[i]; q++) { uint32_t v = rd32(lens + 4 * q); if (v == 0) ok = false; sum += v; }
      if (!ok || (long long)sum != l - 8 - 4ll * nseg[i] - INDEX_TAIL - idx_extra[i] || (uint32_t)sum != rd32(t + 12)) { nseg[i] = 0; continue; }
      if (idx_v2[i]) {
        // the fast path needs the sub-block size this build uses and a sane step size; otherwise only the segment lengths are used
        const uint32_t subb = rd32(lens + 4 * nseg[i]), stepb = rd32(lens + 4 * nseg[i] + 4);
        const bool fast = subb == (uint32_t)IDX_SUB_BYTES && stepb >= 256 && stepb <= (uint32_t)IDX_SUB_BYTES / 2 && (stepb & (stepb - 1)) == 0;
        idx_step[i] = fast ? stepb : 0;
      }
      ipos_by_chunk[i] = ipos[j];
    }
    for (int i = 0; i < n_chunks; i++) if (nseg[i] && ipos_by_chunk[i] < 0) nseg[i] = 0;
    tpos.assign(ipos_by_chunk.begin(), ipos_by_chunk.end());   // reuse: tpos[i] = position of chunk i's index in idx
  }
  c->end();

  if (chunk_status) for (int i = 0; i < n_chunks; i++) chunk_status[i] = 0;
  bool any_bad = false;
  const bool host_io = !comp_is_device || !dst_is_device;
  // a sub-batch must also hold enough independent streams to fill the GPU: chunks without a segment index (e.g.
  // reference-written ones) are ONE serial stream each, so they are batched by count (up to 16 GiB of output).
  // Device-resident calls have nothing to overlap with: they take the largest sub-batches (measured on 600 chunks:
  // 2 GiB 62 GB/s, 4 GiB 75, 8 GiB 88, one 13.9 GB batch 96 — fewer, fuller waves of the block kernels)
  const long long min_streams = 8ll * c->sm_count, hard_limit = std::max<long long>(c->batch_bytes, 16ll << 30);
  const long long sb_limit = host_io ? std::min(c->batch_bytes, c->host_batch_bytes) : hard_limit;
  // index-less chunks with host buffers: equal sub-batches of about par_batch_bytes
  long long par_limit = std::max(sb_limit, c->par_batch_bytes);
  bool small_first = false;                 // several sub-batches of index-less chunks: start with a small one
  {
    long long total_par = 0, max_cb = 0;
    for (int i = 0; i < n_chunks; i++)
      if (!nseg[i]) { long long cb = (chunk_rows[i + 1] - chunk_rows[i]) * row_bytes; total_par += cb; max_cb = std::max(max_cb, cb); }
    const long long n_par = std::max<long long>(1, (total_par + par_limit / 2) / par_limit);
    par_limit = (total_par + n_par - 1) / n_par + max_cb;
    small_first = n_par > 1;
  }
  std::vector<int> sb_first;
  long long max_sb_bytes = 0, max_sb_comp = 0;
  for (int a = 0; a < n_chunks;) {
    sb_first.push_back(a);
    int b = a;
    long long bb = 0, streams = 0;
    while (b < n_chunks && b - a < 60000) {
      long long cb = (chunk_rows[b + 1] - chunk_rows[b]) * row_bytes;
      if (b > a && bb + cb > hard_limit) break;
      // index-less chunks decoded block-parallel have thousands of independent blocks: with host buffers they are
      // batched by bytes so that copies overlap the decode of the neighbouring sub-batches
      const bool par_b = host_io && c->par_inflate && !nseg[b];
      // (the first sub-batch is a quarter of the others: its decode is the one thing the download cannot overlap)
      if (b > a && par_b && bb + cb > ((a == 0 && small_first) ? par_limit / 4 : par_limit)) break;
      if (b > a && !par_b && bb + cb > sb_limit && streams >= min_streams) break;
      bb += cb; streams += nseg[b] ? nseg[b] : 1; b++;
    }
    max_sb_bytes = std::max(max_sb_bytes, bb);
    max_sb_comp = std::max(max_sb_comp, comp_offsets[b] - comp_offsets[a]);
    a = b;
  }
  sb_first.push_back(n_chunks);
  const int n_sb = (int)sb_first.size() - 1;
  Buf* comp_buf[2] = {&c->d_comp, &c->d_comp2};
  Buf* out_buf[2] = {&c->d_out, &c->d_out2};
  if (!comp_is_device) { NEED(c->d_comp, (size_t)max_sb_comp + 256); if (n_sb > 1) NEED(c->d_comp2, (size_t)max_sb_comp + 256); }
  if (!dst_is_device) { NEED(c->d_out, (size_t)max_sb_bytes + 256); if (n_sb > 1) NEED(c->d_out2, (size_t)max_sb_bytes + 256); }
  if (!comp_is_device) {
    CK(cudaEventRecord(c->ev_done, c->stream));
    CK(cudaStreamWaitEvent(c->copy_in, c->ev_done, 0));
    CK(cudaMemcpyAsync(comp_buf[0]->p, comp + comp_offsets[0], (size_t)(comp_offsets[sb_first[1]] - comp_offsets[0]),
                       cudaMemcpyHostToDevice, c->copy_in));
    CK(cudaEventRecord(c->ev_in[0], c->copy_in));
  }
  for (int k = 0; k < n_sb; k++) {
    const int c0 = sb_first[k], c1 = sb_first[k + 1];
    const long long bbytes = (chunk_rows[c1] - chunk_rows[c0]) * row_bytes;
    const int nb = c1 - c0;
    const long long row0 = chunk_rows[c0];
    const long long comp0 = comp_offsets[c0], comp_bytes = comp_offsets[c1] - comp0;
    std::vector<ChunkDesc> cds(nb);
    std::vector<InflateSeg> segs;
    std::vector<AdlerSeg> as;
    std::vector<int> first(nb + 1), first_inf(nb + 1), whole, v2_ids;
    std::vector<SegV2> v2;
    std::vector<uint32_t> want_adler(nb, 0);
    int max_ns = 0;
    const int ASEG = 1 << 16;
    for (int i = 0; i < nb; i++) {
      int g = c0 + i;
      long long ns = chunk_rows[g + 1] - chunk_rows[g], raw = ns * row_bytes;
      cds[i].elem_off = (chunk_rows[g] - row0) * nc;
      cds[i].ns = (int)ns; cds[i].first_seg = 0; cds[i].n_seg = 0; cds[i].pad_ = 0;
      max_ns = std::max(max_ns, (int)ns);
      long long tbase = cds[i].elem_off * itemsize;
      long long cbase = comp_offsets[g] - comp0, clen = comp_offsets[g + 1] - comp_offsets[g];
      first_inf[i] = (int)segs.size();
      if (nseg[g]) {
        const unsigned char* p = idx.data() + tpos[g];
        want_adler[i] = ((uint32_t)p[0] << 24) | (p[1] << 16) | (p[2] << 8) | p[3];
        const unsigned char* lens = p + 4 + (idx_v2[g] ? idx_extra[g] - 8 : 0);
        long long pos = cbase + 2;
        long long tab = cbase + clen - INDEX_TAIL - 4ll * nseg[g] - idx_extra[g];   // the chunk's sub-block table (second format)
        for (int j = 0; j < nseg[g]; j++) {
          InflateSeg s;
          s.in_off = pos; s.in_len = (int)rd32(lens + 4 * j);
          s.out_off = tbase + (long long)j * segb[g];
          s.out_len = (int)std::min<long long>(segb[g], raw - (long long)j * segb[g]);
          s.flags = 0; s.start_bit = 0; s.opos0 = 0; s.pad_ = 0;
          if (idx_step[g] && c->seg_v2 && c->par_inflate && s.in_len < (1 << 28)) {
            SegV2 v;
            v.in_off = s.in_off; v.out_off = s.out_off; v.tab_off = tab; v.in_len = s.in_len; v.out_len = s.out_len;
            v.sub_first = 0; v.step_bytes = idx_step[g];
            v2.push_back(v);
            v2_ids.push_back((int)segs.size());
          }
          tab += 4ll * idx_n_sub(s.out_len);
          pos += s.in_len;
          segs.push_back(s);
        }
      } else {
        InflateSeg s;
        s.in_off = cbase; s.in_len = (int)clen; s.out_off = tbase; s.out_len = (int)raw; s.flags = INF_ZLIB;
        s.start_bit = 0; s.opos0 = 0; s.pad_ = 0;
        whole.push_back((int)segs.size());
        segs.push_back(s);
      }
    }
    first_inf[nb] = (int)segs.size();
    const int n_segs = (int)segs.size();
    NEED(c->d_T, (size_t)bbytes + 16384);
    c->begin(0);
    if (!comp_is_device && k + 1 < n_sb) {
      const int a = sb_first[k + 1], b = sb_first[k + 2];
      CK(cudaMemcpyAsync(comp_buf[(k + 1) & 1]->p, comp + comp_offsets[a], (size_t)(comp_offsets[b] - comp_offsets[a]),
                         cudaMemcpyHostToDevice, c->copy_in));
      CK(cudaEventRecord(c->ev_in[(k + 1) & 1], c->copy_in));
    }
    const unsigned char* dcomp = comp + comp0;
    if (!comp_is_device) {
      CK(cudaStreamWaitEvent(c->stream, c->ev_in[k & 1], 0));
      dcomp = (const unsigned char*)comp_buf[k & 1]->p;
    }
    c->end();
    c->begin(2);
    c->lz_adler.assign(n_segs, 0);
    c->lz_adler_have.assign(n_segs, 0);
    // (the block kernels address bits with 32-bit offsets: streams of 256 MB and more stay with the serial decoder)
    const int PAR_MAX_IN = 1 << 28;
    if (c->par_inflate && !whole.empty()) {
      long long whole_in = 0;
      std::vector<int> fit;
      for (int w : whole) if (segs[w].in_len < PAR_MAX_IN) { whole_in += segs[w].in_len; fit.push_back(w); }
      if (whole_in >= 65536) { int r = par_phase(c, dcomp, segs, fit, (unsigned char*)c->d_T.p); if (r) return r; }
    }
    std::vector<uint32_t> v2_ad;
    std::vector<char> v2_ok;
    if (!v2_ids.empty()) { int r = par_phase_v2(c, dcomp, segs, v2_ids, v2, (unsigned char*)c->d_T.p, v2_ad, v2_ok); if (r) return r; }
    if (c->par_inflate && c->par_indexed && (int)whole.size() < n_segs) {
      std::vector<int> ids;
      size_t wi = 0, vi = 0;
      for (int j = 0; j < n_segs; j++) {
        if (wi < whole.size() && whole[wi] == j) { wi++; continue; }
        if (vi < v2_ids.size() && v2_ids[vi] == j) { vi++; if (segs[j].flags & INF_RESUME) continue; }   // done by the second-format kernels
        if (segs[j].in_len < PAR_MAX_IN) ids.push_back(j);
      }
      int r = par_phase_indexed(c, dcomp, segs, ids, (unsigned char*)c->d_T.p);
      if (r) return r;
    }
    // adler32 of each chunk's transformed bytes: folded on the host from the segments' sums where the second-format
    // kernels produced every segment of the chunk, taken from par_lz_kernel where it produced a plain stream completely,
    // computed by the adler kernels otherwise
    std::vector<uint32_t> host_adler(nb, 0);
    std::vector<char> have_adler(nb, 0);
    {
      size_t vi = 0;
      for (int i = 0; i < nb; i++) {
        bool all = first_inf[i + 1] > first_inf[i];
        uint32_t a = 1;
        for (int j = first_inf[i]; j < first_inf[i + 1]; j++) {
          while (vi < v2_ids.size() && v2_ids[vi] < j) vi++;
          if (vi < v2_ids.size() && v2_ids[vi] == j && v2_ok[vi]) {
            const uint32_t a2 = v2_ad[vi], len2 = (uint32_t)segs[j].out_len;
            const uint32_t s1a = a & 0xffff, s2a = a >> 16, s1b = a2 & 0xffff, s2b = a2 >> 16;
            const uint32_t s1 = (s1a + s1b + ADLER_BASE - 1) % ADLER_BASE;
            const unsigned long long t = (unsigned long long)(len2 % ADLER_BASE) * ((s1a + ADLER_BASE - 1) % ADLER_BASE);
            a = ((uint32_t)((s2a + s2b + t) % ADLER_BASE) << 16) | s1;
          } else { all = false; break; }
        }
        if (!nseg[c0 + i] && first_inf[i + 1] == first_inf[i] + 1 && c->lz_adler_have[first_inf[i]]) {
          all = true; a = c->lz_adler[first_inf[i]];          // a plain stream that par_lz_kernel produced completely
        }
        if (all) { have_adler[i] = 1; host_adler[i] = a; }
        const long long raw = (long long)cds[i].ns * row_bytes, tbase = cds[i].elem_off * itemsize;
        first[i] = (int)as.size();
        if (!all) for (long long o = 0; o < raw; o += ASEG) as.push_back(AdlerSeg{tbase + o, (int)std::min<long long>(ASEG, raw - o), 0});
      }
      first[nb] = (int)as.size();
    }
    const int n_as = (int)as.size();
    size_t o_cd = 0, o_seg = (o_cd + nb * sizeof(ChunkDesc) + 255) & ~(size_t)255;
    size_t o_as = (o_seg + n_segs * sizeof(InflateSeg) + 255) & ~(size_t)255;
    size_t o_first = (o_as + n_as * sizeof(AdlerSeg) + 255) & ~(size_t)255;
    size_t tab_bytes = o_first + (nb + 1) * sizeof(int);
    NEED(c->h_tab, tab_bytes);
    NEED(c->d_tab, tab_bytes);
    char* h = (char*)c->h_tab.p;
    memcpy(h + o_cd, cds.data(), nb * sizeof(ChunkDesc));
    memcpy(h + o_seg, segs.data(), n_segs * sizeof(InflateSeg));
    memcpy(h + o_as, as.data(), n_as * sizeof(AdlerSeg));
    memcpy(h + o_first, first.data(), (nb + 1) * sizeof(int));
    NEED(c->d_status, (size_t)n_segs * 4);
    NEED(c->d_tadler, (size_t)n_segs * 4);
    NEED(c->d_seg_adler, (size_t)n_as * 4 + 64);
    NEED(c->d_chunk_adler, (size_t)nb * 4);
    NEED(c->h_small, (size_t)n_segs * 8 + (size_t)nb * 4 + 128);
    const char* d = (const char*)c->d_tab.p;
    const ChunkDesc* d_cd = (const ChunkDesc*)(d + o_cd);
    { int rc_ = small_copy(c, c->d_tab.p, h, tab_bytes); if (rc_) return rc_; }
    // segments the second-format kernels finished completely need nothing from the serial kernel
    int n_serial = 0;
    for (const InflateSeg& sg : segs)
      if (!((sg.flags & INF_RESUME) && !(sg.flags & INF_ZLIB) && sg.opos0 >= (unsigned)sg.out_len)) n_serial++;
    if (!n_serial) {
      CK(cudaMemsetAsync(c->d_status.p, 0, (size_t)n_segs * 4, c->stream));
    } else if (n_segs >= 6 * c->sm_count) {
      // many short streams: global-memory window, 2 warps per CTA, up to 64 warps per SM
      auto k = inflate_kernel<false, 2>;
      MTS_LAUNCH(k, dim3((n_segs + 1) / 2), dim3(64), 0, c->stream, dcomp, (const InflateSeg*)(d + o_seg), n_segs, (unsigned char*)c->d_T.p, (int*)c->d_status.p, (unsigned*)c->d_tadler.p);
      c->launches++;
    } else {
      // few long streams: shared-memory window, one warp per CTA
      auto k = inflate_kernel<true, 1>;
      MTS_LAUNCH(k, dim3(n_segs), dim3(32), 0, c->stream, dcomp, (const InflateSeg*)(d + o_seg), n_segs, (unsigned char*)c->d_T.p, (int*)c->d_status.p, (unsigned*)c->d_tadler.p);
      c->launches++;
    }
    CKL();
    c->end();
    c->begin(3);
    if (n_as) {
      MTS_LAUNCH(adler_partial_kernel, dim3(n_as), dim3(256), 0, c->stream, (const uint8_t*)c->d_T.p, (const AdlerSeg*)(d + o_as), (uint32_t*)c->d_seg_adler.p);
      CKL();
    }
    MTS_LAUNCH(adler_combine_kernel, dim3((nb + 127) / 128), dim3(128), 0, c->stream, (const AdlerSeg*)(d + o_as), (const uint32_t*)c->d_seg_adler.p, (const int*)(d + o_first), nb, (uint32_t*)c->d_chunk_adler.p);
    CKL();
    c->launches += 2;
    c->end();
    void* outp;
    if (dst_is_device) outp = (char*)dst + row0 * row_bytes;
    else {
      if (k >= 2) CK(cudaStreamWaitEvent(c->stream, c->ev_out[k & 1], 0));   // D2H of sub-batch k-2 has drained it
      outp = out_buf[k & 1]->p;
    }
    c->begin(4);
    int r = launch_inv(c, itemsize, c->d_T.p, outp, d_cd, nb, max_ns, nc, flags, (size_t)(bbytes / itemsize));
    if (r) return r;
    c->end();
    char* hs = (char*)c->h_small.p;
    const size_t so_t = ((size_t)n_segs * 4 + 15) & ~(size_t)15, so_c = so_t + (((size_t)n_segs * 4 + 15) & ~(size_t)15);
    { int rc_ = small_copy(c, hs, c->d_status.p, (size_t)n_segs * 4); if (rc_) return rc_; }
    { int rc_ = small_copy(c, hs + so_t, c->d_tadler.p, (size_t)n_segs * 4); if (rc_) return rc_; }
    { int rc_ = small_copy(c, hs + so_c, c->d_chunk_adler.p, (size_t)nb * 4); if (rc_) return rc_; }
    CK(cudaStreamSynchronize(c->stream));
    if (!dst_is_device) {
      CK(cudaMemcpyAsync((char*)dst + row0 * row_bytes, outp, (size_t)bbytes, cudaMemcpyDeviceToHost, c->copy_out));
      CK(cudaEventRecord(c->ev_out[k & 1], c->copy_out));
    }
    const int* st = (const int*)hs;
    const uint32_t* ta = (const uint32_t*)(hs + so_t);
    const uint32_t* ca = (const uint32_t*)(hs + so_c);
    for (int i = 0; i < nb; i++) {
      int s = 0;
      for (int j = first_inf[i]; j < first_inf[i + 1] && !s; j++) s = st[j];
      if (!s) {
        uint32_t want = nseg[c0 + i] ? want_adler[i] : ta[first_inf[i]];
        if (want != (have_adler[i] ? host_adler[i] : ca[i])) s = INF_BAD_ADLER;
      }
      if (s) any_bad = true;
      if (chunk_status) chunk_status[c0 + i] = s;
    }
  }
  if (!dst_is_device) CK(cudaStreamSynchronize(c->copy_out));
  c->collect_timing();
  if (any_bad && chunk_status && !c->ignore_index) {
    // A chunk that carries something that looks like an index but does not decode with it (bytes after a foreign zlib
    // stream that happen to pass the index checks) is still a valid chunk for zlib, which ignores what follows the
    // stream: decode it again as a plain stream before calling it corrupt.
    any_bad = false;
    for (int i = 0; i < n_chunks; i++) {
      if (!chunk_status[i]) continue;
      if (!nseg[i]) { any_bad = true; continue; }
      const long long one_off[2] = {0, comp_offsets[i + 1] - comp_offsets[i]}, one_rows[2] = {0, chunk_rows[i + 1] - chunk_rows[i]};
      int st = 0;
      c->ignore_index = true;
      const int rc = mtsb_decompress_chunks(c, comp + comp_offsets[i], comp_is_device, one_off, 1, one_rows, nc, itemsize, flags,
                                            (char*)dst + chunk_rows[i] * row_bytes, dst_is_device, &st);
      c->ignore_index = false;
      if (rc != 0 && rc != MTSB_E_CORRUPT) return rc;
      chunk_status[i] = st;
      if (st) any_bad = true;
    }
  }
  if (any_bad) return fail(c, MTSB_E_CORRUPT, "at least one compressed chunk is corrupted");
  return 0;
}

}  // extern "C"
