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
#include "verify.cuh"

using namespace mts;

namespace {

thread_local std::string g_err;
int fail(mtsb_ctx* c, int code, const char* fmt, ...);

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


struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  bool host = false;
  Buf() = default;
  Buf(const Buf&) = delete;
  Buf& operator=(const Buf&) = delete;
  ~Buf() { release(); }
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

// The double-buffered copy pipeline of the host-buffer paths.  Sub-batch k's input goes up on copy_in into in[k & 1]
// while the kernels work on the sub-batch before it, and its output comes down on copy_out from out[k & 1] while they
// work on the next one.  A side whose pair is null is device memory that the kernels use in place.
struct CopyPipe {
  cudaStream_t stream = nullptr, copy_in = nullptr, copy_out = nullptr;   // the kernels' stream, H2D, D2H
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr}, ev_done = nullptr;
  Buf* in[2] = {nullptr, nullptr};     // the buffer pairs of the call in progress
  Buf* out[2] = {nullptr, nullptr};
  Buf* ref[2] = {nullptr, nullptr};
  CopyPipe() = default;
  CopyPipe(const CopyPipe&) = delete;
  bool create(cudaStream_t compute) {
    stream = compute;
    if (cudaStreamCreateWithFlags(&copy_in, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&copy_out, cudaStreamNonBlocking) != cudaSuccess) return false;
    for (int i = 0; i < 2; i++) { cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming); cudaEventCreateWithFlags(&ev_out[i], cudaEventDisableTiming); }
    cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming);
    return true;
  }
  ~CopyPipe() {
    for (int i = 0; i < 2; i++) { if (ev_in[i]) cudaEventDestroy(ev_in[i]); if (ev_out[i]) cudaEventDestroy(ev_out[i]); }
    if (ev_done) cudaEventDestroy(ev_done);
    if (copy_in) cudaStreamDestroy(copy_in);
    if (copy_out) cudaStreamDestroy(copy_out);
  }
  // takes the call's pairs (NEEDed by the caller) and queues the upload of sub-batch 0.  ref0 / ref1: a second input
  // pair (the reference rows of a verify call with a host reference), uploaded with the first and ready with it
  int start(mtsb_ctx* c, Buf* in0, Buf* in1, Buf* out0, Buf* out1, const void* src0, size_t bytes0, Buf* ref0 = nullptr,
            Buf* ref1 = nullptr, const void* ref_src0 = nullptr, size_t ref_bytes0 = 0) {
    in[0] = in0; in[1] = in1; out[0] = out0; out[1] = out1; ref[0] = ref0; ref[1] = ref1;
    if (!in[0] && !ref[0]) return 0;
    // the copy-in stream must not start before work already queued on the caller's stream (e.g. producing `src`)
    CK(cudaEventRecord(ev_done, stream));
    CK(cudaStreamWaitEvent(copy_in, ev_done, 0));
    return upload(c, 0, src0, bytes0, ref_src0, ref_bytes0);
  }
  int upload(mtsb_ctx* c, int k, const void* src, size_t bytes, const void* ref_src = nullptr, size_t ref_bytes = 0) {
    if (!in[0] && !ref[0]) return 0;                 // queues the upload of sub-batch k
    if (in[0]) CK(cudaMemcpyAsync(in[k & 1]->p, src, bytes, cudaMemcpyHostToDevice, copy_in));
    if (ref[0]) CK(cudaMemcpyAsync(ref[k & 1]->p, ref_src, ref_bytes, cudaMemcpyHostToDevice, copy_in));
    CK(cudaEventRecord(ev_in[k & 1], copy_in));
    return 0;
  }
  // p (and r, with a reference pair): sub-batch k's input, once its upload is done
  int input(mtsb_ctx* c, int k, const void*& p, const void** r = nullptr) {
    if (in[0] || ref[0]) CK(cudaStreamWaitEvent(stream, ev_in[k & 1], 0));
    if (in[0]) p = in[k & 1]->p;
    if (ref[0] && r) *r = ref[k & 1]->p;
    return 0;
  }
  int output(mtsb_ctx* c, int k, void*& p) {        // p: where sub-batch k's output goes, once it is free
    if (!out[0]) return 0;
    if (k >= 2) CK(cudaStreamWaitEvent(stream, ev_out[k & 1], 0));   // D2H of sub-batch k-2 has drained it
    p = out[k & 1]->p;
    return 0;
  }
  int download(mtsb_ctx* c, int k, void* dst, size_t bytes) {   // queues the download of sub-batch k, whose kernels are done
    if (!out[0]) return 0;
    CK(cudaMemcpyAsync(dst, out[k & 1]->p, bytes, cudaMemcpyDeviceToHost, copy_out));
    CK(cudaEventRecord(ev_out[k & 1], copy_out));
    return 0;
  }
  int finish(mtsb_ctx* c) { if (out[0]) CK(cudaStreamSynchronize(copy_out)); return 0; }   // waits for the last download
};

// The sub-batches of a call: chunks [first[k], first[k + 1]); max_in / max_out: the largest input / output of one
struct Batches {
  std::vector<int> first;
  long long max_in = 0, max_out = 0;
  int count() const { return (int)first.size() - 1; }
};

}  // namespace

struct mtsb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  long long sm_count = 148;
  std::string err;
  // params
  long long par_inflate = 1;   // decode index-less zlib streams block-parallel (inflate_par.cuh)
  long long par_indexed = 1;    // indexed segments of GPU-written chunks also go through the block kernels
  long long par_cells = -1;     // index-less streams: -1 by stream count, 1 = blocks resolved in parallel into cells, 0 = chain of tiles
  long long par_lz_wide = -1;   // LZ resolve kernel shape: -1 by stream count, 1 = 1024-thread CTAs, 0 = 256-thread CTAs
  long long par_batch_bytes = 2ll << 30;   // host-buffer sub-batch of index-less chunks (output bytes): large enough to amortise the block search
  // last call: survivors of the block search, candidate blocks, chained blocks, streams resumed
  long long par_survivors = 0, par_candidates = 0, par_chained = 0, par_resumed = 0;
  long long seg_bytes = 262144, batch_bytes = 2ll << 30, host_batch_bytes = 512ll << 20, write_index = 1;
  CopyPipe io;
  long long lz_ctas_per_sm = 2;
  // device scratch
  Buf d_pstreams, d_surv, d_cand, d_pcount, d_tokens, d_cells, d_ptab, d_plist, d_pbad;   // block-parallel inflate scratch
  std::vector<uint32_t> lz_adler;   // per segment of the current sub-batch: adler32 left by par_lz_kernel ...
  std::vector<char> lz_adler_have;  // ... where it produced the whole stream
  Buf d_pieces;
  long long par_single_pass = 1;   // par_block_kernel keeps the tokens of its counting pass (see par_decode)
  Buf d_segv2, d_btab, d_subout;                                                          // indexed (second format) segments
  long long seg_v2 = 1;         // indexed segments of the second format go through seg_tokens / seg_resolve
  Buf d_raw, d_raw2, d_out2, d_comp2, d_T, d_tok, d_hist, d_codes, d_hdrs, d_tab, d_so, d_seg_adler, d_chunk_adler, d_chunk_off, d_out,
      d_partial, d_comp, d_status, d_tadler, d_gather, d_subabs, d_subtok, d_invstate, d_invcells;
  Buf d_ref, d_ref2, d_vcount;     // verify: the reference rows of a host reference (a pair), the per-chunk counters
  int inv_cells_isz = 0;           // element size of the launch that last wrote the look-back cells
  long long inv_epoch = 0;         // epoch of the last inv_tile_kernel launch (tags its look-back cells)
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
  ~mtsb_ctx() {
    for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
    if (own_stream) cudaStreamDestroy(stream);
  }
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

// A sub-batch's tables in one blob: each array starts at a 256-byte aligned offset.  stage() fills h_tab, upload()
// copies it to d_tab with one small_copy.
struct TableBlob {
  struct Part { const void* src; size_t off, bytes; };
  std::vector<Part> parts;
  size_t bytes = 0;
  template <class T> size_t add(const std::vector<T>& v) {
    const size_t off = (bytes + 255) & ~(size_t)255;
    parts.push_back(Part{v.data(), off, v.size() * sizeof(T)});
    bytes = off + v.size() * sizeof(T);
    return off;
  }
  int stage(mtsb_ctx* c) const {
    NEED(c->h_tab, bytes);
    NEED(c->d_tab, bytes);
    for (const Part& p : parts) if (p.bytes) memcpy((char*)c->h_tab.p + p.off, p.src, p.bytes);
    return 0;
  }
  int upload(mtsb_ctx* c) const { return small_copy(c, c->d_tab.p, c->h_tab.p, bytes); }
  template <class T> static const T* dev(const mtsb_ctx* c, size_t off) { return (const T*)((const char*)c->d_tab.p + off); }
};

// Device words read back at the end of a step: add() queues a small_copy of each area to the next 16-byte aligned
// offset of h_small (which the caller NEEDs large enough); after sync(), get(i) is the i-th area on the host.
struct ReadBack {
  mtsb_ctx* c;
  std::vector<size_t> off;
  size_t used = 0;
  int rc = 0;
  explicit ReadBack(mtsb_ctx* c_) : c(c_) {}
  void add(const void* dev, size_t bytes) {
    off.push_back(used);
    if (!rc) rc = small_copy(c, (char*)c->h_small.p + used, dev, bytes);
    used += (bytes + 15) & ~(size_t)15;
  }
  int sync() {
    if (rc) return rc;
    CK(cudaStreamSynchronize(c->stream));
    return 0;
  }
  template <class T> const T* get(int i) const { return (const T*)((const char*)c->h_small.p + off[i]); }
};

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

// The compare of a verify sub-batch: decoded rows `dec` against reference rows `ref` (both from the sub-batch's first
// row), per-chunk counters into d_vcount = [count nb][first nb]
template <class T>
int launch_verify_t(mtsb_ctx* c, const void* dec, const void* ref, const ChunkDesc* d_cd, int nb, int max_ns, int nc,
                    double rtol, double atol) {
  const long long tiles = ((long long)max_ns * nc * (long long)sizeof(T) + VERIFY_TILE_BYTES - 1) / VERIFY_TILE_BYTES;
  unsigned long long* cnt = (unsigned long long*)c->d_vcount.p;
  long long* fst = (long long*)c->d_vcount.p + nb;
  CK(cudaMemsetAsync(cnt, 0, (size_t)nb * 8, c->stream));
  CK(cudaMemsetAsync(fst, 0x7f, (size_t)nb * 8, c->stream));
  auto k = verify_kernel<T>;
  MTS_LAUNCH(k, dim3((unsigned)tiles, nb), dim3(VERIFY_THREADS), 0, c->stream, (const T*)dec, (const T*)ref, d_cd, nc, (T)rtol,
             (T)atol, cnt, fst);
  c->launches++;
  CKL();
  return 0;
}
int launch_verify(mtsb_ctx* c, int isz, int flags, const void* dec, const void* ref, const ChunkDesc* d_cd, int nb, int max_ns,
                  int nc, double rtol, double atol) {
  if (flags & FLAG_FLOAT) {
    if (isz == 4) return launch_verify_t<float>(c, dec, ref, d_cd, nb, max_ns, nc, rtol, atol);
    return launch_verify_t<double>(c, dec, ref, d_cd, nb, max_ns, nc, rtol, atol);
  }
  switch (isz) {
    case 1: return launch_verify_t<uint8_t>(c, dec, ref, d_cd, nb, max_ns, nc, 0, 0);
    case 2: return launch_verify_t<uint16_t>(c, dec, ref, d_cd, nb, max_ns, nc, 0, 0);
    case 4: return launch_verify_t<uint32_t>(c, dec, ref, d_cd, nb, max_ns, nc, 0, 0);
  }
  return launch_verify_t<uint64_t>(c, dec, ref, d_cd, nb, max_ns, nc, 0, 0);
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

// mtsb_set_param / mtsb_get_param: the named fields and how a value is checked before it is stored
// (P_RANGE: lo..hi else an error, P_MIN: at least lo else an error, P_CLAMP: clamped to lo..hi, P_BOOL: 0 / 1,
// P_TRI: -1 automatic / 0 / 1, P_WORD: an unsigned 32-bit word, P_READ_ONLY: statistics and properties)
enum ParamRule { P_RANGE, P_MIN, P_CLAMP, P_BOOL, P_TRI, P_WORD, P_READ_ONLY };
struct Param { const char* name; long long mtsb_ctx::*field; ParamRule rule; long long lo, hi; };
const Param PARAMS[] = {
    {"seg_bytes", &mtsb_ctx::seg_bytes, P_RANGE, 4096, 1ll << 30},
    {"batch_bytes", &mtsb_ctx::batch_bytes, P_MIN, 1 << 20, 0},
    {"host_batch_bytes", &mtsb_ctx::host_batch_bytes, P_MIN, 1 << 20, 0},
    {"par_batch_bytes", &mtsb_ctx::par_batch_bytes, P_MIN, 1 << 20, 0},
    {"write_index", &mtsb_ctx::write_index, P_BOOL, 0, 0},
    {"par_inflate", &mtsb_ctx::par_inflate, P_BOOL, 0, 0},
    {"par_indexed", &mtsb_ctx::par_indexed, P_BOOL, 0, 0},
    {"par_single_pass", &mtsb_ctx::par_single_pass, P_BOOL, 0, 0},
    {"seg_v2", &mtsb_ctx::seg_v2, P_BOOL, 0, 0},
    {"inv_single_pass", &mtsb_ctx::inv_single_pass, P_BOOL, 0, 0},
    {"par_cells", &mtsb_ctx::par_cells, P_TRI, 0, 0},
    {"par_lz_wide", &mtsb_ctx::par_lz_wide, P_TRI, 0, 0},
    {"inv_order_block", &mtsb_ctx::inv_order_block, P_CLAMP, 1, 64},
    {"lz_ctas_per_sm", &mtsb_ctx::lz_ctas_per_sm, P_CLAMP, 1, 8},
    {"inv_epoch", &mtsb_ctx::inv_epoch, P_WORD, 0, 0},     // (tests: the wrap of the look-back epochs)
    {"par_survivors", &mtsb_ctx::par_survivors, P_READ_ONLY, 0, 0},
    {"par_candidates", &mtsb_ctx::par_candidates, P_READ_ONLY, 0, 0},
    {"par_chained", &mtsb_ctx::par_chained, P_READ_ONLY, 0, 0},
    {"par_resumed", &mtsb_ctx::par_resumed, P_READ_ONLY, 0, 0},
    {"sm_count", &mtsb_ctx::sm_count, P_READ_ONLY, 0, 0},
};
const Param* find_param(const char* name) {
  for (const Param& p : PARAMS)
    if (!strcmp(p.name, name)) return &p;
  return nullptr;
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
  if (!c->io.create(c->stream)) { fail(nullptr, MTSB_E_CUDA, "cudaStreamCreate failed"); mtsb_destroy(c); return nullptr; }
  if (set_attrs(c)) { g_err = c->err; mtsb_destroy(c); return nullptr; }
  return c;
}

void mtsb_destroy(mtsb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
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
  const Param* p = find_param(name);
  if (!p || p->rule == P_READ_ONLY) return fail(c, MTSB_E_ARG, "unknown parameter %s", name);
  switch (p->rule) {
    case P_RANGE: if (v < p->lo || v > p->hi) return fail(c, MTSB_E_ARG, "%s out of range", name); break;
    case P_MIN: if (v < p->lo) return fail(c, MTSB_E_ARG, "%s too small", name); break;
    case P_CLAMP: v = std::min(std::max(v, p->lo), p->hi); break;
    case P_BOOL: v = v ? 1 : 0; break;
    case P_TRI: v = v < 0 ? -1 : (v ? 1 : 0); break;
    case P_WORD: v = (unsigned)v; break;
    default: break;
  }
  c->*(p->field) = v;
  return 0;
}

long long mtsb_get_param(mtsb_ctx* c, const char* name) {
  if (!c || !name) return MTSB_E_ARG;
  const Param* p = find_param(name);
  if (!p) return MTSB_E_ARG;
  return c->*(p->field);
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
// Compress sub-batches: bounded by batch_bytes; smaller when a host buffer is involved so that copies pipeline with
// kernels.  Device-resident calls have nothing to overlap with: one large sub-batch keeps the persistent match-finder
// CTAs busy to the end (measured on 600 chunks: 2 GiB 99.9, 4 GiB 100.6, one 13.9 GB batch 101.7 GB/s).
// sb_limit: raw bytes per sub-batch (a single larger chunk forms its own)
static Batches plan_encode_batches(const mtsb_ctx* c, int n_chunks, const long long* chunk_rows, long long row_bytes,
                                   int itemsize, int flags, long long sb_limit) {
  Batches sb;
  for (int a = 0; a < n_chunks;) {
    sb.first.push_back(a);
    int b = a;
    long long bb = 0, bd = 0;
    while (b < n_chunks && b - a < 60000) {
      long long ns = chunk_rows[b + 1] - chunk_rows[b], cb = ns * row_bytes;
      if (b > a && bb + cb > sb_limit) break;
      bb += cb; bd += chunk_bound(c, cb, seg_size_for(c, ns, itemsize, flags)); b++;
    }
    sb.max_in = std::max(sb.max_in, bb);
    sb.max_out = std::max(sb.max_out, bd);
    a = b;
  }
  sb.first.push_back(n_chunks);
  return sb;
}

// One compress sub-batch: its chunks, their segments (the work units of the match finder and the encoder) and the
// table blob [ChunkDesc nb][DeflateSeg n_segs][AdlerSeg n_segs][first nb+1]
struct EncodeBatch {
  int nb = 0, max_ns = 0, n_subs = 0;
  long long bound = 0;            // worst-case output
  std::vector<ChunkDesc> cds;
  std::vector<DeflateSeg> segs;
  std::vector<AdlerSeg> as;       // the segments' bytes, for the per-chunk adler32 fold
  std::vector<int> first;         // chunk i's segments: [first[i], first[i + 1])
  TableBlob tab;
  size_t o_cd = 0, o_seg = 0, o_as = 0, o_first = 0;
};

// The part of encode sub-batch [c0, c1) before its table upload: plan and stage the tables, size the scratch.
// inflated: d_T already holds the sub-batch's transformed bytes (recompress), and h_small also takes the encoder's
// per-chunk adler32s.
static int plan_encode_sub_batch(mtsb_ctx* c, const long long* chunk_rows, int nc, int itemsize, int flags, int c0,
                                 int c1, bool inflated, EncodeBatch& b) {
  const long long row_bytes = (long long)nc * itemsize, row0 = chunk_rows[c0];
  b.nb = c1 - c0;
  b.cds.resize(b.nb);
  b.first.resize(b.nb + 1);
  for (int i = 0; i < b.nb; i++) {
    long long ns = chunk_rows[c0 + i + 1] - chunk_rows[c0 + i];
    long long raw = ns * row_bytes;
    long long seg = seg_size_for(c, ns, itemsize, flags);
    int k = (int)((raw + seg - 1) / seg);
    ChunkDesc& cd = b.cds[i];
    cd.elem_off = (chunk_rows[c0 + i] - row0) * nc;
    cd.ns = (int)ns;
    cd.first_seg = (int)b.segs.size();
    cd.n_seg = k;
    cd.pad_ = (int)seg;
    b.first[i] = (int)b.segs.size();
    b.max_ns = std::max(b.max_ns, (int)ns);
    long long base = cd.elem_off * itemsize;
    for (int j = 0; j < k; j++) {
      DeflateSeg s;
      s.in_off = base + (long long)j * seg;
      s.tok_off = s.in_off;
      s.in_len = (int)std::min<long long>(seg, raw - (long long)j * seg);
      s.chunk = i;
      s.flags = (j == 0 ? SEG_FIRST : 0) | (j == k - 1 ? SEG_LAST : 0);
      s.sub_first = b.n_subs;
      b.n_subs += idx_n_sub(s.in_len);
      b.segs.push_back(s);
    }
    b.bound += chunk_bound(c, raw, seg);
  }
  b.first[b.nb] = (int)b.segs.size();
  b.as.resize(b.segs.size());
  for (size_t i = 0; i < b.segs.size(); i++) b.as[i] = AdlerSeg{b.segs[i].in_off, b.segs[i].in_len, 0};
  b.o_cd = b.tab.add(b.cds);
  b.o_seg = b.tab.add(b.segs);
  b.o_as = b.tab.add(b.as);
  b.o_first = b.tab.add(b.first);
  const int nb = b.nb, n_segs = (int)b.segs.size();
  const size_t bbytes = (size_t)((chunk_rows[c1] - row0) * row_bytes);
  if (int r = b.tab.stage(c)) return r;
  if (!inflated) NEED(c->d_T, bbytes + 16384);
  NEED(c->d_tok, bbytes * 2 + 4096);
  NEED(c->d_hist, (size_t)n_segs * HIST_STRIDE * 4);
  NEED(c->d_codes, (size_t)n_segs * CODE_STRIDE * 4);
  NEED(c->d_hdrs, (size_t)n_segs * HDR_WORDS * 4);
  NEED(c->d_so, (size_t)n_segs * sizeof(DeflateSegOut));
  NEED(c->d_seg_adler, (size_t)n_segs * 4);
  NEED(c->d_chunk_adler, (size_t)nb * 4);
  NEED(c->d_chunk_off, (size_t)(nb + 1) * 8);
  NEED(c->d_subabs, (size_t)b.n_subs * 8 + 64);
  NEED(c->d_subtok, (size_t)b.n_subs * 8 + 64);
  NEED(c->h_small, (size_t)(nb + 1) * 8 + (inflated ? (size_t)nb * 4 + 64 : 0));
  return 0;
}

// The kernels that encode one sub-batch (its tables uploaded): forward transform of `raw` into d_T, match finder,
// per-chunk adler32, Huffman tables, output offsets (d_chunk_off), encoder and, with write_index, the index trailers.
// raw == nullptr: d_T already holds the transformed bytes (recompress), there is no transform, and the stages are timed
// in recompress's slots (lz77 4, the rest 5).
static int launch_encode(mtsb_ctx* c, const EncodeBatch& b, const void* raw, int nc, int itemsize, int flags,
                         unsigned char* outp) {
  const int nb = b.nb, n_segs = (int)b.segs.size();
  const ChunkDesc* d_cd = TableBlob::dev<ChunkDesc>(c, b.o_cd);
  const DeflateSeg* d_seg = TableBlob::dev<DeflateSeg>(c, b.o_seg);
  const AdlerSeg* d_as = TableBlob::dev<AdlerSeg>(c, b.o_as);
  const int* d_first = TableBlob::dev<int>(c, b.o_first);
  if (raw) {
    c->begin(1);
    if (int r = launch_fwd(c, itemsize, raw, c->d_T.p, d_cd, nb, b.max_ns, nc, flags)) return r;
    c->end();
  }
  c->begin(raw ? 3 : 4);
  {
    NEED(c->d_invstate, 256);
    CK(cudaMemsetAsync(c->d_invstate.p, 0, 64, c->stream));    // the match finder's segment counter
    const int grid = (int)std::min<long long>(n_segs, c->sm_count * c->lz_ctas_per_sm);
    auto k = itemsize == 2 ? lz77_kernel<2, LZ_NT> : lz77_kernel<1, LZ_NT>;
    const size_t smem = itemsize == 2 ? LzSmem<2, LZ_NT>::total : LzSmem<1, LZ_NT>::total;
    MTS_LAUNCH(k, dim3(grid), dim3(LZ_NT + 32), smem, c->stream, (const unsigned char*)c->d_T.p, d_seg, n_segs, (unsigned short*)c->d_tok.p, (unsigned*)c->d_hist.p, (DeflateSegOut*)c->d_so.p, (unsigned*)c->d_seg_adler.p, c->write_index ? (unsigned long long*)c->d_subtok.p : (unsigned long long*)nullptr, (unsigned*)c->d_invstate.p);
    CKL();
    c->launches++;
  }
  c->end();
  c->begin(raw ? 4 : 5);
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
  return 0;
}

// The rest of encode sub-batch k, its tables uploaded and its input ready: launch_encode into the copy pipeline's
// output, read back the chunk offsets, fill out_offsets and queue the download to dst + total_out, which it advances.
// want_adler (recompress): the adler32 each chunk's inflated bytes had, which the encoder's sums must equal.
static int encode_sub_batch(mtsb_ctx* c, const EncodeBatch& b, int k, int c0, const void* raw, int nc, int itemsize,
                            int flags, const uint32_t* want_adler, void* dst, long long& total_out, long long* out_offsets) {
  const int nb = b.nb;
  void* outp = (unsigned char*)dst + total_out;
  if (int r = c->io.output(c, k, outp)) return r;
  if (int r = launch_encode(c, b, raw, nc, itemsize, flags, (unsigned char*)outp)) return r;
  ReadBack rb(c);
  rb.add(c->d_chunk_off.p, (size_t)(nb + 1) * 8);
  if (want_adler) rb.add(c->d_chunk_adler.p, (size_t)nb * 4);
  if (int r = rb.sync()) return r;
  const long long* co = rb.get<long long>(0);
  if (co[nb] > b.bound) return fail(c, MTSB_E_CAPACITY, "internal: sub-batch output %lld exceeds bound %lld", co[nb], b.bound);
  // the match finder summed the bytes it read: they must be the bytes the decode stages produced and checked
  for (int i = 0; want_adler && i < nb; i++)
    if (rb.get<uint32_t>(1)[i] != want_adler[i])
      return fail(c, MTSB_E_CUDA, "internal: chunk %d: the encoder read bytes with adler32 %08x, the inflated ones have %08x",
                  c0 + i, rb.get<uint32_t>(1)[i], want_adler[i]);
  for (int i = 0; i < nb; i++) out_offsets[c0 + i + 1] = total_out + co[i + 1];
  // the kernels of this sub-batch are complete (synchronised above): drain it on the copy-out stream
  if (int r = c->io.download(c, k, (char*)dst + total_out, (size_t)co[nb])) return r;
  total_out += co[nb];
  return 0;
}

// dst_capacity must hold the worst-case output of every chunk
static int check_capacity(mtsb_ctx* c, int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags,
                          long long dst_capacity) {
  long long need = 0;
  for (int i = 0; i < n_chunks; i++) {
    long long ns = chunk_rows[i + 1] - chunk_rows[i];
    need += chunk_bound(c, ns * nc * itemsize, seg_size_for(c, ns, itemsize, flags));
  }
  if (dst_capacity < need) return fail(c, MTSB_E_CAPACITY, "dst_capacity %lld < bound %lld", dst_capacity, need);
  return 0;
}

int mtsb_compress_chunks(mtsb_ctx* c, const void* src, int src_is_device, int n_chunks, const long long* chunk_rows,
                         int nc, int itemsize, int flags, void* dst, int dst_is_device, long long dst_capacity,
                         long long* out_offsets) {
  if (!valid_common(c, n_chunks, chunk_rows, nc, itemsize) || !src || !dst || !out_offsets)
    return fail(c, MTSB_E_ARG, "compress_chunks: bad arguments");
  cudaSetDevice(c->device);
  c->reset_timing();
  const long long row_bytes = (long long)nc * itemsize;
  if (int r = check_capacity(c, n_chunks, chunk_rows, nc, itemsize, flags, dst_capacity)) return r;

  out_offsets[0] = 0;
  long long total_out = 0;
  const bool host_io = !src_is_device || !dst_is_device;
  const Batches sb = plan_encode_batches(c, n_chunks, chunk_rows, row_bytes, itemsize, flags,
                                         host_io ? std::min(c->batch_bytes, c->host_batch_bytes) : std::max<long long>(c->batch_bytes, 16ll << 30));
  const int n_sb = sb.count();
  if (!src_is_device) { NEED(c->d_raw, (size_t)sb.max_in + 256); if (n_sb > 1) NEED(c->d_raw2, (size_t)sb.max_in + 256); }
  if (!dst_is_device) { NEED(c->d_out, (size_t)sb.max_out + 256); if (n_sb > 1) NEED(c->d_out2, (size_t)sb.max_out + 256); }
  auto sb_src = [&](int k) { return (const char*)src + chunk_rows[sb.first[k]] * row_bytes; };
  auto sb_bytes = [&](int k) { return (size_t)((chunk_rows[sb.first[k + 1]] - chunk_rows[sb.first[k]]) * row_bytes); };
  CopyPipe& io = c->io;
  if (int r = io.start(c, src_is_device ? nullptr : &c->d_raw, &c->d_raw2, dst_is_device ? nullptr : &c->d_out, &c->d_out2, sb_src(0), sb_bytes(0)))
    return r;
  for (int k = 0; k < n_sb; k++) {
    const int c0 = sb.first[k];
    EncodeBatch b;
    if (int r = plan_encode_sub_batch(c, chunk_rows, nc, itemsize, flags, c0, sb.first[k + 1], false, b)) return r;
    c->begin(0);
    if (int r = b.tab.upload(c)) return r;
    // only now queue the next sub-batch's upload: the copy engine serves transfers in submission order, so the small
    // table upload above must not sit behind it
    if (k + 1 < n_sb) {
      if (int r = io.upload(c, k + 1, sb_src(k + 1), sb_bytes(k + 1))) return r;
    }
    const void* raw = sb_src(k);
    if (int r = io.input(c, k, raw)) return r;
    c->end();
    if (int r = encode_sub_batch(c, b, k, c0, raw, nc, itemsize, flags, nullptr, dst, total_out, out_offsets)) return r;
  }
  if (int r = io.finish(c)) return r;
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

// The arguments of one mtsb_decompress_chunks or mtsb_verify_chunks call (verify: the decoded rows go to scratch and are
// compared with `ref`; dst is unused)
struct DecodeArgs {
  const unsigned char* comp; int comp_is_device; const long long* comp_offsets;
  int n_chunks; const long long* chunk_rows; int nc, itemsize, flags;
  void* dst; int dst_is_device; long long row_bytes;
  bool verify = false;
  const void* ref = nullptr; int ref_is_device = 0; double rtol = 0, atol = 0;
  long long* mismatches = nullptr; long long* first_mismatch = nullptr;
};

// What read_indexes found behind a chunk's zlib stream (the index formats are written by trailer_kernel, deflate.cuh).
struct ChunkIndex {
  int n_seg = 0;                 // segments; 0: no usable index, the chunk is decoded as one plain zlib stream
  bool v2 = false;               // second format
  unsigned step = 0;             // second format: the step bytes of its fast path, 0 where the fast path cannot be taken
  long long seg_bytes = 0;       // output bytes of every segment but the last
  long long sub_bytes = 0;       // second format: bytes of the sub-block table and the {sub-block bytes, step bytes} words
  uint32_t adler = 0;            // stored adler32 of the chunk's transformed bytes
  long long tab_off = 0;         // second format: where the sub-block table starts, from the start of the chunk
  const unsigned char* lens = nullptr;   // the n_seg segment lengths (in the buffer read_indexes filled)
};

// Reads the index behind every chunk's zlib stream in two rounds: the 16-byte tails, then the adler32, sub-block table
// and lengths of the chunks whose tail is plausible.  An index is only used when its lengths tile the stream body
// exactly and match its checksum word; `bytes` holds what the records point to.
static int read_indexes(mtsb_ctx* c, const DecodeArgs& a, std::vector<ChunkIndex>& ix, std::vector<unsigned char>& bytes) {
  ix.assign(a.n_chunks, ChunkIndex());
  std::vector<long long> off, pos;
  std::vector<int> len, who;
  std::vector<unsigned char> tails;
  for (int i = 0; i < a.n_chunks; i++) {
    long long l = a.comp_offsets[i + 1] - a.comp_offsets[i];
    if (l >= 2 + 6 + 4 + INDEX_TAIL) { off.push_back(a.comp_offsets[i + 1] - INDEX_TAIL); len.push_back(INDEX_TAIL); who.push_back(i); }
  }
  if (int r = fetch_ranges(c, a.comp, a.comp_is_device, off, len, tails, pos)) return r;
  std::vector<int> who2;
  std::vector<uint32_t> sum_word(a.n_chunks, 0);
  off.clear();
  len.clear();
  for (size_t j = 0; j < who.size(); j++) {
    const unsigned char* t = tails.data() + pos[j];
    int i = who[j];
    long long l = a.comp_offsets[i + 1] - a.comp_offsets[i];
    long long raw = (a.chunk_rows[i + 1] - a.chunk_rows[i]) * a.row_bytes;
    uint32_t sb = rd32(t), k = rd32(t + 4), magic = rd32(t + 8);
    if ((magic != IDX_MAGIC_V1 && magic != IDX_MAGIC_V2) || sb == 0 || k == 0) continue;
    if ((long long)k != (raw + sb - 1) / sb) continue;
    // second format: the sub-block table lies before the k lengths, {sub-block bytes, step bytes} after them
    long long extra = 0;
    if (magic == IDX_MAGIC_V2) {
      long long full = raw / sb, rem = raw - full * sb;
      extra = 8 + 4 * (full * idx_n_sub(sb) + (rem ? idx_n_sub(rem) : 0));
    }
    if (8 + 4ll * k + INDEX_TAIL + extra >= l) continue;
    ChunkIndex& x = ix[i];
    x.n_seg = (int)k; x.seg_bytes = sb; x.sub_bytes = extra; x.v2 = magic == IDX_MAGIC_V2;
    x.tab_off = l - INDEX_TAIL - 4ll * k - extra;
    sum_word[i] = rd32(t + 12);
    off.push_back(a.comp_offsets[i + 1] - INDEX_TAIL - 4ll * k - extra - 4);   // adler32 | [sub table] | k lengths | [2 words]
    len.push_back((int)(4 * k + 4 + extra));
    who2.push_back(i);
  }
  if (int r = fetch_ranges(c, a.comp, a.comp_is_device, off, len, bytes, pos)) return r;
  // validate: lengths must tile the stream body exactly, and match the checksum word
  for (size_t j = 0; j < who2.size(); j++) {
    const int i = who2[j];
    ChunkIndex& x = ix[i];
    const unsigned char* p = bytes.data() + pos[j];
    long long l = a.comp_offsets[i + 1] - a.comp_offsets[i];
    unsigned long long sum = 0;
    bool ok = true;
    const unsigned char* lens = p + 4 + (x.v2 ? x.sub_bytes - 8 : 0);    // after the adler32 and the sub-block table
    for (int q = 0; q < x.n_seg; q++) { uint32_t v = rd32(lens + 4 * q); if (v == 0) ok = false; sum += v; }
    if (!ok || (long long)sum != l - 8 - 4ll * x.n_seg - INDEX_TAIL - x.sub_bytes || (uint32_t)sum != sum_word[i]) { x = ChunkIndex(); continue; }
    x.adler = ((uint32_t)p[0] << 24) | (p[1] << 16) | (p[2] << 8) | p[3];
    x.lens = lens;
    if (x.v2) {
      // the fast path needs the sub-block size this build uses and a sane step size; otherwise only the segment lengths are used
      const uint32_t subb = rd32(lens + 4 * x.n_seg), stepb = rd32(lens + 4 * x.n_seg + 4);
      const bool fast = subb == (uint32_t)IDX_SUB_BYTES && stepb >= 256 && stepb <= (uint32_t)IDX_SUB_BYTES / 2 && (stepb & (stepb - 1)) == 0;
      x.step = fast ? stepb : 0;
    }
  }
  return 0;
}

// Decompress sub-batches.  A sub-batch must also hold enough independent streams to fill the GPU: chunks without a
// segment index (e.g. reference-written ones) are ONE serial stream each, so they are batched by count (up to 16 GiB of
// output).  Device-resident calls have nothing to overlap with: they take the largest sub-batches (measured on 600
// chunks: 2 GiB 62 GB/s, 4 GiB 75, 8 GiB 88, one 13.9 GB batch 96 — fewer, fuller waves of the block kernels).
static Batches plan_decode_batches(const mtsb_ctx* c, const DecodeArgs& a, const std::vector<ChunkIndex>& ix) {
  const bool host_io = !a.comp_is_device || !(a.verify ? a.ref_is_device : a.dst_is_device);
  const long long min_streams = 8ll * c->sm_count, hard_limit = std::max<long long>(c->batch_bytes, 16ll << 30);
  const long long sb_limit = host_io ? std::min(c->batch_bytes, c->host_batch_bytes) : hard_limit;
  // index-less chunks with host buffers: equal sub-batches of about par_batch_bytes
  long long par_limit = std::max(sb_limit, c->par_batch_bytes);
  bool small_first = false;                 // several sub-batches of index-less chunks: start with a small one
  {
    long long total_par = 0, max_cb = 0;
    for (int i = 0; i < a.n_chunks; i++)
      if (!ix[i].n_seg) { long long cb = (a.chunk_rows[i + 1] - a.chunk_rows[i]) * a.row_bytes; total_par += cb; max_cb = std::max(max_cb, cb); }
    const long long n_par = std::max<long long>(1, (total_par + par_limit / 2) / par_limit);
    par_limit = (total_par + n_par - 1) / n_par + max_cb;
    small_first = n_par > 1;
  }
  Batches sb;
  for (int i0 = 0; i0 < a.n_chunks;) {
    sb.first.push_back(i0);
    int i1 = i0;
    long long bb = 0, streams = 0;
    while (i1 < a.n_chunks && i1 - i0 < 60000) {
      long long cb = (a.chunk_rows[i1 + 1] - a.chunk_rows[i1]) * a.row_bytes;
      if (i1 > i0 && bb + cb > hard_limit) break;
      // index-less chunks decoded block-parallel have thousands of independent blocks: with host buffers they are
      // batched by bytes so that copies overlap the decode of the neighbouring sub-batches
      const bool par_b = host_io && c->par_inflate && !ix[i1].n_seg;
      // (the first sub-batch is a quarter of the others: its decode is the one thing the download cannot overlap)
      if (i1 > i0 && par_b && bb + cb > ((i0 == 0 && small_first) ? par_limit / 4 : par_limit)) break;
      if (i1 > i0 && !par_b && bb + cb > sb_limit && streams >= min_streams) break;
      bb += cb; streams += ix[i1].n_seg ? ix[i1].n_seg : 1; i1++;
    }
    sb.max_out = std::max(sb.max_out, bb);
    sb.max_in = std::max(sb.max_in, a.comp_offsets[i1] - a.comp_offsets[i0]);
    i0 = i1;
  }
  sb.first.push_back(a.n_chunks);
  return sb;
}

// One decompress sub-batch: its chunks and their inflate segments, which segments each decode phase takes, and what
// the phases return
struct DecodeBatch {
  int c0 = 0, nb = 0, max_ns = 0;
  std::vector<ChunkDesc> cds;
  std::vector<InflateSeg> segs;
  std::vector<int> first;        // chunk i's segments: [first[i], first[i + 1])
  std::vector<int> whole;        // the segments that are a whole index-less chunk (plain zlib streams)
  std::vector<int> v2_ids;       // the segments the second-format kernels take, described by v2 ...
  std::vector<SegV2> v2;
  std::vector<uint32_t> v2_ad;   // ... and the adler32 of each that they produced (v2_ok)
  std::vector<char> v2_ok;
  std::vector<uint32_t> adler;   // per chunk: the adler32 of its transformed bytes where it is known on the host (have_adler)
  std::vector<char> have_adler;
  std::vector<AdlerSeg> as;      // the bytes the adler kernels sum for the other chunks: chunk i's [as_first[i], as_first[i + 1])
  std::vector<int> as_first;
  size_t o_cd = 0;               // where inflate_stages put the ChunkDesc table in d_tab
};

// Chunks [c0, c1) placed in d_T and in the device copy of the compressed bytes relative to chunk `base` (<= c0): the
// first chunk of the sub-batch whose buffers they are in
static void plan_segments(const mtsb_ctx* c, const DecodeArgs& a, const std::vector<ChunkIndex>& ix, int c0, int c1,
                          DecodeBatch& b, int base) {
  const long long row0 = a.chunk_rows[base], comp0 = a.comp_offsets[base];
  b.c0 = c0;
  b.nb = c1 - c0;
  b.cds.resize(b.nb);
  b.first.resize(b.nb + 1);
  for (int i = 0; i < b.nb; i++) {
    const int g = c0 + i;
    const ChunkIndex& x = ix[g];
    long long ns = a.chunk_rows[g + 1] - a.chunk_rows[g], raw = ns * a.row_bytes;
    ChunkDesc& cd = b.cds[i];
    cd.elem_off = (a.chunk_rows[g] - row0) * a.nc;
    cd.ns = (int)ns; cd.first_seg = 0; cd.n_seg = 0; cd.pad_ = 0;
    b.max_ns = std::max(b.max_ns, (int)ns);
    long long tbase = cd.elem_off * a.itemsize;
    long long cbase = a.comp_offsets[g] - comp0, clen = a.comp_offsets[g + 1] - a.comp_offsets[g];
    b.first[i] = (int)b.segs.size();
    if (!x.n_seg) {
      InflateSeg s;
      s.in_off = cbase; s.in_len = (int)clen; s.out_off = tbase; s.out_len = (int)raw; s.flags = INF_ZLIB;
      s.start_bit = 0; s.opos0 = 0; s.pad_ = 0;
      b.whole.push_back((int)b.segs.size());
      b.segs.push_back(s);
      continue;
    }
    long long pos = cbase + 2;
    long long tab = cbase + x.tab_off;   // the chunk's sub-block table (second format)
    for (int j = 0; j < x.n_seg; j++) {
      InflateSeg s;
      s.in_off = pos; s.in_len = (int)rd32(x.lens + 4 * j);
      s.out_off = tbase + (long long)j * x.seg_bytes;
      s.out_len = (int)std::min<long long>(x.seg_bytes, raw - (long long)j * x.seg_bytes);
      s.flags = 0; s.start_bit = 0; s.opos0 = 0; s.pad_ = 0;
      if (x.step && c->seg_v2 && c->par_inflate && s.in_len < (1 << 28)) {
        SegV2 v;
        v.in_off = s.in_off; v.out_off = s.out_off; v.tab_off = tab; v.in_len = s.in_len; v.out_len = s.out_len;
        v.sub_first = 0; v.step_bytes = x.step;
        b.v2.push_back(v);
        b.v2_ids.push_back((int)b.segs.size());
      }
      tab += 4ll * idx_n_sub(s.out_len);
      pos += s.in_len;
      b.segs.push_back(s);
    }
  }
  b.first[b.nb] = (int)b.segs.size();
}

// Records the block-parallel result `r` of segment `s`: unless no block of it was resolved or its tokens were
// inconsistent (then the serial kernel decodes it from its start), `s` becomes the tail that is left, with `flags`.
static bool resume_tail(mtsb_ctx* c, InflateSeg& s, const ParRes& r, int flags) {
  c->par_chained += r.n_done;
  if (r.n_done == 0 || (r.flags & 2)) return false;
  s.flags = flags;
  s.start_bit = r.tail_bit;
  s.opos0 = r.tail_out;
  c->par_resumed++;
  return true;
}

// The block-parallel decoder for the streams `ps` (segs[ids[i]] each).  blks == nullptr: plain zlib streams, the
// blocks are searched for on the device (find -> validate into per-stream buckets -> sort).  Otherwise blks holds one
// known block per stream (the indexed segments of GPU-written chunks).  No host round trip between the kernels: one
// synchronisation at the end fetches the per-stream results.  The streams whose chain of blocks was resolved are
// rewritten as INF_RESUME tails; the others are left untouched (full serial decode).
static int par_decode(mtsb_ctx* c, const unsigned char* dcomp, std::vector<InflateSeg>& segs, const std::vector<int>& ids,
                      const std::vector<ParStream>& ps, const std::vector<ParBlk>* blks, long long in_total, int max_in,
                      unsigned char* dT) {
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
  if (int r = small_copy(c, c->d_pstreams.p, c->h_tab.p, (size_t)ns * sizeof(ParStream))) return r;
  CK(cudaMemsetAsync(c->d_pcount.p, 0, 256, c->stream));           // [0] survivors, [4..5] token cursor
  const ParStream* d_ps = (const ParStream*)c->d_pstreams.p;
  unsigned* d_cnt = (unsigned*)c->d_pcount.p;
  if (blks) {
    memcpy((char*)c->h_tab.p + o_blk, blks->data(), n_slots * sizeof(ParBlk));
    if (int r = small_copy(c, c->d_plist.p, (char*)c->h_tab.p + o_blk, n_slots * sizeof(ParBlk))) return r;
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
  ReadBack rb(c);
  rb.add(c->d_pcount.p, 64);
  rb.add(c->d_pbad.p, (size_t)ns * sizeof(ParRes));
  if (!blks) rb.add(c->d_cand.p, (size_t)ns * 4);
  if (int r = rb.sync()) return r;
  if (!blks) {
    c->par_survivors += rb.get<unsigned>(0)[0];
    const unsigned* bcount = rb.get<unsigned>(2);
    for (int i = 0; i < ns; i++) c->par_candidates += bcount[i];
  }
  const int zflag = blks ? 0 : INF_ZLIB;
  const ParRes* res = rb.get<ParRes>(1);
  for (int sidx = 0; sidx < ns; sidx++) {
    const ParRes& r = res[sidx];
    InflateSeg& s = segs[ids[sidx]];
    if (!resume_tail(c, s, r, zflag | INF_RESUME | ((r.flags & 1) ? INF_NO_BLOCKS : 0))) continue;
    if ((r.flags & 4) && zflag && r.tail_out == (unsigned)s.out_len && (size_t)ids[sidx] < c->lz_adler.size()) {
      c->lz_adler[ids[sidx]] = r.adler;          // the whole stream went through par_lz_kernel: its adler32 is known
      c->lz_adler_have[ids[sidx]] = 1;
    }
  }
  return 0;
}

// Block-parallel decode of the segments `ids` (indices into segs) through par_decode.  indexed: the indexed segments of
// GPU-written chunks: every segment is one dynamic block at bit 0 followed by the empty stored block that byte-aligns
// the next segment (deflate.cuh), so the blocks are known without any search; a segment stored uncompressed simply
// fails the header parse and stays serial.  Otherwise: whole plain zlib streams, whose blocks are searched for.
static int par_phase(mtsb_ctx* c, const unsigned char* dcomp, std::vector<InflateSeg>& segs, const std::vector<int>& ids,
                     bool indexed, unsigned char* dT) {
  const int ns = (int)ids.size();
  std::vector<ParStream> ps(ns);
  std::vector<ParBlk> blks(indexed ? ns : 0);
  long long in_total = 0;
  int max_in = 0;
  for (int i = 0; i < ns; i++) {
    const InflateSeg& s = segs[ids[i]];
    ps[i].in_off = s.in_off; ps[i].out_off = s.out_off; ps[i].in_len = s.in_len; ps[i].out_len = s.out_len;
    ps[i].first_bit = indexed ? 0 : 16; ps[i].pad_ = 0;     // (after the zlib header)
    if (indexed) {
      ParBlk& b = blks[i];
      b.stream = (unsigned)i; b.bit = 0; b.limit = (unsigned)s.in_len * 8u;
      b.end_bit = 0; b.n_tok = 0; b.out_len = 0; b.flags = 0; b.pad_ = 0; b.tok_off = 0;
    }
    in_total += s.in_len;
    max_in = std::max(max_in, s.in_len);
  }
  return par_decode(c, dcomp, segs, ids, ps, indexed ? &blks : nullptr, in_total, max_in, dT);
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
    if (int r = small_copy(c, c->d_segv2.p, c->h_tab.p, (size_t)ns * sizeof(SegV2))) return r;
    MTS_LAUNCH(seg_tokens_kernel, dim3(ns), dim3(32), 0, c->stream, dcomp, (const SegV2*)c->d_segv2.p, (unsigned*)c->d_tokens.p,
               (uint2*)c->d_btab.p, (SubOut*)c->d_subout.p, (ParRes*)c->d_pbad.p);
    CKL();
    MTS_LAUNCH(seg_resolve_kernel, dim3(ns), dim3(SEG_RES_WARPS * 32), SMEM, c->stream, (const SegV2*)c->d_segv2.p,
               (const unsigned*)c->d_tokens.p, (const uint2*)c->d_btab.p, (const SubOut*)c->d_subout.p, dT, (ParRes*)c->d_pbad.p,
               (unsigned*)c->d_tadler.p);
    CKL();
    c->launches += 2;
    ReadBack rb(c);
    rb.add(c->d_pbad.p, (size_t)ns * sizeof(ParRes));
    rb.add(c->d_tadler.p, (size_t)ns * 4);
    if (int r = rb.sync()) return r;
    const ParRes* res = rb.get<ParRes>(0);
    const uint32_t* ad = rb.get<uint32_t>(1);
    for (int i = 0; i < ns; i++) {
      if (!resume_tail(c, segs[ids[a + i]], res[i], INF_RESUME)) continue;
      seg_ok[a + i] = 1;
      seg_ad[a + i] = ad[i];
    }
    a = b;
  }
  return 0;
}

// (the block kernels address bits with 32-bit offsets: streams of 256 MB and more stay with the serial decoder)
static const int PAR_MAX_IN = 1 << 28;

// The segments the block kernels take as indexed ones: all but the whole streams, the segments the second-format
// kernels turned into tails, and streams too long for them
static std::vector<int> indexed_for_blocks(const DecodeBatch& b) {
  std::vector<int> ids;
  size_t wi = 0, vi = 0;
  for (int j = 0; j < (int)b.segs.size(); j++) {
    if (wi < b.whole.size() && b.whole[wi] == j) { wi++; continue; }
    if (vi < b.v2_ids.size() && b.v2_ids[vi] == j) { vi++; if (b.segs[j].flags & INF_RESUME) continue; }
    if (b.segs[j].in_len < PAR_MAX_IN) ids.push_back(j);
  }
  return ids;
}

// The parallel decode phases of a sub-batch: plain streams, second-format segments, then the other indexed segments
static int par_phases(mtsb_ctx* c, const unsigned char* dcomp, DecodeBatch& b) {
  unsigned char* dT = (unsigned char*)c->d_T.p;
  c->lz_adler.assign(b.segs.size(), 0);
  c->lz_adler_have.assign(b.segs.size(), 0);
  if (c->par_inflate && !b.whole.empty()) {
    long long whole_in = 0;
    std::vector<int> fit;
    for (int w : b.whole) if (b.segs[w].in_len < PAR_MAX_IN) { whole_in += b.segs[w].in_len; fit.push_back(w); }
    if (whole_in >= 65536) { int r = par_phase(c, dcomp, b.segs, fit, false, dT); if (r) return r; }
  }
  if (!b.v2_ids.empty()) { int r = par_phase_v2(c, dcomp, b.segs, b.v2_ids, b.v2, dT, b.v2_ad, b.v2_ok); if (r) return r; }
  if (c->par_inflate && c->par_indexed && b.whole.size() < b.segs.size()) {
    if (int r = par_phase(c, dcomp, b.segs, indexed_for_blocks(b), true, dT)) return r;
  }
  return 0;
}

// adler32 of A | B from adler32(A), adler32(B) and the length of B
static uint32_t adler32_combine(uint32_t a, uint32_t b, uint32_t len_b) {
  const uint32_t s1a = a & 0xffff, s2a = a >> 16, s1b = b & 0xffff, s2b = b >> 16;
  const uint32_t s1 = (s1a + s1b + ADLER_BASE - 1) % ADLER_BASE;
  const unsigned long long t = (unsigned long long)(len_b % ADLER_BASE) * ((s1a + ADLER_BASE - 1) % ADLER_BASE);
  return ((uint32_t)((s2a + s2b + t) % ADLER_BASE) << 16) | s1;
}

// adler32 of each chunk's transformed bytes: folded on the host from the segments' sums where the second-format
// kernels produced every segment of the chunk, taken from par_lz_kernel where it produced a plain stream completely,
// summed by the adler kernels (b.as) otherwise
static void fold_adlers(const mtsb_ctx* c, const DecodeArgs& a, const std::vector<ChunkIndex>& ix, DecodeBatch& b) {
  const int ASEG = 1 << 16;
  b.adler.assign(b.nb, 0);
  b.have_adler.assign(b.nb, 0);
  b.as_first.resize(b.nb + 1);
  size_t vi = 0;
  for (int i = 0; i < b.nb; i++) {
    bool all = b.first[i + 1] > b.first[i];
    uint32_t ad = 1;
    for (int j = b.first[i]; j < b.first[i + 1]; j++) {
      while (vi < b.v2_ids.size() && b.v2_ids[vi] < j) vi++;
      if (vi < b.v2_ids.size() && b.v2_ids[vi] == j && b.v2_ok[vi]) ad = adler32_combine(ad, b.v2_ad[vi], (uint32_t)b.segs[j].out_len);
      else { all = false; break; }
    }
    if (!ix[b.c0 + i].n_seg && b.first[i + 1] == b.first[i] + 1 && c->lz_adler_have[b.first[i]]) {
      all = true; ad = c->lz_adler[b.first[i]];          // a plain stream that par_lz_kernel produced completely
    }
    if (all) { b.have_adler[i] = 1; b.adler[i] = ad; }
    const long long raw = (long long)b.cds[i].ns * a.row_bytes, tbase = b.cds[i].elem_off * a.itemsize;
    b.as_first[i] = (int)b.as.size();
    if (!all) for (long long o = 0; o < raw; o += ASEG) b.as.push_back(AdlerSeg{tbase + o, (int)std::min<long long>(ASEG, raw - o), 0});
  }
  b.as_first[b.nb] = (int)b.as.size();
}

// The serial inflate kernel over the segments (d_segs: their table on the device): it decodes the segments and tails
// the parallel phases left, checks every segment's end and writes its status and, for zlib streams, the trailer's adler32
static int serial_inflate(mtsb_ctx* c, const unsigned char* dcomp, const std::vector<InflateSeg>& segs, const InflateSeg* d_segs) {
  const int n_segs = (int)segs.size();
  // segments the second-format kernels finished completely need nothing from the serial kernel
  int n_serial = 0;
  for (const InflateSeg& sg : segs)
    if (!((sg.flags & INF_RESUME) && !(sg.flags & INF_ZLIB) && sg.opos0 >= (unsigned)sg.out_len)) n_serial++;
  if (!n_serial) {
    CK(cudaMemsetAsync(c->d_status.p, 0, (size_t)n_segs * 4, c->stream));
  } else if (n_segs >= 6 * c->sm_count) {
    // many short streams: global-memory window, 2 warps per CTA, up to 64 warps per SM
    auto k = inflate_kernel<false, 2>;
    MTS_LAUNCH(k, dim3((n_segs + 1) / 2), dim3(64), 0, c->stream, dcomp, d_segs, n_segs, (unsigned char*)c->d_T.p, (int*)c->d_status.p, (unsigned*)c->d_tadler.p);
    c->launches++;
  } else {
    // few long streams: shared-memory window, one warp per CTA
    auto k = inflate_kernel<true, 1>;
    MTS_LAUNCH(k, dim3(n_segs), dim3(32), 0, c->stream, dcomp, d_segs, n_segs, (unsigned char*)c->d_T.p, (int*)c->d_status.p, (unsigned*)c->d_tadler.p);
    c->launches++;
  }
  CKL();
  return 0;
}

// Each chunk's status: its first failing segment's, else INF_BAD_ADLER where the adler32 of its transformed bytes is not
// the stored one (the index's, or the zlib trailer's the serial kernel read: ta).  st: the segments' statuses, ca: the
// adler kernels' sums.  accepted (may be null): per chunk, the stored adler32 that a good chunk matched.
static void chunk_verdicts(const DecodeBatch& b, const std::vector<ChunkIndex>& ix, const int* st, const uint32_t* ta,
                           const uint32_t* ca, int* status, uint32_t* accepted) {
  for (int i = 0; i < b.nb; i++) {
    int s = 0;
    for (int j = b.first[i]; j < b.first[i + 1] && !s; j++) s = st[j];
    if (!s) {
      const ChunkIndex& x = ix[b.c0 + i];
      uint32_t want = x.n_seg ? x.adler : ta[b.first[i]];
      if (want != (b.have_adler[i] ? b.adler[i] : ca[i])) s = INF_BAD_ADLER;
      if (accepted) accepted[i] = want;
    }
    status[b.c0 + i] = s;
  }
}

// The rows of sub-batch k in the caller's `ref` (verify)
static const void* ref_rows(const DecodeArgs& a, const Batches& sb, int k) {
  return (const char*)a.ref + a.chunk_rows[sb.first[k]] * a.row_bytes;
}
static size_t batch_bytes_of(const DecodeArgs& a, const Batches& sb, int k) {
  return (size_t)((a.chunk_rows[sb.first[k + 1]] - a.chunk_rows[sb.first[k]]) * a.row_bytes);
}

// The decode stages that fill d_T for the planned segments of b (dcomp: the device copy of their compressed bytes):
// parallel phases, serial inflate, adler32s.  The statuses, trailer adler32s and sums are left in d_status, d_tadler
// and d_chunk_adler for chunk_verdicts.
static int inflate_stages(mtsb_ctx* c, const DecodeArgs& a, const std::vector<ChunkIndex>& ix, const unsigned char* dcomp,
                          DecodeBatch& b) {
  const int nb = b.nb, n_segs = (int)b.segs.size();
  c->begin(2);
  if (int r = par_phases(c, dcomp, b)) return r;
  fold_adlers(c, a, ix, b);
  TableBlob tab;
  const size_t o_cd = tab.add(b.cds), o_seg = tab.add(b.segs), o_as = tab.add(b.as), o_first = tab.add(b.as_first);
  b.o_cd = o_cd;
  if (int r = tab.stage(c)) return r;
  const int n_as = (int)b.as.size();
  NEED(c->d_status, (size_t)n_segs * 4);
  NEED(c->d_tadler, (size_t)n_segs * 4);
  NEED(c->d_seg_adler, (size_t)n_as * 4 + 64);
  NEED(c->d_chunk_adler, (size_t)nb * 4);
  NEED(c->h_small, (size_t)n_segs * 8 + (size_t)nb * 4 + 128);
  const AdlerSeg* d_as = TableBlob::dev<AdlerSeg>(c, o_as);
  if (int r = tab.upload(c)) return r;
  if (int r = serial_inflate(c, dcomp, b.segs, TableBlob::dev<InflateSeg>(c, o_seg))) return r;
  c->end();
  c->begin(3);
  if (n_as) {
    MTS_LAUNCH(adler_partial_kernel, dim3(n_as), dim3(256), 0, c->stream, (const uint8_t*)c->d_T.p, d_as, (uint32_t*)c->d_seg_adler.p);
    CKL();
  }
  MTS_LAUNCH(adler_combine_kernel, dim3((nb + 127) / 128), dim3(128), 0, c->stream, d_as, (const uint32_t*)c->d_seg_adler.p, TableBlob::dev<int>(c, o_first), nb, (uint32_t*)c->d_chunk_adler.p);
  CKL();
  c->launches += 2;
  c->end();
  return 0;
}

// Sub-batch k up to the filled d_T: its segments, the upload of sub-batch k+1 (and, verify, its reference rows), the
// wait for its own input (dcomp; ref: its reference rows), inflate_stages
static int inflate_batch(mtsb_ctx* c, const DecodeArgs& a, const std::vector<ChunkIndex>& ix, const Batches& sb, int k,
                         DecodeBatch& b, const unsigned char*& dcomp, const void*& ref) {
  CopyPipe& io = c->io;
  const int c0 = sb.first[k], c1 = sb.first[k + 1];
  const long long row0 = a.chunk_rows[c0], bbytes = (a.chunk_rows[c1] - row0) * a.row_bytes;
  plan_segments(c, a, ix, c0, c1, b, c0);
  NEED(c->d_T, (size_t)bbytes + 16384);
  c->begin(0);
  if (k + 1 < sb.count()) {
    const long long n0 = a.comp_offsets[sb.first[k + 1]], n1 = a.comp_offsets[sb.first[k + 2]];
    if (a.verify) {
      if (int r = io.upload(c, k + 1, a.comp + n0, (size_t)(n1 - n0), ref_rows(a, sb, k + 1), batch_bytes_of(a, sb, k + 1))) return r;
    } else if (int r = io.upload(c, k + 1, a.comp + n0, (size_t)(n1 - n0))) {
      return r;
    }
  }
  const void* in = a.comp + a.comp_offsets[c0];
  ref = a.verify ? ref_rows(a, sb, k) : nullptr;
  if (int r = io.input(c, k, in, &ref)) return r;
  dcomp = (const unsigned char*)in;
  c->end();
  return inflate_stages(c, a, ix, dcomp, b);
}

// The rows of b's chunks from d_T into outp (the sub-batch's first row; span_elems: the sub-batch's elements) and,
// verify, their compare with the sub-batch's reference rows `ref`
static int inverse_stages(mtsb_ctx* c, const DecodeArgs& a, const DecodeBatch& b, void* outp, const void* ref,
                          size_t span_elems) {
  const int nb = b.nb;
  const ChunkDesc* d_cd = TableBlob::dev<ChunkDesc>(c, b.o_cd);
  c->begin(4);
  if (int r = launch_inv(c, a.itemsize, c->d_T.p, outp, d_cd, nb, b.max_ns, a.nc, a.flags, span_elems)) return r;
  c->end();
  if (!a.verify) return 0;
  NEED(c->d_vcount, (size_t)nb * 16);
  NEED(c->h_small, b.segs.size() * 8 + (size_t)nb * 20 + 160);
  c->begin(6);
  if (int r = launch_verify(c, a.itemsize, a.flags, outp, ref, d_cd, nb, b.max_ns, a.nc, a.rtol, a.atol)) return r;
  c->end();
  return 0;
}

// One synchronisation for what the stages of b left on the device, then b's statuses (chunk_verdicts, `accepted` as
// there) and, verify, its compare counters
static int batch_verdicts(mtsb_ctx* c, const DecodeArgs& a, const std::vector<ChunkIndex>& ix, const DecodeBatch& b,
                          int* status, uint32_t* accepted = nullptr) {
  const int c0 = b.c0, nb = b.nb, n_segs = (int)b.segs.size();
  ReadBack rb(c);
  rb.add(c->d_status.p, (size_t)n_segs * 4);
  rb.add(c->d_tadler.p, (size_t)n_segs * 4);
  rb.add(c->d_chunk_adler.p, (size_t)nb * 4);
  if (a.verify) rb.add(c->d_vcount.p, (size_t)nb * 16);
  if (int r = rb.sync()) return r;
  chunk_verdicts(b, ix, rb.get<int>(0), rb.get<uint32_t>(1), rb.get<uint32_t>(2), status, accepted);
  if (a.verify) {
    const long long* cnt = rb.get<long long>(3);
    for (int i = 0; i < nb; i++) {
      const bool ok = status[c0 + i] == 0;
      a.mismatches[c0 + i] = ok ? cnt[i] : -1;
      a.first_mismatch[c0 + i] = !ok || cnt[nb + i] == VERIFY_NONE ? -1 : cnt[nb + i];
    }
  }
  return 0;
}

// A chunk that carries something that looks like an index but does not decode with it (bytes after a foreign zlib
// stream that happen to pass the index checks) is still a valid chunk for zlib, which ignores what follows the stream.
// Each such chunk of sub-batch b is inflated again alone as a plain stream into its own place in d_T (dcomp: the
// sub-batch's compressed bytes), its rows go to their place at outp as inverse_stages puts them (outp null: recompress,
// d_T only), and it gets a new verdict.  The sub-batch's buffers are still in their copy-pipeline slots: nothing of it
// has been downloaded yet, and the next uploads go to the other slot.
static int retry_misled(mtsb_ctx* c, const DecodeArgs& a, std::vector<ChunkIndex>& ix, const DecodeBatch& b,
                        const unsigned char* dcomp, void* outp, const void* ref, size_t span_elems, int* status,
                        uint32_t* accepted = nullptr) {
  for (int i = b.c0; i < b.c0 + b.nb; i++) {
    if (!status[i] || !ix[i].n_seg) continue;
    ix[i] = ChunkIndex();
    DecodeBatch one;
    plan_segments(c, a, ix, i, i + 1, one, b.c0);
    if (int r = inflate_stages(c, a, ix, dcomp, one)) return r;
    if (outp) {
      if (int r = inverse_stages(c, a, one, outp, ref, span_elems)) return r;
    }
    if (int r = batch_verdicts(c, a, ix, one, status, accepted ? accepted + (i - b.c0) : nullptr)) return r;
  }
  return 0;
}

// Sub-batch k: inflate_batch, inverse transform, verdicts, retry of misled chunks, download.  Verify: the inverse
// writes to scratch (d_out), the compare follows on the same stream and its counters come back with the verdicts.
static int decode_batch(mtsb_ctx* c, const DecodeArgs& a, std::vector<ChunkIndex>& ix, const Batches& sb, int k,
                        int* status) {
  DecodeBatch b;
  const unsigned char* dcomp = nullptr;
  const void* ref = nullptr;
  if (int r = inflate_batch(c, a, ix, sb, k, b, dcomp, ref)) return r;
  const long long row0 = a.chunk_rows[b.c0], bbytes = (a.chunk_rows[sb.first[k + 1]] - row0) * a.row_bytes;
  const size_t span_elems = (size_t)(bbytes / a.itemsize);
  void* outp = a.verify ? c->d_out.p : (char*)a.dst + row0 * a.row_bytes;
  if (!a.verify) {
    if (int r = c->io.output(c, k, outp)) return r;
  }
  if (int r = inverse_stages(c, a, b, outp, ref, span_elems)) return r;
  if (int r = batch_verdicts(c, a, ix, b, status)) return r;
  if (int r = retry_misled(c, a, ix, b, dcomp, outp, ref, span_elems, status)) return r;
  if (!a.verify) {
    if (int r = c->io.download(c, k, (char*)a.dst + row0 * a.row_bytes, (size_t)bbytes)) return r;
  }
  return 0;
}

// The start of every call that decodes (decompress, verify, recompress): the compressed lengths fit the kernels'
// 32-bit lengths and are not empty; timings and statistics restart; the segment index behind each chunk's zlib stream
// is read (timed in slot 1) into ix, whose records point into ix_bytes; all n_chunks statuses are 0.
static int start_decode_call(mtsb_ctx* c, const char* name, const DecodeArgs& a, int* status,
                             std::vector<ChunkIndex>& ix, std::vector<unsigned char>& ix_bytes) {
  for (int i = 0; i < a.n_chunks; i++) {
    long long l = a.comp_offsets[i + 1] - a.comp_offsets[i];
    if (l < 1 || l > 0x7fffffffll) return fail(c, MTSB_E_ARG, "%s: bad compressed length of chunk %d", name, i);
  }
  cudaSetDevice(c->device);
  c->reset_timing();
  c->par_survivors = c->par_candidates = c->par_chained = c->par_resumed = 0;
  c->begin(1);
  if (int r = read_indexes(c, a, ix, ix_bytes)) return r;
  c->end();
  for (int i = 0; i < a.n_chunks; i++) status[i] = 0;
  return 0;
}

// The body both batch decode entry points share: plan, sub-batches through the copy pipeline
static int decode_call(mtsb_ctx* c, const char* name, const DecodeArgs& a, int* chunk_status) {
  // every chunk's status, also when the caller does not ask for them
  std::vector<int> own_status(chunk_status ? 0 : a.n_chunks);
  int* status = chunk_status ? chunk_status : own_status.data();
  std::vector<ChunkIndex> ix;
  std::vector<unsigned char> ix_bytes;
  if (int r = start_decode_call(c, name, a, status, ix, ix_bytes)) return r;
  const Batches sb = plan_decode_batches(c, a, ix);
  const int n_sb = sb.count();
  if (!a.comp_is_device) { NEED(c->d_comp, (size_t)sb.max_in + 256); if (n_sb > 1) NEED(c->d_comp2, (size_t)sb.max_in + 256); }
  const bool host_rows = a.verify ? !a.ref_is_device : !a.dst_is_device;
  if (host_rows || a.verify) NEED(c->d_out, (size_t)sb.max_out + 256);   // verify: the decoded rows, one buffer
  if (host_rows && !a.verify && n_sb > 1) NEED(c->d_out2, (size_t)sb.max_out + 256);
  if (host_rows && a.verify) { NEED(c->d_ref, (size_t)sb.max_out + 256); if (n_sb > 1) NEED(c->d_ref2, (size_t)sb.max_out + 256); }
  const void* comp0 = a.comp + a.comp_offsets[0];
  const size_t comp_bytes0 = (size_t)(a.comp_offsets[sb.first[1]] - a.comp_offsets[0]);
  Buf* in0 = a.comp_is_device ? nullptr : &c->d_comp;
  int r0 = a.verify ? c->io.start(c, in0, &c->d_comp2, nullptr, nullptr, comp0, comp_bytes0, host_rows ? &c->d_ref : nullptr,
                                  &c->d_ref2, ref_rows(a, sb, 0), batch_bytes_of(a, sb, 0))
                    : c->io.start(c, in0, &c->d_comp2, host_rows ? &c->d_out : nullptr, &c->d_out2, comp0, comp_bytes0);
  if (r0) return r0;
  for (int k = 0; k < n_sb; k++)
    if (int r = decode_batch(c, a, ix, sb, k, status)) return r;
  if (int r = c->io.finish(c)) return r;
  c->collect_timing();
  for (int i = 0; i < a.n_chunks; i++)
    if (status[i]) return fail(c, MTSB_E_CORRUPT, "at least one compressed chunk is corrupted");
  return 0;
}

int mtsb_decompress_chunks(mtsb_ctx* c, const void* comp_, int comp_is_device, const long long* comp_offsets,
                           int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags, void* dst,
                           int dst_is_device, int* chunk_status) {
  if (!valid_common(c, n_chunks, chunk_rows, nc, itemsize) || !comp_ || !comp_offsets || !dst)
    return fail(c, MTSB_E_ARG, "decompress_chunks: bad arguments");
  const DecodeArgs a{(const unsigned char*)comp_, comp_is_device, comp_offsets, n_chunks, chunk_rows, nc, itemsize, flags, dst,
                     dst_is_device, (long long)nc * itemsize};
  return decode_call(c, "decompress_chunks", a, chunk_status);
}

int mtsb_verify_chunks(mtsb_ctx* c, const void* comp, int comp_is_device, const long long* comp_offsets, int n_chunks,
                       const long long* chunk_rows, int nc, int itemsize, int flags, const void* ref, int ref_is_device,
                       double rtol, double atol, long long* mismatches, long long* first_mismatch, int* chunk_status) {
  if (!valid_common(c, n_chunks, chunk_rows, nc, itemsize) || !comp || !comp_offsets || !ref || !mismatches ||
      !first_mismatch || !chunk_status || ((size_t)ref % (size_t)itemsize) || ((flags & FLAG_FLOAT) && itemsize != 4 && itemsize != 8))
    return fail(c, MTSB_E_ARG, "verify_chunks: bad arguments");
  DecodeArgs a{(const unsigned char*)comp, comp_is_device, comp_offsets, n_chunks, chunk_rows, nc, itemsize, flags, nullptr,
               0, (long long)nc * itemsize};
  a.verify = true;
  a.ref = ref; a.ref_is_device = ref_is_device; a.rtol = rtol; a.atol = atol;
  a.mismatches = mismatches; a.first_mismatch = first_mismatch;
  return decode_call(c, "verify_chunks", a, chunk_status);
}

// =============================================================================================== recompress
// Inflate sub-batch k into d_T (the decode stages, no inverse transform), then deflate d_T again (the encode stages, no
// forward transform).  The decode and the encode scratch are used one after the other on one stream, so a sub-batch is
// bounded like a compress sub-batch: batch_bytes of raw bytes, host_batch_bytes with a host buffer.
int mtsb_recompress_chunks(mtsb_ctx* c, const void* comp_, int comp_is_device, const long long* comp_offsets,
                           int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags, void* dst,
                           int dst_is_device, long long dst_capacity, long long* out_offsets, int* chunk_status) {
  if (!valid_common(c, n_chunks, chunk_rows, nc, itemsize) || !comp_ || !comp_offsets || !dst || !out_offsets || !chunk_status)
    return fail(c, MTSB_E_ARG, "recompress_chunks: bad arguments");
  const long long row_bytes = (long long)nc * itemsize;
  const DecodeArgs a{(const unsigned char*)comp_, comp_is_device, comp_offsets, n_chunks, chunk_rows, nc, itemsize, flags,
                     nullptr, 0, row_bytes};
  std::vector<ChunkIndex> ix;
  std::vector<unsigned char> ix_bytes;
  if (int r = start_decode_call(c, "recompress_chunks", a, chunk_status, ix, ix_bytes)) return r;
  if (int r = check_capacity(c, n_chunks, chunk_rows, nc, itemsize, flags, dst_capacity)) return r;

  const bool host_io = !comp_is_device || !dst_is_device;
  const Batches sb = plan_encode_batches(c, n_chunks, chunk_rows, row_bytes, itemsize, flags,
                                         host_io ? std::min(c->batch_bytes, c->host_batch_bytes) : c->batch_bytes);
  const int n_sb = sb.count();
  long long max_comp = 0;
  for (int k = 0; k < n_sb; k++) max_comp = std::max(max_comp, comp_offsets[sb.first[k + 1]] - comp_offsets[sb.first[k]]);
  if (!comp_is_device) { NEED(c->d_comp, (size_t)max_comp + 256); if (n_sb > 1) NEED(c->d_comp2, (size_t)max_comp + 256); }
  if (!dst_is_device) { NEED(c->d_out, (size_t)sb.max_out + 256); if (n_sb > 1) NEED(c->d_out2, (size_t)sb.max_out + 256); }
  CopyPipe& io = c->io;
  if (int r = io.start(c, comp_is_device ? nullptr : &c->d_comp, &c->d_comp2, dst_is_device ? nullptr : &c->d_out, &c->d_out2,
                       a.comp + comp_offsets[0], (size_t)(comp_offsets[sb.first[1]] - comp_offsets[0])))
    return r;
  out_offsets[0] = 0;
  long long total_out = 0;
  bool any_bad = false;
  for (int k = 0; k < n_sb; k++) {
    const int c0 = sb.first[k], c1 = sb.first[k + 1];
    // ---- decode half: inflate into d_T, verdicts
    DecodeBatch b;
    const unsigned char* dcomp = nullptr;
    const void* unused_ref = nullptr;
    if (int r = inflate_batch(c, a, ix, sb, k, b, dcomp, unused_ref)) return r;
    std::vector<uint32_t> adler(b.nb, 0);     // the adler32 each good chunk's stored checksum confirmed
    if (int r = batch_verdicts(c, a, ix, b, chunk_status, adler.data())) return r;
    if (int r = retry_misled(c, a, ix, b, dcomp, nullptr, nullptr, 0, chunk_status, adler.data())) return r;
    for (int i = c0; i < c1; i++) if (chunk_status[i]) any_bad = true;
    if (any_bad) continue;          // the output is undefined: only the statuses of the remaining chunks are wanted

    // ---- encode half: deflate d_T as mtsb_compress_chunks does
    EncodeBatch e;
    if (int r = plan_encode_sub_batch(c, chunk_rows, nc, itemsize, flags, c0, c1, true, e)) return r;
    c->begin(0);
    if (int r = e.tab.upload(c)) return r;
    c->end();
    if (int r = encode_sub_batch(c, e, k, c0, nullptr, nc, itemsize, flags, adler.data(), dst, total_out, out_offsets))
      return r;
  }
  if (int r = io.finish(c)) return r;
  c->collect_timing();
  if (any_bad) return fail(c, MTSB_E_CORRUPT, "at least one compressed chunk is corrupted");
  return 0;
}

}  // extern "C"
