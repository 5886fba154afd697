// transform.cuh — K1 (delta transform + demultiplex) and K4 (inverse: cumulative sums + re-multiplex) kernels,
// plus the adler32 partial/combine kernels that both directions share.
//
// Replaces, bit-exactly for integer dtypes (arithmetic is modular in the element width, SURVEY G4):
//   encode  mtscomp.py:381-394  diff_along_axis(axis=0) -> diff_along_axis(axis=1) -> tobytes(order=chunk_order)
//   decode  mtscomp.py:622-635  frombuffer -> reshape(order) -> cumsum(axis=1) -> cumsum(axis=0) -> ascontiguousarray
// Time and spatial operators act on different axes and commute exactly in modular arithmetic, so the kernels apply
// them in whichever order is cheapest.
//
// HBM layout: raw chunk = row-major (ns, nc) elements; transformed chunk = the deflate input, either channel-major
// ('F': nc runs of ns elements) or row-major ('C'), at the same element offset as the raw chunk.
// Every CTA works on a full-width tile of TT consecutive rows, which is one contiguous span of the row-major side.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace mts {

// Shared-memory row pitch (elements): chosen so a column walk (lane = row) hits 32 distinct banks.
template <class T> __host__ __device__ inline int tile_pitch(int nc) {
  if (sizeof(T) == 1) { int p = (nc + 3) & ~3; if ((p & 4) == 0) p += 4; return p; }
  if (sizeof(T) == 2) { int p = (nc + 1) & ~1; if ((p & 2) == 0) p += 2; return p; }
  return nc | 1;
}

// ------------------------------------------------------------------------------------------------ element arithmetic
// Differences and sums of float32 / float64 elements give the NaN that NumPy gives on x86-64, the hosts that write and
// read these files: a NaN operand comes back quieted (the first one if both are NaN), and a NaN made from numbers
// (inf - inf) is the default NaN with the sign bit set.  The device's own rule (always 0x7fffffff) would change the
// transform bytes, and the decoded bits, of any recording with a NaN in it.  Integers: plain modular arithmetic.
template <class T> __device__ __forceinline__ T nan_as_x86(T, T, T r) { return r; }
template <class F, class U> __device__ __forceinline__ F nan_as_x86_fp(F a, F b, F r, U quiet, U dflt) {
  U u;
  if (a != a) { memcpy(&u, &a, sizeof u); u |= quiet; }
  else if (b != b) { memcpy(&u, &b, sizeof u); u |= quiet; }
  else if (r != r) u = dflt;
  else return r;
  memcpy(&r, &u, sizeof r);
  return r;
}
__device__ __forceinline__ float nan_as_x86(float a, float b, float r) { return nan_as_x86_fp(a, b, r, 0x00400000u, 0xffc00000u); }
__device__ __forceinline__ double nan_as_x86(double a, double b, double r) {
  return nan_as_x86_fp(a, b, r, 0x0008000000000000ull, 0xfff8000000000000ull);
}
template <class T> __device__ __forceinline__ T sub_el(T a, T b) { return nan_as_x86(a, b, (T)(a - b)); }
template <class T> __device__ __forceinline__ T add_el(T a, T b) { return nan_as_x86(a, b, (T)(a + b)); }
// Time difference x[t] - x[t-1].  The chunk's first row is copied, as np.diff's caller does (mtscomp.py:143-159), not
// reduced by a zero: that would quiet a signalling NaN.  (For integers the two are the same.)
template <class T> __device__ __forceinline__ T time_diff(T cur, T prev, bool first_row) {
  return std::is_floating_point<T>::value && first_row ? cur : sub_el(cur, prev);
}

// ------------------------------------------------------------------------------------------------ K1 forward
// Algorithmic traffic: read sizeof(T) + write sizeof(T) per element (the halo row is re-read once per tile: +1/TT).
template <class T>
__global__ void __launch_bounds__(512) fwd_transform_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                            const ChunkDesc* __restrict__ chunks, int nc, int TT,
                                                            int flags) {
  MTS_DYN_SMEM(smem_raw);
  T* s = (T*)smem_raw;
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int t0 = blockIdx.x * TT;
  if (t0 >= ns) return;
  const int rows = min(TT, ns - t0);
  const int P = tile_pitch<T>(nc);
  const T* x = src + cd.elem_off;
  T* y = dst + cd.elem_off;
  const bool td = (flags & FLAG_TIME_DIFF) != 0, sd = (flags & FLAG_SPATIAL_DIFF) != 0;

  // smem row r holds sample t0-1+r; row 0 is zero for the chunk's first tile (never used: time_diff copies that row).
  const long long base = (long long)(t0 - 1) * nc;
  const int n_el = (rows + 1) * nc;
  for (int e = threadIdx.x; e < n_el; e += blockDim.x) {
    int r = e / nc, c = e - r * nc;
    T v = 0;
    if (t0 > 0 || r > 0) v = x[base + e];
    s[r * P + c] = v;
  }
  __syncthreads();

  if (flags & FLAG_ORDER_C) {
    for (int e = threadIdx.x; e < rows * nc; e += blockDim.x) {
      int r = e / nc, c = e - r * nc;
      const T* p = s + (r + 1) * P + c;
      T v = p[0];
      if (td) v = time_diff(v, p[-P], t0 + r == 0);
      if (sd && c > 0) { T w = p[-1]; if (td) w = time_diff(w, p[-P - 1], t0 + r == 0); v = sub_el(v, w); }
      y[(long long)t0 * nc + e] = v;
    }
  } else {
    const int nw = blockDim.x >> 5;
    for (int c = warp_id(); c < nc; c += nw) {
      for (int r = lane_id(); r < rows; r += 32) {
        const T* p = s + (r + 1) * P + c;
        T v = p[0];
        if (td) v = time_diff(v, p[-P], t0 + r == 0);
        if (sd && c > 0) { T w = p[-1]; if (td) w = time_diff(w, p[-P - 1], t0 + r == 0); v = sub_el(v, w); }
        y[(long long)c * ns + t0 + r] = v;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ K4 inverse
// Pass 1: per (tile, channel) sums of the time-diffed stream.  partial[(chunk*max_tiles + tile)*nc + c].
template <class T>
__global__ void __launch_bounds__(512) inv_tile_sums_kernel(const T* __restrict__ in, T* __restrict__ partial,
                                                            const ChunkDesc* __restrict__ chunks, int nc, int TT,
                                                            int max_tiles, int flags) {
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int t0 = blockIdx.x * TT;
  if (t0 >= ns) return;
  const int rows = min(TT, ns - t0);
  const T* x = in + cd.elem_off;
  T* out = partial + ((long long)blockIdx.y * max_tiles + blockIdx.x) * nc;
  if (flags & FLAG_ORDER_C) {
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
      T acc = 0;
      for (int r = 0; r < rows; r++) acc = (T)(acc + x[(long long)(t0 + r) * nc + c]);
      out[c] = acc;
    }
  } else {
    const int nw = blockDim.x >> 5;
    for (int c = warp_id(); c < nc; c += nw) {
      unsigned acc = 0;
      for (int r = lane_id(); r < rows; r += 32) acc += (unsigned)x[(long long)c * ns + t0 + r];
      if (sizeof(T) <= 4) {
        acc = warp_sum(acc);
        if (lane_id() == 0) out[c] = (T)acc;
      }
    }
  }
}
// 64-bit elements need a 64-bit accumulator in the F-order branch above.
template <>
__global__ void __launch_bounds__(512) inv_tile_sums_kernel<uint64_t>(const uint64_t* __restrict__ in,
                                                                      uint64_t* __restrict__ partial,
                                                                      const ChunkDesc* __restrict__ chunks, int nc,
                                                                      int TT, int max_tiles, int flags) {
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int t0 = blockIdx.x * TT;
  if (t0 >= ns) return;
  const int rows = min(TT, ns - t0);
  const uint64_t* x = in + cd.elem_off;
  uint64_t* out = partial + ((long long)blockIdx.y * max_tiles + blockIdx.x) * nc;
  for (int c = threadIdx.x; c < nc; c += blockDim.x) {
    uint64_t acc = 0;
    for (int r = 0; r < rows; r++)
      acc += (flags & FLAG_ORDER_C) ? x[(long long)(t0 + r) * nc + c] : x[(long long)c * ns + t0 + r];
    out[c] = acc;
  }
}

// Pass 2: exclusive scan of the tile sums along time, per channel (tiny).
template <class T>
__global__ void inv_tile_scan_kernel(T* __restrict__ partial, const ChunkDesc* __restrict__ chunks, int nc, int TT,
                                     int max_tiles) {
  const ChunkDesc cd = chunks[blockIdx.y];
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  const int ntiles = (cd.ns + TT - 1) / TT;
  T* p = partial + (long long)blockIdx.y * max_tiles * nc + c;
  T run = 0;
  for (int j = 0; j < ntiles; j++) {
    T v = p[(long long)j * nc];
    p[(long long)j * nc] = run;
    run = (T)(run + v);
  }
}

// Pass 3: tile -> smem, per-channel running sum seeded by the scanned tile sums, optional per-row (spatial) running
// sum, contiguous row-major write.  Traffic: read + write sizeof(T) per element.
template <class T>
__global__ void __launch_bounds__(512) inv_apply_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                        const T* __restrict__ partial,
                                                        const ChunkDesc* __restrict__ chunks, int nc, int TT,
                                                        int max_tiles, int flags) {
  MTS_DYN_SMEM(smem_raw);
  T* s = (T*)smem_raw;
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int t0 = blockIdx.x * TT;
  if (t0 >= ns) return;
  const int rows = min(TT, ns - t0);
  const int P = tile_pitch<T>(nc);
  const T* x = in + cd.elem_off;
  T* y = out + cd.elem_off;
  const int nw = blockDim.x >> 5;

  if (flags & FLAG_ORDER_C) {
    for (int e = threadIdx.x; e < rows * nc; e += blockDim.x) {
      int r = e / nc, c = e - r * nc;
      s[r * P + c] = x[(long long)t0 * nc + e];
    }
  } else {
    for (int c = warp_id(); c < nc; c += nw)
      for (int r = lane_id(); r < rows; r += 32) s[r * P + c] = x[(long long)c * ns + t0 + r];
  }
  __syncthreads();
  if (flags & FLAG_TIME_DIFF) {
    const T* seed = partial + ((long long)blockIdx.y * max_tiles + blockIdx.x) * nc;
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
      T run = seed[c];
      for (int r = 0; r < rows; r++) {
        run = (T)(run + s[r * P + c]);
        s[r * P + c] = run;
      }
    }
    __syncthreads();
  }
  if (flags & FLAG_SPATIAL_DIFF) {
    for (int r = warp_id(); r < rows; r += nw) {
      T carry = 0;
      for (int c0 = 0; c0 < nc; c0 += 32) {
        int c = c0 + lane_id();
        T v = (c < nc) ? s[r * P + c] : (T)0;
        v = (T)(warp_incl_scan(v) + carry);
        if (c < nc) s[r * P + c] = v;
        carry = __shfl_sync(0xffffffffu, v, 31);
      }
    }
    __syncthreads();
  }
  for (int e = threadIdx.x; e < rows * nc; e += blockDim.x) {
    int r = e / nc, c = e - r * nc;
    y[(long long)t0 * nc + e] = s[r * P + c];
  }
}

// ------------------------------------------------------------------------------------------------ fast paths
// Channel-major layouts ('F' order, the reference's default).  The unit of work is one channel x R = 32 / sizeof(T)
// consecutive samples, i.e. one 32-byte sector of the channel-major side.
template <class T> struct ColRun { static const int R = 32 / sizeof(T); };

// Forward transform for the channel-major ('F') layouts, time and/or spatial differences.  A CTA takes a tile of TT
// consecutive rows x all channels, which is ONE contiguous span of the row-major side: it is staged in shared memory by
// a TMA bulk copy (the 16-byte aligned interior; the ragged ends by ordinary loads), together with the row above as
// halo.  A work item is one channel x R rows = one 32-byte sector of the channel-major side: the lanes of a warp take
// consecutive channels, so the shared-memory reads are conflict-free at any row pitch (385 or 384 channels alike),
// and every item leaves as two 128-bit stores.
// A full run of R elements (32 bytes) leaves with the widest stores its address allows (channel runs of an odd number
// of samples are only 8-, 4- or 2-byte aligned); a short run element by element.
template <class T> __device__ __forceinline__ void store_run(T* y, const T (&v)[32 / sizeof(T)], int nr) {
  const int R = 32 / sizeof(T);
  const uintptr_t a = (uintptr_t)y;
  if (nr == R && !(a & 15)) {
    uint4 q[2];
    memcpy(q, v, 32);
    ((uint4*)y)[0] = q[0]; ((uint4*)y)[1] = q[1];
  } else if (nr == R && !(a & 7)) {
    uint2 q[4];
    memcpy(q, v, 32);
#pragma unroll
    for (int i = 0; i < 4; i++) ((uint2*)y)[i] = q[i];
  } else if (nr == R && !(a & 3)) {
    unsigned q[8];
    memcpy(q, v, 32);
#pragma unroll
    for (int i = 0; i < 8; i++) ((unsigned*)y)[i] = q[i];
  } else {
#pragma unroll
    for (int r = 0; r < R; r++) if (r < nr) y[r] = v[r];
  }
}

static const int INV_TILE_MAXT = 448;                 // most threads of a tile kernel (one channel per thread and pass)
template <class T, int G, int J>
__global__ void __launch_bounds__(INV_TILE_MAXT, 2) fwd_tile_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                                    const ChunkDesc* __restrict__ chunks, int nc,
                                                                    int flags) {
  const int R = ColRun<T>::R, TT = G * R;
  MTS_DYN_SMEM(sm);                                    // [0,16) mbarrier, [16, ...) the span (16-byte aligned)
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int t0 = blockIdx.x * TT;
  if (t0 >= ns) return;
  const int rows = min(TT, ns - t0);
  const int halo = t0 > 0 ? 1 : 0;
  const unsigned char* x = (const unsigned char*)(src + cd.elem_off + (long long)(t0 - halo) * nc);
  const unsigned span = (unsigned)((rows + halo) * nc) * (unsigned)sizeof(T);
  const unsigned off0 = (unsigned)((uintptr_t)x & 15);
  unsigned char* data = sm + 16;                       // data[off0 + i] = x[i]
  const unsigned head = min(span, (16 - off0) & 15);   // bytes before the aligned interior
  const unsigned mid = (span - head) & ~15u;
  const mbar_t mbar = mbar_addr((unsigned long long*)sm);
  if (threadIdx.x == 0) {
    mbar_init(mbar);
    if (mid) { mbar_expect_tx(mbar, mid); bulk_g2s(data + off0 + head, x + head, mid, mbar); }
  }
  for (unsigned i = threadIdx.x; i < head; i += blockDim.x) data[off0 + i] = x[i];
  for (unsigned i = head + mid + threadIdx.x; i < span; i += blockDim.x) data[off0 + i] = x[i];
  __syncthreads();                                     // barrier initialised, ragged ends in place
  if (mid) mbar_wait(mbar, 0);

  const T* s = (const T*)(data + off0) + (long long)halo * nc;     // s[r * nc + c] = sample t0 + r, channel c
  const bool td = (flags & FLAG_TIME_DIFF) != 0, sd = (flags & FLAG_SPATIAL_DIFF) != 0;
  T* ychunk = dst + cd.elem_off + t0;
  // a thread owns J channels and walks down the G runs of each: no index arithmetic beyond a pointer step per row
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int c = threadIdx.x + j * blockDim.x;
    if (c >= nc) continue;
    const T* p = s + c;
    const bool left = sd && c > 0;
    // in the reference's order (it matters for floating point): time difference of each column first, then the
    // difference between the two columns (mtscomp.py:381-394)
    T prev = 0, prevl = 0;
    if (td && halo) { prev = p[-nc]; if (left) prevl = p[-nc - 1]; }
    T* y = ychunk + (long long)c * ns;
#pragma unroll
    for (int g = 0; g < G; g++) {
      const int nr = min(R, rows - g * R);
      if (nr <= 0) break;
      T v[R];
      if (nr == R && !left) {
#pragma unroll
        for (int r = 0; r < R; r++) {
          const T cur = p[(long long)(g * R + r) * nc];
          v[r] = td ? time_diff(cur, prev, !halo && g == 0 && r == 0) : cur;
          prev = cur;
        }
      } else {
#pragma unroll
        for (int r = 0; r < R; r++) {
          T cur = 0, curl = 0;
          if (r < nr) { cur = p[(long long)(g * R + r) * nc]; if (left) curl = p[(long long)(g * R + r) * nc - 1]; }
          const bool first = !halo && g == 0 && r == 0;
          T a = td ? time_diff(cur, prev, first) : cur;
          if (left) a = sub_el(a, td ? time_diff(curl, prevl, first) : curl);
          v[r] = a;
          prev = cur; prevl = curl;
        }
      }
      store_run<T>(y + g * R, v, nr);
    }
  }
}

// Inverse transform for the channel-major layouts in ONE pass over the data (read T once, write the output once): a CTA
// takes a tile of TT = G * R rows x all channels.  A thread owns J channels (c = threadIdx.x + j * blockDim.x) and, of
// each, the G runs of R rows of the tile: 32 bytes per run, loaded up front (G * J * 2 128-bit loads in flight per
// thread) and KEPT IN REGISTERS while the carry arrives; so the tile costs one shared-memory store per element (the
// transposition into row order) and nothing else.  Across the tiles of a chunk each channel's carry travels by decoupled
// look-back, channel by channel (no barrier, no fence): per (tile, channel) there is ONE word that holds a value, its
// kind (AGGREGATE of the tile / INCLUSIVE prefix up to its end) and the launch's epoch, so it is written and read
// atomically and words left by earlier launches read as "not there yet" (no clearing between launches).  A thread
// publishes its aggregate as soon as it has it, adds up the aggregates of the predecessors until it meets an inclusive
// one, and publishes its own inclusive value; the predecessor's word is requested before the tile's data, so with many
// chunks in the batch (tiles are handed out by a ticket counter, tile t of every chunk before tile t + 1 of any) it has
// arrived, inclusive, before the data has.  A waiting thread only ever waits for tickets below its own, which are
// running or done.  64-bit elements do not fit a word with their tag: they use separate value and tag arrays and fences.
// The finished rows leave shared memory as one contiguous span (TMA bulk store of the aligned interior).
template <class T> __device__ __forceinline__ void load_run(uint4 (&q)[2], const T* p, int nr) {
  const int R = 32 / sizeof(T);
  const uintptr_t a = (uintptr_t)p;
  if (nr == R && !(a & 15)) {
    q[0] = ((const uint4*)p)[0]; q[1] = ((const uint4*)p)[1];
  } else if (nr == R && !(a & 7)) {
    uint2 h[4];
#pragma unroll
    for (int i = 0; i < 4; i++) h[i] = ((const uint2*)p)[i];
    memcpy(q, h, 32);
  } else if (nr == R && !(a & 3)) {
    unsigned h[8];
#pragma unroll
    for (int i = 0; i < 8; i++) h[i] = ((const unsigned*)p)[i];
    memcpy(q, h, 32);
  } else {
    T v[R];
#pragma unroll
    for (int r = 0; r < R; r++) v[r] = r < nr ? p[r] : (T)0;
    memcpy(q, v, 32);
  }
}

static const unsigned INV_EPOCH_MAX = 0x3fffu;         // epochs 1..INV_EPOCH_MAX, then the host clears the words
template <int SZ> struct InvWord { typedef unsigned type; };
template <> struct InvWord<4> { typedef unsigned long long type; };
template <> struct InvWord<8> { typedef unsigned long long type; };
// bytes of look-back state per (tile, channel)
template <class T> __host__ __device__ inline size_t inv_state_bytes() { return sizeof(T) == 8 ? 24 : sizeof(typename InvWord<sizeof(T)>::type); }

// One channel's look-back cell of one tile.  kind: 0 nothing yet, 1 aggregate, 2 inclusive.
template <class T> struct InvCell {
  typedef typename InvWord<sizeof(T)>::type W;
  static const int VB = 8 * sizeof(T);
  __device__ static __forceinline__ void put(void* base, size_t n_cells, size_t i, unsigned epoch, unsigned kind, T v) {
    if (sizeof(T) == 8) {
      unsigned long long* val = (unsigned long long*)base + (kind == 2 ? n_cells : 0);
      volatile unsigned* tag = (volatile unsigned*)((unsigned long long*)base + 2 * n_cells);
      ((volatile unsigned long long*)val)[i] = (unsigned long long)v;
      __threadfence();
      tag[i] = (epoch << 2) | kind;
    } else {
      ((volatile W*)base)[i] = (W)v | ((W)kind << VB) | ((W)epoch << (VB + 2));
    }
  }
  // kind of the cell in this launch (0: not there yet) and its value
  __device__ static __forceinline__ unsigned get(const void* base, size_t n_cells, size_t i, unsigned epoch, T& v) {
    if (sizeof(T) == 8) {
      const volatile unsigned* tag = (const volatile unsigned*)((const unsigned long long*)base + 2 * n_cells);
      const unsigned t = tag[i];
      if ((t >> 2) != epoch || !(t & 3)) return 0;
      __threadfence();
      v = (T)((const volatile unsigned long long*)base)[((t & 3) == 2 ? n_cells : 0) + i];
      return t & 3;
    } else {
      const W w = ((const volatile W*)base)[i];
      if ((unsigned)(w >> (VB + 2)) != epoch) return 0;
      v = (T)w;
      return (unsigned)(w >> VB) & 3u;
    }
  }
};

template <class T, int G, int J>
__global__ void __launch_bounds__(INV_TILE_MAXT, 2) inv_tile_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                                    const ChunkDesc* __restrict__ chunks, int n_chunks,
                                                                    int nc, int max_tiles, int flags, int order_block,
                                                                    void* cells, unsigned epoch, unsigned* ticket) {
  const int R = ColRun<T>::R, TT = G * R;
  MTS_DYN_SMEM(sm);                                    // [16 bytes][tile: data at offset off0, rows x nc]
  __shared__ unsigned s_ticket;
  if (threadIdx.x == 0) s_ticket = atomicAdd(ticket, 1u);
  __syncthreads();
  const unsigned tk = s_ticket;
  // order_block consecutive tiles of a chunk have consecutive tickets (they run at the same time and read neighbouring
  // pieces of every channel run), then the same tiles of the next chunk, ...
  const unsigned per = (unsigned)order_block * (unsigned)n_chunks, rem = tk % per;
  const int ci = (int)(rem / (unsigned)order_block), tl = (int)(tk / per) * order_block + (int)(rem % (unsigned)order_block);
  const ChunkDesc cd = chunks[ci];
  const int ns = cd.ns;
  const int t0 = tl * TT;
  if (t0 >= ns) return;
  const int rows = min(TT, ns - t0);
  const bool td = (flags & FLAG_TIME_DIFF) != 0, sd = (flags & FLAG_SPATIAL_DIFF) != 0;
  unsigned char* gout = (unsigned char*)(out + cd.elem_off + (long long)t0 * nc);
  const unsigned off0 = (unsigned)((uintptr_t)gout & 15);
  T* s = (T*)(sm + 16 + off0);                         // s[r * nc + c]; 16-byte aligned exactly where the output is
  const T* x = in + cd.elem_off + t0;
  const size_t n_cells = (size_t)n_chunks * max_tiles * nc;
  const size_t cell0 = ((size_t)ci * max_tiles + tl) * nc;           // this tile's cells; the predecessor's are nc below
  // ---- the predecessor's cells are requested first, then the thread's runs -> registers
  T pv[J];
  unsigned pk[J];
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int c = threadIdx.x + j * blockDim.x;
    pv[j] = 0; pk[j] = 0;
    if (td && tl > 0 && c < nc) pk[j] = InvCell<T>::get(cells, n_cells, cell0 - nc + c, epoch, pv[j]);
  }
  uint4 q[J][G][2];
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int c = threadIdx.x + j * blockDim.x;
#pragma unroll
    for (int g = 0; g < G; g++) {
      const int nr = min(R, rows - g * R);
      if (c < nc && nr > 0) load_run<T>(q[j][g], x + (long long)c * ns + g * R, nr);
      else q[j][g][0] = q[j][g][1] = make_uint4(0, 0, 0, 0);
    }
  }
  // ---- aggregate, look-back, running sums in registers, one shared-memory store per element (the transposition)
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int c = threadIdx.x + j * blockDim.x;
    if (c >= nc) continue;
    T a = 0;
    if (td) {
      const bool publish = (long long)(tl + 1) * TT < ns;            // somebody comes after this tile
      T total = 0;
#pragma unroll
      for (int g = 0; g < G; g++) {
        T v[R];
        memcpy(v, q[j][g], 32);
#pragma unroll
        for (int r = 0; r < R; r++) total = (T)(total + v[r]);
      }
      if (publish && pk[j] != 2 && tl > 0) InvCell<T>::put(cells, n_cells, cell0 + c, epoch, 1, total);
      T cy = 0;
      for (int i = tl - 1; i >= 0; i--) {
        T v = pv[j];
        unsigned kind = pk[j];
        pk[j] = 0;                                                   // (the prefetched answer serves the first step only)
        while (kind == 0) {
          kind = InvCell<T>::get(cells, n_cells, ((size_t)ci * max_tiles + i) * nc + c, epoch, v);
#ifdef MTSCOMP_EMU
          if (kind == 0) emu::yield();
#endif
        }
        cy = (T)(cy + v);
        if (kind == 2) break;
      }
      if (publish) InvCell<T>::put(cells, n_cells, cell0 + c, epoch, 2, (T)(cy + total));
      a = cy;
    }
    T* sp = s + c;
#pragma unroll
    for (int g = 0; g < G; g++) {
      T v[R];
      memcpy(v, q[j][g], 32);
      if (rows == TT) {
#pragma unroll
        for (int r = 0; r < R; r++) {
          if (td) { a = (T)(a + v[r]); v[r] = a; }
          sp[(long long)(g * R + r) * nc] = v[r];
        }
      } else {
#pragma unroll
        for (int r = 0; r < R; r++) {
          if (td) { a = (T)(a + v[r]); v[r] = a; }
          if (g * R + r < rows) sp[(long long)(g * R + r) * nc] = v[r];
        }
      }
    }
  }
  __syncthreads();
  if (sd) {
    // per-row running sum over the channels (after the time sums: the two commute in modular arithmetic)
    const int nw = blockDim.x >> 5;
    for (int r = warp_id(); r < rows; r += nw) {
      T cy = 0;
      for (int c0 = 0; c0 < nc; c0 += 32) {
        const int c = c0 + lane_id();
        T v = (c < nc) ? s[r * nc + c] : (T)0;
        v = (T)(warp_incl_scan(v) + cy);
        if (c < nc) s[r * nc + c] = v;
        cy = __shfl_sync(0xffffffffu, v, 31);
      }
    }
    __syncthreads();
  }
  // ---- rows -> global: one contiguous span; 16-byte aligned interior by TMA bulk store, the ragged ends by threads
  const unsigned span = (unsigned)(rows * nc) * (unsigned)sizeof(T);
  const unsigned head = min(span, (16 - off0) & 15), mid = (span - head) & ~15u;
  const unsigned char* sb = (const unsigned char*)s;
  for (unsigned i = threadIdx.x; i < head; i += blockDim.x) gout[i] = sb[i];
  for (unsigned i = head + mid + threadIdx.x; i < span; i += blockDim.x) gout[i] = sb[i];
  if (mid) {
    fence_async_smem();
    __syncthreads();
    if (threadIdx.x == 0) { bulk_s2g(gout + head, sb + head, mid); bulk_s2g_wait(); }
  }
}

// Inverse of the above: per-channel running sum seeded by the scanned tile sums (tile = TT rows, TT % R == 0).
template <class T>
__global__ void __launch_bounds__(128) inv_cols_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                       const T* __restrict__ partial,
                                                       const ChunkDesc* __restrict__ chunks, int nc, int TT,
                                                       int max_tiles, int flags) {
  const int R = ColRun<T>::R;
  const ChunkDesc cd = chunks[blockIdx.z];
  const int ns = cd.ns;
  const int c = blockIdx.y * 128 + (int)threadIdx.x;        // (tiles on x: a long chunk has more than 65535 of them)
  const int t0 = blockIdx.x * TT;
  if (t0 >= ns || c >= nc) return;
  const T* x = in + cd.elem_off + (long long)c * ns;
  T* y = out + cd.elem_off;
  const bool td = (flags & FLAG_TIME_DIFF) != 0;
  T run = td ? partial[((long long)blockIdx.z * max_tiles + blockIdx.x) * nc + c] : (T)0;
  const int tend = min(t0 + TT, ns);
  for (int t = t0; t < tend; t += R) {
    const int rows = min(R, tend - t);
    T v[R];
    if (rows == R && ((uintptr_t)(x + t) & 15) == 0) {
      uint4 a = ((const uint4*)(x + t))[0], b = ((const uint4*)(x + t))[1];
      memcpy(&v[0], &a, 16);
      memcpy(&v[R / 2], &b, 16);
    } else {
      for (int r = 0; r < R; r++) v[r] = (r < rows) ? x[t + r] : (T)0;
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
      if (td) { run = (T)(run + v[r]); v[r] = run; }
      if (r < rows) y[(long long)(t + r) * nc + c] = v[r];
    }
  }
}


// ------------------------------------------------------------------------------------------------ floating point inverse
// float32 / float64 (FLAG_FLOAT): the forward differences are single IEEE subtractions (sub_el, with NumPy's NaNs), so
// the integer kernels above are simply instantiated for float / double.  The inverse is different: np.cumsum
// accumulates sequentially in the array's own precision (mtscomp.py:162-169), and reproducing the reference Reader bit
// for bit means adding in the same order (add_el) — one thread per row (spatial pass, into a scratch copy) and one
// thread per channel (time pass).
template <class T>
__global__ void __launch_bounds__(128) inv_float_space_kernel(const T* __restrict__ in, T* __restrict__ tmp,
                                                              const ChunkDesc* __restrict__ chunks, int nc, int flags) {
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ns) return;
  const T* x = in + cd.elem_off;
  T* y = tmp + cd.elem_off;
  const bool oc = (flags & FLAG_ORDER_C) != 0;
  T acc = 0;
  for (int c = 0; c < nc; c++) {
    const long long i = oc ? (long long)t * nc + c : (long long)c * ns + t;
    const T v = x[i];
    acc = c == 0 ? v : add_el(acc, v);
    y[i] = acc;
  }
}

template <class T>
__global__ void __launch_bounds__(128) inv_float_time_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                             const ChunkDesc* __restrict__ chunks, int nc, int flags) {
  const ChunkDesc cd = chunks[blockIdx.y];
  const int ns = cd.ns;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  const T* x = in + cd.elem_off;
  T* y = out + cd.elem_off;
  const bool oc = (flags & FLAG_ORDER_C) != 0, td = (flags & FLAG_TIME_DIFF) != 0;
  T acc = 0;
  for (int t = 0; t < ns; t++) {
    const T v = x[oc ? (long long)t * nc + c : (long long)c * ns + t];
    acc = (t == 0 || !td) ? v : add_el(acc, v);
    y[(long long)t * nc + c] = acc;
  }
}

// ------------------------------------------------------------------------------------------------ adler32
// One CTA per segment: standalone adler32 of bytes [off, off+len) (i.e. starting from adler = 1).  Segments are
// folded per chunk with zlib's adler32_combine rule (SURVEY Appendix B) by adler_combine_kernel / the deflate scan.
struct AdlerSeg {
  long long off;
  int len;
  int pad_;
};

__global__ void __launch_bounds__(256) adler_partial_kernel(const uint8_t* __restrict__ data,
                                                            const AdlerSeg* __restrict__ segs,
                                                            uint32_t* __restrict__ seg_adler) {
  __shared__ unsigned long long sh_a[8], sh_b[8];
  const AdlerSeg sg = segs[blockIdx.x];
  const uint8_t* p = data + sg.off;
  const unsigned n = (unsigned)sg.len;
  unsigned long long a = 0, b = 0;  // a = sum b_i ; b = sum (n - i) * b_i
  // head bytes up to 4-byte alignment, aligned words, tail bytes
  unsigned head = (unsigned)((4 - ((uintptr_t)p & 3)) & 3);
  if (head > n) head = n;
  const unsigned nwords = (n - head) >> 2;
  const unsigned tail0 = head + (nwords << 2);
  if (threadIdx.x < head) { unsigned v = p[threadIdx.x]; a += v; b += (unsigned long long)(n - threadIdx.x) * v; }
  const uint32_t* w = (const uint32_t*)(p + head);
  for (unsigned i = threadIdx.x; i < nwords; i += blockDim.x) {
    uint32_t v = w[i];
    unsigned b0 = v & 255, b1 = (v >> 8) & 255, b2 = (v >> 16) & 255, b3 = v >> 24;
    unsigned pos = head + (i << 2);
    unsigned sum = b0 + b1 + b2 + b3;
    a += sum;
    b += (unsigned long long)(n - pos) * sum - (b1 + 2 * b2 + 3 * b3);
  }
  if (tail0 + threadIdx.x < n) { unsigned v = p[tail0 + threadIdx.x]; a += v; b += (unsigned long long)(n - tail0 - threadIdx.x) * v; }
  a = warp_sum(a);
  b = warp_sum(b);
  if (lane_id() == 0) { sh_a[warp_id()] = a; sh_b[warp_id()] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long ta = 0, tb = 0;
    for (unsigned i = 0; i < (blockDim.x >> 5); i++) { ta += sh_a[i]; tb += sh_b[i] % ADLER_BASE; }
    uint32_t s1 = (uint32_t)((1 + ta) % ADLER_BASE);
    uint32_t s2 = (uint32_t)((n % ADLER_BASE + tb) % ADLER_BASE);
    seg_adler[blockIdx.x] = (s2 << 16) | s1;
  }
}

__device__ __forceinline__ uint32_t adler_combine(uint32_t a1, uint32_t a2, unsigned len2) {
  uint32_t s1a = a1 & 0xffff, s2a = a1 >> 16, s1b = a2 & 0xffff, s2b = a2 >> 16;
  uint32_t s1 = (s1a + s1b + ADLER_BASE - 1) % ADLER_BASE;
  unsigned long long t = (unsigned long long)(len2 % ADLER_BASE) * ((s1a + ADLER_BASE - 1) % ADLER_BASE);
  uint32_t s2 = (uint32_t)((s2a + s2b + t) % ADLER_BASE);
  return (s2 << 16) | s1;
}

// One thread per chunk: fold the chunk's segment adlers in order.  seg ranges come from first[i] .. first[i+1].
__global__ void adler_combine_kernel(const AdlerSeg* __restrict__ segs, const uint32_t* __restrict__ seg_adler,
                                     const int* __restrict__ first, int n_chunks, uint32_t* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_chunks) return;
  uint32_t a = 1;
  for (int s = first[i]; s < first[i + 1]; s++) a = adler_combine(a, seg_adler[s], (unsigned)segs[s].len);
  out[i] = a;
}

}  // namespace mts
