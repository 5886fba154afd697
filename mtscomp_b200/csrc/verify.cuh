// verify.cuh — the integrity check's compare: decoded rows against the caller's reference rows, on the device.
#pragma once
#include "common.cuh"

namespace mts {

static const int VERIFY_THREADS = 256;
static const int VERIFY_TILE_BYTES = 32768;   // per CTA: a multiple of 16, so every tile of a chunk has its alignment phase
static const long long VERIFY_NONE = 0x7f7f7f7f7f7f7f7fll;   // first-mismatch cell before any CTA found one (memset 0x7f)

// Whether decoded element x fails against reference element y.  Integers: bit inequality.  Floats: NumPy 2's isclose
// body, (|x - y| <= atol + rtol * |y| && isfinite(y)) || x == y, in the element's own precision with each operation
// rounded on its own (no FMA contraction, which would move verdicts at the tolerance's edge).
template <class T> __device__ __forceinline__ bool verify_fails(T x, T y, T, T) { return x != y; }
template <> __device__ __forceinline__ bool verify_fails<float>(float x, float y, float rtol, float atol) {
  const float ay = fabsf(y);
  const bool close = fabsf(__fsub_rn(x, y)) <= __fadd_rn(atol, __fmul_rn(rtol, ay)) && ay <= 3.40282347e+38f;
  return !(close || x == y);
}
template <> __device__ __forceinline__ bool verify_fails<double>(double x, double y, double rtol, double atol) {
  const double ay = fabs(y);
  const bool close = fabs(__dsub_rn(x, y)) <= __dadd_rn(atol, __dmul_rn(rtol, ay)) && ay <= 1.7976931348623157e+308;
  return !(close || x == y);
}

// Grid (tiles, chunks): CTA (t, i) compares elements [t * TILE, (t + 1) * TILE) of chunk i, which starts at element
// cd[i].elem_off of both `dec` and `ref`.  Chunk starts are only itemsize-aligned: where both pointers of a tile have
// the same 16-byte phase the body is read with 16-byte loads between a scalar head and tail, otherwise element by
// element.  count[i] += the CTA's failures and first[i] = min(first[i], index in the chunk of its first one); a CTA
// that finds nothing writes nothing.
template <class T>
__global__ void __launch_bounds__(VERIFY_THREADS) verify_kernel(const T* __restrict__ dec, const T* __restrict__ ref,
                                                               const ChunkDesc* __restrict__ cd, int nc, T rtol, T atol,
                                                               unsigned long long* __restrict__ count,
                                                               long long* __restrict__ first) {
  constexpr int V = 16 / sizeof(T), TILE = VERIFY_TILE_BYTES / sizeof(T);
  constexpr bool IS_FLOAT = T(0.5) != T(0);
  const ChunkDesc d = cd[blockIdx.y];
  const long long n = (long long)d.ns * nc, a = (long long)blockIdx.x * TILE;
  if (a >= n) return;
  const int len = (int)(n - a < TILE ? n - a : TILE);
  const T* x = dec + d.elem_off + a;
  const T* y = ref + d.elem_off + a;
  const unsigned px = (unsigned)((size_t)x & 15), py = (unsigned)((size_t)y & 15);
  int head = len, nv = 0;
  if (px == py) {
    head = (int)(((16 - px) & 15) / sizeof(T));
    if (head > len) head = len;
    nv = (len - head) / V;
  }
  unsigned long long cnt = 0;
  long long fst = VERIFY_NONE;
  const uint4* xv = (const uint4*)(x + head);
  const uint4* yv = (const uint4*)(y + head);
#pragma unroll 4
  for (int v = threadIdx.x; v < nv; v += VERIFY_THREADS) {
    const uint4 p = xv[v], q = yv[v];
    if (!IS_FLOAT && p.x == q.x && p.y == q.y && p.z == q.z && p.w == q.w) continue;
    T pe[V], qe[V];
    memcpy(pe, &p, 16);   // (not a pointer cast: reading a uint4 through T* breaks strict aliasing)
    memcpy(qe, &q, 16);
#pragma unroll
    for (int e = 0; e < V; e++)
      if (verify_fails<T>(pe[e], qe[e], rtol, atol)) {
        cnt++;
        const long long at = a + head + (long long)v * V + e;
        if (at < fst) fst = at;
      }
  }
  // scalar head [0, head) and tail [head + nv * V, len)
  const int body_end = head + nv * V, n_scalar = head + (len - body_end);
  for (int j = threadIdx.x; j < n_scalar; j += VERIFY_THREADS) {
    const int e = j < head ? j : j - head + body_end;
    if (verify_fails<T>(x[e], y[e], rtol, atol)) {
      cnt++;
      if (a + e < fst) fst = a + e;
    }
  }
  if (!__syncthreads_or(cnt != 0)) return;
  __shared__ unsigned long long s_cnt[VERIFY_THREADS / 32];
  __shared__ long long s_fst[VERIFY_THREADS / 32];
  cnt = warp_sum(cnt);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const long long f = __shfl_xor_sync(0xffffffffu, fst, o);
    if (f < fst) fst = f;
  }
  if (lane_id() == 0) { s_cnt[warp_id()] = cnt; s_fst[warp_id()] = fst; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < VERIFY_THREADS / 32; w++) { cnt += s_cnt[w]; if (s_fst[w] < fst) fst = s_fst[w]; }
    atomicAdd(&count[blockIdx.y], cnt);
    atomicMin(&first[blockIdx.y], fst);
  }
}

}  // namespace mts
