// deflate.cuh — K2: parallel DEFLATE encoder (RFC 1951) producing one valid zlib stream (RFC 1950) per chunk.
//
// Replaces `zlib.compress(chunkd.tobytes(order))` at mtscomp.py:394.  The reference Reader only requires that
// zlib.decompress() accepts the stream and returns the transformed bytes (mtscomp.py:619, SURVEY G5), so the encoder
// is free to pick its own parse; the contract is decodability + size <= 1.031x zlib level 6 (north star).
//
// Each chunk's transformed bytes are cut into independent "segments" (fresh 32 KB window, own dynamic-Huffman block,
// closed by an empty stored block so the next segment starts byte-aligned).  Four kernels, split by parallelism shape:
//   lz77_kernel     one CTA / segment : shared-memory hash-chain match finder over a 64 KB data ring, every position
//                                       matched in parallel, lazy parse by pointer doubling, token + histogram output
//   huff_kernel     one warp / segment: length-limited Huffman codes (<=15 / <=7 bits), RLE'd dynamic header, sizes
//   scan_kernel     one CTA           : exclusive prefix of segment byte sizes -> final offsets (packed .cbin layout)
//   encode_kernel   one CTA / segment : code lookup, prefix-sum bit offsets, bit-pack straight into the final stream,
//                                       zlib header / stored fallback / final block / adler32 trailer
#pragma once
#include "common.cuh"

namespace mts {

// ------------------------------------------------------------------------------------------------ tables
struct DeflateSeg {
  long long in_off;     // byte offset of the segment's input in the transformed buffer
  long long tok_off;    // element offset of the segment's token area (capacity = in_len u16 elements)
  int in_len;           // input bytes (> 0)
  int chunk;            // owning chunk (index within the batch)
  int flags;            // SEG_FIRST | SEG_LAST
  int sub_first;        // index of the segment's first sub-block in the batch's sub-block table
};
enum { SEG_FIRST = 1, SEG_LAST = 2 };
// In-band index written after each chunk's zlib stream (zlib.decompress ignores trailing bytes, SURVEY G5), all
// little-endian u32:
//   [sub-block table: for every segment, one entry per sub-block of its input | k segment body lengths |
//    sub-block bytes, step bytes | segment bytes, k, magic "MTS2", sum of the lengths]
// The sub-blocks of a segment begin at the output offsets idx_bound(j) = 0, S/2, S, 2S, 3S, ... (S = IDX_SUB_BYTES; the
// first S bytes, which are mostly literals because the window is still empty, count as two sub-blocks so that all of
// them hold about the same number of codes).  Sub-block j starts with the first token whose output begins at or after
// idx_bound(j); its entry is (bits from the previous sub-block's first token to its own; for j = 0 from the segment's
// first bit) | overshoot << 17, overshoot = output offset of that token - idx_bound(j) (< 258).  "step bytes" states the encoder's STEP RULE: no
// match reads output at or after the beginning of the step (of that many bytes, counted from the segment's start) that
// the match itself starts in.  Files of the first format ("MTSB": k lengths | segment bytes, k, magic, sum) still decode.
static const unsigned IDX_MAGIC_V1 = 0x4253544Du, IDX_MAGIC_V2 = 0x3253544Du;
static const int IDX_SUB_BYTES = 8192;
static const int IDX_MIN_RAW = 2048;       // a chunk of one segment shorter than this gets no index (it would dwarf the stream)
__host__ __device__ inline bool idx_wanted(int n_seg, int first_seg_len) { return !(n_seg == 1 && first_seg_len < IDX_MIN_RAW); }
__host__ __device__ inline int idx_n_sub(long long seg_len) {
  return (int)((seg_len + IDX_SUB_BYTES - 1) / IDX_SUB_BYTES) + (seg_len > IDX_SUB_BYTES / 2 ? 1 : 0);
}
__host__ __device__ inline unsigned idx_bound(unsigned j) { return j == 0 ? 0u : j == 1 ? IDX_SUB_BYTES / 2u : (j - 1) * (unsigned)IDX_SUB_BYTES; }
__host__ __device__ inline unsigned idx_item(unsigned pos) { return (pos >= IDX_SUB_BYTES / 2u ? 1u : 0u) + pos / (unsigned)IDX_SUB_BYTES; }   // sub-block that holds pos
enum { MODE_STORED = 0, MODE_DYNAMIC = 1, MODE_FIXED = 2 };

struct DeflateSegOut {   // written by huff_kernel / scan_kernel, read by encode_kernel
  unsigned n_tok;        // u16 token elements produced by lz77_kernel
  unsigned hdr_bits;     // dynamic header length in bits
  unsigned mode;
  unsigned body_bytes;   // bytes of this segment's deflate data (without zlib header/trailer)
  long long out_off;     // byte offset in the packed output
};

static const int LL_SYMS = 286, D_SYMS = 30, BL_SYMS = 19;
static const int HIST_STRIDE = 320;          // u32 per segment: [0,286) lit/len, [288,318) dist
static const int HDR_WORDS = 192;            // dynamic header capacity (u32) per segment
static const int CODE_STRIDE = 320;          // u32 per segment: code | len<<16, same layout as the histogram


__device__ __forceinline__ void len_symbol(unsigned len, unsigned& sym, unsigned& nb, unsigned& ev) {
  unsigned l = len - 3;
  if (l < 8) { sym = 257 + l; nb = 0; ev = 0; }
  else if (len == 258) { sym = 285; nb = 0; ev = 0; }
  else { nb = 29 - __clz((int)l); sym = 261 + 4 * nb + ((l >> nb) & 3); ev = l & ((1u << nb) - 1); }
}
__device__ __forceinline__ void dist_symbol(unsigned dist, unsigned& sym, unsigned& nb, unsigned& ev) {
  unsigned d = dist - 1;
  if (d < 4) { sym = d; nb = 0; ev = 0; }
  else { nb = 30 - __clz((int)d); sym = 2 * nb + 2 + ((d >> nb) & 1); ev = d & ((1u << nb) - 1); }
}
__device__ __forceinline__ unsigned ll_extra_bits(unsigned sym) {   // sym in [0,286)
  if (sym < 265 || sym == 285) return 0;
  return (sym - 261) >> 2;
}
__device__ __forceinline__ unsigned d_extra_bits(unsigned sym) { return sym < 4 ? 0 : (sym >> 1) - 1; }

// ------------------------------------------------------------------------------------------------ lz77_kernel
// One CTA of NT threads per segment (persistent over segments), several CTAs per SM.  STRIDE = bytes between indexed
// positions ("units"): 2 for int16 streams (matches start at sample boundaries and cover whole samples; the byte in
// between inherits the next sample's match extended backwards), 1 generic.  The segment is processed in steps of NT
// units, one unit per thread, every phase of a step data-parallel over the whole CTA (no serial inserter):
//   (A) lookup   each unit hashes its first 6 bytes (table L) and 4 bytes (table S) and reads its two buckets.  A bucket
//                is one u32 = the two newest units with that hash (newest << 16 | second newest) as of the END OF THE
//                PREVIOUS STEP: units of one step do not see each other (matches nearer than the step are found
//                through the next older entry or not at all; measured cost in DESIGN.md)
//   (C) compare  up to 3 candidates (L newest, L second, S newest) against the unit's 16 bytes held in registers; the
//                longest wins, ties go to the nearer one
//   (B) insert   after a barrier every unit stores (itself << 16 | old newest) into its buckets; where several units of
//                the step share a bucket the highest one must win whatever order the hardware applied the stores in,
//                so after a second barrier each unit that finds a LOWER unit of its step in its bucket atomicMax'es its
//                word in (rare, a few lanes per step).  The result depends on the data only (test_chop determinism).
//   (D) parse    greedy over units, hierarchical: pointer doubling in registers inside each warp, one warp chains the
//                warps' stretches by relaxation, then every warp emits its tokens (ballot prefix) and histogram counts
// Input reaches the 32 KB ring (+ mirror of its first bytes, so that compares never wrap) by TMA bulk copies
// (cp.async.bulk, one elected thread, completion on an mbarrier) issued two steps ahead.
static const int LZ_RING = 32768;
static const int LZ_MIRROR = 288;             // ring[RING + i] mirrors ring[i]: reads of up to 258 + 16 + 4 bytes never wrap
static const unsigned LZ_BIAS = 32768;

template <int STRIDE, int NT> struct LzSmem {
  static const int SEG = NT * STRIDE;         // bytes per step
#ifndef MTS_HL_BITS
#define MTS_HL_BITS 13
#define MTS_HS_BITS 13
#endif
  static const int HL_BITS = MTS_HL_BITS;     // buckets of table L (u32 each)
  static const int HS_BITS = MTS_HS_BITS;     // buckets of table S
  // the piece loaded during step s overwrites ring coordinates up to (s + 3) * SEG - RING; step s + 1 reads back to
  // (s + 1) * SEG - MAXD
  static const int MAXD = LZ_RING - 2 * SEG - 8;           // bytes
  static const int MAXD_UNITS = MAXD / STRIDE;
  static const int NSW = NT / 32;
  static const size_t ring_off = 0;
  static const size_t headl_off = LZ_RING + LZ_MIRROR;     // multiple of 16
  static const size_t heads_off = headl_off + ((size_t)4 << HL_BITS);
  static const size_t xe_off = heads_off + ((size_t)4 << HS_BITS);
  static const size_t hist_off = (xe_off + (size_t)(2 * NT) * 4 + 15) & ~(size_t)15;
  static const size_t misc_off = hist_off + (size_t)HIST_STRIDE * 4;     // two steps of [0..31] element base of each stretch, [32..63] entries, [64] step total
  static const size_t mbar_off = misc_off + 2 * 72 * 4 + 8;              // 8-byte aligned; [2 * 72]: the CTA's next segment
  static const size_t total = mbar_off + 16;
};

__device__ __forceinline__ unsigned ring_load4(const unsigned char* ring, unsigned m) {   // m < LZ_RING
  const unsigned* w = (const unsigned*)(ring + (m & ~3u));
  return __funnelshift_r(w[0], w[1], m << 3);              // w[1] may lie in the mirror
}
__device__ __forceinline__ unsigned lz_hash4(unsigned w, int bits) { return (w * 0x9E3779B1u) >> (32 - bits); }
__device__ __forceinline__ unsigned lz_hash6(unsigned w0, unsigned w1, int bits) {
  return ((w0 * 0x9E3779B1u) ^ ((w1 & 0xffffu) * 0x85EBCA6Bu)) >> (32 - bits);
}

#if defined(MTS_LZ_PROFILE) && !defined(MTSCOMP_EMU)
// development instrumentation: cycles per phase (thread 0 of CTA 0), summed over steps
// [0] steps [1] lookup+compare [2] insert+parse stage 1 [3] settle+chain [4] emit [5] whole step
__device__ unsigned long long g_lz_prof[16];
#define LZ_PROF_T(var) long long var = clock64()
#define LZ_PROF_ADD(i, v) do { if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&g_lz_prof[i], (unsigned long long)(v)); } while (0)
#else
#define LZ_PROF_T(var)
#define LZ_PROF_ADD(i, v)
#endif

// Per-unit state of a step, from the lookup to the insert (M, mm and tokw: to the emit one step later)
struct LzUnit {
  unsigned M, mm, tokw;          // units on the token chain from here (stretch-local mask), matches of the stretch, token
  unsigned hs, hl, cws, cwl;     // buckets and their words as of the end of the previous step
  unsigned ub;                   // unit number (16 bits, biased)
  bool vS, vL;                   // the unit goes into table S / L
};

// (A) lookup, (C) compare and stage 1 of the parse for this thread's unit of the step that starts at s0; u arrives
// zeroed.  FULL: every unit of the step has at least 258 + 16 bytes of input from its position on -- all steps but the
// last one or two of a segment -- so the body is compiled without the bounds tests (slen, lim), which only a step
// near the segment's end needs.
template <int STRIDE, int NT, bool FULL>
__device__ __forceinline__ void lz_find(LzUnit& u, const unsigned char* ring, const unsigned* headL, const unsigned* headS,
                                        unsigned* xs, unsigned s0, unsigned n, unsigned off0, unsigned tid,
                                        unsigned& ad_a, unsigned& ad_c, unsigned long long& ad_b) {
  typedef LzSmem<STRIDE, NT> L;
  const unsigned SEG = L::SEG, RM = LZ_RING - 1, lane = tid & 31, wid = tid >> 5;
  const unsigned* ringw = (const unsigned*)ring;
  const unsigned slen = FULL ? SEG : min(SEG, n - s0);
  // ---- (A) lookup + (C) compare
  const unsigned li = tid * STRIDE;                   // local position in the step
  const unsigned p = s0 + li;
  u.ub = (p / STRIDE + LZ_BIAS) & 0xffffu;
  unsigned mlen = 0, mdist = 0;
  if (FULL || li < slen) {
    const unsigned lim = FULL ? 258u : min(258u, n - p);
    const unsigned pr = (p + off0) & RM;              // ring offset of this unit
    unsigned w0, w1;
    {
      const unsigned* pw = ringw + (pr >> 2);
      const unsigned sh = pr << 3;
      const unsigned t0 = pw[0], t1 = pw[1], t2 = pw[2];
      w0 = __funnelshift_r(t0, t1, sh); w1 = __funnelshift_r(t1, t2, sh);
    }
    u.tokw = STRIDE == 2 ? __byte_perm(w0, 0, 0x4140) : (w0 & 0xffu);   // literal token: the unit's bytes, one per element
    // adler32 of the segment: a = sum of bytes, b = sum of (n - position) * byte
    {
      const unsigned b1 = STRIDE == 2 ? u.tokw >> 16 : 0u, sum = (u.tokw & 0xffu) + b1;
      ad_a += sum; ad_c += b1;
      ad_b += (unsigned long long)(n - p) * sum;
    }
    if (FULL || lim >= 4) {
      u.hs = lz_hash4(w0, L::HS_BITS); u.vS = true; u.cws = headS[u.hs];
      u.vL = FULL || lim >= 6;
      u.hl = u.vL ? lz_hash6(w0, w1, L::HL_BITS) : 0u; u.cwl = headL[u.hl];
      // Candidates: S newest, L newest, L second newest, evaluated without branches so that their loads are in
      // flight together (an unusable candidate compares the unit with itself and is masked).  Fast path over
      // the first 8 bytes: key = matched length class << 16 | ~distance, so that the largest key is the longest
      // match and, among equals, the nearest.
      unsigned bestk = 0;
#pragma unroll
      for (int k = 0; k < 3; k++) {
        const unsigned cand = k == 0 ? u.cws >> 16 : k == 1 ? u.cwl >> 16 : u.cwl & 0xffffu;
        const unsigned du = (u.ub - cand) & 0xffffu;          // any value: q below always lies inside the ring
        // STEP RULE: a match must not read what its own step writes -- its source ends at or before the step's
        // first byte, so cap = dist - li bytes are usable (candidates are units of earlier steps: dist > li; a
        // stale table entry that points into this step is refused).  The decoder relies on it: all the tokens of
        // a step can be resolved at once (seg_resolve_kernel).  A candidate with fewer than 8 usable bytes is not
        // considered at all (so the 8-byte fast path needs no cap, and a long run finds the older candidate
        // whose source is not cut short); the winner's extension is capped below.
        const unsigned dist_k = du * STRIDE;
        const bool ok = du - 1 < (unsigned)L::MAXD_UNITS && (k == 0 || u.vL) && dist_k >= li + 8;
        const unsigned q = (pr - du * STRIDE) & RM;
        const unsigned* qw = ringw + (q >> 2);
        const unsigned sh = q << 3;
        const unsigned t0 = qw[0], t1 = qw[1], t2 = qw[2];
        const unsigned c0 = __funnelshift_r(t0, t1, sh), x1 = __funnelshift_r(t1, t2, sh) ^ w1;
        // length class: 4..8 matched bytes (STRIDE 2: 4, 6, 8) from the trailing zeros of the second word's
        // difference; 8 = the first 8 bytes match (extended below)
        const unsigned tz = (unsigned)__clz((int)__brev(x1));   // 32 when x1 == 0
        const unsigned lc = STRIDE == 2 ? 4u + 2u * (tz >> 4) : 4u + (tz >> 3);
        const unsigned key = (lc << 16) | (0xffffu ^ du);
        bestk = max(bestk, (ok && c0 == w0) ? key : 0u);
      }
      mlen = bestk >> 16;
      if (mlen) {
        mdist = (0xffffu ^ (bestk & 0xffffu)) * STRIDE;
        const unsigned lim2 = min(lim, mdist - li);             // (step rule)
        if (mlen == 8 && lim2 > 8) {
          // the first 8 bytes match: check the next two bytes, which ends it for most; the few matches that go
          // on are compared word by word (no wrap: the mirror covers pr + 258 + 8)
          const unsigned q = (pr - mdist) & RM;
          const bool more = STRIDE == 2 ? *(const unsigned short*)(ring + pr + 8) == *(const unsigned short*)(ring + q + 8)
                                        : ring[pr + 8] == ring[q + 8];
          if (more) {
            unsigned x = 0;
            while (mlen < lim2) {
              x = ring_load4(ring, pr + mlen) ^ ring_load4(ring, q + mlen);
              if (x) break;
              mlen += 4;
            }
            if (x) mlen += (unsigned)(__ffs((int)x) - 1) >> 3;
          }
        }
        mlen = min(mlen, lim2);
        if (STRIDE == 2) mlen &= ~1u;                 // matches cover whole units
        if (mlen < 4) mlen = 0;
        else u.tokw = (0x8000u | mlen) | ((mdist - 1) << 16);
      }
    }
  }
  // ---- (D) greedy parse over units, hierarchical; thread = unit, warp = stretch of 32 units.
  //      Stage 1 (registers, shuffles; here): pointer doubling gives every unit the exit of the token chain that
  //      starts there (where it leaves the stretch) and the mask of the units it visits (= its tokens).
  //      Stage 2 (chain warp): chains the stretches from the carried start (entry + element base per stretch).
  //      Stage 3 (one step later): the warp picks the mask of its entry unit and emits those tokens.
  //      A token is 2 elements (match: length, distance; STRIDE 2 literal: the unit's two bytes) or 1 (STRIDE 1 literal).
  const unsigned nu = (slen + STRIDE - 1) / STRIDE;   // units in this step
  const unsigned sb = wid * 32;
  const unsigned sel = FULL ? 32u : min(sb + 32, nu) > sb ? min(sb + 32, nu) - sb : 0u;   // valid lanes of this stretch
  u.mm = __ballot_sync(0xffffffffu, mlen != 0);
  u.M = 1u << lane;
  unsigned v = lane + (mlen ? mlen / STRIDE : 1u);   // next unit (stretch-local)
#pragma unroll
  for (unsigned r = 0; r < 5; r++) {
    const unsigned tv = __shfl_sync(0xffffffffu, v, v & 31);
    const unsigned tM = __shfl_sync(0xffffffffu, u.M, v & 31);
    if (v < sel) { v = tv; u.M |= tM; }
  }
  const unsigned els = STRIDE == 2 ? 2 * __popc(u.M) : __popc(u.M) + __popc(u.M & u.mm);
  xs[tid] = (sb + v) | (els << 16);
}

template <int STRIDE, int NT>
__global__ void __launch_bounds__(NT + 32, NT <= 512 ? 2 : 1) lz77_kernel(const unsigned char* __restrict__ tbuf,
                                                                          const DeflateSeg* __restrict__ segs, int n_segs,
                                                                          unsigned short* __restrict__ tokens,
                                                                          unsigned* __restrict__ hist,
                                                                          DeflateSegOut* __restrict__ so,
                                                                          unsigned* __restrict__ seg_adler,
                                                                          unsigned long long* __restrict__ sub_tok,
                                                                          unsigned* __restrict__ next_seg) {
  typedef LzSmem<STRIDE, NT> L;
  const unsigned SEG = L::SEG, NSW = L::NSW, RM = LZ_RING - 1;
  const int NALL = NT + 32;                                       // unit threads + the chain warp
  MTS_DYN_SMEM(sm);
  unsigned char* ring = sm + L::ring_off;
  unsigned* headL = (unsigned*)(sm + L::headl_off);
  unsigned* headS = (unsigned*)(sm + L::heads_off);
  unsigned* xe = (unsigned*)(sm + L::xe_off);                    // [step parity][unit]: exit of its stretch | token elements << 16
  unsigned* shist = (unsigned*)(sm + L::hist_off);
  unsigned* misc = (unsigned*)(sm + L::misc_off);                // [step parity][0..31 element base of each stretch, 32..63 entry, 64 step total]
  const mbar_t mbar = mbar_addr((unsigned long long*)(sm + L::mbar_off));
  const unsigned tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned lt = (1u << lane) - 1;
  unsigned phase = 0;                                             // mbarrier phases completed so far (uniform)

  if (tid == 0) mbar_init(mbar);
  __syncthreads();

  // the first segment of a CTA is its block index, the following ones come from a counter (the CTAs drift apart)
  for (int sidx = blockIdx.x; sidx < n_segs;) {
    const DeflateSeg sg = segs[sidx];
    const unsigned n = (unsigned)sg.in_len;
    const unsigned n_steps = (n + SEG - 1) / SEG;
    const unsigned char* in = tbuf + sg.in_off;
    const unsigned off0 = (unsigned)((uintptr_t)in & 15);
    const unsigned char* in16 = in - off0;                   // 16-byte aligned; ring coordinate c holds in16[c]
    unsigned short* tok = tokens + sg.tok_off;
    const unsigned n_ring = n + off0;                        // ring coordinates [off0, n_ring) are real input
    unsigned run_tok = 0;                                    // token elements emitted so far (uniform across the unit threads)
    const unsigned n_sub = sub_tok ? (unsigned)idx_n_sub(n) : 0u;   // index entries of the segment (0: no index wanted)
    unsigned ad_a = 0, ad_c = 0;                             // adler32 partial sums of this thread's units
    unsigned long long ad_b = 0;

    // reset tables (headL and headS are contiguous); pieces 0 and 1 of the input
    for (unsigned i = tid; i < (1u << L::HL_BITS) + (1u << L::HS_BITS); i += NALL) headL[i] = 0;
    for (unsigned i = tid; i < HIST_STRIDE; i += NALL) shist[i] = 0;
    if (tid == 0) {
      const unsigned len = min(2 * SEG, (n_ring + 15) & ~15u), mir = min((unsigned)LZ_MIRROR, len);
      mbar_expect_tx(mbar, len + mir);
      bulk_g2s(ring, in16, len, mbar);
      bulk_g2s(ring + LZ_RING, in16, mir, mbar);
    }
    __syncthreads();

    if (wid == NSW) {
      // ================= chain warp: stage 2 of the parse, one step behind the unit warps' stage 1 and one step ahead
      // of their stage 3 (it works while they look up and compare the next step).  By relaxation (lane = stretch):
      // every lane guesses that its stretch is entered at its first unit, looks up where that chain leaves, and hands
      // the exit to the next lane as ITS entry; repeat until no entry changes.  Lane w is certainly right after w
      // rounds, but greedy parses that start a few units apart merge almost at once, so the exits barely depend on
      // the entries: 2-4 rounds instead of a serial walk.
      unsigned start = 0;                                   // local start unit carried from the previous step
      named_barrier_arrive(1, NALL);
      for (unsigned step = 0; step < n_steps; step++) {
        const unsigned nu = (min(SEG, n - step * SEG) + STRIDE - 1) / STRIDE;
        const unsigned* xs = xe + (step & 1) * NT;
        unsigned* ms = misc + (step & 1) * 72;
        named_barrier(2, NALL);                             // xe[] of this step is complete
        if (start < nu) {
          const unsigned my_se = min((lane + 1) * 32, nu);
          unsigned e = lane == 0 ? start : lane * 32, t = 0;
          for (;;) {
            t = (lane < NSW && e < my_se) ? xs[e] : e;              // exit | elements << 16 (entry beyond the stretch: pass)
            unsigned ne = __shfl_up_sync(0xffffffffu, t & 0xffffu, 1);
            if (lane == 0) ne = start;
            const bool ch = lane < NSW && ne != e;
            e = ne;
            if (!__any_sync(0xffffffffu, ch)) break;
          }
          unsigned acc = lane < NSW ? t >> 16 : 0u;                  // elements emitted by my stretch; inclusive scan
          for (int d = 1; d < 32; d <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, acc, d); if ((int)lane >= d) acc += v; }
          if (lane < NSW) { ms[32 + lane] = e < my_se ? e : 0xffffffffu; ms[lane] = acc - (t >> 16); }
          if (lane == NSW - 1) ms[64] = acc;                         // elements emitted by this step
          start = __shfl_sync(0xffffffffu, t & 0xffffu, NSW - 1) - nu;   // >= 0: where the last token of this step ends
        } else {
          if (lane < NSW) ms[32 + lane] = 0xffffffffu;
          if (lane == 0) ms[64] = 0;
          start -= nu;
        }
        named_barrier_arrive(1, NALL);                      // entries and bases of this step are published
      }
    } else {
    // ================= unit warps
    mbar_wait(mbar, phase & 1); phase++;
    unsigned pM = 0, pmm = 0, ptok = 0;                      // previous step's stage-1 results (emitted one step later)
    for (unsigned step = 0; step <= n_steps; step++) {
      LzUnit u = {};
      LZ_PROF_T(t_step);
      if (step < n_steps) {
        const unsigned s0 = step * SEG;                    // first position of this step
        // piece step + 1 (issued during the previous step) must have landed: this step reads up to s0 + SEG + 294
        if (step > 0 && (step + 1) * SEG < n_ring) { mbar_wait(mbar, phase & 1); phase++; }
        unsigned* xs = xe + (step & 1) * NT;
        if (s0 + SEG + 258 + 16 <= n) lz_find<STRIDE, NT, true>(u, ring, headL, headS, xs, s0, n, off0, tid, ad_a, ad_c, ad_b);
        else lz_find<STRIDE, NT, false>(u, ring, headL, headS, xs, s0, n, off0, tid, ad_a, ad_c, ad_b);
      }
      LZ_PROF_T(t_a);
      named_barrier(1, NALL);                             // #1: every lookup of this step is done; stage 2 of the previous step too

      // ---- (B) insert, first round: any unit of the step becomes the bucket's newest; the next piece of input
      const unsigned myL = (u.ub << 16) | (u.cwl >> 16), myS = (u.ub << 16) | (u.cws >> 16);
      if (u.vL) headL[u.hl] = myL;
      if (u.vS) headS[u.hs] = myS;
      if (tid == 0 && (step + 2) * SEG < n_ring) {
        const unsigned c0 = (step + 2) * SEG, o = c0 & RM;
        const unsigned len = min(SEG, (n_ring - c0 + 15) & ~15u), mir = o == 0 ? min((unsigned)LZ_MIRROR, len) : 0u;
        mbar_expect_tx(mbar, len + mir);
        bulk_g2s(ring + o, in16 + c0, len, mbar);
        if (mir) bulk_g2s(ring + LZ_RING, in16 + c0, mir, mbar);
      }
      // ---- stage 3 of the previous step: emit
      if (step > 0) {
        const unsigned* ms = misc + ((step - 1) & 1) * 72;
        const unsigned entry = ms[32 + wid];
        // (sub-block boundaries are multiples of IDX_SUB_BYTES / 2: only a step that reaches one can hold such a token)
        const unsigned ps = (step - 1) * SEG;
        const bool idx_near = n_sub && ((ps + SEG + 258) / (IDX_SUB_BYTES / 2)) != (ps / (IDX_SUB_BYTES / 2));
        if (entry != 0xffffffffu) {                         // warp-uniform
          const unsigned reach = __shfl_sync(0xffffffffu, pM, entry & 31);
          if ((reach >> lane) & 1u) {
            const unsigned before = reach & lt;
            const unsigned pos = run_tok + ms[wid] + (STRIDE == 2 ? 2 * __popc(before) : __popc(before) + __popc(before & pmm));
            if (idx_near) {
              // in-band index: a token whose output reaches the next sub-block boundary makes its successor the first
              // token of that sub-block; noted as (token element index of the successor) << 9 | output overshoot, the
              // encode kernel turns the element index into a bit offset
              const unsigned pp = (step - 1) * SEG + tid * STRIDE;
              const unsigned pl = (ptok & 0x8000u) ? (ptok & 0x1ffu) : (STRIDE == 2 ? 2u : 1u);
              const unsigned jn = idx_item(pp + pl);
              if (jn != idx_item(pp) && jn < n_sub)
                sub_tok[sg.sub_first + jn] = ((unsigned long long)(pos + ((ptok & 0x8000u) || STRIDE == 2 ? 2u : 1u)) << 9) | (pp + pl - idx_bound(jn));
            }
            if (ptok & 0x8000u) {
              if (STRIDE == 2) *(unsigned*)(tok + pos) = ptok;
              else { tok[pos] = (unsigned short)ptok; tok[pos + 1] = (unsigned short)(ptok >> 16); }
              unsigned sym, nb, ev;
              len_symbol(ptok & 0x1ffu, sym, nb, ev);
              atomicAdd(&shist[sym], 1u);
              dist_symbol((ptok >> 16) + 1, sym, nb, ev);
              atomicAdd(&shist[288 + sym], 1u);
            } else {
              atomicAdd(&shist[ptok & 0xffu], 1u);
              if (STRIDE == 2) {
                *(unsigned*)(tok + pos) = ptok;
                atomicAdd(&shist[ptok >> 16], 1u);
              } else tok[pos] = (unsigned short)ptok;
            }
          }
        }
        run_tok += ms[64];
      }
      if (step == n_steps) break;
      pM = u.M; pmm = u.mm; ptok = u.tokw;
      LZ_PROF_T(t_b);
      named_barrier(2, NALL);                             // #2: first-round stores are visible (and xe[] to the chain warp)

      // ---- (B) insert, second round: a lower unit of this step in my bucket gives way
      if (u.vL) { const unsigned d = (u.ub - (headL[u.hl] >> 16)) & 0xffffu; if (d - 1 < NT - 1) atomicMax(&headL[u.hl], myL); }
      if (u.vS) { const unsigned d = (u.ub - (headS[u.hs] >> 16)) & 0xffffu; if (d - 1 < NT - 1) atomicMax(&headS[u.hs], myS); }
      LZ_PROF_T(t_c);
      named_barrier(3, NT);                               // #3: buckets settled
      LZ_PROF_ADD(0, 1); LZ_PROF_ADD(1, t_a - t_step); LZ_PROF_ADD(2, t_b - t_a); LZ_PROF_ADD(3, t_c - t_b); LZ_PROF_ADD(5, t_c - t_step);
    }
    }

    // ---- segment done: publish histogram + token count (the barrier also keeps the next segment's table reset and
    //      input pieces away from threads still emitting)
    //      adler32 of the segment's bytes (standalone, from adler = 1; folded per chunk by adler_combine_kernel)
    {
      unsigned long long a = ad_a, b = (ad_b - ad_c) % ADLER_BASE;
      a = warp_sum(a); b = warp_sum(b);
      unsigned long long* red = (unsigned long long*)xe;
      if (lane == 0) { red[2 * wid] = a; red[2 * wid + 1] = b; }
    }
    __syncthreads();
    for (unsigned i = tid; i < HIST_STRIDE; i += NALL) hist[(size_t)sidx * HIST_STRIDE + i] = shist[i];
    if (tid == 0) {
      so[sidx].n_tok = run_tok;
      const unsigned long long* red = (const unsigned long long*)xe;
      unsigned long long ta = 0, tb = 0;
      for (unsigned w = 0; w < NSW; w++) { ta += red[2 * w]; tb += red[2 * w + 1]; }
      seg_adler[sidx] = ((unsigned)((n % ADLER_BASE + tb) % ADLER_BASE) << 16) | (unsigned)((1 + ta) % ADLER_BASE);
      misc[2 * 72] = gridDim.x + atomicAdd(next_seg, 1u);
    }
    __syncthreads();
    sidx = (int)misc[2 * 72];
  }
}

// ------------------------------------------------------------------------------------------------ huff_kernel
// One warp per segment.  Package: sort used symbols by frequency (rank sort across lanes), two-queue Huffman merge,
// depth count, zlib-style overflow repair to the length limit, canonical codes (bit-reversed for LSB-first packing).
struct HuffScratch {
  unsigned weight[2 * LL_SYMS];
  unsigned short parent[2 * LL_SYMS];
  unsigned short sorted[LL_SYMS];
  unsigned char depth[2 * LL_SYMS];
  unsigned char lens[LL_SYMS + D_SYMS + 8];
  unsigned char rle_sym[LL_SYMS + D_SYMS + 8];
  unsigned char rle_ext[LL_SYMS + D_SYMS + 8];
  unsigned bl_freq[BL_SYMS];
  unsigned bl_code[BL_SYMS];
  unsigned bl_count[16];
  unsigned next_code[16];
  unsigned hdr[HDR_WORDS];
};

// Builds code lengths for `nsym` symbols with frequencies f[] (u32, >= 2 non-zero entries) limited to maxbits, then
// canonical bit-reversed codes: out[s] = code | len << 16.  All lanes call; lane 0 does the serial parts.
__device__ void build_codes(const unsigned* f, int nsym, int maxbits, unsigned* out, unsigned char* lens_out,
                            HuffScratch* S) {
  const unsigned lane = lane_id();
  // rank sort of used symbols by (freq, symbol)
  int nused = 0;
  for (int s0 = 0; s0 < nsym; s0 += 32) {
    int s = s0 + lane;
    bool used = s < nsym && f[s] > 0;
    nused += __popc(__ballot_sync(0xffffffffu, used));
  }
  for (int s = lane; s < nsym; s += 32) {
    unsigned fs = f[s];
    lens_out[s] = 0;
    if (!fs) continue;
    int rank = 0;
    for (int t = 0; t < nsym; t++) {
      unsigned ft = f[t];
      rank += (ft > 0) && (ft < fs || (ft == fs && t < s));
    }
    S->sorted[rank] = (unsigned short)s;
  }
  __syncwarp();
  if (lane == 0) {
    const int n = nused;
    for (int i = 0; i < n; i++) S->weight[i] = f[S->sorted[i]];
    // two-queue merge: leaves [0,n), internal nodes [n, 2n-1)
    int a = 0, b = n, e = n;
    for (; e < 2 * n - 1; e++) {
      unsigned w = 0;
      for (int k = 0; k < 2; k++) {
        int pick;
        if (a < n && (b >= e || S->weight[a] <= S->weight[b])) pick = a++; else pick = b++;
        w += S->weight[pick];
        S->parent[pick] = (unsigned short)e;
      }
      S->weight[e] = w;
    }
    for (int i = 0; i <= maxbits; i++) S->bl_count[i] = 0;
    const int root = 2 * n - 2;
    S->depth[root] = 0;
    for (int i = root - 1; i >= 0; i--) {
      int d = S->depth[S->parent[i]] + 1;
      if (i < n) S->bl_count[min(d, maxbits)]++;
      S->depth[i] = (unsigned char)min(d, 255);
    }
    // length limiting: clamping deep leaves to maxbits over-subscribes the code by `excess` units of 2^-maxbits;
    // each zlib-style move (one leaf one level down, one clamped leaf becomes its sibling) removes exactly one unit
    long long excess = -(1ll << maxbits);
    for (int b = 1; b <= maxbits; b++) excess += (long long)S->bl_count[b] << (maxbits - b);
    while (excess > 0) {
      int bits = maxbits - 1;
      while (S->bl_count[bits] == 0) bits--;
      S->bl_count[bits]--;
      S->bl_count[bits + 1] += 2;
      S->bl_count[maxbits]--;
      excess--;
    }
    // least frequent symbols take the longest codes
    int i = 0;
    for (int bits = maxbits; bits >= 1; bits--)
      for (unsigned k = 0; k < S->bl_count[bits]; k++) lens_out[S->sorted[i++]] = (unsigned char)bits;
    unsigned code = 0;
    S->bl_count[0] = 0;
    for (int bits = 1; bits <= maxbits; bits++) {
      code = (code + S->bl_count[bits - 1]) << 1;
      S->next_code[bits] = code;
    }
    for (int s = 0; s < nsym; s++) {
      unsigned l = lens_out[s];
      unsigned c = 0;
      if (l) c = __brev(S->next_code[l]++) >> (32 - l);
      out[s] = c | (l << 16);
    }
  }
  __syncwarp();
}

struct BitW {   // serial LSB-first bit writer (lane 0 of huff_kernel)
  unsigned* w;
  unsigned nbits;
  __device__ void put(unsigned v, unsigned n) {
    if (!n) return;
    unsigned i = nbits >> 5, sh = nbits & 31;
    w[i] |= v << sh;
    if (sh + n > 32) w[i + 1] |= v >> (32 - sh);
    nbits += n;
  }
};

__global__ void __launch_bounds__(32) huff_kernel(const DeflateSeg* __restrict__ segs, int n_segs,
                                                  unsigned* __restrict__ hist, unsigned* __restrict__ codes,
                                                  unsigned* __restrict__ hdrs, DeflateSegOut* __restrict__ so) {
  __shared__ HuffScratch S;
  __shared__ unsigned f[HIST_STRIDE];
  __shared__ unsigned c[CODE_STRIDE];
  __shared__ unsigned char bl_len_sh[BL_SYMS + 5];
  __shared__ int sh_nr, sh_hlit, sh_hdist;
  const int sidx = blockIdx.x;
  if (sidx >= n_segs) return;
  const unsigned lane = lane_id();
  for (int i = lane; i < HIST_STRIDE; i += 32) f[i] = hist[(size_t)sidx * HIST_STRIDE + i];
  for (int i = lane; i < HDR_WORDS; i += 32) S.hdr[i] = 0;
  __syncwarp();
  if (lane == 0) {
    f[256] += 1;                                          // end-of-block
    // at least two used symbols per tree (zlib does the same so that every tree is complete)
    int used = 0;
    for (int i = 0; i < LL_SYMS; i++) used += f[i] > 0;
    for (int i = 0; used < 2; i++) if (!f[i]) { f[i] = 1; used++; }
    used = 0;
    for (int i = 0; i < D_SYMS; i++) used += f[288 + i] > 0;
    for (int i = 0; used < 2; i++) if (!f[288 + i]) { f[288 + i] = 1; used++; }
  }
  __syncwarp();
  build_codes(f, LL_SYMS, 15, c, S.lens, &S);
  build_codes(f + 288, D_SYMS, 15, c + 288, S.lens + LL_SYMS, &S);

  // body size in bits under the dynamic codes
  unsigned long long bits = 0;
  for (int s = lane; s < LL_SYMS; s += 32) bits += (unsigned long long)hist[(size_t)sidx * HIST_STRIDE + s] * ((c[s] >> 16) + ll_extra_bits(s));
  for (int s = lane; s < D_SYMS; s += 32) bits += (unsigned long long)hist[(size_t)sidx * HIST_STRIDE + 288 + s] * ((c[288 + s] >> 16) + d_extra_bits(s));
  bits = warp_sum(bits);
  bits += c[256] >> 16;

  if (lane == 0) {
    int hlit = LL_SYMS, hdist = D_SYMS;
    while (hlit > 257 && S.lens[hlit - 1] == 0) hlit--;
    while (hdist > 1 && S.lens[LL_SYMS + hdist - 1] == 0) hdist--;
    // concatenated length sequence, run-length coded with symbols 16/17/18 (RFC 1951 3.2.7)
    unsigned char seq[LL_SYMS + D_SYMS];
    int nseq = 0;
    for (int i = 0; i < hlit; i++) seq[nseq++] = S.lens[i];
    for (int i = 0; i < hdist; i++) seq[nseq++] = S.lens[LL_SYMS + i];
    for (int i = 0; i < BL_SYMS; i++) S.bl_freq[i] = 0;
    int nr = 0;
    for (int i = 0; i < nseq;) {
      int v = seq[i], run = 1;
      while (i + run < nseq && seq[i + run] == v) run++;
      i += run;
      if (v == 0) {
        while (run >= 11) { int r = min(run, 138); S.rle_sym[nr] = 18; S.rle_ext[nr++] = (unsigned char)(r - 11); run -= r; }
        if (run >= 3) { S.rle_sym[nr] = 17; S.rle_ext[nr++] = (unsigned char)(run - 3); run = 0; }
        while (run-- > 0) { S.rle_sym[nr] = 0; S.rle_ext[nr++] = 0; }
      } else {
        S.rle_sym[nr] = (unsigned char)v; S.rle_ext[nr++] = 0; run--;
        while (run >= 3) { int r = min(run, 6); S.rle_sym[nr] = 16; S.rle_ext[nr++] = (unsigned char)(r - 3); run -= r; }
        while (run-- > 0) { S.rle_sym[nr] = (unsigned char)v; S.rle_ext[nr++] = 0; }
      }
    }
    for (int i = 0; i < nr; i++) S.bl_freq[S.rle_sym[i]]++;
    int used = 0;
    for (int i = 0; i < BL_SYMS; i++) used += S.bl_freq[i] > 0;
    for (int i = 0; used < 2; i++) if (!S.bl_freq[i]) { S.bl_freq[i] = 1; used++; }
    sh_nr = nr; sh_hlit = hlit; sh_hdist = hdist;
  }
  __syncwarp();
  const int nr = sh_nr, hlit = sh_hlit, hdist = sh_hdist;
  build_codes(S.bl_freq, BL_SYMS, 7, S.bl_code, bl_len_sh, &S);

  if (lane == 0) {
    static const unsigned char order[BL_SYMS] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int hclen = BL_SYMS;
    while (hclen > 4 && bl_len_sh[order[hclen - 1]] == 0) hclen--;
    BitW bw{S.hdr, 0};
    bw.put(0, 1);             // BFINAL = 0 (the stream is closed by a separate empty final block)
    bw.put(2, 2);             // BTYPE = 10 dynamic
    bw.put((unsigned)(hlit - 257), 5);
    bw.put((unsigned)(hdist - 1), 5);
    bw.put((unsigned)(hclen - 4), 4);
    for (int i = 0; i < hclen; i++) bw.put(bl_len_sh[order[i]], 3);
    for (int i = 0; i < nr; i++) {
      unsigned s = S.rle_sym[i];
      bw.put(S.bl_code[s] & 0xffff, S.bl_code[s] >> 16);
      if (s == 16) bw.put(S.rle_ext[i], 2);
      else if (s == 17) bw.put(S.rle_ext[i], 3);
      else if (s == 18) bw.put(S.rle_ext[i], 7);
    }
    const unsigned n = (unsigned)segs[sidx].in_len;
    unsigned long long dyn_bits = bw.nbits + bits;
    // + empty stored block that byte-aligns the next segment: 3 header bits, pad, 00 00 FF FF
    unsigned dyn_bytes = (unsigned)((dyn_bits + 3 + 7) >> 3) + 4;
    unsigned stored_bytes = n + 5 * ((n + 65534) / 65535);
    DeflateSegOut o = so[sidx];
    o.hdr_bits = bw.nbits;
    if (dyn_bytes < stored_bytes) { o.mode = MODE_DYNAMIC; o.body_bytes = dyn_bytes; }
    else { o.mode = MODE_STORED; o.body_bytes = stored_bytes; }
    so[sidx] = o;
  }
  __syncwarp();
  for (int i = lane; i < CODE_STRIDE; i += 32) codes[(size_t)sidx * CODE_STRIDE + i] = c[i];
  for (int i = lane; i < HDR_WORDS; i += 32) hdrs[(size_t)sidx * HDR_WORDS + i] = S.hdr[i];
}

// ------------------------------------------------------------------------------------------------ scan_kernel
// Single CTA: exclusive prefix of (zlib header + body + trailer) sizes over all segments of the batch, in order.
// Segments of a chunk are contiguous, so chunk_off[] (n_chunks + 1 entries) falls out of the same scan.
__global__ void __launch_bounds__(1024) scan_kernel(const DeflateSeg* __restrict__ segs, int n_segs,
                                                    DeflateSegOut* __restrict__ so, long long* __restrict__ chunk_off,
                                                    int n_chunks, const ChunkDesc* __restrict__ chunks,
                                                    int write_index) {
  __shared__ unsigned long long wsum[32];
  __shared__ unsigned long long carry, tile_total;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n_segs; base += 1024) {
    int i = base + threadIdx.x;
    unsigned long long sz = 0;
    int fl = 0;
    if (i < n_segs) {
      fl = segs[i].flags;
      sz = so[i].body_bytes + ((fl & SEG_FIRST) ? 2 : 0) + ((fl & SEG_LAST) ? 6 : 0);
      if ((fl & SEG_LAST) && write_index) {
        const ChunkDesc cd = chunks[segs[i].chunk];
        const unsigned subs = (unsigned)(segs[i].sub_first + idx_n_sub(segs[i].in_len) - segs[cd.first_seg].sub_first);
        if (idx_wanted(cd.n_seg, segs[cd.first_seg].in_len)) sz += 4ull * subs + 4ull * (unsigned)cd.n_seg + 24;
      }
    }
    unsigned long long incl = warp_incl_scan(sz);
    if (lane_id() == 31) wsum[warp_id()] = incl;
    __syncthreads();
    if (warp_id() == 0) {
      unsigned long long t = wsum[lane_id()];
      unsigned long long ti = warp_incl_scan(t);
      wsum[lane_id()] = ti - t;
      if (lane_id() == 31) tile_total = ti;
    }
    __syncthreads();
    unsigned long long excl = carry + wsum[warp_id()] + incl - sz;
    if (i < n_segs) {
      so[i].out_off = (long long)excl;
      if (fl & SEG_FIRST) chunk_off[segs[i].chunk] = (long long)excl;
      if (i == n_segs - 1) chunk_off[n_chunks] = (long long)(excl + sz);
    }
    __syncthreads();
    if (threadIdx.x == 0) carry += tile_total;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ encode_kernel
static const int ENC_THREADS = 256;
static const int ENC_PER = 8;                              // token elements per thread per tile
static const int ENC_TILE = ENC_THREADS * ENC_PER;
static const int ENC_STAGE_WORDS = ENC_TILE + 64;          // >= tile * 28 bits / 32 + header slack

__device__ __forceinline__ void stage_or(unsigned* stage, unsigned bitpos, unsigned v, unsigned n) {
  if (!n) return;
  unsigned i = bitpos >> 5, sh = bitpos & 31;
  atomicOr(&stage[i], v << sh);
  if (sh + n > 32) atomicOr(&stage[i + 1], v >> (32 - sh));
}

// Flush stage words [0, nwords) to global memory starting at the 4-byte aligned address `gw`; bytes before
// `lo_byte` (absolute address) or at/after `hi_byte` are not touched (they belong to neighbouring segments).
__device__ __forceinline__ void stage_flush(const unsigned* stage, unsigned nwords, unsigned char* gw,
                                            const unsigned char* lo_byte, const unsigned char* hi_byte) {
  for (unsigned i = threadIdx.x; i < nwords; i += blockDim.x) {
    unsigned char* a = gw + 4 * (size_t)i;
    unsigned v = stage[i];
    if (a >= lo_byte && a + 4 <= hi_byte) *(unsigned*)a = v;
    else
      for (int b = 0; b < 4; b++)
        if (a + b >= lo_byte && a + b < hi_byte) a[b] = (unsigned char)(v >> (8 * b));
  }
}

template <bool PAIRS>
__global__ void __launch_bounds__(ENC_THREADS) encode_kernel(const unsigned char* __restrict__ tbuf,
                                                             const DeflateSeg* __restrict__ segs, int n_segs,
                                                             const unsigned short* __restrict__ tokens,
                                                             const unsigned* __restrict__ codes,
                                                             const unsigned* __restrict__ hdrs,
                                                             const DeflateSegOut* __restrict__ so,
                                                             const unsigned* __restrict__ chunk_adler,
                                                             unsigned char* __restrict__ dst,
                                                             const unsigned long long* __restrict__ sub_tok,   // lz77's notes
                                                             unsigned long long* __restrict__ sub_abs) {         // bit offsets
  __shared__ unsigned stage[ENC_STAGE_WORDS];
  __shared__ unsigned code[CODE_STRIDE];
  __shared__ unsigned wtot[ENC_THREADS / 32];
  __shared__ unsigned tile_bits;
  const int sidx = blockIdx.x;
  if (sidx >= n_segs) return;
  const DeflateSeg sg = segs[sidx];
  const DeflateSegOut o = so[sidx];
  const unsigned tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  unsigned char* out = dst + o.out_off;
  const unsigned total = o.body_bytes + ((sg.flags & SEG_FIRST) ? 2 : 0) + ((sg.flags & SEG_LAST) ? 6 : 0);
  unsigned char* const out_end = out + total;   // end of the zlib stream part written by this CTA
  if (sg.flags & SEG_FIRST) {
    if (tid == 0) { out[0] = 0x78; out[1] = 0x9c; }
    out += 2;
  }
  unsigned char* body_end = out + o.body_bytes;
  if ((sg.flags & SEG_LAST) && tid < 6) {
    // empty final fixed-Huffman block (03 00) + adler32 of the whole transformed chunk, big-endian
    unsigned a = chunk_adler[sg.chunk];
    unsigned char t[6] = {0x03, 0x00, (unsigned char)(a >> 24), (unsigned char)(a >> 16), (unsigned char)(a >> 8), (unsigned char)a};
    body_end[tid] = t[tid];
  }
  // sub-block table of this segment: lz77_kernel left (token element index << 9 | output overshoot) for the entries 1..,
  // this kernel replaces the element index by the bit offset of that element (entry 0: the first token); all zero for
  // a stored segment
  const int n_sub = idx_n_sub(sg.in_len);
  if (sub_abs && o.mode == MODE_STORED) for (int j = tid; j < n_sub; j += blockDim.x) sub_abs[sg.sub_first + j] = 0;
  const unsigned char* in = tbuf + sg.in_off;
  if (o.mode == MODE_STORED) {
    unsigned n = (unsigned)sg.in_len;
    for (unsigned b0 = 0, k = 0; b0 < n; b0 += 65535, k++) {
      unsigned len = min(65535u, n - b0);
      unsigned char* q = out + b0 + 5 * (size_t)k;
      if (tid == 0) { q[0] = 0; q[1] = (unsigned char)len; q[2] = (unsigned char)(len >> 8); q[3] = (unsigned char)~len; q[4] = (unsigned char)(~len >> 8); }
      for (unsigned i = tid; i < len; i += blockDim.x) q[5 + i] = in[b0 + i];
    }
    return;
  }
  // ---- dynamic block
  for (unsigned i = tid; i < CODE_STRIDE; i += blockDim.x) code[i] = codes[(size_t)sidx * CODE_STRIDE + i];
  for (unsigned i = tid; i < ENC_STAGE_WORDS; i += blockDim.x) stage[i] = 0;
  __syncthreads();
  unsigned char* gw = (unsigned char*)((uintptr_t)out & ~(uintptr_t)3);   // global address of stage word 0
  unsigned cur = 8 * (unsigned)((uintptr_t)out & 3);                       // bit cursor inside the stage
  // header
  {
    const unsigned* h = hdrs + (size_t)sidx * HDR_WORDS;
    const unsigned hb = o.hdr_bits;
    for (unsigned j = tid; j * 32 < hb; j += blockDim.x) stage_or(stage, cur + 32 * j, h[j], min(32u, hb - 32 * j));
    __syncthreads();
    cur += hb;
    unsigned nw = cur >> 5;
    stage_flush(stage, nw, gw, out, out_end);
    __syncthreads();
    unsigned keep = stage[nw];
    __syncthreads();
    for (unsigned i = tid; i <= nw; i += blockDim.x) stage[i] = 0;
    __syncthreads();
    if (tid == 0) stage[0] = keep;
    gw += 4 * (size_t)nw;
    cur &= 31;
    __syncthreads();
  }
  // Each thread turns 8 token elements into 8 codes of <= 28 bits (PAIRS: the elements come as 4 aligned 32-bit tokens
  // -- length | distance << 16, or two literal bytes -- so there is no dependence on the previous element), the block
  // prefix sum of the bit counts places them, and the thread strings its codes together in a 64-bit register: whole
  // words go to the staging window with plain stores, only the first and the last (shared with the neighbours) by atomicOr.
  const unsigned short* tok = tokens + sg.tok_off;
  const unsigned ntok = o.n_tok;
  unsigned seg_bits = o.hdr_bits;                   // bits of the segment before the tile
  int sub_cur = 1;                                  // next entry of the sub-block table to resolve (uniform) ...
  unsigned note_el = 0xffffffffu, note_ov = 0;      // ... its token element index and overshoot, as lz77_kernel noted them
  if (sub_abs && n_sub > 1) {
    const unsigned long long note = sub_tok[sg.sub_first + 1];
    note_el = (unsigned)(note >> 9); note_ov = (unsigned)(note & 511u);
  }
  if (!sub_abs) sub_cur = n_sub;
  if (sub_abs && tid == 0) sub_abs[sg.sub_first] = (unsigned long long)o.hdr_bits << 9;
  for (unsigned base = 0; base < ntok; base += ENC_TILE) {
    unsigned v[ENC_PER], nb[ENC_PER], mine = 0;
    const unsigned i0 = base + tid * ENC_PER;
    if (PAIRS) {
      uint4 t4 = make_uint4(0, 0, 0, 0);
      if (i0 + ENC_PER <= ntok && !((uintptr_t)(tok + i0) & 15)) t4 = *(const uint4*)(tok + i0);
      else {
        const unsigned* tw = (const unsigned*)(tok + i0);
        if (i0 < ntok) t4.x = tw[0];
        if (i0 + 2 < ntok) t4.y = tw[1];
        if (i0 + 4 < ntok) t4.z = tw[2];
        if (i0 + 6 < ntok) t4.w = tw[3];
      }
      const unsigned tk[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const unsigned e = tk[j];
        unsigned c0, c1, x0 = 0, x1 = 0, e0 = 0, e1 = 0;
        if (e & 0x8000u) {                  // match: length element, distance element
          unsigned sym;
          len_symbol(e & 0x1ffu, sym, x0, e0);
          c0 = code[sym];
          dist_symbol((e >> 16) + 1, sym, x1, e1);
          c1 = code[288 + sym];
        } else { c0 = code[e & 0xffu]; c1 = code[e >> 16]; }
        const bool on = i0 + 2 * j < ntok;
        v[2 * j] = (c0 & 0xffffu) | (e0 << (c0 >> 16));
        nb[2 * j] = on ? (c0 >> 16) + x0 : 0u;
        v[2 * j + 1] = (c1 & 0xffffu) | (e1 << (c1 >> 16));
        nb[2 * j + 1] = on ? (c1 >> 16) + x1 : 0u;
        mine += nb[2 * j] + nb[2 * j + 1];
      }
    } else {
      unsigned prev_el = (i0 > 0 && i0 <= ntok) ? tok[i0 - 1] : 0;
      // bit 15 marks a length element (distance elements are <= 32767), and what follows a length is its distance
      for (int j = 0; j < ENC_PER; j++) {
        unsigned i = i0 + j;
        v[j] = 0; nb[j] = 0;
        if (i < ntok) {
          unsigned e = tok[i];
          if (prev_el & 0x8000u) {            // distance element (follows a length element): closes the match
            unsigned sym, xb, ev;
            dist_symbol(e + 1, sym, xb, ev);
            unsigned c = code[288 + sym];
            v[j] = (c & 0xffff) | (ev << (c >> 16));
            nb[j] = (c >> 16) + xb;
            prev_el = 0;
          } else if (e & 0x8000u) {           // length element
            unsigned sym, xb, ev;
            len_symbol(e & 0x1ff, sym, xb, ev);
            unsigned c = code[sym];
            v[j] = (c & 0xffff) | (ev << (c >> 16));
            nb[j] = (c >> 16) + xb;
            prev_el = e;
          } else {                            // literal
            unsigned c = code[e];
            v[j] = c & 0xffff;
            nb[j] = c >> 16;
            prev_el = e;
          }
          mine += nb[j];
        }
      }
    }
    unsigned incl = warp_incl_scan(mine);
    if (lane == 31) wtot[wid] = incl;
    __syncthreads();
    if (tid == 0) {
      unsigned run = 0;
      for (int w = 0; w < ENC_THREADS / 32; w++) { unsigned t = wtot[w]; wtot[w] = run; run += t; }
      tile_bits = run;
    }
    __syncthreads();
    // sub-block table: the noted token element that falls into this tile gets its bit offset (usually none, at most a few)
    while (note_el < base + ENC_TILE && note_el < ntok) {
      if (note_el >= i0 && note_el < i0 + ENC_PER) {
        unsigned bit = seg_bits + wtot[wid] + incl - mine;
#pragma unroll
        for (unsigned j = 0; j < (unsigned)ENC_PER; j++) bit += j < note_el - i0 ? nb[j] : 0u;
        sub_abs[sg.sub_first + sub_cur] = ((unsigned long long)bit << 9) | note_ov;
      }
      sub_cur++;
      const unsigned long long note = sub_cur < n_sub ? sub_tok[sg.sub_first + sub_cur] : ~0ull;
      note_el = sub_cur < n_sub ? (unsigned)(note >> 9) : 0xffffffffu;
      note_ov = (unsigned)(note & 511u);
    }
    if (mine) {
      const unsigned bp = cur + wtot[wid] + incl - mine;
      unsigned wi = bp >> 5, fill = bp & 31;
      unsigned long long acc = 0;
      bool first = true;
#pragma unroll
      for (int j = 0; j < ENC_PER; j++) {
        acc |= (unsigned long long)v[j] << fill;
        fill += nb[j];
        if (fill >= 32) {
          if (first) { atomicOr(&stage[wi], (unsigned)acc); first = false; } else stage[wi] = (unsigned)acc;
          wi++; acc >>= 32; fill -= 32;
        }
      }
      if (fill) atomicOr(&stage[wi], (unsigned)acc);
    }
    __syncthreads();
    cur += tile_bits;
    seg_bits += tile_bits;
    unsigned nw = cur >> 5;
    stage_flush(stage, nw, gw, out, out_end);
    __syncthreads();
    unsigned keep = stage[nw];
    __syncthreads();
    for (unsigned i = tid; i <= nw + 1; i += blockDim.x) stage[i] = 0;
    __syncthreads();
    if (tid == 0) stage[0] = keep;
    gw += 4 * (size_t)nw;
    cur &= 31;
    __syncthreads();
  }
  // end-of-block, then the empty stored block: 3 zero bits, pad to a byte boundary, 00 00 FF FF
  if (tid == 0) {
    unsigned c = code[256];
    stage_or(stage, cur, c & 0xffff, c >> 16);
    unsigned e = cur + (c >> 16) + 3;
    e = (e + 7) & ~7u;
    stage_or(stage, e + 16, 0xffffu, 16);
    tile_bits = e + 32;
  }
  __syncthreads();
  unsigned endbits = tile_bits;
  stage_flush(stage, (endbits + 31) >> 5, gw, out, body_end);
}

// ------------------------------------------------------------------------------------------------ trailer_kernel
// One CTA per chunk, after encode_kernel: the in-band index (layout at IDX_MAGIC_V2 above) behind the chunk's zlib stream.
__device__ __forceinline__ void put32(unsigned char* p, unsigned v) {
  p[0] = (unsigned char)v; p[1] = (unsigned char)(v >> 8); p[2] = (unsigned char)(v >> 16); p[3] = (unsigned char)(v >> 24);
}
__global__ void __launch_bounds__(128) trailer_kernel(const DeflateSeg* __restrict__ segs, const DeflateSegOut* __restrict__ so,
                                                      const ChunkDesc* __restrict__ chunks, const long long* __restrict__ chunk_off,
                                                      const unsigned long long* __restrict__ sub_abs,
                                                      unsigned char* __restrict__ dst, unsigned step_bytes) {
  const ChunkDesc cd = chunks[blockIdx.x];
  const unsigned k = (unsigned)cd.n_seg;
  const DeflateSeg s0 = segs[cd.first_seg], s1 = segs[cd.first_seg + k - 1];
  if (!idx_wanted(cd.n_seg, s0.in_len)) return;
  const unsigned n_subs = (unsigned)(s1.sub_first + idx_n_sub(s1.in_len) - s0.sub_first);
  unsigned char* ix = dst + chunk_off[blockIdx.x + 1] - (4ull * n_subs + 4ull * k + 24);
  for (unsigned q = threadIdx.x; q < k; q += blockDim.x) {
    const DeflateSeg sg = segs[cd.first_seg + q];
    const int ns = idx_n_sub(sg.in_len);
    for (int j = 0; j < ns; j++) {
      const unsigned long long a = sub_abs[sg.sub_first + j], b = j ? sub_abs[sg.sub_first + j - 1] : 0ull;
      const unsigned delta = (unsigned)((a >> 9) - (b >> 9));
      put32(ix + 4ull * (unsigned)(sg.sub_first - s0.sub_first + j), (delta & 0x1ffffu) | ((unsigned)(a & 511u) << 17));
    }
    put32(ix + 4ull * n_subs + 4ull * q, so[cd.first_seg + q].body_bytes);
  }
  if (threadIdx.x == 0) {
    unsigned sum = 0;
    for (unsigned q = 0; q < k; q++) sum += so[cd.first_seg + q].body_bytes;
    unsigned char* t = ix + 4ull * n_subs + 4ull * k;
    put32(t, IDX_SUB_BYTES); put32(t + 4, step_bytes);
    put32(t + 8, (unsigned)cd.pad_); put32(t + 12, k); put32(t + 16, IDX_MAGIC_V2); put32(t + 20, sum);
  }
}

}  // namespace mts
