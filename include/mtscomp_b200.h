/* mtscomp_b200.h — C ABI of the B200-native per-chunk codec for mtscomp (.cbin / .ch) files.
 *
 * The reference (int-brain-lab/mtscomp) has no FFI: its codec seam is two Python methods whose bodies call NumPy and
 * zlib.  Each entry point below names the reference code it replaces (file:line in the reference's mtscomp.py).  All
 * functions are plain C: pointers, sizes, ints.  Buffers are caller-allocated; `*_is_device` says whether a pointer is
 * a CUDA device pointer on the context's device (1) or host memory (0; pinned memory makes the copies asynchronous).
 * The library owns only its context (stream, scratch, tables).  A context is not re-entrant: one call at a time per
 * context (the Python layer holds a lock; create one context per thread/stream if you want concurrency).
 *
 * Return values: 0 = success, negative = MTSB_E_* below; mtsb_last_error() gives a message for the last failure.
 * There is no CPU fallback: without a usable CUDA device mtsb_create() fails.
 */
#ifndef MTSCOMP_B200_H
#define MTSCOMP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mtsb_ctx mtsb_ctx;

enum {
  MTSB_OK = 0,
  MTSB_E_CUDA = -1,       /* CUDA runtime error */
  MTSB_E_ARG = -2,        /* invalid argument */
  MTSB_E_CAPACITY = -3,   /* destination too small (see mtsb_compress_bound) */
  MTSB_E_NOMEM = -4,      /* device scratch allocation failed */
  MTSB_E_CORRUPT = -5     /* at least one compressed chunk failed to decode; see chunk_status[] */
};

/* transform flags (Writer options do_time_diff / do_spatial_diff / chunk_order, mtscomp.py:250-255) */
enum { MTSB_TIME_DIFF = 1, MTSB_SPATIAL_DIFF = 2, MTSB_ORDER_C = 4,
       MTSB_FLOAT = 8 /* elements are IEEE float32 / float64 (itemsize 4 / 8) instead of integers: the differences are
                         float subtractions and the inverse adds sequentially, as np.diff / np.cumsum do */ };

/* per-chunk decode status (chunk_status[]); non-zero maps to the reference's
 * IOError("Compressed chunk #%d is corrupted.") raised at mtscomp.py:618-621 */
enum {
  MTSB_CHUNK_OK = 0, MTSB_CHUNK_BAD_HEADER = 1, MTSB_CHUNK_BAD_BLOCK = 2, MTSB_CHUNK_BAD_LENGTHS = 3,
  MTSB_CHUNK_BAD_CODE = 4, MTSB_CHUNK_BAD_DISTANCE = 5, MTSB_CHUNK_BAD_SIZE = 6, MTSB_CHUNK_INPUT_OVERRUN = 7,
  MTSB_CHUNK_BAD_STORED = 8, MTSB_CHUNK_BAD_ADLER = 9
};

int mtsb_version(void);
/* Number of CUDA devices visible (0 if none / no driver). */
int mtsb_device_count(void);

/* Context on `device_id`.  `stream` is an existing cudaStream_t to run on (e.g. torch's current stream), or NULL to
 * let the context create its own non-blocking stream.  Returns NULL on failure (call mtsb_last_error(NULL)). */
mtsb_ctx* mtsb_create(int device_id, void* stream);
void mtsb_destroy(mtsb_ctx* ctx);
const char* mtsb_last_error(mtsb_ctx* ctx);
/* Block until everything queued by this context has finished. */
int mtsb_sync(mtsb_ctx* ctx);

/* Tunables (by name): "seg_bytes" target encoder segment size (default 262144), "lz_ctas_per_sm" (resident
 * match-finder CTAs per SM, 2), "write_index" (append the in-band index of segments and sub-blocks after each chunk's
 * zlib stream, 1; with 0 the output is exactly one zlib stream per chunk, as the reference writes it),
 * "batch_bytes" (raw bytes processed per internal sub-batch), "host_batch_bytes" (the same when a host buffer is
 * involved: copies of one sub-batch overlap the kernels of the next), "par_batch_bytes" (host-buffer sub-batch of
 * index-less chunks on the decode side), "par_inflate" (1: block-parallel decoder; 0: serial warp per stream),
 * "par_indexed" (1: indexed segments that the step kernels do not take go through the block kernels), "par_single_pass"
 * (1: the block decoder keeps the tokens of its counting pass instead of decoding every block twice), "seg_v2" (1: indexed
 * segments of the second index format are decoded by seg_tokens_kernel / seg_resolve_kernel), "par_lz_wide"
 * (-1 auto / 0 / 1: shape of the token-resolve kernel), "par_cells" (-1 auto / 0 / 1: resolve the blocks of an
 * index-less stream in parallel — the low-latency path for few streams), "inv_single_pass" (1: channel-major inverse
 * transform in one pass with look-back carries; 0: tile sums + scan + apply), "inv_order_block" (consecutive tiles of a
 * chunk that run together in the single-pass inverse, 2).  Read-only: "par_survivors", "par_candidates", "par_chained",
 * "par_resumed" (what the parallel decoders did in the last call), "sm_count".  Returns MTSB_E_ARG for unknown names. */
int mtsb_set_param(mtsb_ctx* ctx, const char* name, long long value);
long long mtsb_get_param(mtsb_ctx* ctx, const char* name);

/* Worst-case compressed size of ONE chunk of `raw_bytes` bytes with the context's current parameters
 * (stored-block bound + zlib framing + segment index). */
long long mtsb_compress_bound(mtsb_ctx* ctx, long long raw_bytes, long long ns, int nc, int itemsize, int flags);

/* K1 alone — replaces diff_along_axis(axis=0) / diff_along_axis(axis=1) / ndarray.tobytes(order) at
 * mtscomp.py:381-394 (definitions :143-159).  src: row-major (ns, nc) elements of `itemsize` bytes (1, 2, 4 or 8;
 * integer arithmetic modulo 2^(8*itemsize)); dst: the ns*nc*itemsize bytes the reference hands to zlib.compress. */
int mtsb_delta_transform(mtsb_ctx* ctx, const void* src, int src_is_device, long long ns, int nc, int itemsize,
                         int flags, void* dst, int dst_is_device);

/* K4 alone — replaces reshape(order) / cumsum_along_axis(axis=1) / cumsum_along_axis(axis=0) / ascontiguousarray at
 * mtscomp.py:622-635 (definition :162-169).  src: transformed bytes; dst: row-major (ns, nc).  If adler32_out is not
 * NULL it receives adler32(src bytes), computed on the device in the same pass structure the decoder uses. */
int mtsb_inverse_transform(mtsb_ctx* ctx, const void* src, int src_is_device, long long ns, int nc, int itemsize,
                           int flags, void* dst, int dst_is_device, uint32_t* adler32_out);

/* Batched encoder — replaces Writer.compress_batch / Writer._compress_chunk (mtscomp.py:375-423): for each chunk i,
 * rows [chunk_rows[i], chunk_rows[i+1]) of the row-major (chunk_rows[n_chunks], nc) array at `src` are transformed and
 * deflated into one zlib stream.  The streams are written back to back at `dst` exactly as they appear in a .cbin;
 * out_offsets[i] (n_chunks + 1 host int64 entries, out_offsets[0] = 0) are the reference's chunk_offsets relative to
 * this batch (mtscomp.py:453-480).  chunk_rows[0] must be 0.  dst_capacity must be >= the sum of mtsb_compress_bound()
 * over the chunks. */
int mtsb_compress_chunks(mtsb_ctx* ctx, const void* src, int src_is_device, int n_chunks, const long long* chunk_rows,
                         int nc, int itemsize, int flags, void* dst, int dst_is_device, long long dst_capacity,
                         long long* out_offsets);

/* Batched decoder — replaces Reader.decompress_chunks / Reader.read_chunk after the pread (mtscomp.py:618-650): chunk i
 * is the zlib stream comp[comp_offsets[i] : comp_offsets[i+1]] (host int64 offsets, any origin) and decodes to rows
 * [chunk_rows[i], chunk_rows[i+1]) of the row-major (chunk_rows[n_chunks], nc) array at `dst`.  Streams written by
 * mtsb_compress_chunks with write_index=1 are decoded through their index (a lane per 8 KB sub-block, all tokens of a
 * step at once); any other valid zlib stream (e.g. written by the reference) by the block-parallel decoder, which
 * finds the deflate blocks itself; what neither takes is decoded serially by one warp, which also decides what is
 * corrupt.  A chunk whose trailing bytes look like an index but do not decode with it is decoded again as a plain
 * stream (zlib ignores what follows a stream, so such a chunk is valid), whether or not chunk_status is given.
 * chunk_status (n_chunks host ints, may be NULL) receives MTSB_CHUNK_*; the call returns MTSB_E_CORRUPT if any chunk
 * is corrupt. */
int mtsb_decompress_chunks(mtsb_ctx* ctx, const void* comp, int comp_is_device, const long long* comp_offsets,
                           int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags, void* dst,
                           int dst_is_device, int* chunk_status);

/* Integrity check — replaces the per-chunk compare of check() (mtscomp.py:866-888).  Chunk i is decoded exactly as
 * mtsb_decompress_chunks decodes it and compared on the device with rows [chunk_rows[i], chunk_rows[i+1]) of the
 * row-major array `ref` (host or device, itemsize-aligned); the decoded rows are not returned.  Integers: bit equality.
 * MTSB_FLOAT: np.isclose(decoded, ref, rtol, atol) per element, evaluated as NumPy 2 evaluates it for Python-float
 * tolerances: (|x - y| <= atol + rtol * |y| && isfinite(y)) || x == y in the element's precision, with atol and rtol
 * rounded to it.  mismatches[i] / first_mismatch[i] (n_chunks host int64): elements that fail, and the element index
 * within chunk i of the first one (-1: none).  chunk_status as in mtsb_decompress_chunks (never NULL here); a chunk
 * that does not decode gets -1 in both arrays and the call returns MTSB_E_CORRUPT. */
int mtsb_verify_chunks(mtsb_ctx* ctx, const void* comp, int comp_is_device, const long long* comp_offsets,
                       int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags,
                       const void* ref, int ref_is_device, double rtol, double atol,
                       long long* mismatches, long long* first_mismatch, int* chunk_status);

/* Re-encode: chunk i is the zlib stream comp[comp_offsets[i] : comp_offsets[i+1]], as mtsb_decompress_chunks takes it.
 * It is inflated on the device to its transformed bytes, and those bytes are deflated again exactly as
 * mtsb_compress_chunks deflates a chunk with the context's current parameters (write_index, seg_bytes, ...).  There is no
 * inverse or forward transform.  The new stream inflates to the same bytes, so it has the same adler32 and decodes to
 * exactly what chunk i decodes to.  Output: packed at dst, out_offsets as in mtsb_compress_chunks; dst_capacity must be
 * >= the sum of mtsb_compress_bound.  flags: the file's, as for mtsb_decompress_chunks (the ORDER_C bit sets the
 * encoder's segments).  chunk_status as in mtsb_decompress_chunks, never NULL.  A chunk that does not decode makes the
 * call return MTSB_E_CORRUPT, and dst / out_offsets are then undefined.  If the bytes the encoder read do not have
 * the adler32 the decode accepted for a chunk, the call returns MTSB_E_CUDA with an "internal:" message naming it.
 * Sub-batches hold at most "batch_bytes" raw bytes ("host_batch_bytes" when comp or dst is host memory).  Peak device
 * scratch: about 3 bytes per raw byte of the largest sub-batch (the transformed bytes and the match finder's tokens),
 * plus the decoder's scratch, which is about 9.6 bytes per compressed byte of plain zlib streams (2 bytes per raw byte
 * more for a sub-batch of 16 streams or fewer) and about 2.3 bytes per raw byte of indexed ones; with host buffers, two
 * compressed inputs and two output bounds on top.  For AP-like int16 data (0.38 compressed bytes per raw byte) that is
 * about 7 bytes per raw byte, 14 GiB at the default batch_bytes. */
int mtsb_recompress_chunks(mtsb_ctx* ctx, const void* comp, int comp_is_device, const long long* comp_offsets,
                           int n_chunks, const long long* chunk_rows, int nc, int itemsize, int flags,
                           void* dst, int dst_is_device, long long dst_capacity, long long* out_offsets,
                           int* chunk_status);

/* Device-time (ms, CUDA events on the context's stream) of the stages of the last compress / decompress / verify /
 * recompress call:
 * out[0..7] = {h2d, transform, adler, lz77, huffman+scan, encode, d2h, total} for compress,
 *             {h2d, plan, inflate, adler, inverse, d2h, 0, total} for decompress,
 *             {h2d, plan, inflate, adler, inverse, 0, compare, total} for verify,
 *             {h2d, plan, inflate, adler, lz77, adler+huffman+scan+encode+trailer, 0, total} for recompress (its
 *             downloads overlap the next sub-batch on a copy stream and are not timed).  Returns the number filled. */
int mtsb_last_timings(mtsb_ctx* ctx, float* out, int n);
/* Number of kernels launched by the last compress / decompress / verify / recompress / transform call. */
long long mtsb_last_launches(mtsb_ctx* ctx);

/* Pinned host memory helpers (so that Python can stage file data without torch). */
void* mtsb_host_alloc(long long bytes);
void mtsb_host_free(void* p);
/* Plain device memory helpers for callers that keep data resident (bench, tests). */
void* mtsb_device_alloc(mtsb_ctx* ctx, long long bytes);
void mtsb_device_free(mtsb_ctx* ctx, void* p);
int mtsb_memcpy(mtsb_ctx* ctx, void* dst, const void* src, long long bytes, int kind /*1 H2D, 2 D2H, 3 D2D*/);

#ifdef __cplusplus
}
#endif
#endif
