/*
 * dcae_rans.h -- C ABI of libdcae_rans.so: the CPU range coder the DCAE entropy-model hot path feeds
 * (SURVEY.md section 8f, rows N1/N2).
 *
 * What it replaces.  The reference codes its symbols with compressai's `ans` extension (third-party, un-vendored,
 * unpinned: README.md:30): `BufferedRansEncoder.encode_with_indexes(symbols, indexes, cdf, cdf_lengths, offsets)`
 * + `flush()` at /root/reference/models/dcae.py:722, 755-756 and `RansDecoder.set_stream / decode_stream` at
 * dcae.py:875-876, 893.  Its source is not in /root/reference, so this is a restatement of the published algorithm
 * (ryg_rans 64-bit rANS, 32-bit renormalisation, 16-bit probability precision, symbols coded in reverse so that
 * the decoder reads forward; out-of-range symbols leave through a 4-bit bypass code behind the sentinel symbol
 * `cdf_length - 2`), pinned by round trips and by the coder contract; byte compatibility with compressai streams is
 * the intent and cannot be verified offline.
 *
 * Differences from the Python-list interface: symbols / indexes are plain arrays (int32, or the packed int16 / uint8
 * that dcae_pack_symbols produces on the device, so the D2H buffer is coded without any conversion), the CDF table is
 * one row-major int32 matrix [n_cdfs, cdf_stride] (`GaussianConditional._quantized_cdf`, dcae.py:718).
 *
 * All pointers are HOST pointers.  Return 0 on success, negative on error (dcae_rans_last_error()).
 */
#ifndef DCAE_RANS_H_
#define DCAE_RANS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { DCAE_RANS_OK = 0, DCAE_RANS_E_INVALID = -1, DCAE_RANS_E_STREAM = -2 };

/* element types of the symbol / index arrays */
enum { DCAE_RANS_I32 = 0, DCAE_RANS_I16 = 1, DCAE_RANS_U8 = 2 };

const char* dcae_rans_last_error(void);

/* CDF tables shared by encoder and decoder calls: cdfs [n_cdfs, cdf_stride] int32 row-major, cdf_sizes [n_cdfs]
 * (entries used per row, `_cdf_length`), offsets [n_cdfs] (`_offset`).  dcae.py:718-720. */
typedef struct {
  const int32_t* cdfs; int32_t cdf_stride;
  const int32_t* cdf_sizes;
  const int32_t* offsets;
  int32_t n_cdfs;
} dcae_rans_tables;

/* ---- compressai.ans.BufferedRansEncoder ------------------------------------------------------------------- */
typedef struct dcae_rans_encoder dcae_rans_encoder;
dcae_rans_encoder* dcae_rans_encoder_create(void);
void dcae_rans_encoder_destroy(dcae_rans_encoder* e);
/* encode_with_indexes (dcae.py:755): appends n symbols to the buffer; may be called repeatedly before flush. */
int dcae_rans_encoder_encode_with_indexes(dcae_rans_encoder* e, const void* symbols, int32_t symbols_type,
                                          const void* indexes, int32_t indexes_type, int64_t n,
                                          const dcae_rans_tables* t);
/* flush (dcae.py:756): codes the buffered symbols in reverse and returns the stream size in bytes; the bytes stay
 * owned by the encoder until the next encode / flush / destroy and are read with dcae_rans_encoder_bytes(). */
int64_t dcae_rans_encoder_flush(dcae_rans_encoder* e);
const uint8_t* dcae_rans_encoder_bytes(const dcae_rans_encoder* e);

/* ---- compressai.ans.RansDecoder ---------------------------------------------------------------------------- */
typedef struct dcae_rans_decoder dcae_rans_decoder;
dcae_rans_decoder* dcae_rans_decoder_create(void);
void dcae_rans_decoder_destroy(dcae_rans_decoder* d);
/* set_stream (dcae.py:876): copies the stream. */
int dcae_rans_decoder_set_stream(dcae_rans_decoder* d, const uint8_t* bytes, int64_t n_bytes);
/* decode_stream (dcae.py:893): decodes the next n symbols; out: int32 [n]. */
int dcae_rans_decoder_decode_stream(dcae_rans_decoder* d, const void* indexes, int32_t indexes_type, int64_t n,
                                    const dcae_rans_tables* t, int32_t* out);

/* ---- ilv1: the interleaved y-stream format, one string per image (opt-in; the reference format above is the default) --
 * The same steps as the coder above (same tables, sentinel and 4-bit bypass, same per-step arithmetic); only the
 * assignment of symbols to states and the order of the words differ, so that up to 32 lanes decode in parallel.
 *   string  = u8 version (1), u8 L (lanes: 1, 2, 4, 8, 16 or 32), u16 0, u32 bytes of segment s (s = 0..4), segments
 *   segment = L final states (u64, lane order), then one shared stream of u32 words      (all fields little-endian)
 * Symbol j of a slice (the [64, h, w] slice of one image flattened) is coded by lane j % L at step j / L.  The words
 * are in the order the decoder consumes them: step ascending, then sub-operation ascending (0 = the symbol, then the
 * bypass count and digit steps), then lane ascending; only lanes whose step renormalises take a word.  With L = 1 a
 * segment is byte-identical to what dcae_rans_encoder_flush writes for the slice.  Cost: 4 + 5 (4 + 8 L) bytes per
 * image (the reference format: 8).  csrc/rans_gpu.cu (libdcae_b200.so) codes the same bytes on the GPU.
 *
 * symbols / indexes / out: int32 [5, n] (slice-major, n symbols per slice).  _encode writes the string into out and
 * returns its length (<= dcae_rans_ilv_max_bytes(n, lanes)), or a negative code if it does not fit `capacity`.
 * _decode: DCAE_RANS_E_STREAM for a malformed, truncated or corrupt string (a segment must also end with every word
 * consumed and every lane back in its initial state), DCAE_RANS_E_INVALID for bad arguments or indexes. */
int64_t dcae_rans_ilv_max_bytes(int64_t n, int32_t lanes);
int64_t dcae_rans_ilv_encode(const int32_t* symbols, const int32_t* indexes, int64_t n, int32_t lanes,
                             const dcae_rans_tables* t, uint8_t* out, int64_t capacity);
int dcae_rans_ilv_decode(const uint8_t* bytes, int64_t n_bytes, const int32_t* indexes, int64_t n,
                         const dcae_rans_tables* t, int32_t* out);

/* ---- compressai._CXX.pmf_to_quantized_cdf (used by GaussianConditional.update(), dcae.py:616-621) --------- */
/* pmf [n] (non-negative, finite) -> cdf [n + 1] with cdf[0] = 0, cdf[n] = 2^precision, strictly increasing. */
int dcae_pmf_to_quantized_cdf(const float* pmf, int32_t n, int32_t precision, int32_t* cdf);

#ifdef __cplusplus
}
#endif
#endif /* DCAE_RANS_H_ */
