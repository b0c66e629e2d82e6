// libdcae_rans.so: 64-bit rANS coder for the symbols / indexes the slice loop emits (include/dcae_rans.h).
//
// Stream format (the published ryg_rans "rans64" scheme that compressai's `ans` extension wraps; the calls it stands in
// for are /root/reference/models/dcae.py:722, 755-756, 875-876, 893):
//   state x in [2^31, 2^63), 32-bit words, probabilities in 16 bits; coding symbol (start, freq):
//     x' = (x / freq) << 16 | (x % freq) + start, after emitting the low word of x while x >= ((2^31 >> 16) << 32) * freq.
//   Symbols are coded last-to-first into a buffer that grows downwards, so the decoder reads words upwards and returns
//   symbols first-to-last.  A value outside [0, cdf_size - 2) is coded as the sentinel `cdf_size - 2` followed by a
//   bypass tail of 4-bit digits: the digit count in unary-of-15s, then the digits of 2*(v - max) or -2*v - 1, low first.
// Host code only; one stream per encoder object.  dcae_rans_ilv_*: the interleaved format ilv1 (include/dcae_rans.h), the
// same steps spread over up to 32 states; the host reference of the sm_100a kernels in rans_gpu.cu.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <new>
#include <numeric>
#include <vector>

#include "dcae_rans.h"

namespace {

constexpr int kProbBits = 16;
constexpr int kBypassBits = 4;
constexpr uint32_t kBypassMax = (1u << kBypassBits) - 1;
constexpr uint64_t kLow = 1ull << 31;

thread_local char g_err[256] = "";
int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

inline int32_t load_elem(const void* p, int32_t type, int64_t i) {
  switch (type) {
    case DCAE_RANS_I16: return static_cast<const int16_t*>(p)[i];
    case DCAE_RANS_U8: return static_cast<const uint8_t*>(p)[i];
    default: return static_cast<const int32_t*>(p)[i];
  }
}

bool tables_ok(const dcae_rans_tables* t) {
  return t && t->cdfs && t->cdf_sizes && t->offsets && t->n_cdfs > 0 && t->cdf_stride >= 3;
}

// One coding step waiting for flush(): freq == 0 marks a bypass digit held in `start`.
struct Step {
  uint16_t start;
  uint16_t freq;
};

// Appends the coding steps of one symbol (decode order: the symbol, then the bypass count and digits) to `steps`.
int push_symbol(int32_t sym, int32_t k, const dcae_rans_tables* t, std::vector<Step>& steps, const char* what, int64_t i) {
  if (k < 0 || k >= t->n_cdfs) return fail(DCAE_RANS_E_INVALID, "%s: index %d outside [0, %d) at %lld", what, k, t->n_cdfs, (long long)i);
  const int32_t size = t->cdf_sizes[k];
  if (size < 3 || size > t->cdf_stride) return fail(DCAE_RANS_E_INVALID, "%s: cdf_sizes[%d] = %d", what, k, size);
  const int32_t* cdf = t->cdfs + (int64_t)k * t->cdf_stride;
  const int32_t sentinel = size - 2;
  int64_t v = (int64_t)sym - t->offsets[k];
  uint64_t raw = 0;
  if (v < 0) {
    raw = (uint64_t)(-2 * v - 1);
    v = sentinel;
  } else if (v >= sentinel) {
    raw = (uint64_t)(2 * (v - sentinel));
    v = sentinel;
  }
  const uint32_t lo = (uint32_t)cdf[v], hi = (uint32_t)cdf[v + 1];
  if (hi <= lo || hi > (1u << kProbBits)) return fail(DCAE_RANS_E_INVALID, "%s: cdf row %d is not increasing at %lld", what, k, (long long)v);
  // freq = 65536 (a one-symbol table) does not fit 16 bits; it cannot occur with a sentinel present
  steps.push_back({(uint16_t)lo, (uint16_t)(hi - lo)});
  if (v == sentinel) {
    int digits = 0;
    while ((raw >> (digits * kBypassBits)) != 0) ++digits;
    int rest = digits;
    for (; rest >= (int)kBypassMax; rest -= (int)kBypassMax) steps.push_back({(uint16_t)kBypassMax, 0});
    steps.push_back({(uint16_t)rest, 0});
    for (int j = 0; j < digits; ++j) steps.push_back({(uint16_t)((raw >> (j * kBypassBits)) & kBypassMax), 0});
  }
  return DCAE_RANS_OK;
}

// Encoder half of one step: renormalise (emit the low word through `emit`) then code the step into x.
template <class Emit>
inline void put(uint64_t& x, Step s, Emit emit) {
  if (s.freq) {
    const uint64_t limit = ((kLow >> kProbBits) << 32) * s.freq;
    if (x >= limit) {
      emit((uint32_t)x);
      x >>= 32;
    }
    x = ((x / s.freq) << kProbBits) + (x % s.freq) + s.start;
  } else {   // bypass digit: a uniform symbol of 2^-4, i.e. freq = 2^(16 - 4) in 16-bit terms
    const uint64_t limit = ((kLow >> kProbBits) << 32) * (1u << (kProbBits - kBypassBits));
    if (x >= limit) {
      emit((uint32_t)x);
      x >>= 32;
    }
    x = (x << kBypassBits) | s.start;
  }
}

}  // namespace

struct dcae_rans_encoder {
  std::vector<Step> steps;
  std::vector<uint32_t> words;   // filled from the back
  size_t first = 0;              // index of the first valid word after flush()
};

struct dcae_rans_decoder {
  std::vector<uint32_t> words;
  size_t pos = 0;
  uint64_t x = 0;
  bool primed = false;
  uint32_t next() { return pos < words.size() ? words[pos++] : 0u; }   // reading past the end yields zeros, never UB
};

extern "C" const char* dcae_rans_last_error(void) { return g_err; }

extern "C" dcae_rans_encoder* dcae_rans_encoder_create(void) { return new (std::nothrow) dcae_rans_encoder; }
extern "C" void dcae_rans_encoder_destroy(dcae_rans_encoder* e) { delete e; }

extern "C" int dcae_rans_encoder_encode_with_indexes(dcae_rans_encoder* e, const void* symbols, int32_t symbols_type,
                                                     const void* indexes, int32_t indexes_type, int64_t n,
                                                     const dcae_rans_tables* t) {
  if (!e || n < 0 || (n > 0 && (!symbols || !indexes)) || !tables_ok(t)) return fail(DCAE_RANS_E_INVALID, "encode_with_indexes: bad arguments");
  e->steps.reserve(e->steps.size() + (size_t)n + 16);
  for (int64_t i = 0; i < n; ++i) {
    const int rc = push_symbol(load_elem(symbols, symbols_type, i), load_elem(indexes, indexes_type, i), t, e->steps, "encode_with_indexes", i);
    if (rc != DCAE_RANS_OK) return rc;
  }
  return DCAE_RANS_OK;
}

extern "C" int64_t dcae_rans_encoder_flush(dcae_rans_encoder* e) {
  if (!e) return fail(DCAE_RANS_E_INVALID, "flush: null encoder");
  // every step emits at most one word; + 2 for the final state
  e->words.assign(e->steps.size() + 2, 0u);
  size_t w = e->words.size();
  uint64_t x = kLow;
  for (size_t i = e->steps.size(); i-- > 0;) put(x, e->steps[i], [&](uint32_t v) { e->words[--w] = v; });
  e->words[--w] = (uint32_t)(x >> 32);
  e->words[--w] = (uint32_t)x;
  e->first = w;
  e->steps.clear();
  return (int64_t)((e->words.size() - w) * sizeof(uint32_t));
}

extern "C" const uint8_t* dcae_rans_encoder_bytes(const dcae_rans_encoder* e) {
  return e ? reinterpret_cast<const uint8_t*>(e->words.data() + e->first) : nullptr;
}

extern "C" dcae_rans_decoder* dcae_rans_decoder_create(void) { return new (std::nothrow) dcae_rans_decoder; }
extern "C" void dcae_rans_decoder_destroy(dcae_rans_decoder* d) { delete d; }

extern "C" int dcae_rans_decoder_set_stream(dcae_rans_decoder* d, const uint8_t* bytes, int64_t n_bytes) {
  if (!d || !bytes || n_bytes < 8 || n_bytes % 4 != 0) return fail(DCAE_RANS_E_STREAM, "set_stream: a stream is at least 8 bytes and a multiple of 4 (got %lld)", (long long)n_bytes);
  d->words.resize((size_t)n_bytes / 4);
  memcpy(d->words.data(), bytes, (size_t)n_bytes);
  d->pos = 0;
  d->x = (uint64_t)d->next();
  d->x |= (uint64_t)d->next() << 32;
  d->primed = true;
  return DCAE_RANS_OK;
}

namespace {
inline uint32_t take_bits(dcae_rans_decoder* d) {
  const uint32_t v = (uint32_t)(d->x & kBypassMax);
  d->x >>= kBypassBits;
  if (d->x < kLow) d->x = (d->x << 32) | d->next();
  return v;
}
}  // namespace

extern "C" int dcae_rans_decoder_decode_stream(dcae_rans_decoder* d, const void* indexes, int32_t indexes_type, int64_t n,
                                               const dcae_rans_tables* t, int32_t* out) {
  if (!d || n < 0 || (n > 0 && (!indexes || !out)) || !tables_ok(t)) return fail(DCAE_RANS_E_INVALID, "decode_stream: bad arguments");
  if (!d->primed) return fail(DCAE_RANS_E_STREAM, "decode_stream: set_stream was not called");
  const uint64_t mask = (1ull << kProbBits) - 1;
  for (int64_t i = 0; i < n; ++i) {
    const int32_t k = load_elem(indexes, indexes_type, i);
    if (k < 0 || k >= t->n_cdfs) return fail(DCAE_RANS_E_INVALID, "decode_stream: index %d outside [0, %d) at %lld", k, t->n_cdfs, (long long)i);
    const int32_t size = t->cdf_sizes[k];
    if (size < 3 || size > t->cdf_stride) return fail(DCAE_RANS_E_INVALID, "decode_stream: cdf_sizes[%d] = %d", k, size);
    const int32_t* cdf = t->cdfs + (int64_t)k * t->cdf_stride;
    const int32_t sentinel = size - 2;
    const uint32_t slot = (uint32_t)(d->x & mask);
    // first entry greater than the slot, minus one (rows are increasing: binary search instead of the linear scan)
    const int32_t* it = std::upper_bound(cdf, cdf + size, (int32_t)slot);
    int32_t s = (int32_t)(it - cdf) - 1;
    if (s < 0 || s > sentinel) return fail(DCAE_RANS_E_STREAM, "decode_stream: corrupt stream (slot %u outside cdf row %d)", slot, k);
    const uint32_t lo = (uint32_t)cdf[s], freq = (uint32_t)cdf[s + 1] - lo;
    d->x = (uint64_t)freq * (d->x >> kProbBits) + slot - lo;
    if (d->x < kLow) d->x = (d->x << 32) | d->next();
    int64_t v = s;
    if (s == sentinel) {
      uint32_t digit = take_bits(d);
      int64_t digits = digit;
      while (digit == kBypassMax) {
        digit = take_bits(d);
        digits += digit;
        if (digits > 64) return fail(DCAE_RANS_E_STREAM, "decode_stream: corrupt bypass length");
      }
      uint64_t raw = 0;
      for (int64_t j = 0; j < digits; ++j) raw |= (uint64_t)take_bits(d) << (j * kBypassBits);
      v = (int64_t)(raw >> 1);
      v = (raw & 1) ? -v - 1 : v + sentinel;
    }
    out[i] = (int32_t)(v + t->offsets[k]);
  }
  return DCAE_RANS_OK;
}

// ---- ilv1: interleaved lanes, one string per image (include/dcae_rans.h) -------------------------------------------
namespace {
constexpr int kIlvSlices = 5;
constexpr int kIlvHeader = 4 + 4 * kIlvSlices;
constexpr int kIlvMaxSteps = 11;   // int32 symbol and offset: |v| < 2^32, so raw < 2^33 = 9 digits, 1 count step, 1 symbol

bool ilv_lanes_ok(int32_t lanes) { return lanes >= 1 && lanes <= 32 && (lanes & (lanes - 1)) == 0; }
void put_u32(uint8_t* p, uint32_t v) { memcpy(p, &v, 4); }
uint32_t get_u32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
}  // namespace

extern "C" int64_t dcae_rans_ilv_max_bytes(int64_t n, int32_t lanes) {
  if (n < 0 || !ilv_lanes_ok(lanes)) return fail(DCAE_RANS_E_INVALID, "ilv_max_bytes: bad arguments (lanes must be 1, 2, 4, 8, 16 or 32)");
  return kIlvHeader + kIlvSlices * (8 * (int64_t)lanes + 4 * kIlvMaxSteps * n);
}

extern "C" int64_t dcae_rans_ilv_encode(const int32_t* symbols, const int32_t* indexes, int64_t n, int32_t lanes,
                                        const dcae_rans_tables* t, uint8_t* out, int64_t capacity) {
  if (n < 0 || (n > 0 && (!symbols || !indexes)) || !tables_ok(t) || !out || !ilv_lanes_ok(lanes))
    return fail(DCAE_RANS_E_INVALID, "ilv_encode: bad arguments (lanes must be 1, 2, 4, 8, 16 or 32)");
  std::vector<uint8_t> buf(kIlvHeader, 0);
  buf[0] = 1;
  buf[1] = (uint8_t)lanes;
  std::vector<Step> steps;
  std::vector<int64_t> first((size_t)n + 1);
  std::vector<uint32_t> words;
  for (int s = 0; s < kIlvSlices; ++s) {
    steps.clear();
    for (int64_t j = 0; j < n; ++j) {
      first[j] = (int64_t)steps.size();
      const int rc = push_symbol(symbols[s * n + j], indexes[s * n + j], t, steps, "ilv_encode", s * n + j);
      if (rc != DCAE_RANS_OK) return rc;
    }
    first[n] = (int64_t)steps.size();
    // the decoder's order is (step t, sub-operation k, lane) ascending: walk it backwards, collecting words reversed
    words.clear();
    uint64_t x[32];
    for (int l = 0; l < lanes; ++l) x[l] = kLow;
    for (int64_t tt = (n + lanes - 1) / lanes; tt-- > 0;) {
      int64_t kmax = 0;
      for (int l = 0; l < lanes && tt * lanes + l < n; ++l) kmax = std::max(kmax, first[tt * lanes + l + 1] - first[tt * lanes + l]);
      for (int64_t k = kmax; k-- > 0;)
        for (int l = lanes; l-- > 0;) {
          const int64_t j = tt * lanes + l;
          if (j < n && k < first[j + 1] - first[j]) put(x[l], steps[first[j] + k], [&](uint32_t v) { words.push_back(v); });
        }
    }
    const size_t at = buf.size();
    buf.resize(at + 8 * (size_t)lanes + 4 * words.size());
    memcpy(buf.data() + at, x, 8 * (size_t)lanes);
    uint8_t* w = buf.data() + at + 8 * (size_t)lanes;
    for (size_t i = words.size(); i-- > 0; w += 4) put_u32(w, words[i]);
    put_u32(buf.data() + 4 + 4 * s, (uint32_t)(buf.size() - at));
  }
  if ((int64_t)buf.size() > capacity) return fail(DCAE_RANS_E_INVALID, "ilv_encode: %lld bytes do not fit the %lld given", (long long)buf.size(), (long long)capacity);
  memcpy(out, buf.data(), buf.size());
  return (int64_t)buf.size();
}

extern "C" int dcae_rans_ilv_decode(const uint8_t* bytes, int64_t n_bytes, const int32_t* indexes, int64_t n,
                                    const dcae_rans_tables* t, int32_t* out) {
  if (!bytes || n_bytes < 0 || n < 0 || (n > 0 && (!indexes || !out)) || !tables_ok(t)) return fail(DCAE_RANS_E_INVALID, "ilv_decode: bad arguments");
  if (n_bytes < kIlvHeader) return fail(DCAE_RANS_E_STREAM, "ilv_decode: truncated header (%lld bytes)", (long long)n_bytes);
  const int lanes = bytes[1];
  uint64_t total = kIlvHeader;
  for (int s = 0; s < kIlvSlices; ++s) total += get_u32(bytes + 4 + 4 * s);
  if (bytes[0] != 1 || !ilv_lanes_ok(lanes) || bytes[2] != 0 || bytes[3] != 0 || total != (uint64_t)n_bytes)
    return fail(DCAE_RANS_E_STREAM, "ilv_decode: bad header");
  const uint64_t mask = (1ull << kProbBits) - 1;
  const uint8_t* seg = bytes + kIlvHeader;
  for (int s = 0; s < kIlvSlices; ++s) {
    const uint32_t seg_bytes = get_u32(bytes + 4 + 4 * s);
    if (seg_bytes < 8u * lanes || (seg_bytes - 8u * lanes) % 4) return fail(DCAE_RANS_E_STREAM, "ilv_decode: bad size of segment %d", s);
    uint64_t x[32];
    memcpy(x, seg, 8 * (size_t)lanes);
    const uint8_t* words = seg + 8 * lanes;
    const uint32_t n_words = (seg_bytes - 8u * lanes) / 4;
    uint32_t w = 0;
    const int32_t* idx = indexes + s * n;
    int32_t* sym = out + s * n;
    // per lane: phase 0 = symbol, 1 = bypass count, 2 = bypass digits, 3 = done
    int phase[32], count[32], got[32];
    uint64_t raw[32];
    for (int64_t tt = 0; tt * lanes < n; ++tt) {
      for (int l = 0; l < lanes; ++l) phase[l] = tt * lanes + l < n ? 0 : 3;
      for (bool any = true; any;) {            // one sub-operation per pass, lanes ascending
        any = false;
        for (int l = 0; l < lanes; ++l) {
          if (phase[l] == 3) continue;
          any = true;
          const int64_t j = tt * lanes + l;
          const int32_t k = idx[j];
          if (k < 0 || k >= t->n_cdfs) return fail(DCAE_RANS_E_INVALID, "ilv_decode: index %d outside [0, %d) at %lld", k, t->n_cdfs, (long long)(s * n + j));
          const int32_t size = t->cdf_sizes[k];
          if (size < 3 || size > t->cdf_stride) return fail(DCAE_RANS_E_INVALID, "ilv_decode: cdf_sizes[%d] = %d", k, size);
          const int32_t sentinel = size - 2;
          if (phase[l] == 0) {
            const int32_t* cdf = t->cdfs + (int64_t)k * t->cdf_stride;
            const uint32_t slot = (uint32_t)(x[l] & mask);
            const int32_t v = (int32_t)(std::upper_bound(cdf, cdf + size, (int32_t)slot) - cdf) - 1;
            if (v < 0 || v > sentinel) return fail(DCAE_RANS_E_STREAM, "ilv_decode: corrupt stream (slot %u outside cdf row %d)", slot, k);
            const uint32_t lo = (uint32_t)cdf[v], freq = (uint32_t)cdf[v + 1] - lo;
            x[l] = (uint64_t)freq * (x[l] >> kProbBits) + slot - lo;
            if (v == sentinel) {
              phase[l] = 1;
              count[l] = got[l] = 0;
              raw[l] = 0;
            } else {
              sym[j] = v + t->offsets[k];
              phase[l] = 3;
            }
          } else {
            const uint32_t d = (uint32_t)(x[l] & kBypassMax);
            x[l] >>= kBypassBits;
            if (phase[l] == 1) {
              count[l] += (int)d;
              if (count[l] > 16) return fail(DCAE_RANS_E_STREAM, "ilv_decode: corrupt bypass length");
              if (d != kBypassMax) phase[l] = 2;
            } else {
              raw[l] |= (uint64_t)d << (got[l]++ * kBypassBits);
            }
            if (phase[l] == 2 && got[l] == count[l]) {
              int64_t v = (int64_t)(raw[l] >> 1);
              v = (raw[l] & 1) ? -v - 1 : v + sentinel;
              sym[j] = (int32_t)(v + t->offsets[k]);
              phase[l] = 3;
            }
          }
          if (x[l] < kLow) {
            if (w >= n_words) return fail(DCAE_RANS_E_STREAM, "ilv_decode: segment %d is truncated", s);
            x[l] = (x[l] << 32) | get_u32(words + 4 * (size_t)w++);
          }
        }
      }
    }
    if (w != n_words) return fail(DCAE_RANS_E_STREAM, "ilv_decode: segment %d has %u words left over", s, n_words - w);
    for (int l = 0; l < lanes; ++l)
      if (x[l] != kLow) return fail(DCAE_RANS_E_STREAM, "ilv_decode: segment %d does not end in the initial state", s);
    seg += seg_bytes;
  }
  return DCAE_RANS_OK;
}

extern "C" int dcae_pmf_to_quantized_cdf(const float* pmf, int32_t n, int32_t precision, int32_t* cdf) {
  if (!pmf || !cdf || n <= 0 || precision < 1 || precision > 16) return fail(DCAE_RANS_E_INVALID, "pmf_to_quantized_cdf: bad arguments");
  if (n > (1 << precision)) return fail(DCAE_RANS_E_INVALID, "pmf_to_quantized_cdf: %d symbols do not fit %d bits", n, precision);
  const uint32_t one = 1u << precision;
  std::vector<uint32_t> c((size_t)n + 1);
  c[0] = 0;
  uint64_t total = 0;
  for (int i = 0; i < n; ++i) {
    if (!(pmf[i] >= 0.f) || !std::isfinite(pmf[i])) return fail(DCAE_RANS_E_INVALID, "pmf_to_quantized_cdf: pmf[%d] is negative or not finite", i);
    c[i + 1] = (uint32_t)std::round(pmf[i] * (float)one);
    total += c[i + 1];
  }
  if (total == 0) return fail(DCAE_RANS_E_INVALID, "pmf_to_quantized_cdf: pmf sums to zero");
  uint64_t run = 0;
  for (int i = 1; i <= n; ++i) {          // renormalise every frequency to the 2^precision total (floor), then accumulate
    run += ((uint64_t)one * c[i]) / total;
    c[i] = (uint32_t)run;
  }
  c[n] = one;
  for (int i = 0; i < n; ++i) {
    if (c[i] != c[i + 1]) continue;
    // a zero-frequency symbol: take one count from the cheapest symbol that can spare it and shift the entries between
    uint32_t best = ~0u;
    int donor = -1;
    for (int j = 0; j < n; ++j) {
      const uint32_t f = c[j + 1] - c[j];
      if (f > 1 && f < best) { best = f; donor = j; }
    }
    if (donor < 0) return fail(DCAE_RANS_E_INVALID, "pmf_to_quantized_cdf: no symbol can donate a count");
    if (donor < i) for (int j = donor + 1; j <= i; ++j) --c[j];
    else for (int j = i + 1; j <= donor; ++j) ++c[j];
  }
  for (int i = 0; i <= n; ++i) cdf[i] = (int32_t)c[i];
  return DCAE_RANS_OK;
}
