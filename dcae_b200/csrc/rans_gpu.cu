// The interleaved y-stream format ilv1 (include/dcae_rans.h) coded on the GPU: the same per-step arithmetic as the host
// coder (csrc/rans_coder.cpp: 64-bit rANS, 32-bit renormalisation, 16-bit probabilities, sentinel + 4-bit bypass), with
// the L lanes of one slice segment held by the L threads of one warp.
//   Encode: one warp per (image, slice), all of them in one launch per phase.  The decoder consumes words in the order
//   (step t, sub-operation k, lane) ascending, so the encoder walks t, k and the lanes backwards; at each (t, k) the
//   lanes that renormalise are found with __ballot_sync and each takes the slot given by the popcount of the higher
//   lanes in the ballot.  Phase 1 only counts the words, a one-thread pass turns the counts into segment sizes, image
//   offsets and headers, and phase 2 repeats phase 1 and stores every word at its final place.  No atomics: the bytes
//   are a function of the input.
//   Decode: one warp per image for one slice, inside the slice loop of decompress (indexes in, int32 symbols out).
//   Every read is checked against the image's string and segment; a malformed or corrupt string sets the image's status
//   word, fills the image's symbols with 0 and stops that image, and later slices of it are skipped.
#include "common.cuh"

namespace dcae {

constexpr int ILV_THREADS = 128;
constexpr int ILV_WARPS = ILV_THREADS / 32;
constexpr int ILV_SLICES = 5;
constexpr int ILV_HEADER = 4 + 4 * ILV_SLICES;
constexpr int ILV_MAX_STEPS = 11;     // see dcae_rans_ilv_max_bytes: 1 symbol + 1 count + 9 digits for int32 values
constexpr uint64_t kLow = 1ull << 31;
constexpr unsigned kFull = 0xffffffffu;

__host__ __device__ inline bool ilv_lanes_ok(int32_t lanes) { return lanes >= 1 && lanes <= 32 && (lanes & (lanes - 1)) == 0; }

// The coding steps of one symbol (rans_coder.cpp push_symbol): step 0 codes (start, freq); a sentinel symbol is
// followed by ncount bypass count steps and `digits` bypass digit steps of raw.
struct IlvSymbol {
  uint32_t start, freq;
  int steps, ncount, digits;
  uint64_t raw;
};

__device__ __forceinline__ int ilv_prepare(int32_t sym, int32_t k, const dcae_coder_tables& t, IlvSymbol& s) {
  if (k < 0 || k >= t.n_cdfs) return DCAE_ILV_E_INDEX;
  const int32_t size = __ldg(t.cdf_sizes + k);
  if (size < 3 || size > t.cdf_stride) return DCAE_ILV_E_TABLE;
  const int32_t sentinel = size - 2;
  int64_t v = (int64_t)sym - __ldg(t.offsets + k);
  s.raw = 0;
  if (v < 0) {
    s.raw = (uint64_t)(-2 * v - 1);
    v = sentinel;
  } else if (v >= sentinel) {
    s.raw = (uint64_t)(2 * (v - sentinel));
    v = sentinel;
  }
  const int32_t* cdf = t.cdfs + (int64_t)k * t.cdf_stride;
  const uint32_t lo = (uint32_t)__ldg(cdf + v), hi = (uint32_t)__ldg(cdf + v + 1);
  if (hi <= lo || hi > 65536u) return DCAE_ILV_E_TABLE;
  s.start = lo;
  s.freq = hi - lo;
  s.steps = 1;
  s.ncount = s.digits = 0;
  if (v == sentinel) {
    while (s.digits < 16 && (s.raw >> (4 * s.digits)) != 0) ++s.digits;
    s.ncount = s.digits / 15 + 1;
    s.steps = 1 + s.ncount + s.digits;
  }
  return DCAE_ILV_OK;
}

// Encoder half of step k of a symbol: whether it renormalises first (emitting the low word of x), then the coding step.
__device__ __forceinline__ bool ilv_needs_word(uint64_t x, const IlvSymbol& s, int k) {
  const uint64_t freq = k == 0 ? s.freq : 4096u;             // a bypass digit is a uniform symbol of 2^-4
  return x >= (freq << 47);                                   // ((kLow >> 16) << 32) * freq
}
__device__ __forceinline__ uint64_t ilv_put(uint64_t x, const IlvSymbol& s, int k) {
  if (k == 0) return ((x / s.freq) << 16) + (x % s.freq) + s.start;
  uint32_t v;
  if (k <= s.ncount) v = k < s.ncount ? 15u : (uint32_t)(s.digits - 15 * (s.ncount - 1));
  else v = (uint32_t)(s.raw >> (4 * (k - s.ncount - 1))) & 15u;
  return (x << 4) | v;
}

struct IlvScratch {
  uint32_t* words;        // [B * 5] words of each (image, slice) segment
  int32_t* seg_status;    // [B * 5]
  int64_t* image_offsets; // [B + 1]
};

inline size_t ilv_scratch_layout(int32_t B, IlvScratch* sc, void* base) {
  const size_t n = (size_t)B * ILV_SLICES;
  const size_t o_status = n * 4, o_offsets = (n * 8 + 7) / 8 * 8, total = o_offsets + ((size_t)B + 1) * 8;
  if (sc) {
    char* p = static_cast<char*>(base);
    sc->words = reinterpret_cast<uint32_t*>(p);
    sc->seg_status = reinterpret_cast<int32_t*>(p + o_status);
    sc->image_offsets = reinterpret_cast<int64_t*>(p + o_offsets);
  }
  return total;
}

template <bool WRITE>
__global__ void __launch_bounds__(ILV_THREADS) ilv_encode_kernel(const dcae_ilv_enc_args a, const IlvScratch sc) {
  const int warp = blockIdx.x * ILV_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (warp >= a.B * ILV_SLICES) return;                                  // warp-uniform
  const int b = warp / ILV_SLICES, s = warp % ILV_SLICES, L = a.lanes;
  const int64_t n = 64ll * a.h * a.w;
  const int32_t* sym = a.symbols + ((int64_t)s * a.B + b) * n;
  const int32_t* idx = a.indexes + ((int64_t)s * a.B + b) * n;
  uint32_t* seg = nullptr;                                              // phase 2: L states (u64 as 2 x u32), then words
  uint32_t top = 0;                                                     // phase 1: words so far; phase 2: words left
  if (WRITE) {
    if (sc.seg_status[warp] != DCAE_ILV_OK) return;
    int64_t off = sc.image_offsets[b] + ILV_HEADER;
    for (int q = 0; q < s; ++q) off += 8ll * L + 4ll * sc.words[b * ILV_SLICES + q];
    seg = reinterpret_cast<uint32_t*>(a.out + off);
    top = sc.words[warp];
  }
  const unsigned ge = kFull << lane;                                    // this lane and the higher ones
  uint64_t x = kLow;
  int err = DCAE_ILV_OK;
  for (int64_t t = (n + L - 1) / L - 1; t >= 0; --t) {
    const int64_t j = t * L + lane;
    IlvSymbol y;
    int steps = 0, e = DCAE_ILV_OK;
    if (lane < L && j < n) {
      e = ilv_prepare(__ldg(sym + j), __ldg(idx + j), a.tables, y);
      steps = e == DCAE_ILV_OK ? y.steps : 0;
    }
    err = __reduce_max_sync(kFull, e);
    if (err != DCAE_ILV_OK) break;
    for (int k = __reduce_max_sync(kFull, steps) - 1; k >= 0; --k) {
      const bool act = k < steps;
      const bool need = act && ilv_needs_word(x, y, k);
      const unsigned m = __ballot_sync(kFull, need);
      if (WRITE) {
        if (need) seg[2 * L + top - __popc(m & ge)] = (uint32_t)x;
        top -= __popc(m);
      } else {
        top += __popc(m);
      }
      if (act) x = ilv_put(need ? x >> 32 : x, y, k);
    }
  }
  if (!WRITE) {
    if (lane == 0) {
      sc.words[warp] = top;
      sc.seg_status[warp] = err;
    }
  } else if (lane < L) {                                               // the final states lead the segment
    seg[2 * lane] = (uint32_t)x;
    seg[2 * lane + 1] = (uint32_t)(x >> 32);
  }
}

// segment sizes, per-image status (first failing slice), image offsets and headers; one thread, B x 5 steps
__global__ void ilv_encode_scan_kernel(const dcae_ilv_enc_args a, const IlvScratch sc) {
  if (threadIdx.x != 0) return;
  int64_t off = 0;
  for (int b = 0; b < a.B; ++b) {
    uint32_t* head = reinterpret_cast<uint32_t*>(a.out + off);
    head[0] = 1u | ((uint32_t)a.lanes << 8);
    int32_t st = DCAE_ILV_OK;
    int64_t len = ILV_HEADER;
    for (int s = 0; s < ILV_SLICES; ++s) {
      const uint32_t bytes = 8u * a.lanes + 4u * sc.words[b * ILV_SLICES + s];
      a.sizes[b * ILV_SLICES + s] = bytes;
      head[1 + s] = bytes;
      len += bytes;
      if (st == DCAE_ILV_OK) st = sc.seg_status[b * ILV_SLICES + s];
    }
    a.status[b] = st;
    sc.image_offsets[b] = off;
    off += len;
  }
  sc.image_offsets[a.B] = off;
}

__global__ void __launch_bounds__(ILV_THREADS) ilv_decode_kernel(const dcae_ilv_dec_args a) {
  const int b = blockIdx.x * ILV_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= a.B) return;                                                 // warp-uniform
  const int64_t n = 64ll * a.h * a.w;
  int32_t* out = a.symbols + (int64_t)b * n;
  const int32_t* idx = a.indexes + (int64_t)b * n;
  int err = a.status[b];
  // header: every field is checked before a byte of the body is read
  const int64_t beg = a.bounds[2 * b], len = a.bounds[2 * b + 1] - beg;
  int L = 1, W = 0;
  int64_t seg = 0;
  if (err == DCAE_ILV_OK) {
    err = DCAE_ILV_E_HEADER;
    if (beg >= 0 && beg % 4 == 0 && len >= ILV_HEADER) {
      const uint32_t* head = reinterpret_cast<const uint32_t*>(a.strings + beg);
      const uint32_t h0 = head[0];
      L = (int)((h0 >> 8) & 0xff);
      uint64_t total = ILV_HEADER;
      bool ok = (h0 & 0xff) == 1u && (h0 >> 16) == 0u && ilv_lanes_ok(L);
      for (int s = 0; s < ILV_SLICES; ++s) {
        const uint32_t bytes = head[1 + s];
        ok = ok && bytes >= 8u * L && (bytes - 8u * L) % 4 == 0;
        if (s < a.slice) seg += bytes;
        if (s == a.slice) W = (int)((bytes - 8u * L) / 4);
        total += bytes;
      }
      if (ok && total == (uint64_t)len) err = DCAE_ILV_OK;
    }
  }
  if (err == DCAE_ILV_OK) {
    const uint8_t* base = a.strings + beg + ILV_HEADER + seg;
    const uint32_t* words = reinterpret_cast<const uint32_t*>(base + 8ll * L);
    uint64_t x = kLow;
    if (lane < L) x = (uint64_t)reinterpret_cast<const uint32_t*>(base)[2 * lane] | ((uint64_t)reinterpret_cast<const uint32_t*>(base)[2 * lane + 1] << 32);
    const unsigned lt = (1u << lane) - 1u;
    int pos = 0;
    for (int64_t t = 0; t * L < n && err == DCAE_ILV_OK; ++t) {
      const int64_t j = t * L + lane;
      // phase 0 = symbol, 1 = bypass count, 2 = bypass digits, 3 = done
      int phase = (lane < L && j < n) ? 0 : 3, e = DCAE_ILV_OK, count = 0, got = 0, k = 0, sentinel = 0;
      uint64_t raw = 0;
      const int32_t* cdf = nullptr;
      if (phase == 0) {
        k = __ldg(idx + j);
        int32_t size = 0;
        if (k < 0 || k >= a.tables.n_cdfs) e = DCAE_ILV_E_INDEX;
        else if ((size = __ldg(a.tables.cdf_sizes + k)) < 3 || size > a.tables.cdf_stride) e = DCAE_ILV_E_TABLE;
        sentinel = size - 2;
        cdf = a.tables.cdfs + (int64_t)k * a.tables.cdf_stride;
        if (e != DCAE_ILV_OK) phase = 3;
      }
      while (__any_sync(kFull, phase != 3)) {            // one sub-operation per pass, lanes in order of the ballot
        const bool did = phase != 3;
        if (phase == 0) {
          const int32_t slot = (int32_t)(x & 0xffffu);
          int lo = 0, hi = sentinel + 2;                   // first entry above the slot, minus one
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(cdf + mid) > slot) hi = mid; else lo = mid + 1;
          }
          const int v = lo - 1;
          const int32_t c0 = v >= 0 && v <= sentinel ? __ldg(cdf + v) : 0, c1 = v >= 0 && v <= sentinel ? __ldg(cdf + v + 1) : 0;
          if (v < 0 || v > sentinel || c1 <= c0) {
            e = DCAE_ILV_E_CORRUPT;
            phase = 3;
          } else {
            x = (uint64_t)(uint32_t)(c1 - c0) * (x >> 16) + (uint32_t)(slot - c0);
            if (v == sentinel) phase = 1;
            else {
              out[j] = v + __ldg(a.tables.offsets + k);
              phase = 3;
            }
          }
        } else if (phase != 3) {
          const int d = (int)(x & 15u);
          x >>= 4;
          if (phase == 1) {
            count += d;
            if (count > 16) {
              e = DCAE_ILV_E_CORRUPT;
              phase = 3;
            } else if (d != 15) {
              phase = 2;
            }
          } else {
            raw |= (uint64_t)d << (4 * got++);
          }
          if (phase == 2 && got == count) {
            int64_t v = (int64_t)(raw >> 1);
            v = (raw & 1) ? -v - 1 : v + sentinel;
            out[j] = (int32_t)(v + __ldg(a.tables.offsets + k));
            phase = 3;
          }
        }
        const bool need = did && e == DCAE_ILV_OK && x < kLow;
        const unsigned m = __ballot_sync(kFull, need);
        if (need) {
          const int p = pos + __popc(m & lt);
          if (p < W) x = (x << 32) | __ldg(words + p);
          else e = DCAE_ILV_E_CORRUPT;
        }
        pos += __popc(m);
        if (e != DCAE_ILV_OK) phase = 3;
      }
      err = __reduce_max_sync(kFull, e);
    }
    // a segment ends with every word consumed and every lane back in the encoder's initial state
    if (err == DCAE_ILV_OK && (pos != W || !__all_sync(kFull, x == kLow))) err = DCAE_ILV_E_CORRUPT;
  }
  if (err != DCAE_ILV_OK) {
    __syncwarp();
    for (int64_t j = lane; j < n; j += 32) out[j] = 0;
    if (lane == 0) a.status[b] = err;
  }
}

}  // namespace dcae

extern "C" size_t dcae_ilv_encode_scratch_bytes(int32_t B, int32_t h, int32_t w, int32_t lanes) {
  (void)h; (void)w; (void)lanes;
  return B < 0 ? 0 : dcae::ilv_scratch_layout(B, nullptr, nullptr);
}

extern "C" int64_t dcae_ilv_encode_max_bytes(int32_t B, int32_t h, int32_t w, int32_t lanes) {
  if (B < 0 || h < 0 || w < 0 || !dcae::ilv_lanes_ok(lanes)) return -1;
  return (int64_t)B * (dcae::ILV_HEADER + dcae::ILV_SLICES * (8ll * lanes + 4ll * dcae::ILV_MAX_STEPS * 64ll * h * w));
}

namespace {
bool tables_ok(const dcae_coder_tables& t) { return t.cdfs && t.cdf_sizes && t.offsets && t.n_cdfs > 0 && t.cdf_stride >= 3; }
}  // namespace

extern "C" int dcae_ilv_encode(const dcae_ilv_enc_args* a, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(a, "dcae_ilv_encode: null arguments");
  DCAE_REQUIRE(ilv_lanes_ok(a->lanes), "dcae_ilv_encode: lanes = %d (1, 2, 4, 8, 16 or 32)", a->lanes);
  DCAE_REQUIRE(a->B >= 0 && a->h >= 0 && a->w >= 0 && (int64_t)a->h * a->w <= (1ll << 20), "dcae_ilv_encode: bad shape");
  DCAE_REQUIRE(tables_ok(a->tables), "dcae_ilv_encode: bad coder tables");
  if (a->B == 0) return DCAE_OK;
  DCAE_REQUIRE(a->symbols && a->indexes && a->sizes && a->status && a->out && a->scratch, "dcae_ilv_encode: null pointer");
  DCAE_REQUIRE((reinterpret_cast<uintptr_t>(a->out) & 3u) == 0 && (reinterpret_cast<uintptr_t>(a->scratch) & 7u) == 0,
               "dcae_ilv_encode: out must be 4-byte and scratch 8-byte aligned");
  DCAE_REQUIRE(a->out_capacity >= dcae_ilv_encode_max_bytes(a->B, a->h, a->w, a->lanes), "dcae_ilv_encode: out_capacity below dcae_ilv_encode_max_bytes");
  IlvScratch sc;
  DCAE_REQUIRE(a->scratch_bytes >= ilv_scratch_layout(a->B, &sc, a->scratch), "dcae_ilv_encode: scratch below dcae_ilv_encode_scratch_bytes");
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const unsigned blocks = (unsigned)((a->B * ILV_SLICES + ILV_WARPS - 1) / ILV_WARPS);
  ilv_encode_kernel<false><<<blocks, ILV_THREADS, 0, (cudaStream_t)stream>>>(*a, sc);
  DCAE_LAUNCH_CHECK();
  ilv_encode_scan_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(*a, sc);
  DCAE_LAUNCH_CHECK();
  ilv_encode_kernel<true><<<blocks, ILV_THREADS, 0, (cudaStream_t)stream>>>(*a, sc);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_ilv_decode(const dcae_ilv_dec_args* a, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(a, "dcae_ilv_decode: null arguments");
  DCAE_REQUIRE(a->slice >= 0 && a->slice < ILV_SLICES, "dcae_ilv_decode: slice %d outside [0, 5)", a->slice);
  DCAE_REQUIRE(a->B >= 0 && a->h >= 0 && a->w >= 0 && (int64_t)a->h * a->w <= (1ll << 20), "dcae_ilv_decode: bad shape");
  DCAE_REQUIRE(tables_ok(a->tables), "dcae_ilv_decode: bad coder tables");
  if (a->B == 0) return DCAE_OK;
  DCAE_REQUIRE(a->strings && a->bounds && a->indexes && a->symbols && a->status, "dcae_ilv_decode: null pointer");
  DCAE_REQUIRE((reinterpret_cast<uintptr_t>(a->strings) & 3u) == 0, "dcae_ilv_decode: strings must be 4-byte aligned");
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  ilv_decode_kernel<<<(unsigned)((a->B + ILV_WARPS - 1) / ILV_WARPS), ILV_THREADS, 0, (cudaStream_t)stream>>>(*a);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
