// Shared host/device helpers for libdcae_b200.so (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/dcae_b200.h"

namespace dcae {

// thread-local error string behind dcae_last_error()
void set_error(const char* fmt, ...);
// every kernel launch goes through this counter (bench `gpu_launches`)
extern thread_local int64_t g_launches;
inline void count_launch(int n = 1) { g_launches += n; }

#define DCAE_REQUIRE(cond, ...)                     \
  do {                                              \
    if (!(cond)) {                                  \
      ::dcae::set_error(__VA_ARGS__);               \
      return DCAE_E_INVALID;                        \
    }                                               \
  } while (0)

#define DCAE_CUDA(call)                                                                    \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      ::dcae::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                        __LINE__);                                                         \
      return DCAE_E_CUDA;                                                                  \
    }                                                                                      \
  } while (0)

#define DCAE_LAUNCH_CHECK()                                                                      \
  do {                                                                                           \
    ::dcae::count_launch();                                                                      \
    cudaError_t e__ = cudaPeekAtLastError();                                                     \
    if (e__ != cudaSuccess) {                                                                    \
      ::dcae::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__,   \
                        __LINE__);                                                               \
      return DCAE_E_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

#define DCAE_TRY(call)          \
  do {                          \
    int rc__ = (call);          \
    if (rc__ != DCAE_OK) return rc__; \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// exact (erf-form) GELU as torch.nn.GELU() computes it in fp32: 0.5 x (1 + erf(x / sqrt 2))
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// The same function for the tensor-core epilogues, where SIMT issue slots are the scarce resource: branch-free,
// ~15 instructions instead of erff's two divergent paths.  With t = |x| / sqrt 2 clamped to 4.3 and
// erfc(t) = 2^(-t R(t)) (R: degree-7 minimax fit, absolute error of erfc weighted), gelu(x) = x - 0.5 x erfc(t) for
// x >= 0 and 0.5 x erfc(t) for x < 0 -- no 1 + erf cancellation on the negative side.  Max |error| against the exact
// function 2.7e-7 over [-12, 12] (torch's fp32 erf form: 1.2e-6); fit and check: tools/fit_gelu.py.
__device__ __forceinline__ float gelu_fast(float x) {
  const float t = fminf(fabsf(x) * 0.70710678118654752440f, 4.3f);
  float r = 4.535862899501808e-05f;
  r = fmaf(r, t, -0.0004455076123122126f);
  r = fmaf(r, t, 0.0014894407941028476f);
  r = fmaf(r, t, 0.0007746322662569582f);
  r = fmaf(r, t, -0.02825368382036686f);
  r = fmaf(r, t, 0.14848162233829498f);
  r = fmaf(r, t, 0.9184163808822632f);
  r = fmaf(r, t, 1.6279085874557495f);
  // -t r >= -32: outside exp2f's denormal fix-up, so the bare MUFU.EX2 gives the same bits in 1 instruction instead of 4
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-t * r));
  const float he = 0.5f * x * e;
  return x >= 0.f ? x - he : he;
}

// v -> (hi, lo) fp16 with v ~= hi + lo to 22 bits; saturating (never inf)
__device__ __forceinline__ void f16_split(float v, unsigned short& h, unsigned short& l) {
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(h) : "f"(v));
  const float hf = __half2float(__ushort_as_half(h));
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(l) : "f"(v - hf));
}
// two values at once, packed {a -> low half, b -> high half}: F2FP.PACK_AB + 2 HADD2.F32 + 2 FADD + F2FP.PACK_AB, i.e.
// 3 instructions per element and no PRMT (the scalar form is 5); same roundings as f16_split, bit for bit
__device__ __forceinline__ void f16_split2(float a, float b, uint32_t& h, uint32_t& l) {
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(b), "f"(a));
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&h));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(b - hf.y), "f"(a - hf.x));
}
// four consecutive columns of one row into both planes (two 8-byte stores); p pre-offset to the window
__device__ __forceinline__ void store_planes4(const dcae_planes& p, int64_t row, int col, float4 v) {
  uint2 hv, lv;
  f16_split2(v.x, v.y, hv.x, lv.x);
  f16_split2(v.z, v.w, hv.y, lv.y);
  *reinterpret_cast<uint2*>(static_cast<__half*>(p.hi) + row * p.ld + col) = hv;
  *reinterpret_cast<uint2*>(static_cast<__half*>(p.lo) + row * p.ld + col) = lv;
}
inline bool planes_ok(const dcae_planes* p) {
  return p == nullptr || p->hi == nullptr ||
         (p->lo != nullptr && p->ld % 4 == 0 && (reinterpret_cast<uintptr_t>(p->hi) & 7u) == 0 && (reinterpret_cast<uintptr_t>(p->lo) & 7u) == 0);
}
inline dcae_planes planes_or_null(const dcae_planes* p) {
  dcae_planes z; z.hi = nullptr; z.lo = nullptr; z.ld = 0;
  return (p && p->hi) ? *p : z;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// RAII event pair around one public op when profiling is on (dcae_profile_start/stop)
struct ProfileScope {
  ProfileScope(int family, double work, void* stream);
  ~ProfileScope();
  int slot;
  void* stream;
};

bool profiling_on();

// internal cross-file entry points
int gemm_simt(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, cudaStream_t s);
int gemm_tcgen05(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int passes, cudaStream_t s);
int gemm_tcgen05_f16x3(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int passes, cudaStream_t s);
int dict_attention_tcgen05(const float* q, int64_t q_ld, const dcae_dict_kv* kv, int64_t T, float* out, int64_t out_ld,
                           dcae_planes out16, int passes, cudaStream_t s);
int dict_attention_tcgen05_f16(const dcae_planes* q16, const dcae_dict_kv* kv, int64_t T, float* out, int64_t out_ld,
                               dcae_planes out16, cudaStream_t s);
int layernorm_any(const float* x, int64_t x_ld, const float* gamma, const float* beta, int C, int64_t T, float* out, int64_t out_ld,
                  dcae_planes o16, cudaStream_t s);
int dict_attention_simt(const float* q, int64_t q_ld, const float* Kh, const float* Vh, const float* head_scale,
                        int64_t T, float* out, int64_t out_ld, cudaStream_t s);

}  // namespace dcae
