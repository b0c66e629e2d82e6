// Token-major fp32 helper kernels of the dictionary cross-attention module
// (/root/reference/models/dcae.py:300-336, 386-448, 479-509): LayerNorm, GELU, depthwise 3x3,
// spatial-attention gate, NCHW <-> token-major transposes.  All HBM-bound: float4 accesses,
// channel-contiguous thread mapping, no atomics.
#include "common.cuh"

namespace dcae {

// ---------------------------------------------------------------------------------------------
// LayerNorm: one warp per token, C % 128 == 0, C <= 1024.  Two-pass (mean, then centred variance).
// ---------------------------------------------------------------------------------------------
template <int V>  // V = C / 128 float4 per lane
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int64_t x_ld,
                                                        const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, int64_t T,
                                                        float* __restrict__ out, int64_t out_ld, const dcae_planes o16) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  constexpr int C = V * 128;
  const float4* xr = reinterpret_cast<const float4*>(x + t * x_ld);
  float4 v[V];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    v[k] = __ldg(xr + lane + 32 * k);
    s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  }
  const float mean = warp_sum(s) * (1.0f / C);
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    float a = v[k].x - mean, b = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / C) + 1e-5f);
  float4* orow = reinterpret_cast<float4*>(out + t * out_ld);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float4 g = __ldg(g4 + lane + 32 * k), b = __ldg(b4 + lane + 32 * k);
    float4 o;
    o.x = (v[k].x - mean) * rstd * g.x + b.x;
    o.y = (v[k].y - mean) * rstd * g.y + b.y;
    o.z = (v[k].z - mean) * rstd * g.z + b.z;
    o.w = (v[k].w - mean) * rstd * g.w + b.w;
    if (out) orow[lane + 32 * k] = o;
    if (o16.hi) store_planes4(o16, t, (lane + 32 * k) * 4, o);
  }
}

__global__ void __launch_bounds__(256) gelu_kernel(const float* __restrict__ x, int64_t x_ld, int C4, int64_t n4,
                                                   float* __restrict__ out, int64_t out_ld, const dcae_planes o16) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / C4;
    const int c = (int)(i - t * C4) * 4;
    float4 v = __ldg(reinterpret_cast<const float4*>(x + t * x_ld + c));
    v.x = gelu_erf(v.x); v.y = gelu_erf(v.y); v.z = gelu_erf(v.z); v.w = gelu_erf(v.w);
    if (out) *reinterpret_cast<float4*>(out + t * out_ld + c) = v;
    if (o16.hi) store_planes4(o16, t, c, v);
  }
}

// ---------------------------------------------------------------------------------------------
// Depthwise 3x3 (stride 1, zero pad 1) on the token grid; weights tap-major [9, C].
// out = act(dw(x) + bias) * gate
// Each thread owns 4 channels of DX horizontally adjacent tokens: a 3 x (DX + 2) input patch is read
// once (4.5 float4 loads per output at DX = 4 instead of 9), consecutive threads take consecutive channel
// groups so every load/store is a coalesced 16-byte access.  DX = 4 (72 registers) measured 8 % / 23 % faster than
// DX = 8 (104 registers, 25 % occupancy) on the 640- / 1280-channel GLU launch, DX = 2 slower again.
// ---------------------------------------------------------------------------------------------
constexpr int DW_ROWS = 4;      // token rows per block
constexpr int DX = 4;           // tokens per thread

// grid = (ceil(C4 / 32), ceil(h / DW_ROWS), B * ceil(w / DX)); block = 32 channel groups x DW_ROWS token rows, so the
// three input rows a thread needs are shared with its neighbours in the block through L1.
// ACT: 0 none, 1 GELU (erff form, the fp32 path), 2 GELU through gelu_fast (planes-only output, i.e. the tensor-core
// modes: measured issue-bound on erff, 67% issue utilisation at 25% occupancy, before the switch).
// All element offsets are 32-bit (the host checks that every tensor spans < 2^32 elements): one IMAD per access and one
// IMAD.WIDE onto the 64-bit base, instead of the 64-bit multiply chains that made integer work 45 % of the kernel
// (round 1: 69 instructions per output element, 16 of them FFMA).
template <int ACT>
__global__ void __launch_bounds__(32 * DW_ROWS) dwconv3x3_kernel(const float* __restrict__ x, uint32_t x_ld,
                                                        const float* __restrict__ wt, const float* __restrict__ bias,
                                                        int C4, int B, int h, int w,
                                                        const float* __restrict__ gate, uint32_t gate_ld,
                                                        float* __restrict__ out, uint32_t out_ld, const dcae_planes o16) {
  const int xg = (w + DX - 1) / DX;
  const uint32_t C = (uint32_t)C4 * 4;
  const int c4 = blockIdx.x * 32 + (threadIdx.x & 31);
  const int yy = blockIdx.y * DW_ROWS + (threadIdx.x >> 5);
  const int b = blockIdx.z / xg;
  const int x0 = (blockIdx.z - b * xg) * DX;
  if (c4 >= C4 || yy >= h) return;
  const uint32_t c = (uint32_t)c4 * 4;
  const float* xb = x + c;
  float4 k[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) k[t] = __ldg(reinterpret_cast<const float4*>(wt + (uint32_t)t * C + c));
  const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + c));
  float4 acc[DX];
#pragma unroll
  for (int j = 0; j < DX; ++j) acc[j] = bv;
  const uint32_t img = (uint32_t)b * (uint32_t)h;
  const bool interior = x0 >= 1 && x0 + DX + 1 <= w;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int y2 = yy + dy;
    if ((unsigned)y2 >= (unsigned)h) continue;
    const uint32_t row = (img + (uint32_t)y2) * (uint32_t)w;          // token index of (b, y2, 0)
    float4 p[DX + 2];
    if (interior) {        // block-uniform: the whole DX + 2 window lies inside the row (10 of 12 column groups at w = 48)
      const float* pr = xb + (row + (uint32_t)(x0 - 1)) * x_ld;
#pragma unroll
      for (int j = 0; j < DX + 2; ++j) p[j] = __ldg(reinterpret_cast<const float4*>(pr + (uint32_t)j * x_ld));
    } else {
#pragma unroll
      for (int j = 0; j < DX + 2; ++j) {
        const int x2 = x0 - 1 + j;
        p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if ((unsigned)x2 < (unsigned)w) p[j] = __ldg(reinterpret_cast<const float4*>(xb + (row + (uint32_t)x2) * x_ld));
      }
    }
#pragma unroll
    for (int j = 0; j < DX; ++j) {
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const float4 kk = k[(dy + 1) * 3 + dx];
        const float4 v = p[j + dx];
        acc[j].x = fmaf(v.x, kk.x, acc[j].x); acc[j].y = fmaf(v.y, kk.y, acc[j].y);
        acc[j].z = fmaf(v.z, kk.z, acc[j].z); acc[j].w = fmaf(v.w, kk.w, acc[j].w);
      }
    }
  }
  const uint32_t t0 = (img + (uint32_t)yy) * (uint32_t)w + (uint32_t)x0;
  const uint32_t p_ld = (uint32_t)o16.ld;
  __half* const hi = static_cast<__half*>(o16.hi);
  __half* const lo = static_cast<__half*>(o16.lo);
#pragma unroll
  for (int j = 0; j < DX; ++j) {
    if (x0 + j >= w) break;
    const uint32_t t = t0 + (uint32_t)j;
    float4 a = acc[j];
    if (ACT == 1) { a.x = gelu_erf(a.x); a.y = gelu_erf(a.y); a.z = gelu_erf(a.z); a.w = gelu_erf(a.w); }
    if (ACT == 2) { a.x = gelu_fast(a.x); a.y = gelu_fast(a.y); a.z = gelu_fast(a.z); a.w = gelu_fast(a.w); }
    if (gate != nullptr) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gate + (t * gate_ld + c)));
      a.x *= g.x; a.y *= g.y; a.z *= g.z; a.w *= g.w;
    }
    if (out) *reinterpret_cast<float4*>(out + (t * out_ld + c)) = a;
    if (hi) {
      uint2 hv, lv;
      f16_split2(a.x, a.y, hv.x, lv.x);
      f16_split2(a.z, a.w, hv.y, lv.y);
      const uint32_t o = t * p_ld + c;
      *reinterpret_cast<uint2*>(hi + o) = hv;
      *reinterpret_cast<uint2*>(lo + o) = lv;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Spatial attention gate.  Pass 1: per-token channel mean and max.  Pass 2: 7x7 conv over the
// 2-channel stats map, sigmoid, out = s_out * gate + res_scale * x0.
// ---------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(256) channel_stats_kernel(const float* __restrict__ x, int64_t x_ld, int64_t T,
                                                            float* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const float4* xr = reinterpret_cast<const float4*>(x + t * x_ld);
  float s = 0.f, m = -INFINITY;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float4 v = __ldg(xr + lane + 32 * k);
    s += (v.x + v.y) + (v.z + v.w);
    m = fmaxf(fmaxf(m, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
  }
  s = warp_sum(s);
  m = warp_max(m);
  if (lane == 0) {
    stats[2 * t] = s * (1.0f / (V * 128));
    stats[2 * t + 1] = m;
  }
}

template <int V>
__global__ void __launch_bounds__(256) spatial_gate_kernel(const float* __restrict__ s_out, int64_t s_ld,
                                                           const float* __restrict__ x0, int64_t x0_ld,
                                                           const float* __restrict__ res_scale,
                                                           const float* __restrict__ w7,
                                                           const float* __restrict__ stats, int B, int h, int w,
                                                           float* __restrict__ out, int64_t out_ld,
                                                           const float* __restrict__ ln_gamma, const float* __restrict__ ln_beta,
                                                           const dcae_planes ln16) {
  const int lane = threadIdx.x & 31;
  const int64_t T = (int64_t)B * h * w;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const int xx = (int)(t % w);
  const int yy = (int)((t / w) % h);
  float acc = 0.f;
  for (int k = lane; k < 98; k += 32) {
    const int ch = k / 49, r = k - ch * 49;
    const int dy = r / 7 - 3, dx = r % 7 - 3;
    if ((unsigned)(yy + dy) < (unsigned)h && (unsigned)(xx + dx) < (unsigned)w)
      acc = fmaf(__ldg(w7 + k), __ldg(stats + 2 * (t + dy * w + dx) + ch), acc);
  }
  acc = warp_sum(acc);
  const float gate = 1.0f / (1.0f + expf(-acc));
  const float4* sr = reinterpret_cast<const float4*>(s_out + t * s_ld);
  const float4* xr = reinterpret_cast<const float4*>(x0 + t * x0_ld);
  const float4* rs = reinterpret_cast<const float4*>(res_scale);
  float4* orow = reinterpret_cast<float4*>(out + t * out_ld);
  float4 v[V];
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float4 a = __ldg(sr + lane + 32 * k), b = __ldg(xr + lane + 32 * k), r = __ldg(rs + lane + 32 * k);
    float4 o;
    o.x = a.x * gate + b.x * r.x; o.y = a.y * gate + b.y * r.y;
    o.z = a.z * gate + b.z * r.z; o.w = a.w * gate + b.w * r.w;
    orow[lane + 32 * k] = o;
    v[k] = o;
  }
  if (ln16.hi == nullptr) return;
  // fused LayerNorm of the row just produced (lnx of dcae.py:487): the warp holds all C values, so the separate
  // layernorm launch and its re-read of the row go away.  Same two-pass arithmetic as layernorm_kernel: same bits.
  constexpr int C = V * 128;
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < V; ++k) s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  const float mean = warp_sum(s) * (1.0f / C);
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    float a = v[k].x - mean, b = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / C) + 1e-5f);
  const float4* g4 = reinterpret_cast<const float4*>(ln_gamma);
  const float4* b4 = reinterpret_cast<const float4*>(ln_beta);
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float4 g = __ldg(g4 + lane + 32 * k), b = __ldg(b4 + lane + 32 * k);
    float4 o;
    o.x = (v[k].x - mean) * rstd * g.x + b.x;
    o.y = (v[k].y - mean) * rstd * g.y + b.y;
    o.z = (v[k].z - mean) * rstd * g.z + b.z;
    o.w = (v[k].w - mean) * rstd * g.w + b.w;
    store_planes4(ln16, t, (lane + 32 * k) * 4, o);
  }
}

// ---------------------------------------------------------------------------------------------
// [B, C, HW] <-> [B*HW, ld] transposes through a 32x33 shared tile.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) nchw_to_tokens_kernel(const T* __restrict__ src, int C, int64_t HW,
                                                             T* __restrict__ dst, int64_t dst_ld) {
  __shared__ T tile[32][33];
  const int b = blockIdx.z;
  const int64_t p0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r;
    const int64_t p = p0 + tx;
    tile[r][tx] = (c < C && p < HW) ? src[((int64_t)b * C + c) * HW + p] : T(0);
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int64_t p = p0 + r;
    const int c = c0 + tx;
    if (c < C && p < HW) dst[((int64_t)b * HW + p) * dst_ld + c] = tile[tx][r];
  }
}

// fp32 NCHW -> token-major fp16 hi/lo planes (and optionally fp32), same 32x33 tile transpose
__global__ void __launch_bounds__(256) nchw_to_token_planes_kernel(const float* __restrict__ src, int C, int64_t HW,
                                                                   float* __restrict__ dst, int64_t dst_ld, const dcae_planes o16) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int64_t p0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r;
    const int64_t p = p0 + tx;
    tile[r][tx] = (c < C && p < HW) ? src[((int64_t)b * C + c) * HW + p] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int64_t p = p0 + r;
    const int c = c0 + tx;
    if (c < C && p < HW) {
      const float v = tile[tx][r];
      const int64_t t = (int64_t)b * HW + p;
      if (dst) dst[t * dst_ld + c] = v;
      unsigned short h, l;
      f16_split(v, h, l);
      static_cast<__half*>(o16.hi)[t * o16.ld + c] = __ushort_as_half(h);
      static_cast<__half*>(o16.lo)[t * o16.ld + c] = __ushort_as_half(l);
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256) tokens_to_nchw_kernel(const T* __restrict__ src, int64_t src_ld, int C,
                                                             int64_t HW, T* __restrict__ dst) {
  __shared__ T tile[32][33];
  const int b = blockIdx.z;
  const int64_t p0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int64_t p = p0 + r;
    const int c = c0 + tx;
    tile[r][tx] = (c < C && p < HW) ? src[((int64_t)b * HW + p) * src_ld + c] : T(0);
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r;
    const int64_t p = p0 + tx;
    if (c < C && p < HW) dst[((int64_t)b * C + c) * HW + p] = tile[tx][r];
  }
}

__global__ void split_tf32_kernel(const float* __restrict__ w, float* __restrict__ hi, float* __restrict__ lo, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = w[i];
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
    const float hf = __uint_as_float(h);
    uint32_t l;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - hf));
    hi[i] = hf;
    lo[i] = __uint_as_float(l);
  }
}

static inline unsigned grid_for(int64_t n, int threads) {
  int64_t b = (n + threads - 1) / threads;
  const int64_t cap = (int64_t)num_sms() * 16;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace dcae

using namespace dcae;

extern "C" int dcae_op_layernorm(const float* x, int64_t x_ld, const float* gamma, const float* beta, int32_t C,
                                 int64_t T, float* out, int64_t out_ld, const dcae_planes* out16, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const dcae_planes o16 = planes_or_null(out16);
  DCAE_REQUIRE(x && gamma && beta && (out || o16.hi) && planes_ok(out16), "dcae_op_layernorm: null pointer / bad planes");
  DCAE_REQUIRE(aligned16(x) && aligned16(out) && aligned16(gamma) && aligned16(beta) && x_ld % 4 == 0 && out_ld % 4 == 0,
               "dcae_op_layernorm: 16-byte alignment required");
  if (T == 0) return DCAE_OK;
  // the dictionary module's widths (multiples of 128) keep their fully unrolled kernel; the transform stacks'
  // 96 / 144 / 192 channels (dcae.py:349,352) take the guarded one in transform_kernels.cu
  if (C % 128 != 0 || C < 128 || C > 1024) return layernorm_any(x, x_ld, gamma, beta, C, T, out, out_ld, o16, (cudaStream_t)stream);
  const unsigned blocks = (unsigned)((T + 7) / 8);
  cudaStream_t s = (cudaStream_t)stream;
  switch (C / 128) {
#define LN_CASE(V) case V: layernorm_kernel<V><<<blocks, 256, 0, s>>>(x, x_ld, gamma, beta, T, out, out_ld, o16); break;
    LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(5) LN_CASE(6) LN_CASE(7) LN_CASE(8)
#undef LN_CASE
  }
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_op_gelu(const float* x, int64_t x_ld, int32_t C, int64_t T, float* out, int64_t out_ld,
                            const dcae_planes* out16, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const dcae_planes o16 = planes_or_null(out16);
  DCAE_REQUIRE(x && (out || o16.hi) && planes_ok(out16) && C % 4 == 0 && x_ld % 4 == 0 && out_ld % 4 == 0 && aligned16(x) && aligned16(out), "dcae_op_gelu: bad arguments");
  if (T == 0) return DCAE_OK;
  const int64_t n4 = T * (C / 4);
  gelu_kernel<<<grid_for(n4, 256), 256, 0, (cudaStream_t)stream>>>(x, x_ld, C / 4, n4, out, out_ld, o16);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_op_dwconv3x3(const float* x, int64_t x_ld, const float* wt, const float* bias, int32_t C, int32_t B,
                                 int32_t h, int32_t w, int32_t act, const float* gate, int64_t gate_ld, float* out,
                                 int64_t out_ld, const dcae_planes* out16, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const dcae_planes o16 = planes_or_null(out16);
  DCAE_REQUIRE(x && wt && bias && (out || o16.hi) && planes_ok(out16), "dcae_op_dwconv3x3: null pointer / bad planes");
  DCAE_REQUIRE(C % 4 == 0 && x_ld % 4 == 0 && out_ld % 4 == 0 && (gate == nullptr || gate_ld % 4 == 0), "dcae_op_dwconv3x3: C and lds must be multiples of 4");
  DCAE_REQUIRE(aligned16(x) && aligned16(wt) && aligned16(bias) && aligned16(out) && aligned16(gate), "dcae_op_dwconv3x3: 16-byte alignment required");
  DCAE_REQUIRE(act == DCAE_ACT_NONE || act == DCAE_ACT_GELU, "dcae_op_dwconv3x3: act must be NONE or GELU");
  if ((int64_t)B * h * w == 0) return DCAE_OK;
  {
    const int64_t T = (int64_t)B * h * w, lim = 1ll << 32;
    DCAE_REQUIRE(T * x_ld < lim && T * out_ld < lim && T * gate_ld < lim && T * o16.ld < lim && x_ld < lim && out_ld < lim && gate_ld < lim,
                 "dcae_op_dwconv3x3: tensors of 2^32 elements or more are not supported (32-bit offsets)");
  }
  const int xg = (w + DX - 1) / DX;
  DCAE_REQUIRE((int64_t)B * xg <= 65535 && (h + DW_ROWS - 1) / DW_ROWS <= 65535, "dcae_op_dwconv3x3: token grid too large");
  dim3 grid((unsigned)((C / 4 + 31) / 32), (unsigned)((h + DW_ROWS - 1) / DW_ROWS), (unsigned)(B * xg));
  const int variant = act == DCAE_ACT_NONE ? 0 : (out == nullptr ? 2 : 1);
#define DW_LAUNCH(A) dwconv3x3_kernel<A><<<grid, 32 * DW_ROWS, 0, (cudaStream_t)stream>>>(x, (uint32_t)x_ld, wt, bias, C / 4, B, h, w, gate, (uint32_t)gate_ld, out, (uint32_t)out_ld, o16)
  if (variant == 0) DW_LAUNCH(0); else if (variant == 1) DW_LAUNCH(1); else DW_LAUNCH(2);
#undef DW_LAUNCH
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_op_spatial_gate(const float* s_out, int64_t s_ld, const float* x0, int64_t x0_ld,
                                    const float* res_scale, const float* w7, int32_t C, int32_t B, int32_t h, int32_t w,
                                    float* stats, float* out, int64_t out_ld, void* stream) {
  return dcae_op_spatial_gate_ln(s_out, s_ld, x0, x0_ld, res_scale, w7, C, B, h, w, stats, out, out_ld, nullptr, nullptr, nullptr, stream);
}

extern "C" int dcae_op_spatial_gate_ln(const float* s_out, int64_t s_ld, const float* x0, int64_t x0_ld,
                                       const float* res_scale, const float* w7, int32_t C, int32_t B, int32_t h, int32_t w,
                                       float* stats, float* out, int64_t out_ld, const float* ln_gamma, const float* ln_beta,
                                       const dcae_planes* ln_out16, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const dcae_planes ln16 = planes_or_null(ln_out16);
  DCAE_REQUIRE(s_out && x0 && res_scale && w7 && stats && out, "dcae_op_spatial_gate: null pointer");
  DCAE_REQUIRE(!ln16.hi || (ln_gamma && ln_beta && planes_ok(ln_out16) && aligned16(ln_gamma) && aligned16(ln_beta)), "dcae_op_spatial_gate_ln: LayerNorm output planes need gamma / beta (16-byte aligned)");
  DCAE_REQUIRE(C % 128 == 0 && C >= 128 && C <= 1024, "dcae_op_spatial_gate: C=%d must be a multiple of 128 in [128,1024]", C);
  DCAE_REQUIRE(aligned16(s_out) && aligned16(x0) && aligned16(res_scale) && aligned16(out) && s_ld % 4 == 0 && x0_ld % 4 == 0 && out_ld % 4 == 0,
               "dcae_op_spatial_gate: 16-byte alignment required");
  const int64_t T = (int64_t)B * h * w;
  if (T == 0) return DCAE_OK;
  const unsigned blocks = (unsigned)((T + 7) / 8);
  cudaStream_t s = (cudaStream_t)stream;
  switch (C / 128) {
#define SG_CASE(V)                                                                                               \
  case V:                                                                                                        \
    channel_stats_kernel<V><<<blocks, 256, 0, s>>>(s_out, s_ld, T, stats);                                       \
    count_launch();                                                                                              \
    spatial_gate_kernel<V><<<blocks, 256, 0, s>>>(s_out, s_ld, x0, x0_ld, res_scale, w7, stats, B, h, w, out, out_ld, ln_gamma, ln_beta, ln16); \
    break;
    SG_CASE(1) SG_CASE(2) SG_CASE(3) SG_CASE(4) SG_CASE(5) SG_CASE(6) SG_CASE(7) SG_CASE(8)
#undef SG_CASE
  }
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

template <typename T>
static int transpose_in(const T* src, int32_t B, int32_t C, int64_t HW, T* dst, int64_t dst_ld, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  DCAE_REQUIRE(src && dst && B >= 0 && C >= 0 && HW >= 0 && dst_ld >= C, "nchw_to_tokens: bad arguments");
  if (B == 0 || C == 0 || HW == 0) return DCAE_OK;
  DCAE_REQUIRE(B <= 65535 && (C + 31) / 32 <= 65535, "nchw_to_tokens: B or C too large");
  dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  nchw_to_tokens_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(src, C, HW, dst, dst_ld);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
template <typename T>
static int transpose_out(const T* src, int64_t src_ld, int32_t B, int32_t C, int64_t HW, T* dst, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  DCAE_REQUIRE(src && dst && B >= 0 && C >= 0 && HW >= 0 && src_ld >= C, "tokens_to_nchw: bad arguments");
  if (B == 0 || C == 0 || HW == 0) return DCAE_OK;
  DCAE_REQUIRE(B <= 65535 && (C + 31) / 32 <= 65535, "tokens_to_nchw: B or C too large");
  dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  tokens_to_nchw_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(src, src_ld, C, HW, dst);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_op_nchw_to_tokens(const float* src, int32_t B, int32_t C, int64_t HW, float* dst, int64_t dst_ld,
                                      const dcae_planes* dst16, void* stream) {
  if (dst16 == nullptr || dst16->hi == nullptr) return transpose_in<float>(src, B, C, HW, dst, dst_ld, stream);
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  DCAE_REQUIRE(src && planes_ok(dst16) && B >= 0 && C >= 0 && HW >= 0, "nchw_to_tokens(planes): bad arguments");
  if (B == 0 || C == 0 || HW == 0) return DCAE_OK;
  dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  nchw_to_token_planes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, C, HW, dst, dst_ld, *dst16);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
extern "C" int dcae_op_tokens_to_nchw(const float* src, int64_t src_ld, int32_t B, int32_t C, int64_t HW, float* dst, void* stream) {
  return transpose_out<float>(src, src_ld, B, C, HW, dst, stream);
}
extern "C" int dcae_op_tokens_to_nchw_i32(const int32_t* src, int64_t src_ld, int32_t B, int32_t C, int64_t HW, int32_t* dst, void* stream) {
  return transpose_out<int32_t>(src, src_ld, B, C, HW, dst, stream);
}
extern "C" int dcae_op_nchw_to_tokens_i32(const int32_t* src, int32_t B, int32_t C, int64_t HW, int32_t* dst, int64_t dst_ld, void* stream) {
  return transpose_in<int32_t>(src, B, C, HW, dst, dst_ld, stream);
}

// ---- coder hand-off (SURVEY 8f N1): int32 symbols / indexes -> int16 / uint8, 16 bytes in, 6 bytes out per 4 elements ----
// Symbols outside int16 saturate and are counted (the coder's bypass path needs the int32 value: the caller falls back
// to the int32 tensor when the count is not zero); indexes are < 256 by construction (table size <= 256).
__global__ void __launch_bounds__(256) pack_symbols_kernel(const int4* __restrict__ sym, const int4* __restrict__ idx, int64_t n4,
                                                           short4* __restrict__ sym16, uchar4* __restrict__ idx8,
                                                           unsigned long long* __restrict__ overflow) {
  unsigned int bad = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int4 v = __ldg(sym + i), j = __ldg(idx + i);
    bad += (v.x < -32768 || v.x > 32767) + (v.y < -32768 || v.y > 32767) + (v.z < -32768 || v.z > 32767) + (v.w < -32768 || v.w > 32767);
    sym16[i] = make_short4((short)max(-32768, min(32767, v.x)), (short)max(-32768, min(32767, v.y)),
                           (short)max(-32768, min(32767, v.z)), (short)max(-32768, min(32767, v.w)));
    idx8[i] = make_uchar4((unsigned char)j.x, (unsigned char)j.y, (unsigned char)j.z, (unsigned char)j.w);
  }
  bad = (unsigned int)__reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(overflow, (unsigned long long)bad);
}

extern "C" int dcae_pack_symbols(const int32_t* symbols, const int32_t* indexes, int64_t n, int16_t* symbols16, uint8_t* indexes8,
                                 unsigned long long* overflow_count, void* stream) {
  DCAE_REQUIRE(symbols && indexes && symbols16 && indexes8 && overflow_count && n >= 0 && n % 4 == 0, "dcae_pack_symbols: bad arguments (n must be a multiple of 4)");
  DCAE_REQUIRE(aligned16(symbols) && aligned16(indexes) && (reinterpret_cast<uintptr_t>(symbols16) & 7u) == 0 && (reinterpret_cast<uintptr_t>(indexes8) & 3u) == 0,
               "dcae_pack_symbols: alignment");
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  DCAE_CUDA(cudaMemsetAsync(overflow_count, 0, sizeof(unsigned long long), (cudaStream_t)stream));
  if (n == 0) return DCAE_OK;
  pack_symbols_kernel<<<grid_for(n / 4, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const int4*>(symbols), reinterpret_cast<const int4*>(indexes), n / 4,
                                                                           reinterpret_cast<short4*>(symbols16), reinterpret_cast<uchar4*>(indexes8), overflow_count);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

// ---- fp16 operand-plane range check (DCAE_MATH_F16X3) -----------------------------------------------------
// Activations are converted to hi/lo planes with cvt.rn.satfinite: a magnitude above 65504 is silently clamped.
// This kernel counts the elements of a planes window whose hi half sits at the clamp (|hi| == 0x7bff) or is not
// finite; the slice loop runs it behind every producer when range checking is on (validation of a new checkpoint).
__global__ void count_f16_clamped_kernel(const __half* __restrict__ hi, int64_t ld, int64_t rows, int32_t cols, unsigned long long* counter) {
  unsigned long long n = 0;
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    const unsigned short b = __half_as_ushort(hi[r * ld + (i - r * cols)]) & 0x7fffu;
    n += b >= 0x7bffu;
  }
  n = __reduce_add_sync(0xffffffffu, (unsigned)n);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(counter, n);
}

extern "C" int dcae_count_f16_clamped(const dcae_planes* planes, int64_t T, int32_t cols, unsigned long long* counter, void* stream) {
  DCAE_REQUIRE(planes && planes->hi && counter && T >= 0 && cols >= 0, "dcae_count_f16_clamped: bad arguments");
  if (T == 0 || cols == 0) return DCAE_OK;
  count_f16_clamped_kernel<<<grid_for(T * cols, 256), 256, 0, (cudaStream_t)stream>>>(static_cast<const __half*>(planes->hi), planes->ld, T, cols, counter);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_split_tf32(const float* w, float* w_hi, float* w_lo, int64_t n, void* stream) {
  DCAE_REQUIRE(w && w_hi && w_lo && n >= 0, "dcae_split_tf32: bad arguments");
  if (n == 0) return DCAE_OK;
  split_tf32_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(w, w_hi, w_lo, n);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
