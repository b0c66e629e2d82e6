// Hyper-latent entropy model (SURVEY 8f N3, first part): compressai's EntropyBottleneck as the reference uses it for z
// (/root/reference/models/dcae.py:629-633 forward, :705-706 compress, :861 decompress) in one pass:
//   out    = round(z - median) + median   (EVAL)  |  z + noise (NOISE)  |  float(symbols) + median (DECODE)
//   lik    = max(sigmoid(L(out + 1/2)) - sigmoid(L(out - 1/2)), lik_bound)
//   L(v)   = the per-channel monotone network 1 -> 3 -> 3 -> 3 -> 3 -> 1 of the factorised prior (Balle et al. 2018):
//            h = softplus(M_i) h + b_i;  h += tanh(f_i) * tanh(h)  for i < 4
//   sym    = int32(round(z - median)),  z_hat = out
// softplus(M_i) and tanh(f_i) are constant per weight load: the host packs them once, 58 floats per channel.
// One block works on one (image, channel) row of h*w elements with the channel's 58 parameters in shared memory.
#include "common.cuh"

namespace dcae {

constexpr int EB_THREADS = 128;
constexpr int EB_PARAMS = 58;   // matrices 3 + 9 + 9 + 9 + 3, biases 3 + 3 + 3 + 3 + 1, factors 3 + 3 + 3 + 3
// offsets inside the packed row
constexpr int EB_M0 = 0, EB_M1 = 3, EB_M2 = 12, EB_M3 = 21, EB_M4 = 30, EB_B0 = 33, EB_B1 = 36, EB_B2 = 39, EB_B3 = 42, EB_B4 = 45,
              EB_F0 = 46, EB_F1 = 49, EB_F2 = 52, EB_F3 = 55;

__device__ __forceinline__ float eb_logits(float v, const float* p) {
  float h[3], g[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    h[k] = p[EB_M0 + k] * v + p[EB_B0 + k];
    h[k] += p[EB_F0 + k] * tanhf(h[k]);
  }
#pragma unroll
  for (int layer = 0; layer < 3; ++layer) {
    const float* m = p + EB_M1 + 9 * layer;
    const float* b = p + EB_B1 + 3 * layer;
    const float* f = p + EB_F1 + 3 * layer;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      g[k] = m[3 * k] * h[0] + m[3 * k + 1] * h[1] + m[3 * k + 2] * h[2] + b[k];
      g[k] += f[k] * tanhf(g[k]);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) h[k] = g[k];
  }
  return p[EB_M4] * h[0] + p[EB_M4 + 1] * h[1] + p[EB_M4 + 2] * h[2] + p[EB_B4];
}

__device__ __forceinline__ float eb_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(EB_THREADS) eb_fused_kernel(const dcae_eb_args a) {
  __shared__ float p[EB_PARAMS];
  const int row = blockIdx.x;                  // image * C + channel
  const int c = row % a.C;
  for (int i = threadIdx.x; i < EB_PARAMS; i += EB_THREADS) p[i] = a.params[(int64_t)c * EB_PARAMS + i];
  __syncthreads();
  const float med = a.medians[c];
  const int64_t base = (int64_t)row * a.HW;
  for (int64_t i = (int64_t)blockIdx.y * EB_THREADS + threadIdx.x; i < a.HW; i += (int64_t)gridDim.y * EB_THREADS) {
    float r, out;
    if (a.mode == DCAE_GC_DECODE) {
      r = (float)a.sym_in[base + i];
      out = r + med;
    } else {
      const float z = a.z[base + i];
      r = rintf(z - med);                      // torch.round: half to even
      out = a.mode == DCAE_GC_NOISE ? z + a.noise[base + i] : r + med;
    }
    if (a.sym) a.sym[base + i] = (int)r;
    if (a.z_hat) a.z_hat[base + i] = r + med;  // ste_round(z - median) + median (dcae.py:631-633) == the dequantised value
    if (a.lik) {
      const float lower = eb_logits(out - 0.5f, p), upper = eb_logits(out + 0.5f, p);
      const float lk = eb_sigmoid(upper) - eb_sigmoid(lower);
      a.lik[base + i] = (lk != lk) ? lk : fmaxf(lk, a.lik_bound);
    }
  }
}

}  // namespace dcae

extern "C" int dcae_eb_fused(const dcae_eb_args* a, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(a && a->params && a->medians, "dcae_eb_fused: null parameters");
  DCAE_REQUIRE(a->mode >= DCAE_GC_EVAL && a->mode <= DCAE_GC_DECODE, "dcae_eb_fused: bad mode %d", a->mode);
  DCAE_REQUIRE(a->B >= 0 && a->C > 0 && a->HW >= 0 && (int64_t)a->B * a->C < (1ll << 31), "dcae_eb_fused: bad shape");
  DCAE_REQUIRE(a->mode == DCAE_GC_DECODE ? a->sym_in != nullptr : a->z != nullptr, "dcae_eb_fused: missing input for mode %d", a->mode);
  DCAE_REQUIRE(a->mode != DCAE_GC_NOISE || a->noise != nullptr, "dcae_eb_fused: NOISE mode needs a noise tensor");
  DCAE_REQUIRE(a->mode != DCAE_GC_DECODE || a->lik == nullptr, "dcae_eb_fused: DECODE produces no likelihood");
  if (a->B == 0 || a->HW == 0) return DCAE_OK;
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  int64_t chunks = (a->HW + EB_THREADS - 1) / EB_THREADS;
  if (chunks > 64) chunks = 64;
  dim3 grid((unsigned)(a->B * a->C), (unsigned)chunks);
  eb_fused_kernel<<<grid, EB_THREADS, 0, (cudaStream_t)stream>>>(*a);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

namespace dcae {

// ---- backward of the likelihood (training: train.py:165-179 differentiates the rate of z through compressai's
// EntropyBottleneck.forward) ------------------------------------------------------------------------------------------
// Per element the two evaluations L(out +- 1/2) are recomputed with every layer's output h and tanh value t kept in
// registers, then differentiated layer by layer:
//   dU = g' s(U) s(-U),  dLo = -g' s(Lo) s(-Lo)            (s = sigmoid; g' = g where lik_raw >= lik_bound or g < 0)
//   h = a + f tanh(a):  da = dh (1 + f (1 - t^2)),  df += dh t,  db += da,  dM += da h_prev^T,  dh_prev = M^T da
// The bound test uses lik_raw = |s(sU) - s(sLo)| with s = -sign(U + Lo) (compressai's mirrored form): above the median
// s(U) - s(Lo) is a difference of two numbers near 1 and cancels to 0 or 6e-8 in fp32 where the true value is far
// below the bound; the mirrored form keeps its relative accuracy on both sides.
// One block per channel: each thread accumulates the 58 parameter gradients of its elements (element order fixed by
// the shape), then a fixed xor-butterfly inside each warp and the warps in index order.  No atomics, every grad_z
// element has one writer and depends on its own element only.
constexpr int EBB_THREADS = 256;

__device__ __forceinline__ float eb_logits_trace(float v, const float* p, float (&h)[4][3], float (&t)[4][3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float a = p[EB_M0 + k] * v + p[EB_B0 + k];
    t[0][k] = tanhf(a);
    h[0][k] = a + p[EB_F0 + k] * t[0][k];
  }
#pragma unroll
  for (int l = 1; l < 4; ++l) {
    const float* m = p + EB_M1 + 9 * (l - 1);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float a = m[3 * k] * h[l - 1][0] + m[3 * k + 1] * h[l - 1][1] + m[3 * k + 2] * h[l - 1][2] + p[EB_B0 + 3 * l + k];
      t[l][k] = tanhf(a);
      h[l][k] = a + p[EB_F0 + 3 * l + k] * t[l][k];
    }
  }
  return p[EB_M4] * h[3][0] + p[EB_M4 + 1] * h[3][1] + p[EB_M4 + 2] * h[3][2] + p[EB_B4];
}

// accumulates dL/dparams of one evaluation L(v) with dL/dL = d into g[58]; returns dL/dv
__device__ __forceinline__ float eb_logits_backward(float d, float v, const float* p, const float (&h)[4][3], const float (&t)[4][3],
                                                   float (&g)[EB_PARAMS]) {
  float dh[3], da[3];
  g[EB_B4] += d;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    g[EB_M4 + j] += d * h[3][j];
    dh[j] = d * p[EB_M4 + j];
  }
#pragma unroll
  for (int l = 3; l >= 1; --l) {
    const float* m = p + EB_M1 + 9 * (l - 1);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      da[k] = dh[k] * (1.0f + p[EB_F0 + 3 * l + k] * (1.0f - t[l][k] * t[l][k]));
      g[EB_F0 + 3 * l + k] += dh[k] * t[l][k];
      g[EB_B0 + 3 * l + k] += da[k];
#pragma unroll
      for (int j = 0; j < 3; ++j) g[EB_M1 + 9 * (l - 1) + 3 * k + j] += da[k] * h[l - 1][j];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) dh[j] = da[0] * m[j] + da[1] * m[3 + j] + da[2] * m[6 + j];
  }
  float dv = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    da[k] = dh[k] * (1.0f + p[EB_F0 + k] * (1.0f - t[0][k] * t[0][k]));
    g[EB_F0 + k] += dh[k] * t[0][k];
    g[EB_B0 + k] += da[k];
    g[EB_M0 + k] += da[k] * v;
    dv += da[k] * p[EB_M0 + k];
  }
  return dv;
}

__global__ void __launch_bounds__(EBB_THREADS) eb_backward_kernel(const dcae_eb_bwd_args a) {
  __shared__ float p[EB_PARAMS];
  __shared__ float part[EBB_THREADS / 32][EB_PARAMS];
  const int c = blockIdx.x;
  for (int i = threadIdx.x; i < EB_PARAMS; i += EBB_THREADS) p[i] = a.params[(int64_t)c * EB_PARAMS + i];
  __syncthreads();
  const float med = a.medians[c];
  const bool noisy = a.mode == DCAE_GC_NOISE;
  float g[EB_PARAMS];
#pragma unroll
  for (int k = 0; k < EB_PARAMS; ++k) g[k] = 0.f;
  const int64_t n = (int64_t)a.B * a.HW;
  for (int64_t e = threadIdx.x; e < n; e += EBB_THREADS) {
    const int64_t b = e / a.HW;
    const int64_t idx = (b * a.C + c) * a.HW + (e - b * a.HW);
    const float z = a.z[idx];
    const float out = noisy ? z + a.noise[idx] : rintf(z - med) + med;
    float hu[4][3], tu[4][3], hl[4][3], tl[4][3];
    const float up = eb_logits_trace(out + 0.5f, p, hu, tu), lo = eb_logits_trace(out - 0.5f, p, hl, tl);
    const float s = (up + lo > 0.f) ? -1.f : 1.f;
    const float raw = fabsf(eb_sigmoid(s * up) - eb_sigmoid(s * lo));
    const float gl = a.grad_lik[idx];
    const float gp = (raw >= a.lik_bound || gl < 0.f) ? gl : 0.f;
    const float d_up = gp * eb_sigmoid(up) * eb_sigmoid(-up), d_lo = -gp * eb_sigmoid(lo) * eb_sigmoid(-lo);
    const float dv = eb_logits_backward(d_up, out + 0.5f, p, hu, tu, g) + eb_logits_backward(d_lo, out - 0.5f, p, hl, tl, g);
    a.grad_z[idx] = noisy ? dv : 0.f;              // EVAL: torch.round passes no gradient
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < EB_PARAMS; ++k) {
    float v = g[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) part[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < EB_PARAMS) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < EBB_THREADS / 32; ++w) v += part[w][threadIdx.x];
    a.grad_params[(int64_t)c * EB_PARAMS + threadIdx.x] = v;
  }
}

}  // namespace dcae

extern "C" int dcae_eb_backward(const dcae_eb_bwd_args* a, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(a && a->params && a->medians && a->z && a->grad_lik, "dcae_eb_backward: null input");
  DCAE_REQUIRE(a->grad_z && a->grad_params, "dcae_eb_backward: null output");
  DCAE_REQUIRE(a->mode == DCAE_GC_EVAL || a->mode == DCAE_GC_NOISE, "dcae_eb_backward: bad mode %d (EVAL or NOISE)", a->mode);
  DCAE_REQUIRE(a->mode != DCAE_GC_NOISE || a->noise != nullptr, "dcae_eb_backward: NOISE mode needs a noise tensor");
  DCAE_REQUIRE(a->B >= 0 && a->C > 0 && a->HW >= 0 && a->C < (1 << 30), "dcae_eb_backward: bad shape");
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  eb_backward_kernel<<<(unsigned)a->C, EBB_THREADS, 0, (cudaStream_t)stream>>>(*a);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
