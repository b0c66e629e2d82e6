// Token-major kernels of the transform stacks around the entropy model (SURVEY 8f N3 / N4:
// /root/reference/models/dcae.py:152-383 blocks, :541-582 g_a / g_s / h_a / h_z_s1 / h_z_s2):
//   * window attention of the Swin blocks (WMSA, dcae.py:228-298): W and SW (cyclic shift + mask) windows,
//     relative position bias, softmax in registers, no sim / probs tensor in HBM;
//   * LayerNorm for any channel count (the dictionary module's LayerNorm kernel needs C % 128 == 0);
//   * space-to-depth / depth-to-space: a stride-2 convolution is a stride-1 3x3 convolution over the 2x2
//     space-to-depth image and a stride-2 transposed convolution is a stride-1 3x3 convolution producing the four
//     output phases (weights re-indexed at pack time, dcae_b200/transforms.py), so both run on the 3x3 implicit
//     GEMM (kernel 2) unchanged.
// All HBM-bound, fp32 in / fp32 (+ optional fp16 hi/lo planes) out, no atomics, deterministic.
#include <math.h>

#include "common.cuh"

namespace dcae {
namespace {

__device__ __forceinline__ void store_plane1(const dcae_planes& p, int64_t row, int col, float v) {
  unsigned short h, l;
  f16_split(v, h, l);
  static_cast<unsigned short*>(p.hi)[row * p.ld + col] = h;
  static_cast<unsigned short*>(p.lo)[row * p.ld + col] = l;
}

// ---------------------------------------------------------------------------------------------
// LayerNorm, one warp per token, any C % 4 == 0 up to 1024 (V = ceil(C / 128) float4 per lane).
// ---------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(256) layernorm_any_kernel(const float* __restrict__ x, int64_t x_ld, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, int C4, int64_t T, float* __restrict__ out,
                                                            int64_t out_ld, const dcae_planes o16) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const float4* xr = reinterpret_cast<const float4*>(x + t * x_ld);
  float4 v[V];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const int c = lane + 32 * k;
    v[k] = c < C4 ? __ldg(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  }
  const float inv_c = 1.0f / (float)(4 * C4);
  const float mean = warp_sum(s) * inv_c;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    if (lane + 32 * k < C4) {
      const float a = v[k].x - mean, b = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * inv_c + 1e-5f);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const int c = lane + 32 * k;
    if (c < C4) {
      const float4 g = __ldg(g4 + c), b = __ldg(b4 + c);
      float4 o;
      o.x = (v[k].x - mean) * rstd * g.x + b.x;
      o.y = (v[k].y - mean) * rstd * g.y + b.y;
      o.z = (v[k].z - mean) * rstd * g.z + b.z;
      o.w = (v[k].w - mean) * rstd * g.w + b.w;
      if (out) *reinterpret_cast<float4*>(out + t * out_ld + 4 * c) = o;
      if (o16.hi) store_planes4(o16, t, 4 * c, o);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Window attention (dcae.py:262-291).  One block per window, heads in sequence.  Four threads share a pair of query
// rows (i2, i2 + PP/2): thread (i2, c4) owns the keys j = c4 + 4 jj.  The two query rows live in registers, K and V of
// the head in shared memory (rows padded to HD + 4 floats: 16-byte aligned and conflict-free for the float4 reads), so
// every float4 of K / V read from shared memory feeds 8 FMAs (two rows x four dims); logits / probabilities stay in
// registers, no sim / probs tensor exists in HBM.
// ---------------------------------------------------------------------------------------------
struct WinArgs {
  const float* qkv; int64_t ld; int q_col, k_col, v_col;
  int n_heads, shift, B, h, w, nwx, nwy;
  const float* rel;            // [n_heads, 2P-1, 2P-1]
  float scale;
  float* out; int64_t out_ld; dcae_planes o16;
};

template <int HD, int P>
__global__ void __launch_bounds__(2 * P * P) window_attention_kernel(const WinArgs a) {
  constexpr int PP = P * P, HALF = PP / 2, NJ = PP / 4, LDS = HD + 4, R = 2 * P - 1, DQ = HD / 4, NT = 2 * PP;
  __shared__ __align__(16) float sk[PP * LDS];
  __shared__ __align__(16) float sv[PP * LDS];
  __shared__ float sbias[R * R];
  __shared__ int64_t stok[PP];
  const int tid = threadIdx.x, i2 = tid >> 2, c4 = tid & 3;
  const int wx = (int)(blockIdx.x % a.nwx), wy = (int)(blockIdx.x / a.nwx), b = (int)blockIdx.y;
  // rolled[r] = x[(r + shift) mod size] (torch.roll by -shift, dcae.py:270); the result goes back to the same token (:289)
  if (tid < PP) {
    int yy = wy * P + tid / P + a.shift; if (yy >= a.h) yy -= a.h;
    int xx = wx * P + tid % P + a.shift; if (xx >= a.w) xx -= a.w;
    stok[tid] = ((int64_t)b * a.h + yy) * a.w + xx;
  }
  // SW mask (generate_mask, dcae.py:244-260): in the last window row / column the wrapped part may not see the rest
  const bool last_row = a.shift > 0 && wy == a.nwy - 1, last_col = a.shift > 0 && wx == a.nwx - 1;
  const int sp = P - a.shift;
  int py[2], px[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) { py[r] = (i2 + r * HALF) / P; px[r] = (i2 + r * HALF) % P; }
  __syncthreads();
  const int64_t tok[2] = {stok[i2], stok[i2 + HALF]};
  for (int e = 0; e < a.n_heads; ++e) {
    __syncthreads();                       // the previous head is done with sk / sv / sbias
    for (int idx = tid; idx < PP * DQ; idx += NT) {
      const int t = idx / DQ, d4 = idx - t * DQ;
      const float* row = a.qkv + stok[t] * a.ld + e * HD + 4 * d4;
      *reinterpret_cast<float4*>(sk + t * LDS + 4 * d4) = __ldg(reinterpret_cast<const float4*>(row + a.k_col));
      *reinterpret_cast<float4*>(sv + t * LDS + 4 * d4) = __ldg(reinterpret_cast<const float4*>(row + a.v_col));
    }
    for (int t = tid; t < R * R; t += NT) sbias[t] = __ldg(a.rel + (int64_t)e * R * R + t);
    float q[2][HD];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const float4* qp = reinterpret_cast<const float4*>(a.qkv + tok[r] * a.ld + a.q_col + e * HD);
#pragma unroll
      for (int d4 = 0; d4 < DQ; ++d4) {
        const float4 v = __ldg(qp + d4);
        q[r][4 * d4] = v.x; q[r][4 * d4 + 1] = v.y; q[r][4 * d4 + 2] = v.z; q[r][4 * d4 + 3] = v.w;
      }
    }
    __syncthreads();
    float s[2][NJ];
    float m[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int jj = 0; jj < NJ; ++jj) {
      const int j = c4 + 4 * jj;
      float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
      for (int d4 = 0; d4 < DQ; ++d4) {
        const float4 kv = *reinterpret_cast<const float4*>(sk + j * LDS + 4 * d4);
        acc0 = fmaf(q[0][4 * d4], kv.x, acc0); acc1 = fmaf(q[1][4 * d4], kv.x, acc1);
        acc0 = fmaf(q[0][4 * d4 + 1], kv.y, acc0); acc1 = fmaf(q[1][4 * d4 + 1], kv.y, acc1);
        acc0 = fmaf(q[0][4 * d4 + 2], kv.z, acc0); acc1 = fmaf(q[1][4 * d4 + 2], kv.z, acc1);
        acc0 = fmaf(q[0][4 * d4 + 3], kv.w, acc0); acc1 = fmaf(q[1][4 * d4 + 3], kv.w, acc1);
      }
      const int qy = j / P, qx = j % P;
      const float acc[2] = {acc0, acc1};
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const float v = acc[r] * a.scale + sbias[(py[r] - qy + P - 1) * R + (px[r] - qx + P - 1)];
        const bool masked = (last_row && ((py[r] < sp) != (qy < sp))) || (last_col && ((px[r] < sp) != (qx < sp)));
        s[r][jj] = masked ? -INFINITY : v;
        m[r] = fmaxf(m[r], s[r][jj]);
      }
    }
    float inv[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      m[r] = fmaxf(m[r], __shfl_xor_sync(0xffffffffu, m[r], 1));
      m[r] = fmaxf(m[r], __shfl_xor_sync(0xffffffffu, m[r], 2));
      float sum = 0.f;
#pragma unroll
      for (int jj = 0; jj < NJ; ++jj) {
        s[r][jj] = expf(s[r][jj] - m[r]);
        sum += s[r][jj];
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      inv[r] = 1.0f / sum;
    }
    float o[2][HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) { o[0][d] = 0.f; o[1][d] = 0.f; }
#pragma unroll
    for (int jj = 0; jj < NJ; ++jj) {
      const int j = c4 + 4 * jj;
      const float p0 = s[0][jj] * inv[0], p1 = s[1][jj] * inv[1];
#pragma unroll
      for (int d4 = 0; d4 < DQ; ++d4) {
        const float4 vv = *reinterpret_cast<const float4*>(sv + j * LDS + 4 * d4);
        o[0][4 * d4] = fmaf(p0, vv.x, o[0][4 * d4]); o[1][4 * d4] = fmaf(p1, vv.x, o[1][4 * d4]);
        o[0][4 * d4 + 1] = fmaf(p0, vv.y, o[0][4 * d4 + 1]); o[1][4 * d4 + 1] = fmaf(p1, vv.y, o[1][4 * d4 + 1]);
        o[0][4 * d4 + 2] = fmaf(p0, vv.z, o[0][4 * d4 + 2]); o[1][4 * d4 + 2] = fmaf(p1, vv.z, o[1][4 * d4 + 2]);
        o[0][4 * d4 + 3] = fmaf(p0, vv.w, o[0][4 * d4 + 3]); o[1][4 * d4 + 3] = fmaf(p1, vv.w, o[1][4 * d4 + 3]);
      }
    }
    // sum over the four key owners of the row pair, then thread c4 keeps and writes dims [c4 DQ, (c4 + 1) DQ)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float mine[DQ];
#pragma unroll
      for (int d = 0; d < HD; ++d) {
        float v = o[r][d];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if (d / DQ == c4) mine[d % DQ] = v;
      }
      const int col = e * HD + c4 * DQ;
      if (a.out) {
        float* op = a.out + tok[r] * a.out_ld + col;
        if (DQ == 2) *reinterpret_cast<float2*>(op) = make_float2(mine[0], mine[1]);
        else {
#pragma unroll
          for (int d4 = 0; d4 < DQ / 4; ++d4) *reinterpret_cast<float4*>(op + 4 * d4) = make_float4(mine[4 * d4], mine[4 * d4 + 1], mine[4 * d4 + 2], mine[4 * d4 + 3]);
        }
      }
      if (a.o16.hi) {
        if (DQ == 2) {
          uint32_t hw, lw;
          f16_split2(mine[0], mine[1], hw, lw);
          *reinterpret_cast<uint32_t*>(static_cast<__half*>(a.o16.hi) + tok[r] * a.o16.ld + col) = hw;
          *reinterpret_cast<uint32_t*>(static_cast<__half*>(a.o16.lo) + tok[r] * a.o16.ld + col) = lw;
        } else {
#pragma unroll
          for (int d4 = 0; d4 < DQ / 4; ++d4)
            store_planes4(a.o16, tok[r], col + 4 * d4, make_float4(mine[4 * d4], mine[4 * d4 + 1], mine[4 * d4 + 2], mine[4 * d4 + 3]));
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// The same operator for 8x8 windows on the warp-level tensor-core path: S = Q K^T and O = P V as m16n8k8 TF32 MMAs with
// the 3-pass hi/lo split (a_lo b_hi + a_hi b_lo + a_hi b_hi, fp32 accumulate: 21 significant bits per operand, the same
// class of accuracy as the f16x3 GEMMs).  One block = one window = 4 warps, warp w owns query rows [16 w, 16 w + 16) (window
// rows 2 w and 2 w + 1) against all 64 keys; K and V of the head sit in shared memory already split into TF32 hi / lo
// (rows padded to HD + 4 words: conflict-free fragment loads).  The probabilities never change registers between the two
// products: with the key order inside a k-step chosen as (2t, 2t + 1) <-> slots (t, t + 4), the C fragment of S IS the A
// fragment of P V.  [A 64-token window is too small a tile for tcgen05 (M = 128 per instruction and a TMEM round trip per
// head); the SIMT kernel above measured 15 TFLOP/s, bound by shared-memory reads.]
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float to_tf32(float v) {
  uint32_t o;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(o) : "f"(v));
  return __uint_as_float(o);
}
__device__ __forceinline__ void mma_tf32_16x8x8(float (&d)[4], const float (&a)[4], float b0, float b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(__float_as_uint(a[0])), "r"(__float_as_uint(a[1])), "r"(__float_as_uint(a[2])), "r"(__float_as_uint(a[3])),
                 "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}

template <int HD>
__global__ void __launch_bounds__(128) window_attention_mma_kernel(const WinArgs a, int C) {
  // heads are walked in groups of G (GW = G HD contiguous q / k / v columns per shared-memory fill).  G = 32 / HD was measured
  // (one fill and one barrier pair per 32 columns): head_dim 8 lost 16 % because 41 KB of shared memory per block leave 5
  // blocks per SM instead of 16; G = 1 it is
  constexpr int P = 8, PP = 64, G = 1, GW = G * HD, LDS = GW + 4, R = 2 * P - 1, KSTEPS = HD / 8, NT = 128;
  __shared__ __align__(16) float skh[PP * LDS], skl[PP * LDS], svh[PP * LDS], svl[PP * LDS];
  __shared__ float sbias[G * R * R];
  __shared__ int64_t stok[PP];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wx = (int)(blockIdx.x % a.nwx), wy = (int)(blockIdx.x / a.nwx), b = (int)blockIdx.y;
  if (tid < PP) {
    int yy = wy * P + tid / P + a.shift; if (yy >= a.h) yy -= a.h;
    int xx = wx * P + tid % P + a.shift; if (xx >= a.w) xx -= a.w;
    stok[tid] = ((int64_t)b * a.h + yy) * a.w + xx;
  }
  const bool last_row = a.shift > 0 && wy == a.nwy - 1, last_col = a.shift > 0 && wx == a.nwx - 1;
  const int sp = P - a.shift;
  // this thread's two query rows: window position (py, px) = (2 warp + r, g)
  const int py0 = 2 * warp, px = g;
  __syncthreads();
  const int64_t tok0 = stok[16 * warp + g], tok1 = stok[16 * warp + g + 8];
  for (int e0 = 0; e0 < a.n_heads; e0 += G) {
    __syncthreads();                       // the previous group is done with shared memory
    for (int idx = tid; idx < PP * (GW / 4); idx += NT) {
      const int tk = idx / (GW / 4), d4 = idx - tk * (GW / 4);
      const int col = e0 * HD + 4 * d4;                       // column inside the q / k / v segment (a tail group ends at C)
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (col < C) {
        const float* row = a.qkv + stok[tk] * a.ld + col;
        kv = __ldg(reinterpret_cast<const float4*>(row + a.k_col));
        vv = __ldg(reinterpret_cast<const float4*>(row + a.v_col));
      }
      float4 kh, kl, vh, vl;
      kh.x = to_tf32(kv.x); kh.y = to_tf32(kv.y); kh.z = to_tf32(kv.z); kh.w = to_tf32(kv.w);
      kl.x = to_tf32(kv.x - kh.x); kl.y = to_tf32(kv.y - kh.y); kl.z = to_tf32(kv.z - kh.z); kl.w = to_tf32(kv.w - kh.w);
      vh.x = to_tf32(vv.x); vh.y = to_tf32(vv.y); vh.z = to_tf32(vv.z); vh.w = to_tf32(vv.w);
      vl.x = to_tf32(vv.x - vh.x); vl.y = to_tf32(vv.y - vh.y); vl.z = to_tf32(vv.z - vh.z); vl.w = to_tf32(vv.w - vh.w);
      *reinterpret_cast<float4*>(skh + tk * LDS + 4 * d4) = kh;
      *reinterpret_cast<float4*>(skl + tk * LDS + 4 * d4) = kl;
      *reinterpret_cast<float4*>(svh + tk * LDS + 4 * d4) = vh;
      *reinterpret_cast<float4*>(svl + tk * LDS + 4 * d4) = vl;
    }
    for (int i = tid; i < G * R * R; i += NT) sbias[i] = (e0 + i / (R * R) < a.n_heads) ? __ldg(a.rel + (int64_t)e0 * R * R + i) : 0.f;
    __syncthreads();
#pragma unroll 1
    for (int eg = 0; eg < G; ++eg) {
      const int e = e0 + eg;
      if (e >= a.n_heads) break;
      const int hc = eg * HD;              // the head's first column inside the group tile
      // Q fragments (A operand, 16 x 8 per k-step): a0 = (g, t), a1 = (g + 8, t), a2 = (g, t + 4), a3 = (g + 8, t + 4)
      float qh[KSTEPS][4], ql[KSTEPS][4];
      {
        const float* q0 = a.qkv + tok0 * a.ld + a.q_col + e * HD;
        const float* q1 = a.qkv + tok1 * a.ld + a.q_col + e * HD;
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const float v[4] = {__ldg(q0 + 8 * ks + t), __ldg(q1 + 8 * ks + t), __ldg(q0 + 8 * ks + t + 4), __ldg(q1 + 8 * ks + t + 4)};
#pragma unroll
          for (int i = 0; i < 4; ++i) { qh[ks][i] = to_tf32(v[i]); ql[ks][i] = to_tf32(v[i] - qh[ks][i]); }
        }
      }
      // S = Q K^T: 8 key tiles of 8; B fragment b0 = K[key n0 + g][8 ks + t], b1 = K[key n0 + g][8 ks + t + 4]
      float sc[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int i = 0; i < 4; ++i) sc[nt][i] = 0.f;
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const int o = (8 * nt + g) * LDS + hc + 8 * ks + t;
          const float bh0 = skh[o], bh1 = skh[o + 4], bl0 = skl[o], bl1 = skl[o + 4];
          mma_tf32_16x8x8(sc[nt], ql[ks], bh0, bh1);
          mma_tf32_16x8x8(sc[nt], qh[ks], bl0, bl1);
          mma_tf32_16x8x8(sc[nt], qh[ks], bh0, bh1);
        }
      }
      // C fragment: c0 = (g, 2t), c1 = (g, 2t + 1), c2 = (g + 8, 2t), c3 = (g + 8, 2t + 1) of key tile nt -> key (qy, qx) = (nt, 2t + i)
      const float* bias = sbias + eg * R * R;
      float m0 = -INFINITY, m1 = -INFINITY;
      if (last_row || last_col) {          // block-uniform: only the last window row / column of an SW layer carries a mask
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = i >> 1, qx = 2 * t + (i & 1), py = py0 + r, qy = nt;
            const float v = sc[nt][i] * a.scale + bias[(py - qy + P - 1) * R + (px - qx + P - 1)];
            const bool masked = (last_row && ((py < sp) != (qy < sp))) || (last_col && ((px < sp) != (qx < sp)));
            sc[nt][i] = masked ? -INFINITY : v;
          }
        }
      } else {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = i >> 1, qx = 2 * t + (i & 1), py = py0 + r, qy = nt;
            sc[nt][i] = sc[nt][i] * a.scale + bias[(py - qy + P - 1) * R + (px - qx + P - 1)];
          }
        }
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        m0 = fmaxf(m0, fmaxf(sc[nt][0], sc[nt][1]));
        m1 = fmaxf(m1, fmaxf(sc[nt][2], sc[nt][3]));
      }
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        sc[nt][0] = expf(sc[nt][0] - m0); sc[nt][1] = expf(sc[nt][1] - m0);
        sc[nt][2] = expf(sc[nt][2] - m1); sc[nt][3] = expf(sc[nt][3] - m1);
        s0 += sc[nt][0] + sc[nt][1];
        s1 += sc[nt][2] + sc[nt][3];
      }
      s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
      const float i0 = 1.0f / s0, i1 = 1.0f / s1;
      // O = P V: k-step j = key tile j with slot t <-> key 8j + 2t, slot t + 4 <-> key 8j + 2t + 1, so that the A fragment
      // (a0, a1, a2, a3) is (c0, c2, c1, c3) of S; B fragment b0 = V[8j + 2t][n0 + g], b1 = V[8j + 2t + 1][n0 + g]
      float oc[KSTEPS][4];
#pragma unroll
      for (int nd = 0; nd < KSTEPS; ++nd) {
#pragma unroll
        for (int i = 0; i < 4; ++i) oc[nd][i] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float pv[4] = {sc[j][0], sc[j][2], sc[j][1], sc[j][3]};          // unnormalised (max-subtracted: in (0, 1]); 1 / sum goes onto O
        float ph[4], pl[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { ph[i] = to_tf32(pv[i]); pl[i] = to_tf32(pv[i] - ph[i]); }
#pragma unroll
        for (int nd = 0; nd < KSTEPS; ++nd) {
          const int o = (8 * j + 2 * t) * LDS + hc + 8 * nd + g;
          const float bh0 = svh[o], bh1 = svh[o + LDS], bl0 = svl[o], bl1 = svl[o + LDS];
          mma_tf32_16x8x8(oc[nd], pl, bh0, bh1);
          mma_tf32_16x8x8(oc[nd], ph, bl0, bl1);
          mma_tf32_16x8x8(oc[nd], ph, bh0, bh1);
        }
      }
      // rows g (tok0) and g + 8 (tok1), dims 8 nd + 2t, 2t + 1
#pragma unroll
      for (int nd = 0; nd < KSTEPS; ++nd) {
        oc[nd][0] *= i0; oc[nd][1] *= i0; oc[nd][2] *= i1; oc[nd][3] *= i1;
        const int col = e * HD + 8 * nd + 2 * t;
        if (a.out) {
          *reinterpret_cast<float2*>(a.out + tok0 * a.out_ld + col) = make_float2(oc[nd][0], oc[nd][1]);
          *reinterpret_cast<float2*>(a.out + tok1 * a.out_ld + col) = make_float2(oc[nd][2], oc[nd][3]);
        }
        if (a.o16.hi) {
          uint32_t hw, lw;
          f16_split2(oc[nd][0], oc[nd][1], hw, lw);
          *reinterpret_cast<uint32_t*>(static_cast<__half*>(a.o16.hi) + tok0 * a.o16.ld + col) = hw;
          *reinterpret_cast<uint32_t*>(static_cast<__half*>(a.o16.lo) + tok0 * a.o16.ld + col) = lw;
          f16_split2(oc[nd][2], oc[nd][3], hw, lw);
          *reinterpret_cast<uint32_t*>(static_cast<__half*>(a.o16.hi) + tok1 * a.o16.ld + col) = hw;
          *reinterpret_cast<uint32_t*>(static_cast<__half*>(a.o16.lo) + tok1 * a.o16.ld + col) = lw;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Backward of the window attention.  Per window and head, s = 1 / sqrt(hd): S and P recomputed as the forward does (same
// bias, SW mask, max-subtracted exponentials); dP = dO V^T; D_i = sum_j P_ij dP_ij; dS = P o (dP - D); dQ = s dS K,
// dK = s dS^T Q, dV = P^T dO; drel[e, dy, dx] = sum of dS over the (query, key) pairs at that offset.
// Determinism without atomics: every token belongs to one window, so each dq / dk / dv element has one writer; block b walks
// heads in order and, per head, the windows b, b + gridDim.x, ... (flattened over the batch) in order, accumulates its drel
// bins in registers (thread tid owns bins tid, tid + NT, ...) and writes them to part[b][e][bin]; a second launch adds the
// partials in block order.  The grid depends on the shape only (wattn_bwd_blocks).
// ---------------------------------------------------------------------------------------------
constexpr int WATTN_BWD_MAX_BLOCKS = 1184;         // 148 SMs x 8

inline int64_t wattn_bwd_blocks(int64_t n_windows) { return n_windows < WATTN_BWD_MAX_BLOCKS ? n_windows : WATTN_BWD_MAX_BLOCKS; }

struct WinBwdArgs {
  const float* qkv; int64_t ld; int q_col, k_col, v_col;
  int n_heads, shift, h, w, nwx, nwy;
  int64_t n_win;               // B * nwx * nwy
  const float* rel;            // [n_heads, 2P-1, 2P-1]
  float scale;
  const float* dout; int64_t dout_ld;
  float* dqkv; int64_t dqkv_ld;
  float* part;                 // [gridDim.x, n_heads, (2P-1)^2]
};

// window `win` (flattened b, wy, wx) -> its tokens (rolled by the SW shift) into stok, and (wy, wx)
template <int P>
__device__ __forceinline__ void window_tokens(const WinBwdArgs& a, int64_t win, int64_t* stok, int& wy, int& wx) {
  const int64_t nw = (int64_t)a.nwx * a.nwy;
  const int b = (int)(win / nw), wi = (int)(win - b * nw);
  wx = wi % a.nwx; wy = wi / a.nwx;
  for (int p = threadIdx.x; p < P * P; p += blockDim.x) {
    int yy = wy * P + p / P + a.shift; if (yy >= a.h) yy -= a.h;
    int xx = wx * P + p % P + a.shift; if (xx >= a.w) xx -= a.w;
    stok[p] = ((int64_t)b * a.h + yy) * a.w + xx;
  }
}

// sum of dS over the pairs at bin = (dy + P - 1) * R + (dx + P - 1): query (py, px), key (py - dy, px - dx); dS(i, j) = ds[j * ld + i]
template <int P>
__device__ __forceinline__ float rel_bin_sum(const float* dsT, int ld, int bin) {
  constexpr int R = 2 * P - 1;
  const int dy = bin / R - (P - 1), dx = bin % R - (P - 1);
  float s = 0.f;
  for (int py = dy > 0 ? dy : 0; py < (dy < 0 ? P + dy : P); ++py)
    for (int px = dx > 0 ? dx : 0; px < (dx < 0 ? P + dx : P); ++px)
      s += dsT[((py - dy) * P + (px - dx)) * ld + py * P + px];
  return s;
}

// 4x4 windows (the hyper path): FFMA, one window of PP = 16 tokens per block iteration, everything in shared memory
template <int HD, int P>
__global__ void __launch_bounds__(128) window_attention_bwd_kernel(const WinBwdArgs a) {
  constexpr int PP = P * P, R = 2 * P - 1, NT = 128, LD = HD + 1, LP = PP + 1, NB = (R * R + NT - 1) / NT;
  __shared__ float sq[PP * LD], sk[PP * LD], sv[PP * LD], sdo[PP * LD];
  __shared__ float sp[PP * LP], sdsT[PP * LP];        // P[i][j] at i * LP + j; dS transposed: dS[i][j] at j * LP + i
  __shared__ float sdp[PP * LP];
  __shared__ float sbias[R * R];
  __shared__ int64_t stok[PP];
  const int tid = threadIdx.x, sp_edge = P - a.shift;
  for (int e = 0; e < a.n_heads; ++e) {
    float acc[NB];
#pragma unroll
    for (int r = 0; r < NB; ++r) acc[r] = 0.f;
    for (int64_t win = blockIdx.x; win < a.n_win; win += gridDim.x) {
      __syncthreads();                     // the previous window is done with shared memory
      int wy, wx;
      window_tokens<P>(a, win, stok, wy, wx);
      for (int i = tid; i < R * R; i += NT) sbias[i] = __ldg(a.rel + (int64_t)e * R * R + i);
      __syncthreads();
      for (int idx = tid; idx < PP * HD; idx += NT) {
        const int t = idx / HD, d = idx - t * HD;
        const float* row = a.qkv + stok[t] * a.ld + e * HD + d;
        sq[t * LD + d] = __ldg(row + a.q_col);
        sk[t * LD + d] = __ldg(row + a.k_col);
        sv[t * LD + d] = __ldg(row + a.v_col);
        sdo[t * LD + d] = __ldg(a.dout + stok[t] * a.dout_ld + e * HD + d);
      }
      __syncthreads();
      const bool last_row = a.shift > 0 && wy == a.nwy - 1, last_col = a.shift > 0 && wx == a.nwx - 1;
      for (int pr = tid; pr < PP * PP; pr += NT) {
        const int i = pr / PP, j = pr - i * PP;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) {
          s = fmaf(sq[i * LD + d], sk[j * LD + d], s);
          dp = fmaf(sdo[i * LD + d], sv[j * LD + d], dp);
        }
        const int py = i / P, px = i % P, qy = j / P, qx = j % P;
        const bool masked = (last_row && ((py < sp_edge) != (qy < sp_edge))) || (last_col && ((px < sp_edge) != (qx < sp_edge)));
        sp[i * LP + j] = masked ? -INFINITY : s * a.scale + sbias[(py - qy + P - 1) * R + (px - qx + P - 1)];
        sdp[i * LP + j] = dp;
      }
      __syncthreads();
      if (tid < PP) {                      // softmax, D and dS of query row tid
        const int i = tid;
        float m = -INFINITY;
        for (int j = 0; j < PP; ++j) m = fmaxf(m, sp[i * LP + j]);
        float sum = 0.f;
        for (int j = 0; j < PP; ++j) { const float v = expf(sp[i * LP + j] - m); sp[i * LP + j] = v; sum += v; }
        const float inv = 1.0f / sum;
        float D = 0.f;
        for (int j = 0; j < PP; ++j) { sp[i * LP + j] *= inv; D = fmaf(sp[i * LP + j], sdp[i * LP + j], D); }
        for (int j = 0; j < PP; ++j) sdsT[j * LP + i] = sp[i * LP + j] * (sdp[i * LP + j] - D);
      }
      __syncthreads();
      for (int idx = tid; idx < PP * HD; idx += NT) {
        const int t = idx / HD, d = idx - t * HD;
        float gq = 0.f, gk = 0.f, gv = 0.f;
#pragma unroll
        for (int j = 0; j < PP; ++j) {
          gq = fmaf(sdsT[j * LP + t], sk[j * LD + d], gq);
          gk = fmaf(sdsT[t * LP + j], sq[j * LD + d], gk);
          gv = fmaf(sp[j * LP + t], sdo[j * LD + d], gv);
        }
        float* o = a.dqkv + stok[t] * a.dqkv_ld + e * HD + d;
        o[a.q_col] = gq * a.scale;
        o[a.k_col] = gk * a.scale;
        o[a.v_col] = gv;
      }
#pragma unroll
      for (int r = 0; r < NB; ++r)
        if (tid + r * NT < R * R) acc[r] += rel_bin_sum<P>(sdsT, LP, tid + r * NT);
    }
#pragma unroll
    for (int r = 0; r < NB; ++r)
      if (tid + r * NT < R * R) a.part[((int64_t)blockIdx.x * a.n_heads + e) * R * R + tid + r * NT] = acc[r];
  }
}

// 8x8 windows: the products on m16n8k8 TF32 MMAs with the 3-pass hi/lo split, like window_attention_mma_kernel.  4 warps;
// warp w owns query rows [16 w, 16 w + 16) for S, dP, dS and dQ (P, dP, D and dS never leave registers: the C fragment of
// dP = dO V^T has the layout of S, and dS is then the A fragment of dS K with the forward's key-slot order), and key rows
// [16 w, 16 w + 16) for dK = dS^T Q and dV = P^T dO, whose A operands go through shared memory transposed.  Q, K, V, dO
// of the head sit in shared memory as fp32 (split into hi / lo at fragment load).
template <int HD>
__host__ __device__ constexpr int wattn_bwd_mma_smem_floats() { return 4 * 64 * (HD + 4) + 2 * 64 * 72 + 228; }

__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) { hi = to_tf32(v); lo = to_tf32(v - hi); }

// d += a b, 3 passes (a_lo b_hi + a_hi b_lo + a_hi b_hi)
__device__ __forceinline__ void mma3_tf32(float (&d)[4], const float (&ah)[4], const float (&al)[4], float b0, float b1) {
  float bh0, bl0, bh1, bl1;
  split_tf32(b0, bh0, bl0);
  split_tf32(b1, bh1, bl1);
  mma_tf32_16x8x8(d, al, bh0, bh1);
  mma_tf32_16x8x8(d, ah, bl0, bl1);
  mma_tf32_16x8x8(d, ah, bh0, bh1);
}

template <int HD>
__global__ void __launch_bounds__(128) window_attention_bwd_mma_kernel(const WinBwdArgs a) {
  constexpr int P = 8, PP = 64, R = 2 * P - 1, LDS = HD + 4, LDT = 72, KSTEPS = HD / 8, NT = 128;
  extern __shared__ __align__(16) float smem[];
  float* sq = smem;
  float* sk = sq + PP * LDS;
  float* sv = sk + PP * LDS;
  float* sdo = sv + PP * LDS;
  float* spT = sdo + PP * LDS;             // P transposed: P[i][j] at j * LDT + i
  float* sdsT = spT + PP * LDT;            // dS transposed
  float* sbias = sdsT + PP * LDT;          // R * R (228 floats keep stok 16-byte aligned)
  int64_t* stok = reinterpret_cast<int64_t*>(sbias + 228);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int r0 = 16 * warp + g, r1 = r0 + 8;          // this thread's query rows (and key rows in the dK / dV phase)
  const int py0 = 2 * warp, px = g, sp_edge = P - a.shift;
  for (int e = 0; e < a.n_heads; ++e) {
    float acc[2] = {0.f, 0.f};
    for (int64_t win = blockIdx.x; win < a.n_win; win += gridDim.x) {
      __syncthreads();
      int wy, wx;
      window_tokens<P>(a, win, stok, wy, wx);
      for (int i = tid; i < R * R; i += NT) sbias[i] = __ldg(a.rel + (int64_t)e * R * R + i);
      __syncthreads();
      for (int idx = tid; idx < PP * (HD / 4); idx += NT) {
        const int tk = idx / (HD / 4), d4 = idx - tk * (HD / 4);
        const float* row = a.qkv + stok[tk] * a.ld + e * HD + 4 * d4;
        *reinterpret_cast<float4*>(sq + tk * LDS + 4 * d4) = __ldg(reinterpret_cast<const float4*>(row + a.q_col));
        *reinterpret_cast<float4*>(sk + tk * LDS + 4 * d4) = __ldg(reinterpret_cast<const float4*>(row + a.k_col));
        *reinterpret_cast<float4*>(sv + tk * LDS + 4 * d4) = __ldg(reinterpret_cast<const float4*>(row + a.v_col));
        *reinterpret_cast<float4*>(sdo + tk * LDS + 4 * d4) =
            __ldg(reinterpret_cast<const float4*>(a.dout + stok[tk] * a.dout_ld + e * HD + 4 * d4));
      }
      __syncthreads();
      // S = Q K^T and dP = dO V^T (C fragment: c0 = (g, 2t), c1 = (g, 2t + 1), c2 = (g + 8, 2t), c3 = (g + 8, 2t + 1) of key tile nt)
      float sc[8][4], dp[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { sc[nt][i] = 0.f; dp[nt][i] = 0.f; }
      }
#pragma unroll
      for (int ks = 0; ks < KSTEPS; ++ks) {
        float qh[4], ql[4], oh[4], ol[4];
        const int c = 8 * ks + t;
        const float qa[4] = {sq[r0 * LDS + c], sq[r1 * LDS + c], sq[r0 * LDS + c + 4], sq[r1 * LDS + c + 4]};
        const float oa[4] = {sdo[r0 * LDS + c], sdo[r1 * LDS + c], sdo[r0 * LDS + c + 4], sdo[r1 * LDS + c + 4]};
#pragma unroll
        for (int i = 0; i < 4; ++i) { split_tf32(qa[i], qh[i], ql[i]); split_tf32(oa[i], oh[i], ol[i]); }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int o = (8 * nt + g) * LDS + c;
          mma3_tf32(sc[nt], qh, ql, sk[o], sk[o + 4]);
          mma3_tf32(dp[nt], oh, ol, sv[o], sv[o + 4]);
        }
      }
      const bool last_row = a.shift > 0 && wy == a.nwy - 1, last_col = a.shift > 0 && wx == a.nwx - 1;
      float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = i >> 1, qx = 2 * t + (i & 1), py = py0 + r, qy = nt;
          const float v = sc[nt][i] * a.scale + sbias[(py - qy + P - 1) * R + (px - qx + P - 1)];
          const bool masked = (last_row && ((py < sp_edge) != (qy < sp_edge))) || (last_col && ((px < sp_edge) != (qx < sp_edge)));
          sc[nt][i] = masked ? -INFINITY : v;
        }
        m0 = fmaxf(m0, fmaxf(sc[nt][0], sc[nt][1]));
        m1 = fmaxf(m1, fmaxf(sc[nt][2], sc[nt][3]));
      }
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        sc[nt][0] = expf(sc[nt][0] - m0); sc[nt][1] = expf(sc[nt][1] - m0);
        sc[nt][2] = expf(sc[nt][2] - m1); sc[nt][3] = expf(sc[nt][3] - m1);
        s0 += sc[nt][0] + sc[nt][1];
        s1 += sc[nt][2] + sc[nt][3];
      }
      s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
      const float i0 = 1.0f / s0, i1 = 1.0f / s1;
      float D0 = 0.f, D1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        sc[nt][0] *= i0; sc[nt][1] *= i0; sc[nt][2] *= i1; sc[nt][3] *= i1;
        D0 = fmaf(sc[nt][0], dp[nt][0], fmaf(sc[nt][1], dp[nt][1], D0));
        D1 = fmaf(sc[nt][2], dp[nt][2], fmaf(sc[nt][3], dp[nt][3], D1));
      }
      D0 += __shfl_xor_sync(0xffffffffu, D0, 1); D0 += __shfl_xor_sync(0xffffffffu, D0, 2);
      D1 += __shfl_xor_sync(0xffffffffu, D1, 1); D1 += __shfl_xor_sync(0xffffffffu, D1, 2);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        dp[nt][0] = sc[nt][0] * (dp[nt][0] - D0); dp[nt][1] = sc[nt][1] * (dp[nt][1] - D0);
        dp[nt][2] = sc[nt][2] * (dp[nt][2] - D1); dp[nt][3] = sc[nt][3] * (dp[nt][3] - D1);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int key = 8 * nt + 2 * t + (i & 1), q = (i >> 1) ? r1 : r0;
          spT[key * LDT + q] = sc[nt][i];
          sdsT[key * LDT + q] = dp[nt][i];
        }
      }
      // dQ = s dS K: k-step j = key tile j, slot t <-> key 8j + 2t, slot t + 4 <-> key 8j + 2t + 1 (A = (c0, c2, c1, c3) of dS)
      {
        float gq[KSTEPS][4];
#pragma unroll
        for (int nd = 0; nd < KSTEPS; ++nd) {
#pragma unroll
          for (int i = 0; i < 4; ++i) gq[nd][i] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float av[4] = {dp[j][0], dp[j][2], dp[j][1], dp[j][3]};
          float ah[4], al[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) split_tf32(av[i], ah[i], al[i]);
#pragma unroll
          for (int nd = 0; nd < KSTEPS; ++nd) {
            const int o = (8 * j + 2 * t) * LDS + 8 * nd + g;
            mma3_tf32(gq[nd], ah, al, sk[o], sk[o + LDS]);
          }
        }
#pragma unroll
        for (int nd = 0; nd < KSTEPS; ++nd) {
          const int col = a.q_col + e * HD + 8 * nd + 2 * t;
          *reinterpret_cast<float2*>(a.dqkv + stok[r0] * a.dqkv_ld + col) = make_float2(gq[nd][0] * a.scale, gq[nd][1] * a.scale);
          *reinterpret_cast<float2*>(a.dqkv + stok[r1] * a.dqkv_ld + col) = make_float2(gq[nd][2] * a.scale, gq[nd][3] * a.scale);
        }
      }
      __syncthreads();                     // P^T and dS^T complete
      // dV = P^T dO and dK = s dS^T Q for key rows r0 / r1: k-step ks over queries, slot t <-> query 8ks + 2t, t + 4 <-> 8ks + 2t + 1
      {
        float gk[KSTEPS][4], gv[KSTEPS][4];
#pragma unroll
        for (int nd = 0; nd < KSTEPS; ++nd) {
#pragma unroll
          for (int i = 0; i < 4; ++i) { gk[nd][i] = 0.f; gv[nd][i] = 0.f; }
        }
#pragma unroll 2
        for (int ks = 0; ks < 8; ++ks) {
          const int c = 8 * ks + 2 * t;
          const float pa[4] = {spT[r0 * LDT + c], spT[r1 * LDT + c], spT[r0 * LDT + c + 1], spT[r1 * LDT + c + 1]};
          const float da[4] = {sdsT[r0 * LDT + c], sdsT[r1 * LDT + c], sdsT[r0 * LDT + c + 1], sdsT[r1 * LDT + c + 1]};
          float ph[4], pl[4], dh[4], dl[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) { split_tf32(pa[i], ph[i], pl[i]); split_tf32(da[i], dh[i], dl[i]); }
#pragma unroll
          for (int nd = 0; nd < KSTEPS; ++nd) {
            const int o = c * LDS + 8 * nd + g;
            mma3_tf32(gv[nd], ph, pl, sdo[o], sdo[o + LDS]);
            mma3_tf32(gk[nd], dh, dl, sq[o], sq[o + LDS]);
          }
        }
#pragma unroll
        for (int nd = 0; nd < KSTEPS; ++nd) {
          const int cd = e * HD + 8 * nd + 2 * t;
          float* o0 = a.dqkv + stok[r0] * a.dqkv_ld + cd;
          float* o1 = a.dqkv + stok[r1] * a.dqkv_ld + cd;
          *reinterpret_cast<float2*>(o0 + a.k_col) = make_float2(gk[nd][0] * a.scale, gk[nd][1] * a.scale);
          *reinterpret_cast<float2*>(o1 + a.k_col) = make_float2(gk[nd][2] * a.scale, gk[nd][3] * a.scale);
          *reinterpret_cast<float2*>(o0 + a.v_col) = make_float2(gv[nd][0], gv[nd][1]);
          *reinterpret_cast<float2*>(o1 + a.v_col) = make_float2(gv[nd][2], gv[nd][3]);
        }
      }
      acc[0] += rel_bin_sum<P>(sdsT, LDT, tid);
      if (tid + NT < R * R) acc[1] += rel_bin_sum<P>(sdsT, LDT, tid + NT);
    }
    float* part = a.part + ((int64_t)blockIdx.x * a.n_heads + e) * R * R;
    part[tid] = acc[0];
    if (tid + NT < R * R) part[tid + NT] = acc[1];
  }
}

// drel[i] = sum over blocks b in order of part[b][i]
__global__ void __launch_bounds__(256) rel_partials_reduce_kernel(const float* __restrict__ part, int n_blocks, int n, float* __restrict__ drel) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int b = 0; b < n_blocks; ++b) s += part[(int64_t)b * n + i];
  drel[i] = s;
}

// ---------------------------------------------------------------------------------------------
// space-to-depth: out[(b, y', x'), (sy*2 + sx) * Cs + c] = x[(b, 2y' + sy, 2x' + sx), c]  (0 outside / for c >= C)
// depth-to-space: out[(b, 2y + py, 2x + px), c] = x[(b, y, x), (py*2 + px) * Cs + c]     (0 for C <= c < Cpad)
// one thread per output float4 (scalar variant when a channel count is not a multiple of 4)
// ---------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256) space_to_depth_kernel(const float* __restrict__ x, int64_t ld, int C, int Cs, int B, int h, int w,
                                                             int h2, int w2, float* __restrict__ out, int64_t out_ld, const dcae_planes o16) {
  const int cv = Cs / VEC;                     // vectors per sub-pixel slot
  const int64_t n = (int64_t)B * h2 * w2 * 4 * cv;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * VEC;
    int64_t r = idx / cv;
    const int sub = (int)(r & 3); r >>= 2;
    const int x2 = (int)(r % w2); r /= w2;
    const int y2 = (int)(r % h2);
    const int b = (int)(r / h2);
    const int yy = 2 * y2 + (sub >> 1), xx = 2 * x2 + (sub & 1);
    const int64_t ot = ((int64_t)b * h2 + y2) * w2 + x2;
    const bool in = yy < h && xx < w;
    const float* src = x + (((int64_t)b * h + yy) * w + xx) * ld + c;
    if (VEC == 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (in && c + 3 < C) v = __ldg(reinterpret_cast<const float4*>(src));
      else if (in && c < C) { v.x = __ldg(src); if (c + 1 < C) v.y = __ldg(src + 1); if (c + 2 < C) v.z = __ldg(src + 2); }
      if (out) *reinterpret_cast<float4*>(out + ot * out_ld + sub * Cs + c) = v;
      if (o16.hi) store_planes4(o16, ot, sub * Cs + c, v);
    } else {
      const float v = (in && c < C) ? __ldg(src) : 0.f;
      if (out) out[ot * out_ld + sub * Cs + c] = v;
      if (o16.hi) store_plane1(o16, ot, sub * Cs + c, v);
    }
  }
}

template <int VEC>
__global__ void __launch_bounds__(256) depth_to_space_kernel(const float* __restrict__ x, int64_t ld, int Cs, int C, int Cpad, int B, int h, int w,
                                                             float* __restrict__ out, int64_t out_ld, const dcae_planes o16) {
  const int cv = Cpad / VEC;
  const int H = 2 * h, W = 2 * w;
  const int64_t n = (int64_t)B * H * W * cv;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * VEC;
    int64_t r = idx / cv;
    const int X = (int)(r % W); r /= W;
    const int Y = (int)(r % H);
    const int b = (int)(r / H);
    const int sub = (Y & 1) * 2 + (X & 1);
    const float* src = x + (((int64_t)b * h + (Y >> 1)) * w + (X >> 1)) * ld + sub * Cs + c;
    const int64_t ot = ((int64_t)b * H + Y) * W + X;
    if (VEC == 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c + 3 < C) v = __ldg(reinterpret_cast<const float4*>(src));
      else if (c < C) { v.x = __ldg(src); if (c + 1 < C) v.y = __ldg(src + 1); if (c + 2 < C) v.z = __ldg(src + 2); }
      if (out) *reinterpret_cast<float4*>(out + ot * out_ld + c) = v;
      if (o16.hi) store_planes4(o16, ot, c, v);
    } else {
      const float v = c < C ? __ldg(src) : 0.f;
      if (out) out[ot * out_ld + c] = v;
      if (o16.hi) store_plane1(o16, ot, c, v);
    }
  }
}

inline unsigned grid_cap(int64_t n, int threads) {
  int64_t b = (n + threads - 1) / threads;
  const int64_t cap = (int64_t)num_sms() * 16;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

// called by dcae_op_layernorm (elementwise_kernels.cu) for channel counts its C % 128 == 0 kernel does not take
int layernorm_any(const float* x, int64_t x_ld, const float* gamma, const float* beta, int C, int64_t T, float* out, int64_t out_ld,
                  dcae_planes o16, cudaStream_t s) {
  DCAE_REQUIRE(C % 4 == 0 && C >= 4 && C <= 1024, "dcae_op_layernorm: C=%d must be a multiple of 4 in [4,1024]", C);
  const unsigned blocks = (unsigned)((T + 7) / 8);
  const int C4 = C / 4;
  switch ((C4 + 31) / 32) {
#define LN_CASE(V) case V: layernorm_any_kernel<V><<<blocks, 256, 0, s>>>(x, x_ld, gamma, beta, C4, T, out, out_ld, o16); break;
    LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(5) LN_CASE(6) LN_CASE(7) LN_CASE(8)
#undef LN_CASE
  }
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae

using namespace dcae;

extern "C" int dcae_op_window_attention(const float* qkv, int64_t ld, int32_t q_col, int32_t k_col, int32_t v_col, int32_t C,
                                        int32_t head_dim, int32_t window, int32_t shift, const float* rel_bias, int32_t B, int32_t h,
                                        int32_t w, float* out, int64_t out_ld, const dcae_planes* out16, void* stream) {
  ProfileScope prof(DCAE_PROF_ATTN, 4.0 * (double)B * h * w * (double)window * window * (double)C, stream);
  const dcae_planes o16 = planes_or_null(out16);
  DCAE_REQUIRE(qkv && rel_bias && (out || o16.hi) && planes_ok(out16), "dcae_op_window_attention: null pointer / bad planes");
  DCAE_REQUIRE((window == 4 || window == 8) && (head_dim == 8 || head_dim == 16 || head_dim == 32),
               "dcae_op_window_attention: window %d / head_dim %d not supported (window 4 or 8, head_dim 8, 16 or 32)", window, head_dim);
  DCAE_REQUIRE(C > 0 && C % head_dim == 0, "dcae_op_window_attention: C=%d is not a multiple of head_dim=%d", C, head_dim);
  DCAE_REQUIRE(B >= 0 && h > 0 && w > 0 && h % window == 0 && w % window == 0,
               "dcae_op_window_attention: the token grid %dx%d must be a multiple of the window %d (dcae.py:271)", h, w, window);
  DCAE_REQUIRE(shift == 0 || shift == window / 2, "dcae_op_window_attention: shift must be 0 (W) or window/2 (SW)");
  DCAE_REQUIRE(q_col >= 0 && k_col >= 0 && v_col >= 0 && q_col + C <= ld && k_col + C <= ld && v_col + C <= ld && (!out || out_ld >= C),
               "dcae_op_window_attention: column windows exceed the leading dimension");
  DCAE_REQUIRE(B <= 65535, "dcae_op_window_attention: batch too large");
  DCAE_REQUIRE(aligned16(qkv) && ld % 4 == 0 && q_col % 4 == 0 && k_col % 4 == 0 && v_col % 4 == 0 && aligned16(out) && out_ld % 4 == 0,
               "dcae_op_window_attention: qkv / out must be 16-byte aligned with ld and column offsets multiples of 4");
  if (B == 0) return DCAE_OK;
  WinArgs a;
  a.qkv = qkv; a.ld = ld; a.q_col = q_col; a.k_col = k_col; a.v_col = v_col;
  a.n_heads = C / head_dim; a.shift = shift; a.B = B; a.h = h; a.w = w; a.nwx = w / window; a.nwy = h / window;
  a.rel = rel_bias; a.scale = 1.0f / sqrtf((float)head_dim);
  a.out = out; a.out_ld = out_ld; a.o16 = o16;
  const dim3 grid((unsigned)(a.nwx * a.nwy), (unsigned)B);
  cudaStream_t s = (cudaStream_t)stream;
  // 8x8 windows: the warp-MMA kernel (3 x TF32); 4x4 windows: the FFMA kernel
  if (window == 8) {
    if (head_dim == 8) window_attention_mma_kernel<8><<<grid, 128, 0, s>>>(a, C);
    else if (head_dim == 16) window_attention_mma_kernel<16><<<grid, 128, 0, s>>>(a, C);
    else window_attention_mma_kernel<32><<<grid, 128, 0, s>>>(a, C);
  } else {
    if (head_dim == 8) window_attention_kernel<8, 4><<<grid, 32, 0, s>>>(a);
    else if (head_dim == 16) window_attention_kernel<16, 4><<<grid, 32, 0, s>>>(a);
    else window_attention_kernel<32, 4><<<grid, 32, 0, s>>>(a);
  }
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" size_t dcae_window_attention_backward_scratch_bytes(int32_t B, int32_t h, int32_t w, int32_t C, int32_t head_dim, int32_t window) {
  if (B <= 0 || window <= 0 || head_dim <= 0 || C <= 0 || h < window || w < window) return 0;
  const int64_t n_win = (int64_t)B * (h / window) * (w / window);
  const int64_t R = 2 * window - 1;
  return (size_t)(wattn_bwd_blocks(n_win) * (C / head_dim) * R * R * (int64_t)sizeof(float));
}

extern "C" int dcae_op_window_attention_backward(const float* qkv, int64_t ld, int32_t q_col, int32_t k_col, int32_t v_col, int32_t C,
                                                 int32_t head_dim, int32_t window, int32_t shift, const float* rel_bias, int32_t B, int32_t h,
                                                 int32_t w, const float* dout, int64_t dout_ld, float* dqkv, int64_t dqkv_ld, float* drel,
                                                 void* scratch, size_t scratch_bytes, void* stream) {
  ProfileScope prof(DCAE_PROF_ATTN, 10.0 * B * h * w * (double)window * window * (double)C, stream);
  DCAE_REQUIRE(qkv && rel_bias && dout && dqkv && drel, "dcae_op_window_attention_backward: null pointer");
  DCAE_REQUIRE((window == 4 || window == 8) && (head_dim == 8 || head_dim == 16 || head_dim == 32),
               "dcae_op_window_attention_backward: window %d / head_dim %d not supported (window 4 or 8, head_dim 8, 16 or 32)", window, head_dim);
  DCAE_REQUIRE(C > 0 && C % head_dim == 0, "dcae_op_window_attention_backward: C=%d is not a multiple of head_dim=%d", C, head_dim);
  DCAE_REQUIRE(B >= 0 && h > 0 && w > 0 && h % window == 0 && w % window == 0,
               "dcae_op_window_attention_backward: the token grid %dx%d must be a multiple of the window %d", h, w, window);
  DCAE_REQUIRE(shift == 0 || shift == window / 2, "dcae_op_window_attention_backward: shift must be 0 (W) or window/2 (SW)");
  DCAE_REQUIRE(q_col >= 0 && k_col >= 0 && v_col >= 0 && q_col + C <= ld && k_col + C <= ld && v_col + C <= ld && q_col + C <= dqkv_ld &&
                   k_col + C <= dqkv_ld && v_col + C <= dqkv_ld && dout_ld >= C,
               "dcae_op_window_attention_backward: column windows exceed the leading dimension");
  DCAE_REQUIRE(abs(q_col - k_col) >= C && abs(q_col - v_col) >= C && abs(k_col - v_col) >= C,
               "dcae_op_window_attention_backward: the q / k / v column windows overlap");
  DCAE_REQUIRE(aligned16(qkv) && aligned16(dout) && aligned16(dqkv) && ld % 4 == 0 && dout_ld % 4 == 0 && dqkv_ld % 4 == 0 && q_col % 4 == 0 &&
                   k_col % 4 == 0 && v_col % 4 == 0,
               "dcae_op_window_attention_backward: qkv / dout / dqkv must be 16-byte aligned with ld and column offsets multiples of 4");
  DCAE_REQUIRE((int64_t)B * h * w < (1ll << 31), "dcae_op_window_attention_backward: too many tokens");
  if (B == 0) return DCAE_OK;
  const size_t need = dcae_window_attention_backward_scratch_bytes(B, h, w, C, head_dim, window);
  DCAE_REQUIRE(scratch && scratch_bytes >= need && aligned16(scratch),
               "dcae_op_window_attention_backward: scratch of %zu bytes (16-byte aligned) needed, %zu given", need, scratch ? scratch_bytes : (size_t)0);
  WinBwdArgs a;
  a.qkv = qkv; a.ld = ld; a.q_col = q_col; a.k_col = k_col; a.v_col = v_col;
  a.n_heads = C / head_dim; a.shift = shift; a.h = h; a.w = w; a.nwx = w / window; a.nwy = h / window;
  a.n_win = (int64_t)B * a.nwx * a.nwy;
  a.rel = rel_bias; a.scale = 1.0f / sqrtf((float)head_dim);
  a.dout = dout; a.dout_ld = dout_ld; a.dqkv = dqkv; a.dqkv_ld = dqkv_ld;
  a.part = static_cast<float*>(scratch);
  const int blocks = (int)wattn_bwd_blocks(a.n_win);
  cudaStream_t s = (cudaStream_t)stream;
  if (window == 8) {
#define WBWD_MMA(HD)                                                                                                     \
  {                                                                                                                      \
    constexpr int bytes = wattn_bwd_mma_smem_floats<HD>() * 4 + 64 * 8;                                                  \
    DCAE_CUDA(cudaFuncSetAttribute(window_attention_bwd_mma_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)); \
    window_attention_bwd_mma_kernel<HD><<<blocks, 128, bytes, s>>>(a);                                                   \
  }
    if (head_dim == 8) WBWD_MMA(8)
    else if (head_dim == 16) WBWD_MMA(16)
    else WBWD_MMA(32)
#undef WBWD_MMA
  } else {
    if (head_dim == 8) window_attention_bwd_kernel<8, 4><<<blocks, 128, 0, s>>>(a);
    else if (head_dim == 16) window_attention_bwd_kernel<16, 4><<<blocks, 128, 0, s>>>(a);
    else window_attention_bwd_kernel<32, 4><<<blocks, 128, 0, s>>>(a);
  }
  DCAE_LAUNCH_CHECK();
  const int n = a.n_heads * (2 * window - 1) * (2 * window - 1);
  rel_partials_reduce_kernel<<<(n + 255) / 256, 256, 0, s>>>(a.part, blocks, n, drel);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_op_space_to_depth(const float* x, int64_t ld, int32_t C, int32_t Cs, int32_t B, int32_t h, int32_t w, float* out,
                                      int64_t out_ld, const dcae_planes* out16, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const dcae_planes o16 = planes_or_null(out16);
  DCAE_REQUIRE(x && (out || o16.hi) && planes_ok(out16), "dcae_op_space_to_depth: null pointer / bad planes");
  DCAE_REQUIRE(C > 0 && Cs >= C && Cs % 4 == 0 && ld >= C && (!out || out_ld >= 4 * Cs) && (!o16.hi || o16.ld >= 4 * Cs) && out_ld % 4 == 0 && aligned16(out),
               "dcae_op_space_to_depth: need C <= Cs, Cs %% 4 == 0, out_ld >= 4 Cs (multiple of 4), 16-byte aligned output");
  DCAE_REQUIRE(B >= 0 && h > 0 && w > 0, "dcae_op_space_to_depth: bad token grid");
  const int h2 = (h + 1) / 2, w2 = (w + 1) / 2;
  const int64_t n4 = (int64_t)B * h2 * w2 * Cs;      // float4 outputs (4 sub-pixels x Cs / 4)
  if (n4 == 0) return DCAE_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (ld % 4 == 0 && aligned16(x))
    space_to_depth_kernel<4><<<grid_cap(n4, 256), 256, 0, s>>>(x, ld, C, Cs, B, h, w, h2, w2, out, out_ld, o16);
  else
    space_to_depth_kernel<1><<<grid_cap(n4 * 4, 256), 256, 0, s>>>(x, ld, C, Cs, B, h, w, h2, w2, out, out_ld, o16);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_op_depth_to_space(const float* x, int64_t ld, int32_t Cs, int32_t C, int32_t Cpad, int32_t B, int32_t h, int32_t w,
                                      float* out, int64_t out_ld, const dcae_planes* out16, void* stream) {
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const dcae_planes o16 = planes_or_null(out16);
  DCAE_REQUIRE(x && (out || o16.hi) && planes_ok(out16), "dcae_op_depth_to_space: null pointer / bad planes");
  DCAE_REQUIRE(C > 0 && Cs >= C && Cpad >= C && ld >= 4 * Cs && (!out || out_ld >= Cpad) && (!o16.hi || o16.ld >= Cpad),
               "dcae_op_depth_to_space: need C <= Cs, C <= Cpad <= out_ld, ld >= 4 Cs");
  DCAE_REQUIRE(B >= 0 && h > 0 && w > 0, "dcae_op_depth_to_space: bad token grid");
  const int64_t n = (int64_t)B * 4 * h * w * Cpad;
  if (n == 0) return DCAE_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (Cpad % 4 == 0 && Cs % 4 == 0 && ld % 4 == 0 && out_ld % 4 == 0 && aligned16(x) && aligned16(out))
    depth_to_space_kernel<4><<<grid_cap(n / 4, 256), 256, 0, s>>>(x, ld, Cs, C, Cpad, B, h, w, out, out_ld, o16);
  else
    depth_to_space_kernel<1><<<grid_cap(n, 256), 256, 0, s>>>(x, ld, Cs, C, Cpad, B, h, w, out, out_ld, o16);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
