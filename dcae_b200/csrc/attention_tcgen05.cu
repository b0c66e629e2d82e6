// Kernel 1: fused dictionary cross-attention core on tcgen05 / TMEM / TMA
// (/root/reference/models/dcae.py:489-501):
//   per head e (20 heads, 32 channels):  out[t, e, :] = softmax_j(q[t, e, :] . K[e, j, :] * scale_e) V[e, j, :]
// with 128 dictionary entries.  The reference materialises sim and probs ([B, 20, HW, 128], 10 KB per
// token) in HBM twice; here they never leave the SM:
//
//   TMA:      Q_e tile [128 tokens x 32] of the q buffer, K_e [128 x 32] and V_e^T [32 x 128] (hi/lo)
//   MMA 1:    S[128 x 128] = Q_e K_e^T            -> TMEM columns [0, 128)        (kind::tf32)
//   softmax:  one thread per token row: tcgen05.ld its 128 logits, scale, max, exp, sum -- all in
//             registers, no shuffles -- then P (hi/lo TF32 split) back to TMEM with tcgen05.st
//   MMA 2:    O[128 x 32] = P V_e   with the A operand read straight from TMEM, V_e^T from smem
//   epilogue: the same thread scales its O row by 1/sum and writes 128 contiguous bytes.
//
// PASSES == 3: error-compensated TF32 (q, k, p, v each split into hi + lo; 3 MMAs per product) so the
// result matches fp32 to ~1e-6; PASSES == 1: plain TF32.
// Warps: 0 = TMA, 1 = MMA issuer + TMEM owner, 2..5 = softmax (one row per thread), 6..9 = Q splitters.
// S(e+1) is issued while the softmax warps work on head e; all waits are bounded (trap, never hang).
#include "common.cuh"
#include "tc_common.cuh"

namespace dcae {

namespace {

constexpr int AT_M = 128;        // tokens per tile
constexpr int AT_HEADS = 20, AT_HD = 32, AT_ND = 128;
constexpr int AT_THREADS = 448;   // warps: 0 TMA, 1 MMA, 2-9 softmax (two column halves x four TMEM quarters), 10-13 Q splitters
constexpr int AT_TILE = AT_M * AT_HD * 4;   // 16 KB: every operand tile of a head has this size
constexpr int AT_MAX_STAGES = 4;
// TMEM columns
constexpr uint32_t TM_S = 0, TM_PHI = 128, TM_PLO = 256, TM_O = 384;

struct AtParams {
  const float* head_scale;
  dcae_planes out16;
  float* out;
  int64_t out_ld;
  int64_t T;
  int tiles, stages;
  uint32_t stage_bytes;
};

template <int PASSES>
__global__ void __launch_bounds__(AT_THREADS, 1)
dict_attention_tcgen05_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_khi,
                              const __grid_constant__ CUtensorMap map_klo, const __grid_constant__ CUtensorMap map_vhi,
                              const __grid_constant__ CUtensorMap map_vlo, const AtParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[AT_MAX_STAGES], ready_bar[AT_MAX_STAGES], empty_bar[AT_MAX_STAGES];
  __shared__ __align__(8) uint64_t s_full, s_free, p_ready, o_full;
  __shared__ uint32_t tmem_base_slot;
  __shared__ float xm[2][2][AT_M], xl[2][2][AT_M];    // row max / row sum of each column half, double-buffered by head parity

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp: provably uniform
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&ready_bar[s]), 128);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&s_full), 1);
    mbar_init(smem_u32(&s_free), 256);
    mbar_init(smem_u32(&p_ready), 256);
    mbar_init(smem_u32(&o_full), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc<1>(smem_u32(&tmem_base_slot), 512);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_slot;

  // stage layout: [Q(hi) | Q_lo | K_hi | K_lo | Vt_hi | Vt_lo]   (1-pass: [Q | K_hi | Vt_hi])
  const uint32_t off_qlo = AT_TILE;
  const uint32_t off_khi = (PASSES == 3) ? 2 * AT_TILE : AT_TILE;
  const uint32_t off_klo = off_khi + AT_TILE;
  const uint32_t off_vhi = (PASSES == 3) ? 4 * AT_TILE : 2 * AT_TILE;
  const uint32_t off_vlo = off_vhi + AT_TILE;
  const int my_tiles = (p.tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int total = my_tiles * AT_HEADS;     // (tile, head) work items of this CTA, in order

  if (warp == 0) {
    {
      // ===================== TMA producer (warp-uniform; one elected lane issues, see elect_one) =====================
      for (int g = 0; g < total; ++g) {
        const int stage = g % p.stages;
        const uint32_t phase = (g / p.stages) & 1;
        const int tile = blockIdx.x + (g / AT_HEADS) * gridDim.x, head = g % AT_HEADS;
        mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
        const uint32_t sb = smem0 + stage * p.stage_bytes;
        const uint32_t fb = smem_u32(&full_bar[stage]);
        if (elect_one()) {
          mbar_expect_tx(fb, (PASSES == 3 ? 5 : 3) * AT_TILE);
          tma_load_2d(sb, &map_q, fb, head * AT_HD, tile * AT_M);
          tma_load_2d(sb + off_khi, &map_khi, fb, 0, head * AT_ND);
          if (PASSES == 3) tma_load_2d(sb + off_klo, &map_klo, fb, 0, head * AT_ND);
#pragma unroll
          for (int c = 0; c < 4; ++c) {      // V^T [32 x 128] as four K-major [32 x 32] chunks
            tma_load_2d(sb + off_vhi + c * 4096, &map_vhi, fb, c * 32, head * AT_HD);
            if (PASSES == 3) tma_load_2d(sb + off_vlo + c * 4096, &map_vlo, fb, c * 32, head * AT_HD);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer (warp-uniform; one elected lane issues) =====================
      const uint32_t idesc_s = make_idesc_tf32(AT_M, AT_ND);    // S: N = 128
      const uint32_t idesc_o = make_idesc_tf32(AT_M, AT_HD);    // O: N = 32
      auto issue_s = [&](int g) {
        const int stage = g % p.stages;
        mbar_wait(smem_u32(PASSES == 3 ? &ready_bar[stage] : &full_bar[stage]), (g / p.stages) & 1);
        mbar_wait(smem_u32(&s_free), (g & 1) ^ 1);               // softmax warps hold S(g-1) in registers
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sb = smem0 + stage * p.stage_bytes;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < AT_HD / 8; ++k) {
            const uint32_t ko = k * 32;
            const uint64_t q_hi = make_smem_desc(sb + ko), k_hi = make_smem_desc(sb + off_khi + ko);
            if (PASSES == 3) {
              const uint64_t q_lo = make_smem_desc(sb + off_qlo + ko), k_lo = make_smem_desc(sb + off_klo + ko);
              mma_tf32(tmem + TM_S, q_lo, k_hi, idesc_s, k != 0);
              mma_tf32(tmem + TM_S, q_hi, k_lo, idesc_s, 1);
              mma_tf32(tmem + TM_S, q_hi, k_hi, idesc_s, 1);
            } else {
              mma_tf32(tmem + TM_S, q_hi, k_hi, idesc_s, k != 0);
            }
          }
          mma_commit(smem_u32(&s_full));
        }
        __syncwarp();
      };
      if (total > 0) issue_s(0);
      for (int g = 0; g < total; ++g) {
        if (g + 1 < total) issue_s(g + 1);                        // overlaps the softmax of head g
        const int stage = g % p.stages;
        const uint32_t sb = smem0 + stage * p.stage_bytes;
        mbar_wait(smem_u32(&p_ready), g & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < AT_ND / 8; ++j) {
            const uint32_t vo = (j >> 2) * 4096 + (j & 3) * 32;
            const uint64_t v_hi = make_smem_desc(sb + off_vhi + vo);
            if (PASSES == 3) {
              const uint64_t v_lo = make_smem_desc(sb + off_vlo + vo);
              mma_tf32_ts(tmem + TM_O, tmem + TM_PLO + j * 8, v_hi, idesc_o, j != 0);
              mma_tf32_ts(tmem + TM_O, tmem + TM_PHI + j * 8, v_lo, idesc_o, 1);
              mma_tf32_ts(tmem + TM_O, tmem + TM_PHI + j * 8, v_hi, idesc_o, 1);
            } else {
              mma_tf32_ts(tmem + TM_O, tmem + TM_PHI + j * 8, v_hi, idesc_o, j != 0);
            }
          }
          mma_commit(smem_u32(&empty_bar[stage]));
          mma_commit(smem_u32(&o_full));
        }
        __syncwarp();
      }
    }
  } else if (warp < 10) {
    // ===================== softmax warps: one token row per PAIR of threads =====================
    // Warp w and w + 4 own the same 32 TMEM lanes (rows); each takes 64 of the 128 dictionary columns, so every
    // scheduler has two softmax warps to alternate between and the unrolled body is half as long.  Row max and row
    // sum cross the pair through shared memory with one 64-thread named barrier per head.
    const int quarter = warp & 3, hf = (warp - 2) >> 2;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    constexpr int HC = AT_ND / 2;     // columns per thread
    auto pair_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory"); };
    // O(g-1) is read back only after the exponentials of head g are done, so the PV MMAs of head g-1 run
    // underneath the softmax arithmetic of head g (and S(g+1) underneath that of head g, see the MMA warp).
    // Each thread of the pair writes 16 of the head's 32 output columns.
    auto write_out = [&](int g) {
      const int tile = blockIdx.x + (g / AT_HEADS) * gridDim.x, head = g % AT_HEADS;
      const float inv = 1.0f / (xl[g & 1][0][r] + xl[g & 1][1][r]);
      mbar_wait(smem_u32(&o_full), g & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      uint32_t o0[16];
      tmem_ld16_nowait(lane_addr + TM_O + hf * 16, o0);
      tmem_ld_wait();
      const int64_t token = (int64_t)tile * AT_M + r;
      if (token < p.T) {
        const int col = head * AT_HD + hf * 16;
        float4* dst = p.out ? reinterpret_cast<float4*>(p.out + token * p.out_ld + col) : nullptr;
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 a = make_float4(__uint_as_float(o0[j]) * inv, __uint_as_float(o0[j + 1]) * inv,
                                       __uint_as_float(o0[j + 2]) * inv, __uint_as_float(o0[j + 3]) * inv);
          if (dst) dst[j / 4] = a;
          if (p.out16.hi) store_planes4(p.out16, token, col + j, a);
        }
      }
    };
    for (int g = 0; g < total; ++g) {
      const int head = g % AT_HEADS;
      // softmax(sim * scale) = 2^(t - max t) / sum with t = sim * (scale * log2 e): one FMUL, one FADD and one MUFU.EX2
      // per element (ex2.approx: 2^-22 relative); max and sum as 8 independent chains.
      const float sc = __ldg(p.head_scale + head) * 1.4426950408889634f;
      mbar_wait(smem_u32(&s_full), g & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      float s[HC];
      {
        uint32_t raw[HC];
#pragma unroll
        for (int c = 0; c < HC / 16; ++c) tmem_ld16_nowait(lane_addr + TM_S + hf * HC + c * 16, raw + c * 16);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < HC; ++j) s[j] = __uint_as_float(raw[j]) * sc;   // sim * scale (dcae.py:498), log2 domain
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(smem_u32(&s_free));                           // S may be overwritten by head g+1
      float m8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) m8[j] = s[j];
#pragma unroll
      for (int j = 8; j < HC; ++j) m8[j & 7] = fmaxf(m8[j & 7], s[j]);
      float mx = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
      xm[g & 1][hf][r] = mx;
      pair_sync();                                              // also orders xl(g-1) of the partner before write_out(g-1)
      mx = fmaxf(mx, xm[g & 1][hf ^ 1][r]);
      float l8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < HC; ++j) {
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(s[j] - mx));
        s[j] = e;
        l8[j & 7] += e;
      }
      if (g > 0) write_out(g - 1);                              // also guarantees PV(g-1) has finished reading P
      xl[g & 1][hf][r] = ((l8[0] + l8[1]) + (l8[2] + l8[3])) + ((l8[4] + l8[5]) + (l8[6] + l8[7]));
#pragma unroll
      for (int c = 0; c < HC / 16; ++c) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float e = s[c * 16 + j];
          const float h = (PASSES == 3) ? tf32_rna(e) : e;
          hi[j] = __float_as_uint(h);
          lo[j] = __float_as_uint(tf32_rna(e - h));
        }
        tmem_st16(lane_addr + TM_PHI + hf * HC + c * 16, hi);
        if (PASSES == 3) tmem_st16(lane_addr + TM_PLO + hf * HC + c * 16, lo);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(smem_u32(&p_ready));
    }
    if (total > 0) {
      pair_sync();
      write_out(total - 1);
    }
  } else {
    // ===================== Q splitters (3-pass): q -> (q_hi in place, q_lo) =====================
    if (PASSES == 3) {
      const int st = threadIdx.x - 320;   // 0..127
      for (int g = 0; g < total; ++g) {
        const int stage = g % p.stages;
        mbar_wait(smem_u32(&full_bar[stage]), (g / p.stages) & 1);
        const uint32_t sb = smem0 + stage * p.stage_bytes;
#pragma unroll
        for (int i = 0; i < AT_TILE / 16 / 128; ++i) {
          const uint32_t off = (uint32_t)(st + i * 128) * 16;
          float4 v;
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(sb + off));
          float4 hi, lo;
          hi.x = tf32_rna(v.x); hi.y = tf32_rna(v.y); hi.z = tf32_rna(v.z); hi.w = tf32_rna(v.w);
          lo.x = tf32_rna(v.x - hi.x); lo.y = tf32_rna(v.y - hi.y); lo.z = tf32_rna(v.z - hi.z); lo.w = tf32_rna(v.w - hi.w);
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sb + off), "f"(hi.x), "f"(hi.y), "f"(hi.z), "f"(hi.w) : "memory");
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sb + off_qlo + off), "f"(lo.x), "f"(lo.y), "f"(lo.z), "f"(lo.w) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(smem_u32(&ready_bar[stage]));
      }
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) tmem_dealloc<1>(tmem, 512);
}

}  // namespace

int dict_attention_tcgen05(const float* q, int64_t q_ld, const dcae_dict_kv* kv, int64_t T, float* out, int64_t out_ld,
                           dcae_planes out16, int passes, cudaStream_t s) {
  DCAE_REQUIRE(kv->Kh_hi && kv->Vt_hi && (passes == 1 || (kv->Kh_lo && kv->Vt_lo)),
               "dict_attention(tcgen05): dictionary K/V have no TF32 split (Kh_hi/Kh_lo/Vt_hi/Vt_lo)");
  if (T == 0) return DCAE_OK;
  AtParams p;
  p.head_scale = kv->head_scale;
  p.out = out; p.out_ld = out_ld; p.T = T;
  p.out16 = out16;
  p.tiles = (int)((T + AT_M - 1) / AT_M);
  p.stage_bytes = (passes == 3 ? 6 : 3) * AT_TILE;
  p.stages = (passes == 3) ? 2 : 4;
  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024;
  CUtensorMap mq, mkh, mkl, mvh, mvl;
  {
    cuuint64_t dims[2] = {(cuuint64_t)q_ld, (cuuint64_t)T};
    cuuint64_t str[1] = {(cuuint64_t)q_ld * 4};
    cuuint32_t box[2] = {AT_HD, AT_M};
    DCAE_TRY(encode_map(&mq, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, q, 2, dims, str, box));
  }
  {
    cuuint64_t dims[2] = {AT_HD, (cuuint64_t)AT_HEADS * AT_ND};
    cuuint64_t str[1] = {AT_HD * 4};
    cuuint32_t box[2] = {AT_HD, AT_ND};
    DCAE_TRY(encode_map(&mkh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, kv->Kh_hi, 2, dims, str, box));
    if (passes == 3) DCAE_TRY(encode_map(&mkl, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, kv->Kh_lo, 2, dims, str, box)); else mkl = mkh;
  }
  {
    cuuint64_t dims[2] = {AT_ND, (cuuint64_t)AT_HEADS * AT_HD};
    cuuint64_t str[1] = {AT_ND * 4};
    cuuint32_t box[2] = {32, AT_HD};
    DCAE_TRY(encode_map(&mvh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, kv->Vt_hi, 2, dims, str, box));
    if (passes == 3) DCAE_TRY(encode_map(&mvl, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, kv->Vt_lo, 2, dims, str, box)); else mvl = mvh;
  }
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(dict_attention_tcgen05_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(dict_attention_tcgen05_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  });
  DCAE_CUDA(attr_err);
  const int ctas = p.tiles < num_sms() ? p.tiles : num_sms();
  if (passes == 3) dict_attention_tcgen05_kernel<3><<<ctas, AT_THREADS, smem, s>>>(mq, mkh, mkl, mvh, mvl, p);
  else dict_attention_tcgen05_kernel<1><<<ctas, AT_THREADS, smem, s>>>(mq, mkh, mkl, mvh, mvl, p);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae
