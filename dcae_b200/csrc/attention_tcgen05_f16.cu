// Kernel 1, fp16-plane variant (DCAE_MATH_F16X3): fused dictionary cross-attention core on tcgen05 / TMEM / TMA
// (/root/reference/models/dcae.py:489-501):
//   per head e (20 heads, 32 channels):  out[t, e, :] = softmax_j(q[t, e, :] . K[e, j, :] * scale_e) V[e, j, :]
// with 128 dictionary entries; sim / probs never leave the SM.
//
// Same 22-bit hi/lo arithmetic as the f16x3 GEMM (kind::f16, 3 MMAs per product), fed by planes:
//   q planes   : written by the q_trans GEMM epilogue (no in-kernel split warps)
//   K planes   : k(LN(dt)) as it is, [128 entries, 640]: a 128-byte row holds the 32 dims of TWO heads, so one
//                SWIZZLE_128B box {64, 128} is the K tile of a head pair and head e uses the k-steps 2(e&1), 2(e&1)+1
//   V^T planes : LN(dt)^T [640, 128 entries]; box {64 entries, 64 rows} x 2 chunks per head pair
// Against the TF32 kernel: half the operand bytes per head (48 instead of 96 KB), so four heads are in flight
// instead of two; half the MMA instructions; P is stored as packed fp16 hi/lo INTO the columns of the S it came
// from, which leaves room to double-buffer S/P and O in TMEM (2 x 128 + 2 x 32 columns) -- QK(g+2) is issued right
// behind PV(g) with no barrier in between (one issuing thread, in-order tensor pipe).
//
//   S[128 x 128] = Q_e K_e^T                      2 k-steps x 3 passes, TMEM buffer g & 1
//   softmax       TWO warp groups in ping-pong: group 0 owns the even head steps (S/P buffer 0, O buffer 0), group 1 the
//                 odd ones, so the dependent chain of one head (TMEM load -> max -> exchange -> ex2 -> pack -> TMEM store)
//                 overlaps the other head's instead of following it (the chain, not a pipe, set the 5.3 k-cycle head
//                 step: 8 and 16 warps on ONE head measured the same).  Inside a group two threads per token row
//                 (64 columns each), log2-domain, ex2.approx; P' = 1024 * 2^(t - max) so that p_lo stays a normal fp16;
//                 the factor cancels against the row sum
//   O[128 x 32]  = P V_e                           8 k-steps x 3 passes, A operand (P) straight from TMEM
//   epilogue      each thread of the pair scales 16 of the 32 O columns by descale_v / sum and writes them
// Warps: 0 = TMA, 1 = MMA issuer + TMEM owner, 2..9 = softmax group 0, 10..17 = softmax group 1.  All waits are bounded
// (trap, never hang).
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_common.cuh"

#include <mutex>

namespace dcae {

namespace {

constexpr int AF_M = 128;                         // tokens per tile
constexpr int AF_HEADS = 20, AF_HD = 32, AF_ND = 128;
constexpr int AF_SUB = 2;                         // softmax threads per token row inside a group (column halves of 64)
constexpr int AF_GROUPS = 2;                      // ping-pong softmax groups: group = head step & 1
constexpr int AF_THREADS = 64 + AF_GROUPS * AF_SUB * 128;     // warps 0 TMA, 1 MMA, then AF_GROUPS x AF_SUB x 4 softmax warps
constexpr int AF_QK_BYTES = AF_M * 128;           // 16 KB: a [128 x 64 halfs] tile (Q or K of a head pair, one plane)
constexpr int AF_V_BYTES = 64 * 128;              // 8 KB: V^T chunk [64 rows (2 heads x 32 dims) x 64 entries], one plane
constexpr int AF_STAGE = 4 * AF_QK_BYTES + 4 * AF_V_BYTES;   // 96 KB per head PAIR
constexpr int AF_STAGES = 2;
// TMEM columns: S/P buffers at 0 and 128, O buffers at 256 and 288
constexpr uint32_t TF_SP = 0, TF_O = 256;

struct AfParams {
  const float* head_scale;
  dcae_planes out16;
  float* out;
  int64_t out_ld;
  int64_t T;
  int tiles;
  float k_descale, v_descale;
};

__global__ void __launch_bounds__(AF_THREADS, 1)
dict_attention_f16_kernel(const __grid_constant__ CUtensorMap map_qh, const __grid_constant__ CUtensorMap map_ql,
                          const __grid_constant__ CUtensorMap map_kh, const __grid_constant__ CUtensorMap map_kl,
                          const __grid_constant__ CUtensorMap map_vh, const __grid_constant__ CUtensorMap map_vl, const AfParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[AF_STAGES], empty_bar[AF_STAGES];
  __shared__ __align__(8) uint64_t s_full[2], p_ready[2], o_full[2], o_free[2];
  __shared__ uint32_t tmem_base_slot;
  // row max of each column range per group; row sums double-buffered by the group's own step parity (write_out of the
  // previous head reads them while the current head's are written)
  __shared__ float xm[AF_GROUPS][AF_SUB][AF_M], xl[AF_GROUPS][2][AF_SUB][AF_M];

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp: provably uniform
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;

  if (threadIdx.x == 0) {
    for (int s = 0; s < AF_STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&s_full[b]), 1);
      mbar_init(smem_u32(&p_ready[b]), AF_SUB * 128);
      mbar_init(smem_u32(&o_full[b]), 1);
      mbar_init(smem_u32(&o_free[b]), AF_SUB * 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc<1>(smem_u32(&tmem_base_slot), 512);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_slot;

  // stage (one head pair): [Q_hi | Q_lo | K_hi | K_lo | Vt_hi chunk0, chunk1 | Vt_lo chunk0, chunk1]
  constexpr uint32_t OFF_QL = AF_QK_BYTES, OFF_KH = 2 * AF_QK_BYTES, OFF_KL = 3 * AF_QK_BYTES;
  constexpr uint32_t OFF_VH = 4 * AF_QK_BYTES, OFF_VL = OFF_VH + 2 * AF_V_BYTES;
  // Work item = one HEAD PAIR of one tile (1 920 items at config #2, 13 per CTA): splitting at tile granularity
  // leaves 192 tiles on 148 SMs, i.e. 44 CTAs with two tiles and 104 with one.  Item i of this CTA is the global
  // pair blockIdx.x + i * gridDim.x -> (tile, head pair); the head-step pipeline runs across items unchanged.
  constexpr int HP = AF_HEADS / 2;
  const int all_pairs = p.tiles * HP;
  const int my_pairs = (all_pairs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int total = my_pairs * 2;            // head steps of this CTA, in order; always even

  if (warp == 0) {
    {
      // ===================== TMA producer: one stage per head pair (warp-uniform, one elected lane issues) =====================
      for (int pr = 0; pr < total / 2; ++pr) {
        const int stage = pr % AF_STAGES;
        const uint32_t phase = (pr / AF_STAGES) & 1;
        const int gp = (int)blockIdx.x + pr * (int)gridDim.x;
        const int tile = gp / HP, hp = gp % HP;
        mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
        const uint32_t sb = smem0 + stage * AF_STAGE;
        const uint32_t fb = smem_u32(&full_bar[stage]);
        if (elect_one()) {
          mbar_expect_tx(fb, AF_STAGE);
          tma_load_2d(sb, &map_qh, fb, hp * 64, tile * AF_M);
          tma_load_2d(sb + OFF_QL, &map_ql, fb, hp * 64, tile * AF_M);
          tma_load_2d(sb + OFF_KH, &map_kh, fb, hp * 64, 0);
          tma_load_2d(sb + OFF_KL, &map_kl, fb, hp * 64, 0);
#pragma unroll
          for (int c = 0; c < 2; ++c) {      // V^T rows of the pair, entries 64c .. 64c + 63
            tma_load_2d(sb + OFF_VH + c * AF_V_BYTES, &map_vh, fb, c * 64, hp * 64);
            tma_load_2d(sb + OFF_VL + c * AF_V_BYTES, &map_vl, fb, c * 64, hp * 64);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer (warp-uniform, one elected lane issues) =====================
      const uint32_t idesc_s = make_idesc_f16(AF_M, AF_ND);     // S: N = 128
      const uint32_t idesc_o = make_idesc_f16(AF_M, AF_HD);     // O: N = 32
      auto issue_s = [&](int g) {                                 // S(g) -> buffer g & 1
        const int pr = g >> 1, stage = pr % AF_STAGES;
        if ((g & 1) == 0) mbar_wait(smem_u32(&full_bar[stage]), (pr / AF_STAGES) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sb = smem0 + stage * AF_STAGE;
        const uint32_t d = tmem + TF_SP + (uint32_t)(g & 1) * 128;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const uint32_t ko = (uint32_t)((g & 1) * 2 + k) * 32;    // this head's 32 dims inside the pair's 128-byte rows
            const uint64_t q_hi = make_smem_desc(sb + ko), q_lo = make_smem_desc(sb + OFF_QL + ko);
            const uint64_t k_hi = make_smem_desc(sb + OFF_KH + ko), k_lo = make_smem_desc(sb + OFF_KL + ko);
            mma_f16(d, q_lo, k_hi, idesc_s, k != 0);
            mma_f16(d, q_hi, k_lo, idesc_s, 1);
            mma_f16(d, q_hi, k_hi, idesc_s, 1);
          }
          mma_commit(smem_u32(&s_full[g & 1]));
        }
        __syncwarp();
      };
      if (total > 0) { issue_s(0); issue_s(1); }
      for (int g = 0; g < total; ++g) {
        const int b = g & 1, pr = g >> 1, stage = pr % AF_STAGES;
        const uint32_t sb = smem0 + stage * AF_STAGE;
        mbar_wait(smem_u32(&p_ready[b]), (g >> 1) & 1);
        if (g >= 2) mbar_wait(smem_u32(&o_free[b]), ((g >> 1) & 1) ^ 1);      // O(g-2) has been read back
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t pa = tmem + TF_SP + (uint32_t)b * 128;                  // P_hi words at +0, P_lo words at +64
        const uint32_t od = tmem + TF_O + (uint32_t)b * 32;
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < AF_ND / 16; ++j) {
            // V^T rows of this head: 32 rows = 4 KB into the pair's chunk; k-step j: chunk j >> 2, 32 bytes per step
            const uint32_t vo = (uint32_t)(j >> 2) * AF_V_BYTES + (uint32_t)b * 4096 + (uint32_t)(j & 3) * 32;
            const uint64_t v_hi = make_smem_desc(sb + OFF_VH + vo), v_lo = make_smem_desc(sb + OFF_VL + vo);
            mma_f16_ts(od, pa + 64 + j * 8, v_hi, idesc_o, j != 0);
            mma_f16_ts(od, pa + j * 8, v_lo, idesc_o, 1);
            mma_f16_ts(od, pa + j * 8, v_hi, idesc_o, 1);
          }
          mma_commit(smem_u32(&o_full[b]));
          if (b == 1) mma_commit(smem_u32(&empty_bar[stage]));                 // both heads of the pair are done with the stage
        }
        __syncwarp();
        if (g + 2 < total) issue_s(g + 2);                                      // overwrites P(g): in order behind PV(g)
      }
    }
  } else {
    // ===================== softmax warps: AF_SUB threads per token row =====================
    // Warps w, w + 4, w + 8, ... own the same 32 TMEM lanes (rows); each takes 128 / AF_SUB dictionary columns, so every
    // scheduler has AF_SUB softmax warps to alternate between.  Row max and row sum cross the group through shared
    // memory with one named barrier (AF_SUB x 32 threads) per head.
    const int quarter = warp & 3, sub = ((warp - 2) >> 2) % AF_SUB, group = (warp - 2) / (4 * AF_SUB);
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    constexpr int HC = AF_ND / AF_SUB;     // columns per thread (32)
    constexpr int OC = AF_HD / AF_SUB;     // output columns per thread (8)
    auto row_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + group * 4 + quarter), "n"(AF_SUB * 32) : "memory"); };
    auto write_out = [&](int g) {
      const int gp = (int)blockIdx.x + (g >> 1) * (int)gridDim.x;
      const int tile = gp / HP, head = (gp % HP) * 2 + (g & 1);
      float l = 0.f;
#pragma unroll
      for (int q = 0; q < AF_SUB; ++q) l += xl[g & 1][(g >> 1) & 1][q][r];
      const float inv = p.v_descale / l;
      mbar_wait(smem_u32(&o_full[g & 1]), (g >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      uint32_t o0[OC];
#pragma unroll
      for (int c = 0; c < OC / 8; ++c) tmem_ld8_nowait(lane_addr + TF_O + (uint32_t)(g & 1) * 32 + sub * OC + c * 8, o0 + c * 8);
      tmem_ld_wait();
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(smem_u32(&o_free[g & 1]));
      const int64_t token = (int64_t)tile * AF_M + r;
      if (token < p.T) {
        const int col = head * AF_HD + sub * OC;
        float4* dst = p.out ? reinterpret_cast<float4*>(p.out + token * p.out_ld + col) : nullptr;
#pragma unroll
        for (int j = 0; j < OC; j += 4) {
          const float4 a = make_float4(__uint_as_float(o0[j]) * inv, __uint_as_float(o0[j + 1]) * inv,
                                       __uint_as_float(o0[j + 2]) * inv, __uint_as_float(o0[j + 3]) * inv);
          if (dst) dst[j / 4] = a;
          if (p.out16.hi) store_planes4(p.out16, token, col + j, a);
        }
      }
    };
    int last = -1;
    for (int g = group; g < total; g += AF_GROUPS) {
      const int b = g & 1;                                 // == group: each group keeps to its own S/P and O buffers
      const int head = (((int)blockIdx.x + (g >> 1) * (int)gridDim.x) % HP) * 2 + b;
      // softmax(sim * scale) = 2^(t - max t) / sum, t = acc * (k_descale * scale * log2 e)
      const float sc = __ldg(p.head_scale + head) * p.k_descale * 1.4426950408889634f;
      mbar_wait(smem_u32(&s_full[b]), (g >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      float s[HC];
      {
        uint32_t raw[HC];
#pragma unroll
        for (int c = 0; c < HC / 16; ++c) tmem_ld16_nowait(lane_addr + TF_SP + (uint32_t)b * 128 + sub * HC + c * 16, raw + c * 16);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < HC; ++j) s[j] = __uint_as_float(raw[j]) * sc;
      }
      float m8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) m8[j] = s[j];
#pragma unroll
      for (int j = 8; j < HC; ++j) m8[j & 7] = fmaxf(m8[j & 7], s[j]);
      float mx = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
      xm[b][sub][r] = mx;
      row_sync();           // every thread of the row holds its S columns in registers now: P may overwrite S; orders xl(g-1) too
#pragma unroll
      for (int q = 0; q < AF_SUB; ++q) mx = fmaxf(mx, xm[b][q][r]);
      mx -= 10.0f;                                         // P' = 1024 * P
      float l8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < HC; ++j) {
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(s[j] - mx));
        s[j] = e;
        l8[j & 7] += e;
      }
      if (last >= 0) write_out(last);                      // this group's previous head: its PV has had a whole head step
      last = g;
      xl[b][(g >> 1) & 1][sub][r] = ((l8[0] + l8[1]) + (l8[2] + l8[3])) + ((l8[4] + l8[5]) + (l8[6] + l8[7]));
      // packed fp16 pairs: word w = (P'[2w], P'[2w+1]); P_hi at columns [0, 64), P_lo at [64, 128) of the S/P buffer
      {
#pragma unroll
        for (int c = 0; c < HC / 32; ++c) {
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f16_split2(s[32 * c + 2 * j], s[32 * c + 2 * j + 1], hi[j], lo[j]);
          tmem_st16(lane_addr + TF_SP + (uint32_t)b * 128 + sub * (HC / 2) + c * 16, hi);
          tmem_st16(lane_addr + TF_SP + (uint32_t)b * 128 + 64 + sub * (HC / 2) + c * 16, lo);
        }
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(smem_u32(&p_ready[b]));
    }
    if (last >= 0) {
      row_sync();
      write_out(last);
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) tmem_dealloc<1>(tmem, 512);
}

}  // namespace

int dict_attention_tcgen05_f16(const dcae_planes* q16, const dcae_dict_kv* kv, int64_t T, float* out, int64_t out_ld,
                               dcae_planes out16, cudaStream_t s) {
  DCAE_REQUIRE(q16 && q16->hi && q16->lo, "dict_attention(f16x3): the query must be given as fp16 planes (q16)");
  DCAE_REQUIRE(kv->K16_hi && kv->K16_lo && kv->Vt16_hi && kv->Vt16_lo && kv->k_descale > 0.f && kv->v_descale > 0.f,
               "dict_attention(f16x3): dictionary K / V^T have no fp16 planes (K16_*, Vt16_*, *_descale)");
  DCAE_REQUIRE(aligned16(q16->hi) && aligned16(q16->lo) && q16->ld % 8 == 0 && q16->ld >= AF_HEADS * AF_HD,
               "dict_attention(f16x3): q planes must be 16-byte aligned with ld %% 8 == 0 and ld >= 640");
  if (T == 0) return DCAE_OK;
  AfParams p;
  p.head_scale = kv->head_scale;
  p.out = out; p.out_ld = out_ld; p.T = T;
  p.out16 = out16;
  p.tiles = (int)((T + AF_M - 1) / AF_M);
  p.k_descale = kv->k_descale; p.v_descale = kv->v_descale;
  CUtensorMap mqh, mql, mkh, mkl, mvh, mvl;
  const cuuint64_t D = (cuuint64_t)AF_HEADS * AF_HD;
  constexpr CUtensorMapDataType F16 = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  {
    cuuint64_t dims[2] = {D, (cuuint64_t)T};
    cuuint64_t str[1] = {(cuuint64_t)q16->ld * 2};
    cuuint32_t box[2] = {64, AF_M};
    DCAE_TRY(encode_map(&mqh, F16, q16->hi, 2, dims, str, box));
    DCAE_TRY(encode_map(&mql, F16, q16->lo, 2, dims, str, box));
  }
  {
    cuuint64_t dims[2] = {D, AF_ND};
    cuuint64_t str[1] = {D * 2};
    cuuint32_t box[2] = {64, AF_ND};
    DCAE_TRY(encode_map(&mkh, F16, kv->K16_hi, 2, dims, str, box));
    DCAE_TRY(encode_map(&mkl, F16, kv->K16_lo, 2, dims, str, box));
  }
  {
    cuuint64_t dims[2] = {AF_ND, D};
    cuuint64_t str[1] = {AF_ND * 2};
    cuuint32_t box[2] = {64, 64};
    DCAE_TRY(encode_map(&mvh, F16, kv->Vt16_hi, 2, dims, str, box));
    DCAE_TRY(encode_map(&mvl, F16, kv->Vt16_lo, 2, dims, str, box));
  }
  const size_t smem = (size_t)AF_STAGES * AF_STAGE + 1024;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(dict_attention_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AF_STAGES * AF_STAGE + 1024);
  });
  DCAE_CUDA(attr_err);
  const int ctas = p.tiles * (AF_HEADS / 2) < num_sms() ? p.tiles * (AF_HEADS / 2) : num_sms();
  dict_attention_f16_kernel<<<ctas, AF_THREADS, smem, s>>>(mqh, mql, mkh, mkl, mvh, mvl, p);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae
