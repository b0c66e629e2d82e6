// DCAE_MATH_F16X3: the dense / implicit-conv GEMM on fp16 hi/lo operand PLANES (tcgen05 kind::f16).
//
// Why (profiles/r01, Little's-law reading of the stage sweeps): the mainloop feed is capped at about
// (shared memory in flight) / (TMA latency ~ 3700 clk) ~ 55 B/clk/SM whatever the tile shape, so the lever is
// flops per operand byte.  An fp32 value a is carried as a_hi = fp16(a), a_lo = fp16(a - a_hi): 22 significant
// bits in 4 bytes (the same accuracy and the same bytes as the TF32 split), but the fp16 MMA runs at twice
// the TF32 rate and a 128-byte swizzle row holds K = 64 instead of 32 -- half the bytes per flop -- and the
// planes come straight from TMA, so the in-kernel split warps (and their latency in the stage turnaround)
// disappear.  Per k-step the MMA warp issues a_lo*w_hi + a_hi*w_lo + a_hi*w_hi into the fp32 TMEM accumulator.
//
// Range: activations are converted with saturation (|a| > 65504 clamps instead of becoming inf; the layers
// of this model are O(1..1e2)).  Weights are pre-scaled by a power of two so that w_lo stays out of the
// fp16 subnormal range; the epilogue multiplies by the exact inverse.
//
// Same structure as gemm_tcgen05.cu otherwise: TMA 4-D boxes (3x3 taps = shifted boxes, hardware zero
// fill), persistent CTAs, <= 96-MMA accumulation chains in two alternating TMEM buffers summed in fp32
// registers (RZ-accumulator fix), epilogue overlapped with the next tile.
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace dcae {

namespace {

constexpr int BM = 128;
constexpr int BK16 = 64;                 // fp16 per k-block = 128 B = one swizzle row
constexpr int UMMA_K16 = 16;
constexpr int A16_BYTES = BM * BK16 * 2; // 16 KB per plane tile
constexpr int MAX_STAGES = 8;
constexpr int NTHREADS = 384;            // warps 0-3 control (TMA, MMA, 2 idle), 4-11 drain / epilogue
constexpr int NDRAIN = 256;
constexpr int REGS_CTRL = 40, REGS_DRAIN = 216;   // 128*40 + 256*216 <= 65536
constexpr int CHUNK_MMAS = 96;
constexpr uint32_t SMEM_LIMIT = 227 * 1024;
// epilogue staging per drain group (the 4 warps that own the same 32-column blocks):
// [fp32 block 128 x 128 B, SWIZZLE_128B | fp16 hi 128 x 64 B, SWIZZLE_64B | fp16 lo]
// one 16 KB buffer per group, used for the fp32 block and then (if both are requested) for the two fp16 planes
constexpr uint32_t STG_O32 = 0, STG_HI = 0, STG_LO = 8192, STG_BYTES = 16384;

struct F16Params {
  dcae_epilogue e;
  int N, KB;                 // KB = taps * (Kp / 64)
  int cblk_per_tap, taps;
  int B, h, w;
  TokenTiling tt;
  int BN, stages, tmem_cols;
  int n_tiles_n, total_tiles, chunk_kb;
  float descale;
  int has_o32, has_o16, has_o16a;
  int fuse_b;                // single CTA, BN <= 128: one N = 2 BN MMA covers a_hi x [b_hi; b_lo], see the MMA issuer
  int passes;                // 3 = hi/lo error-compensated (fp32-level accuracy); 1 = DCAE_MATH_F16: a_hi x b_hi only, lo planes never loaded
  uint32_t stage_bytes, b_bytes;
};


// drain of one chunk; FUSED: the accumulator of block blk is the sum of columns blk*32 (a_hi b_hi + a_lo b_hi) and
// BN + blk*32 (a_hi b_lo)
template <int NB>
__device__ __forceinline__ void drain_chunk_f16(float* acc, uint32_t taddr, int half, int BN, bool first, bool fused_rt) {
  const bool fused = (NB == 2) && fused_rt;     // BN <= 128 only: the NB = 4 instantiation never carries the second range
#pragma unroll
  for (int g = 0; g < NB; ++g) {
    const int blk = 2 * g + half;
    if (blk * 32 < BN) {                      // warp-uniform
      uint32_t raw[32], raw2[32];
      tmem_ld16_nowait(taddr + blk * 32, raw);
      tmem_ld16_nowait(taddr + blk * 32 + 16, raw + 16);
      if (fused) {
        tmem_ld16_nowait(taddr + BN + blk * 32, raw2);
        tmem_ld16_nowait(taddr + BN + blk * 32 + 16, raw2 + 16);
      }
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        float v = __uint_as_float(raw[j]);
        if (fused) v = __fadd_rn(v, __uint_as_float(raw2[j]));
        acc[g * 32 + j] = first ? v : __fadd_rn(acc[g * 32 + j], v);
      }
    }
  }
}

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Epilogue of one tile through shared-memory staging and TMA tensor stores.  The thread owns tile row r; each of
// its 32-column blocks goes bias / addend / activation / residual in registers, then into the group's staging
// buffer in the swizzled box layout (conflict-free st.shared.v4), and one thread issues the bulk store(s):
// full 128-byte lines, ragged tiles clipped by the hardware, no per-thread global address arithmetic.
// One instance, run-time activation: the three branches are disjoint loops (nothing for ptxas to if-convert into
// "evaluate erf AND tanh"), and the epilogue must stay SMALL -- see the note at the block loop.
__device__ __forceinline__ void finalize_block(float* r, const dcae_epilogue& e, int act, bool row_ok, int64_t token, int n0,
                                               float bias_lane, float rs_lane) {
  // bias / res_scale of column n0 + lane were loaded by this lane before the accumulator wait (a global load issued
  // here would pay the loaded L2 latency on the critical path of every block); broadcast by shuffle.
#pragma unroll
  for (int j = 0; j < 32; ++j) r[j] += __shfl_sync(0xffffffffu, bias_lane, j);
  if (e.addend && row_ok) {
    const float4* ap = reinterpret_cast<const float4*>(e.addend + token * e.addend_ld + n0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 ad = __ldg(ap + j);
      r[4 * j] += ad.x; r[4 * j + 1] += ad.y; r[4 * j + 2] += ad.z; r[4 * j + 3] += ad.w;
    }
  }
  if (act == DCAE_ACT_GELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = gelu_fast(r[j]);
  } else if (act == DCAE_ACT_HALF_TANH) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = 0.5f * tanhf(r[j]);
  } else if (act == DCAE_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = fmaxf(r[j], 0.f);
  }
  if (e.residual) {
    const float4* rp = reinterpret_cast<const float4*>(e.residual + token * e.residual_ld + n0);
#pragma unroll
    for (int hq = 0; hq < 2; ++hq) {                 // two halves: 16 registers of loads in flight, not 32
      float4 rv[4];
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < 4; ++j) rv[j] = __ldg(rp + 4 * hq + j);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = 16 * hq + 4 * j;
        const float s0 = __shfl_sync(0xffffffffu, rs_lane, c), s1 = __shfl_sync(0xffffffffu, rs_lane, c + 1);
        const float s2 = __shfl_sync(0xffffffffu, rs_lane, c + 2), s3 = __shfl_sync(0xffffffffu, rs_lane, c + 3);
        if (row_ok) {
          r[c] = fmaf(rv[j].x, s0, r[c]); r[c + 1] = fmaf(rv[j].y, s1, r[c + 1]);
          r[c + 2] = fmaf(rv[j].z, s2, r[c + 2]); r[c + 3] = fmaf(rv[j].w, s3, r[c + 3]);
        }
      }
    }
  }
}
// row `row` of a [128 x 32] fp32 block into the SWIZZLE_128B box layout (128-byte rows)
__device__ __forceinline__ void stage_f32(const float* v, int row, uint32_t stg) {
  const uint32_t base = stg + STG_O32 + (uint32_t)row * 128;
#pragma unroll
  for (int c = 0; c < 8; ++c)
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(base + (uint32_t)((c ^ (row & 7)) << 4)),
                 "f"(v[4 * c]), "f"(v[4 * c + 1]), "f"(v[4 * c + 2]), "f"(v[4 * c + 3]) : "memory");
}
// the same row as fp16 hi / lo planes, each a [128 x 32] block in the SWIZZLE_64B box layout (64-byte rows)
__device__ __forceinline__ void stage_f16(const float* v, int row, uint32_t stg) {
  const uint32_t bh = stg + STG_HI + (uint32_t)row * 64, bl = stg + STG_LO + (uint32_t)row * 64;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      f16_split2(v[8 * c + 2 * q], v[8 * c + 2 * q + 1], hw[q], lw[q]);
    }
    const uint32_t off = (uint32_t)((c ^ ((row >> 1) & 3)) << 4);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(bh + off), "r"(hw[0]), "r"(hw[1]), "r"(hw[2]), "r"(hw[3]) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(bl + off), "r"(lw[0]), "r"(lw[1]), "r"(lw[2]), "r"(lw[3]) : "memory");
  }
}

// ---- fp32 window -> fp16 hi/lo planes [T, Kp] (HBM-bound, one float4 -> two 8-byte stores) -------------
__global__ void __launch_bounds__(256) split_f16_planes_kernel(const float* __restrict__ x, int64_t ld, int col0, int k0, int col1,
                                                               int kc, int Kp, int64_t T, __half* __restrict__ hi, __half* __restrict__ lo) {
  const int g4 = Kp >> 2;
  const int64_t n = T * g4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / g4;
    const int c = (int)(i - t * g4) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < kc) {
      const int col = (c < k0) ? (col0 + c) : (col1 + (c - k0));
      v = __ldg(reinterpret_cast<const float4*>(x + t * ld + col));
    }
    const float f[4] = {v.x, v.y, v.z, v.w};
    __half h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned short hb, lb;
      asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(hb) : "f"(f[k]));
      h[k] = __ushort_as_half(hb);
      const float r = f[k] - __half2float(h[k]);
      asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(lb) : "f"(r));
      l[k] = __ushort_as_half(lb);
    }
    *reinterpret_cast<uint2*>(hi + t * Kp + c) = *reinterpret_cast<const uint2*>(h);
    *reinterpret_cast<uint2*>(lo + t * Kp + c) = *reinterpret_cast<const uint2*>(l);
  }
}

__global__ void __launch_bounds__(256) split_f16_weight_kernel(const float* __restrict__ w, int N, int taps, int kc, int Kp, float scale,
                                                               __half* __restrict__ hi, __half* __restrict__ lo) {
  const int64_t n = (int64_t)N * taps * Kp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % Kp);
    const int64_t r = i / Kp;              // row * taps + tap
    float v = 0.f;
    if (c < kc) v = w[r * kc + c] * scale;
    const __half h = __float2half_rn(v);
    hi[i] = h;
    lo[i] = __float2half_rn(v - __half2float(h));
  }
}

// PAIR = false: one CTA per 128-token tile.  PAIR = true: thread-block pair (cta_group::2): the pair computes a
// 256-token x BN tile with M = 256 MMAs issued by the leader; each CTA loads its own A planes and HALF of the weight
// planes (BN/2 rows), TMA completion of both CTAs is credited to the leader's full barrier, tcgen05.commit is
// multicast to both CTAs, the drain warps of both CTAs release the leader's TMEM-empty barrier.
// NB = 32-column blocks per drain group and tile: 2 for BN <= 128 (64 accumulator registers), 4 up to BN = 256
template <bool PAIR, int NB>
__device__ __forceinline__ void gemm_f16x3_body(const CUtensorMap& map_ah, const CUtensorMap& map_al, const CUtensorMap& map_bh,
                                                const CUtensorMap& map_bl, const CUtensorMap& map_o32, const CUtensorMap& map_oh,
                                                const CUtensorMap& map_ol, const CUtensorMap& map_oha, const CUtensorMap& map_ola,
                                                const F16Params& p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp: provably uniform
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t rank = PAIR ? __shfl_sync(0xffffffffu, cluster_ctarank(), 0) : 0u;
  const bool leader = rank == 0;
  const int unit = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;          // which persistent worker (CTA or pair)
  const int nunits = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[b]), PAIR ? 2 * NDRAIN : NDRAIN);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ah) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_al) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bl) : "memory");
  }
  if (warp == 1) tmem_alloc<PAIR ? 2 : 1>(smem_u32(&tmem_base_slot), p.tmem_cols);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (PAIR) cluster_sync_all();     // the peer's barriers exist before anything signals them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  // per-stage smem: [A_hi | A_lo | B_hi | B_lo] (single pass: [A_hi | B_hi]); the two epilogue staging buffers follow the stages
  const uint32_t off_al = A16_BYTES, off_bh = (p.passes == 3 ? 2 : 1) * A16_BYTES, off_bl = off_bh + p.b_bytes;
  const uint32_t stg_base = smem0 + (uint32_t)p.stages * p.stage_bytes;
  const int n_chunks = (p.KB + p.chunk_kb - 1) / p.chunk_kb;

  auto tile_coords = [&](int t, int& b, int& y0, int& x0, int& n0) {
    const int nt = t % p.n_tiles_n;
    int mt = PAIR ? (t / p.n_tiles_n) * 2 + (int)rank : t / p.n_tiles_n;   // b may reach B for a pair's odd tail tile
    const int tile_x = mt % p.tt.tiles_x; mt /= p.tt.tiles_x;
    const int tile_y = mt % p.tt.tiles_y;
    b = mt / p.tt.tiles_y;
    x0 = tile_x * p.tt.TW; y0 = tile_y * p.tt.TH; n0 = nt * p.BN;
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
    if (warp == 0) {
      // ===================== TMA producer (warp-uniform; one elected lane issues) =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int t = unit; t < p.total_tiles; t += nunits) {
        int b, y0, x0, n0;
        tile_coords(t, b, y0, x0, n0);
        for (int kb = 0; kb < p.KB; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t sbase = smem0 + stage * p.stage_bytes;
          const uint32_t fb = smem_u32(&full_bar[stage]);
          const int tap = kb / p.cblk_per_tap;
          const int c = (kb - tap * p.cblk_per_tap) * BK16;
          int dy = 0, dx = 0;
          if (p.taps == 9) { dy = tap / 3 - 1; dx = tap % 3 - 1; }
          const int nrow = n0 + (int)rank * (p.BN >> 1);
          if (elect_one()) {
            const bool lo_too = p.passes == 3;
            const uint32_t bytes = (lo_too ? 2u : 1u) * (A16_BYTES + p.b_bytes);
            if (PAIR) {
              if (leader) mbar_expect_tx(fb, 2 * bytes);      // bytes landing in BOTH CTAs
              tma_load_4d_2sm(sbase, &map_ah, fb, c, x0 + dx, y0 + dy, b);
              if (lo_too) tma_load_4d_2sm(sbase + off_al, &map_al, fb, c, x0 + dx, y0 + dy, b);
              tma_load_2d_2sm(sbase + off_bh, &map_bh, fb, kb * BK16, nrow);
              if (lo_too) tma_load_2d_2sm(sbase + off_bl, &map_bl, fb, kb * BK16, nrow);
            } else {
              mbar_expect_tx(fb, bytes);
              tma_load_4d(sbase, &map_ah, fb, c, x0 + dx, y0 + dy, b);
              if (lo_too) tma_load_4d(sbase + off_al, &map_al, fb, c, x0 + dx, y0 + dy, b);
              tma_load_2d(sbase + off_bh, &map_bh, fb, kb * BK16, n0);
              if (lo_too) tma_load_2d(sbase + off_bl, &map_bl, fb, kb * BK16, n0);
            }
          }
          __syncwarp();
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    } else if (warp == 1 && leader) {
      // ===================== MMA issuer (the leader CTA of a pair; warp-uniform, one elected lane issues) =====================
      const uint32_t idesc = make_idesc_f16((PAIR ? 2 : 1) * BM, p.BN);
      const uint32_t idesc2 = make_idesc_f16(BM, 2 * p.BN);   // fuse_b: N = 2 BN
      int stage = 0;
      uint32_t phase = 0, gchunk = 0;
      for (int t = unit; t < p.total_tiles; t += nunits) {
        for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
          const uint32_t buf = gchunk & 1;
          if (PAIR) mbar_wait_cluster(smem_u32(&tmem_empty_bar[buf]), ((gchunk >> 1) & 1) ^ 1); else mbar_wait(smem_u32(&tmem_empty_bar[buf]), ((gchunk >> 1) & 1) ^ 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tmem_acc = tmem_base + buf * (uint32_t)(p.fuse_b ? 2 * p.BN : p.BN);
          const int kb_end = min(p.KB, (ck + 1) * p.chunk_kb);
          for (int kb = ck * p.chunk_kb; kb < kb_end; ++kb) {
            if (PAIR) mbar_wait_cluster(smem_u32(&full_bar[stage]), phase); else mbar_wait(smem_u32(&full_bar[stage]), phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sbase = smem0 + stage * p.stage_bytes;
            const uint32_t first = (kb == ck * p.chunk_kb) ? 0u : 1u;
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < BK16 / UMMA_K16; ++k) {
                const uint32_t koff = k * UMMA_K16 * 2;
                const uint64_t a_hi = make_smem_desc(sbase + koff), a_lo = make_smem_desc(sbase + off_al + koff);
                const uint64_t b_hi = make_smem_desc(sbase + off_bh + koff), b_lo = make_smem_desc(sbase + off_bl + koff);
                if (p.passes == 1) {
                  if (PAIR) mma_f16_2sm(tmem_acc, a_hi, b_hi, idesc, first | (uint32_t)(k != 0));
                  else mma_f16(tmem_acc, a_hi, b_hi, idesc, first | (uint32_t)(k != 0));
                } else if (PAIR) {
                  mma_f16_2sm(tmem_acc, a_lo, b_hi, idesc, first | (uint32_t)(k != 0));
                  mma_f16_2sm(tmem_acc, a_hi, b_lo, idesc, 1);
                  mma_f16_2sm(tmem_acc, a_hi, b_hi, idesc, 1);
                } else if (p.fuse_b) {
                  // b_lo sits right behind b_hi in the stage, so ONE N = 2 BN instruction computes a_hi x [b_hi; b_lo]
                  // into columns [0, BN) | [BN, 2 BN): the A tile is read from shared memory twice per k-step, not 3 times
                  mma_f16(tmem_acc, a_hi, b_hi, idesc2, first | (uint32_t)(k != 0));
                  mma_f16(tmem_acc, a_lo, b_hi, idesc, 1);
                } else {
                  mma_f16(tmem_acc, a_lo, b_hi, idesc, first | (uint32_t)(k != 0));
                  mma_f16(tmem_acc, a_hi, b_lo, idesc, 1);
                  mma_f16(tmem_acc, a_hi, b_hi, idesc, 1);
                }
              }
              if (PAIR) mma_commit_2sm(smem_u32(&empty_bar[stage])); else mma_commit(smem_u32(&empty_bar[stage]));
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          if (elect_one()) {
            if (PAIR) mma_commit_2sm(smem_u32(&tmem_full_bar[buf])); else mma_commit(smem_u32(&tmem_full_bar[buf]));
          }
          __syncwarp();
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_DRAIN));
    // ===================== drain + epilogue warps =====================
    const int quarter = warp & 3;
    const int half = (warp - 4) >> 2;
    uint32_t gchunk = 0;
    for (int t = unit; t < p.total_tiles; t += nunits) {
      EpiTile et;
      tile_coords(t, et.b, et.y0, et.x0, et.n0);
      et.B = p.B; et.h = p.h; et.w = p.w; et.tw_shift = p.tt.tw_shift; et.N = p.N; et.BN = p.BN;
      float acc[NB * 32];
      float bias_l[NB], rs_l[NB];          // column (block g, lane) of bias / res_scale, see finalize_block
#pragma unroll
      for (int g = 0; g < NB; ++g) {
        const int n = et.n0 + (2 * g + half) * 32 + lane;
        const bool ok = (2 * g + half) * 32 < p.BN && n < p.N;
        bias_l[g] = (p.e.bias && ok) ? __ldg(p.e.bias + n) : 0.f;
        rs_l[g] = (p.e.residual && p.e.res_scale && ok) ? __ldg(p.e.res_scale + n) : 1.f;
      }
      for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
        const uint32_t buf = gchunk & 1;
        mbar_wait(smem_u32(&tmem_full_bar[buf]), (gchunk >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        drain_chunk_f16<NB>(acc, tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)(p.fuse_b ? 2 * p.BN : p.BN), half, p.BN, ck == 0, p.fuse_b != 0);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        if (PAIR) mbar_arrive_cluster(smem_u32(&tmem_empty_bar[buf]), 0); else mbar_arrive(smem_u32(&tmem_empty_bar[buf]));
      }
      // ---- epilogue: registers -> swizzled staging -> TMA tensor store, one 32-column block at a time ----
      // A ROLLED loop with one copy of the body.  Fully unrolled (4 blocks x 3 activations x 3 outputs) the kernel was
      // 350 KB of straight-line SASS that each warp runs once per tile: instruction fetch, not arithmetic, set the
      // epilogue time (every phase measured 10-20x its instruction count; role-counter logs under profiles/r01).  The
      // accumulator registers need static indices, so the block's 32 values are selected into r[] first.
      const dcae_epilogue& e = p.e;
      const int act_cols = (e.act_cols <= 0 || e.act_cols > p.N) ? p.N : e.act_cols;
      const int row = quarter * 32 + lane;
      const int yy = et.y0 + (row >> p.tt.tw_shift), xx = et.x0 + (row & ((1 << p.tt.tw_shift) - 1));
      const bool row_ok = yy < p.h && xx < p.w && et.b < p.B;
      const int64_t token = ((int64_t)et.b * p.h + yy) * p.w + xx;
      const uint32_t stg = stg_base + (uint32_t)half * STG_BYTES;
      const bool issuer = quarter == 0 && lane == 0;
#pragma unroll 1
      for (int g = 0; g < NB; ++g) {
        const int blk = 2 * g + half;
        const int nb0 = et.n0 + blk * 32;
        if (blk * 32 >= p.BN || nb0 >= p.N) break;              // uniform over the group; ragged last N tile
        const int act = (nb0 < act_cols) ? e.act : DCAE_ACT_NONE;
        // the block to process is always acc[0..32) / bias_l[0]: processed in place, then the queue shifts down
        // (static register indices in a rolled loop without a second copy of the block)
        float* r = acc;
        const float bias_lane = bias_l[0], rs_lane = rs_l[0];
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] *= p.descale;          // exact: power of two
        finalize_block(r, e, act, row_ok, token, nb0, bias_lane, rs_lane);
        // output o: 0 = fp32, 1 = fp16 planes, 2 = fp16 planes of act2(result), the next layer's GELU prologue.
        // One staging round each: wait until the previous store has read the buffer, stage, make the writes visible
        // to the async proxy, and let one thread issue the bulk store(s).
#pragma unroll 1
        for (int o = 0; o < 3; ++o) {
          if (!(o == 0 ? p.has_o32 : o == 1 ? p.has_o16 : p.has_o16a)) continue;
          if (o == 2 && e.act2 == DCAE_ACT_GELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = gelu_fast(r[j]);
          }
          if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          named_bar_sync(1 + half, 128);
          if (o == 0) stage_f32(r, row, stg); else stage_f16(r, row, stg);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          named_bar_sync(1 + half, 128);
          if (issuer) {
            if (o == 0) {
              tma_store_4d(&map_o32, stg + STG_O32, nb0, et.x0, et.y0, et.b);
            } else {
              tma_store_4d(o == 1 ? &map_oh : &map_oha, stg + STG_HI, nb0, et.x0, et.y0, et.b);
              tma_store_4d(o == 1 ? &map_ol : &map_ola, stg + STG_LO, nb0, et.x0, et.y0, et.b);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
#pragma unroll
        for (int i = 0; i < (NB - 1) * 32; ++i) acc[i] = acc[i + 32];
#pragma unroll
        for (int q = 0; q < NB - 1; ++q) { bias_l[q] = bias_l[q + 1]; rs_l[q] = rs_l[q + 1]; }
      }
    }
    if (quarter == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all stores landed before exit
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (PAIR) cluster_sync_all();     // neither CTA may free TMEM / exit while the pair still uses its smem or TMEM
  if (warp == 1) tmem_dealloc<PAIR ? 2 : 1>(tmem_base, p.tmem_cols);
}

template <int NB>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_f16x3_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                  const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                  const __grid_constant__ CUtensorMap map_o32, const __grid_constant__ CUtensorMap map_oh,
                  const __grid_constant__ CUtensorMap map_ol, const __grid_constant__ CUtensorMap map_oha,
                  const __grid_constant__ CUtensorMap map_ola, const F16Params p) {
  gemm_f16x3_body<false, NB>(map_ah, map_al, map_bh, map_bl, map_o32, map_oh, map_ol, map_oha, map_ola, p);
}

template <int NB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
gemm_f16x3_pair_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                       const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                       const __grid_constant__ CUtensorMap map_o32, const __grid_constant__ CUtensorMap map_oh,
                       const __grid_constant__ CUtensorMap map_ol, const __grid_constant__ CUtensorMap map_oha,
                       const __grid_constant__ CUtensorMap map_ola, const F16Params p) {
  gemm_f16x3_body<true, NB>(map_ah, map_al, map_bh, map_bl, map_o32, map_oh, map_ol, map_oha, map_ola, p);
}

inline int pad64(int v) { return (v + 63) / 64 * 64; }

}  // namespace

int gemm_tcgen05_f16x3(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int passes, cudaStream_t s) {
  const int kc = a->k0 + a->k1, Kp = pad64(kc);
  const int64_t T = (int64_t)a->B * a->h * a->w;
  DCAE_REQUIRE(w->w16_hi && w->w16_lo && w->K16 == a->taps * Kp && w->descale > 0.f,
               "gemm(f16x3): weight has no fp16 planes (dcae_split_f16_weight) or K16=%d != taps*pad64(kc)=%d", w->K16, a->taps * Kp);
  const bool direct = a->src16.hi != nullptr;     // the producer already wrote fp16 planes: no split pass
  DCAE_REQUIRE(direct || (a->base && a->planes != nullptr && a->planes_bytes >= dcae_planes_bytes(T, kc) && (reinterpret_cast<uintptr_t>(a->planes) & 127u) == 0),
               "gemm(f16x3): operand.planes scratch missing, misaligned (128 B) or smaller than dcae_planes_bytes()");
  DCAE_REQUIRE(!direct || (a->k1 == 0 && a->src16.lo && a->src16.ld % 8 == 0 && a->col0 % 8 == 0 &&
                           (reinterpret_cast<uintptr_t>(a->src16.hi) & 15u) == 0 && (reinterpret_cast<uintptr_t>(a->src16.lo) & 15u) == 0),
               "gemm(f16x3): src16 planes need one segment, 16-byte aligned planes and col0 / ld multiples of 8");
  DCAE_REQUIRE(e->act_cols <= 0 || e->act_cols >= w->N || e->act_cols % 32 == 0, "gemm(f16x3): act_cols must be a multiple of 32");
  DCAE_REQUIRE(e->out || e->out16.hi || e->out16_act.hi, "gemm(f16x3): no output");
  if (T == 0) return DCAE_OK;
  __half* hi = direct ? static_cast<__half*>(a->src16.hi) + a->col0 : static_cast<__half*>(a->planes);
  __half* lo = direct ? static_cast<__half*>(a->src16.lo) + a->col0 : hi + T * Kp;
  const int64_t ldp = direct ? a->src16.ld : Kp;
  if (!direct) {
    const int64_t n = T * (Kp / 4);
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    if (blocks > cap) blocks = cap;
    split_f16_planes_kernel<<<(unsigned)blocks, 256, 0, s>>>(a->base, a->ld, a->col0, a->k0, a->col1, kc, Kp, T, hi, lo);
    DCAE_LAUNCH_CHECK();
  }
  F16Params p;
  p.e = *e;
  p.N = w->N;
  p.taps = a->taps;
  p.cblk_per_tap = Kp / BK16;
  p.KB = a->taps * p.cblk_per_tap;
  p.B = a->B; p.h = a->h; p.w = a->w;
  p.tt = token_tiling(a->h, a->w);
  const int m_tiles = p.tt.tiles_x * p.tt.tiles_y * a->B;
  // A/B sweeps (profiles/r01/gemm_f16_pair_ab.jsonl, layer_times_bn_pair_sweep3.log): pairs win where the mainloop is
  // long or wide (cc1, proj, fc1, the K = 2 016 conv layers); everything else runs single-CTA with BN <= 128 so that
  // the fused [b_hi; b_lo] MMA applies (N = 320 -> 128 + 128 + 64 ragged beats 2 x 160 by 20 %, N = 224 likewise).
  // single pass: the mainloop moves a third of the flops per operand byte less... per k-block a 128 x 128 tile is 256 tensor
  // cycles against 32 KB of operands (128 B/clk, twice what the L2 -> SM path feeds), so every layer that can takes
  // M = 256 pairs with the widest N tile (each CTA loads half of the weight rows: 62 B/clk at BN = 256)
  // The arithmetic (fused or three-MMA accumulation order) follows want_pair, a function of the layer shape only, so
  // that a result never depends on the batch size (a 1-tile problem cannot pair but keeps the pair path's order).
  const bool want_pair = passes == 1 ? w->N >= 128 : ((int64_t)a->taps * Kp >= 2048 || w->N >= 2048);
  const bool pair = want_pair && m_tiles >= 2;
  p.BN = 0;
  p.passes = passes;
  if (!want_pair) {
    p.BN = w->N >= 128 ? 128 : w->N;
  } else if (passes == 1) {              // least padded work, then the widest tile (N = 640 -> 4 x 160, 672 -> 3 x 224)
    int best = 1 << 30;
    for (int bn = 256; bn >= 128; bn -= 32) {
      const int padded = (w->N + bn - 1) / bn * bn;
      if (padded < best) { best = padded; p.BN = bn; }
    }
  } else {
    // 256 and 128 first: with the 32 KB of epilogue staging, 128 keeps three 64 KB stages in flight; then the largest
    // divisor (672 -> 224).  profiles/r01/gemm_f16_sweep.jsonl
    static const int order[] = {256, 128, 224, 192, 160, 96, 64, 32};
    for (int bn : order)
      if (w->N % bn == 0) { p.BN = bn; break; }
  }
  DCAE_REQUIRE(p.BN > 0 && p.BN % 32 == 0, "gemm(f16x3): N=%d must be a multiple of 32", w->N);
  p.n_tiles_n = (w->N + p.BN - 1) / p.BN;      // a ragged last tile reads zero-filled weight rows and stores clipped
  p.fuse_b = (!want_pair && p.BN <= 128 && passes == 3) ? 1 : 0;
  const int acc_cols = 2 * (p.fuse_b ? 2 * p.BN : p.BN);          // two chunk buffers
  p.tmem_cols = acc_cols <= 64 ? 64 : acc_cols <= 128 ? 128 : acc_cols <= 256 ? 256 : 512;
  p.total_tiles = p.n_tiles_n * (pair ? (m_tiles + 1) / 2 : m_tiles);
  p.chunk_kb = CHUNK_MMAS / (passes == 1 ? 4 : p.fuse_b ? 8 : 12);      // accumulation chain per column: 1, 2 (fused) or 3 MMAs per K = 16 step, 4 steps per k-block
  p.descale = w->descale;
  p.b_bytes = (uint32_t)(pair ? p.BN / 2 : p.BN) * BK16 * 2;     // a pair's CTA holds half of the weight rows
  p.stage_bytes = (passes == 3 ? 2 : 1) * (A16_BYTES + p.b_bytes);
  p.stages = (int)((SMEM_LIMIT - 2048 - 2 * STG_BYTES) / p.stage_bytes);
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  if (p.stages > p.KB) p.stages = p.KB;
  DCAE_REQUIRE(p.stages >= 1, "gemm(f16x3): tile does not fit in shared memory");
  const size_t smem = (size_t)p.stages * p.stage_bytes + 2 * STG_BYTES + 1024;
  p.has_o32 = e->out != nullptr;
  p.has_o16 = e->out16.hi != nullptr;
  p.has_o16a = e->out16_act.hi != nullptr;
  DCAE_REQUIRE(!p.has_o16a || e->act2 == DCAE_ACT_NONE || e->act2 == DCAE_ACT_GELU, "gemm(f16x3): act2 must be NONE or GELU");

  CUtensorMap map_ah, map_al, map_bh, map_bl, map_o32, map_oh, map_ol, map_oha, map_ola;
  {
    // output boxes {32 columns, TW, TH, 1}; dims[0] = N clips a ragged last block, (w, h) clip ragged token tiles
    cuuint32_t box[4] = {32, (cuuint32_t)p.tt.TW, (cuuint32_t)p.tt.TH, 1};
    cuuint64_t dims[4] = {(cuuint64_t)w->N, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->B};
    if (p.has_o32) {
      DCAE_REQUIRE(aligned16(e->out) && e->out_ld % 4 == 0, "gemm(f16x3): fp32 output must be 16-byte aligned with ld %% 4 == 0");
      cuuint64_t str[3] = {(cuuint64_t)e->out_ld * 4, (cuuint64_t)e->out_ld * 4 * a->w, (cuuint64_t)e->out_ld * 4 * a->w * a->h};
      DCAE_TRY(encode_map(&map_o32, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, e->out, 4, dims, str, box));
    }
    if (p.has_o16) {
      DCAE_REQUIRE(aligned16(e->out16.hi) && aligned16(e->out16.lo) && e->out16.ld % 8 == 0, "gemm(f16x3): output planes must be 16-byte aligned with ld %% 8 == 0");
      cuuint64_t str[3] = {(cuuint64_t)e->out16.ld * 2, (cuuint64_t)e->out16.ld * 2 * a->w, (cuuint64_t)e->out16.ld * 2 * a->w * a->h};
      DCAE_TRY(encode_map(&map_oh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, e->out16.hi, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B));
      DCAE_TRY(encode_map(&map_ol, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, e->out16.lo, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B));
    }
    if (p.has_o16a) {
      DCAE_REQUIRE(aligned16(e->out16_act.hi) && aligned16(e->out16_act.lo) && e->out16_act.ld % 8 == 0, "gemm(f16x3): out16_act planes must be 16-byte aligned with ld %% 8 == 0");
      cuuint64_t str[3] = {(cuuint64_t)e->out16_act.ld * 2, (cuuint64_t)e->out16_act.ld * 2 * a->w, (cuuint64_t)e->out16_act.ld * 2 * a->w * a->h};
      DCAE_TRY(encode_map(&map_oha, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, e->out16_act.hi, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B));
      DCAE_TRY(encode_map(&map_ola, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, e->out16_act.lo, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B));
    }
  }
  {
    // dims[0] = Kp: a window that is not a multiple of 64 wide over-reads into the next columns (zero weights there)
    cuuint64_t dims[4] = {(cuuint64_t)Kp, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->B};
    cuuint64_t str[3] = {(cuuint64_t)ldp * 2, (cuuint64_t)ldp * 2 * a->w, (cuuint64_t)ldp * 2 * a->w * a->h};
    cuuint32_t box[4] = {BK16, (cuuint32_t)p.tt.TW, (cuuint32_t)p.tt.TH, 1};
    DCAE_TRY(encode_map(&map_ah, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, hi, 4, dims, str, box));
    DCAE_TRY(encode_map(&map_al, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, lo, 4, dims, str, box));
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)w->K16, (cuuint64_t)w->N};
    cuuint64_t str[1] = {(cuuint64_t)w->K16 * 2};
    cuuint32_t box[2] = {BK16, (cuuint32_t)(pair ? p.BN / 2 : p.BN)};
    DCAE_TRY(encode_map(&map_bh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, w->w16_hi, 2, dims, str, box));
    DCAE_TRY(encode_map(&map_bl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, w->w16_lo, 2, dims, str, box));
  }
  if (!p.has_o32) map_o32 = map_bh;       // unused by the kernel
  if (!p.has_o16) { map_oh = map_bh; map_ol = map_bh; }
  if (!p.has_o16a) { map_oha = map_bh; map_ola = map_bh; }
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    const void* kernels[4] = {(const void*)gemm_f16x3_kernel<2>, (const void*)gemm_f16x3_kernel<4>,
                              (const void*)gemm_f16x3_pair_kernel<2>, (const void*)gemm_f16x3_pair_kernel<4>};
    for (int i = 0; i < 4 && attr_err == cudaSuccess; ++i)
      attr_err = cudaFuncSetAttribute(kernels[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT - 1024);
  });
  DCAE_CUDA(attr_err);
  const int n_ctas = pair ? 2 * (p.total_tiles < num_sms() / 2 ? p.total_tiles : num_sms() / 2)
                          : (p.total_tiles < num_sms() ? p.total_tiles : num_sms());
  // the pair kernel's cluster shape is fixed at compile time (__cluster_dims__)
  const bool nb2 = p.BN <= 128;
  const auto kernel = pair ? (nb2 ? gemm_f16x3_pair_kernel<2> : gemm_f16x3_pair_kernel<4>)
                           : (nb2 ? gemm_f16x3_kernel<2> : gemm_f16x3_kernel<4>);
  kernel<<<n_ctas, NTHREADS, smem, s>>>(map_ah, map_al, map_bh, map_bl, map_o32, map_oh, map_ol, map_oha, map_ola, p);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae

extern "C" int64_t dcae_planes_bytes(int64_t T, int32_t cols) {
  const int64_t Kp = (cols + 63) / 64 * 64;
  return 2 * T * Kp * 2 + 256;
}

extern "C" int dcae_split_f16_weight(const float* w, int32_t N, int32_t taps, int32_t kc, float scale, void* hi, void* lo, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(w && hi && lo && N > 0 && taps > 0 && kc > 0 && scale > 0.f, "dcae_split_f16_weight: bad arguments");
  const int Kp = (kc + 63) / 64 * 64;
  const int64_t n = (int64_t)N * taps * Kp;
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  split_f16_weight_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(w, N, taps, kc, Kp, scale, static_cast<__half*>(hi), static_cast<__half*>(lo));
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}
