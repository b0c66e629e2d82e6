// PTX wrappers shared by the tcgen05 kernels (GEMM and dictionary attention): mbarrier, TMA,
// UMMA descriptors, tcgen05.mma / commit / ld / st, TF32 rounding, tensor-map encoding.
#pragma once
#include <cuda.h>

#include <mutex>

#include "common.cuh"

namespace dcae {
namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  uint64_t t0 = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    if ((++spins & 1023u) == 0) {          // never hang the GPU on a protocol bug: trap after 2 s
      uint64_t now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) __trap();
    }
  }
}
// the same wait with cluster-scope acquire: the data guarded by the barrier was written (or signalled) by the peer CTA
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  uint64_t t0 = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    if ((++spins & 1023u) == 0) {
      uint64_t now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// One lane of a CONVERGED warp.  The tcgen05 / TMA issue roles run warp-uniform and only the issue instructions sit under
// this predicate: issued from `if (lane == 0)` instead, every operand of UTCHMMA / UTMALDG (they take uniform registers)
// goes through a VOTEU / ELECT / R2UR.BROADCAST waterfall loop -- measured 14 SASS instructions per MMA for the lone
// issuing thread = 84-108 cycles per 64-cycle MMA.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr) {
  // K-major, SWIZZLE_128B: rows of 128 B, 8-row atoms 1024 B apart (SBO), LBO unused (=1), version 1
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float tf32_rna(float v) {
  uint32_t o;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(o) : "f"(v));
  return __uint_as_float(o);
}

__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  // A operand from TMEM (128 lanes x K 32-bit columns), B from shared memory
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  // A operand from TMEM: 128 lanes x 8 columns per K = 16 step (two fp16 per 32-bit column), B from shared memory
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
// ---- thread-block-pair (cta_group::2) variants ----------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of this cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t local_bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_bar), "r"(rank));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;   // clears the CTA-rank bit: the barrier of the pair's leader CTA
// TMA loads whose completion bytes are credited to the LEADER CTA's mbarrier (both CTAs of the pair issue them)
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void mma_tf32_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_f16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit: one arrival on the barrier at this offset in BOTH CTAs of the pair once all prior MMAs retire
__device__ __forceinline__ void mma_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// TMEM allocation by one whole warp (CG = 1: this CTA; CG = 2: the same columns in both CTAs of the pair).  The
// base address is written to the shared-memory word at `slot`.
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t ncols) {
  static_assert(CG == 1 || CG == 2, "cta_group is 1 or 2");
  if (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {
  static_assert(CG == 1 || CG == 2, "cta_group is 1 or 2");
  if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}

__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N) {
  // D = F32 (bits 4-5), A = B = TF32 (bits 7-9, 10-12), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
  // D = F32 (bits 4-5), A = B = F16 (format 0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- drain + epilogue shared by the GEMM kernels ---------------------------------------------------
// Drain thread layout: warp `quarter` (= warp % 4) owns TMEM lanes [32q, 32q+32) = 32 tile rows, one per
// lane.  The BN accumulator columns are cut into 32-column blocks; the two warps of a quarter take the even
// / odd blocks (<= 4 each, 128 running sums per thread).
constexpr int EPI_BLOCKS = 4;

// r[j] of lane i = M[i][j]  ->  r[j] of lane i = M[j][i]   (5 butterfly stages, 80 shuffles)
__device__ __forceinline__ void warp_transpose32(float* r, int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if ((j & s) == 0) {
        const float send = up ? r[j] : r[j | s];
        const float recv = __shfl_xor_sync(0xffffffffu, send, s);
        if (up) r[j] = recv; else r[j | s] = recv;
      }
    }
  }
}

// acc (+)= the chain partial sitting in TMEM at taddr (this warp's lane quarter, start of the chain buffer).
// Both tcgen05.ld of a 32-column block are in flight per wait (more would spill next to the 128 running sums).
__device__ __forceinline__ void drain_chunk(float* acc, uint32_t taddr, int half, int BN, bool first) {
#pragma unroll
  for (int g = 0; g < EPI_BLOCKS; ++g) {
    const int blk = 2 * g + half;
    uint32_t raw[32];
    if (blk * 32 < BN) {                        // warp-uniform
      tmem_ld16_nowait(taddr + blk * 32, raw);
      tmem_ld16_nowait(taddr + blk * 32 + 16, raw + 16);
    }
    tmem_ld_wait();
    if (blk * 32 < BN) {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float v = __uint_as_float(raw[j]);
        acc[g * 32 + j] = first ? v : __fadd_rn(acc[g * 32 + j], v);
      }
    }
  }
}

struct EpiTile {
  int b, y0, x0, n0;        // image, tile origin on the token grid, first output column
  int B, h, w, tw_shift, N, BN;
};

// Row-per-lane epilogue of one 32-column block held in r[0..32): bias / addend / activation / scaled residual, eight
// 16-byte stores per thread.  One instance with a run-time activation whose branches are disjoint loops (nothing for
// ptxas to if-convert into "evaluate erf AND tanh for every element"), called from a ROLLED block loop: fully unrolled
// (4 blocks x 3 activations) the epilogue was straight-line code that every warp ran once per tile, and instruction
// fetch set its time (see DESIGN.md, kernel 2).
__device__ __forceinline__ void epi_block(float* r, const dcae_epilogue& e, int act, int64_t token, int n0) {
  if (e.bias) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 bv = __ldg(reinterpret_cast<const float4*>(e.bias + n0 + j));
      r[j] += bv.x; r[j + 1] += bv.y; r[j + 2] += bv.z; r[j + 3] += bv.w;
    }
  }
  if (e.addend) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 ad = __ldg(reinterpret_cast<const float4*>(e.addend + token * e.addend_ld + n0 + j));
      r[j] += ad.x; r[j + 1] += ad.y; r[j + 2] += ad.z; r[j + 3] += ad.w;
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
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 rv = __ldg(reinterpret_cast<const float4*>(e.residual + token * e.residual_ld + n0 + j));
      float4 rs = make_float4(1.f, 1.f, 1.f, 1.f);
      if (e.res_scale) rs = __ldg(reinterpret_cast<const float4*>(e.res_scale + n0 + j));
      r[j] = fmaf(rv.x, rs.x, r[j]); r[j + 1] = fmaf(rv.y, rs.y, r[j + 1]);
      r[j + 2] = fmaf(rv.z, rs.z, r[j + 2]); r[j + 3] = fmaf(rv.w, rs.w, r[j + 3]);
    }
  }
  float* orow = e.out ? e.out + token * e.out_ld + n0 : nullptr;
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    const float4 v = make_float4(r[j], r[j + 1], r[j + 2], r[j + 3]);
    if (orow) *reinterpret_cast<float4*>(orow + j) = v;
    if (e.out16.hi) store_planes4(e.out16, token, n0 + j, v);
  }
}

// out = act(acc + bias + addend) + residual * res_scale for this thread's row.  act_cols (columns that get the
// activation) must be a multiple of 32 when it is smaller than N: a 32-column block is all-or-nothing.  The
// accumulator registers need static indices, so the block being processed is always acc[0..32) and the queue
// shifts down by register moves after each block (acc is consumed).
__device__ __forceinline__ void epilogue_store(float* acc, const dcae_epilogue& e, const EpiTile& t, int quarter, int half, int lane) {
  const int act_cols = (e.act_cols <= 0 || e.act_cols > t.N) ? t.N : e.act_cols;
  const int row = quarter * 32 + lane;
  const int yy = t.y0 + (row >> t.tw_shift), xx = t.x0 + (row & ((1 << t.tw_shift) - 1));
  if (t.b >= t.B || yy >= t.h || xx >= t.w) return;
  const int64_t token = ((int64_t)t.b * t.h + yy) * t.w + xx;
#pragma unroll 1
  for (int g = 0; g < EPI_BLOCKS; ++g) {
    const int blk = 2 * g + half;
    if (blk * 32 >= t.BN) break;
    const int nb0 = t.n0 + blk * 32;
    epi_block(acc, e, (nb0 < act_cols) ? e.act : DCAE_ACT_NONE, token, nb0);
#pragma unroll
    for (int i = 0; i < (EPI_BLOCKS - 1) * 32; ++i) acc[i] = acc[i + 32];
  }
}

// ---- host: cuTensorMapEncodeTiled through the runtime's driver entry point (no libcuda link) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

// rank-1..5 tiled map of `dtype` elements; dims / box innermost first, strides_bytes for dims 1..rank-1
int encode_map(CUtensorMap* m, CUtensorMapDataType dtype, const void* base, int rank, const cuuint64_t* dims,
               const cuuint64_t* strides_bytes, const cuuint32_t* box, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return DCAE_E_CUDA;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (data type %d, rank %d, dims %llu %llu, box %u %u)", (int)r,
              (int)dtype, rank, (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return DCAE_E_CUDA;
  }
  return DCAE_OK;
}

// ---- host: token tiling of the GEMMs ----
// 128 tokens per tile as a TH x TW box inside one image; minimise the number of tiles
void pick_tile(int h, int w, int* TH, int* TW) {
  int best = 1 << 30;
  for (int tw = 128; tw >= 1; tw >>= 1) {
    const int th = 128 / tw;
    const int tiles = ((h + th - 1) / th) * ((w + tw - 1) / tw);
    // prefer wide-ish boxes (tw = 16) on ties: longer contiguous rows per TMA line group
    if (tiles < best || (tiles == best && tw == 16)) { best = tiles; *TH = th; *TW = tw; }
  }
}

// token tile t_x + tiles_x * t_y covers rows [t_y * TH, +TH) and columns [t_x * TW, +TW) of an image; tile row r is
// image row r >> tw_shift, column r & (TW - 1)
struct TokenTiling {
  int TH, TW, tw_shift, tiles_x, tiles_y;
};
TokenTiling token_tiling(int h, int w) {
  TokenTiling t;
  pick_tile(h, w, &t.TH, &t.TW);
  t.tw_shift = 0;
  while ((1 << t.tw_shift) < t.TW) ++t.tw_shift;
  t.tiles_x = (w + t.TW - 1) / t.TW;
  t.tiles_y = (h + t.TH - 1) / t.TH;
  return t;
}

}  // namespace
}  // namespace dcae
