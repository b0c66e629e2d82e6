// tcgen05 / TMEM / TMA GEMM for the dense layers of the entropy model (Linear, 1x1 conv and 3x3
// conv as implicit GEMM; /root/reference/models/dcae.py:482-507, :584-611).
//
//   acc[128 tokens, BN] (fp32, TMEM)  +=  A[128, 32] (smem, K-major, SWIZZLE_128B) * W[BN, 32]^T
//
// * A tile = one TMA 4-D box {32 ch, TW, TH, 1} of the token-major activation viewed as
//   [B][h][w][ld]; the 3x3 taps are the same box shifted by (dy, dx) with hardware zero fill
//   outside the image -- the convolution padding costs nothing and no im2col buffer exists.
// * kind::tf32 MMA, M = 128, N = BN (<= 256), K = 8 per instruction, fp32 accumulate in TMEM.
// * PASSES == 3 (DCAE_MATH_TF32X3): fp32-level accuracy on the TF32 pipe.  Four "split" warps
//   rewrite each landed A tile in place as a_hi = tf32(a) and store a_lo = tf32(a - a_hi) next to
//   it; weights are pre-split (w_hi, w_lo) once per weight load.  Per k-step the MMA warp issues
//   a_lo*w_hi + a_hi*w_lo + a_hi*w_hi.  The dropped a_lo*w_lo term is O(2^-22).
// * PASSES == 1 (DCAE_MATH_TF32): operands go TMA -> MMA untouched (hardware truncates to TF32).
// * warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2..5 = split warps, then the
//   epilogue (tcgen05.ld 32x32b -> bias / addend / GELU / 0.5 tanh / scaled residual -> st.global).
//
// Thread-block-pair variant (tcgen05 cta_group::2, 3-pass only).  With one CTA per tile the 3-pass mainloop
// needs ~58 B/clk/SM from L2 (A + B_hi + B_lo per k-block) and only 2-3 stages fit in shared memory; the sweep
// in profiles/r01/gemm_knobs_v2.jsonl shows it starving.  Two CTAs (one SM pair) compute a 256-token x BN tile
// with M = 256 MMAs issued by the leader CTA: each CTA loads its own 128-token A tile and only HALF of the
// weight tile (BN/2 rows), so the weight traffic and its shared-memory footprint are halved (BN = 256: 64 KB
// per stage -> 3 stages, 31 B/clk/SM) while the MMA instruction does twice the work per issue.
//
// Every mbarrier wait is bounded: a protocol bug traps instead of hanging the GPU.
#include <cuda.h>

#include <mutex>

#include "common.cuh"
#include "tc_common.cuh"

namespace dcae {

namespace {

constexpr int BM = 128;        // tokens per tile (TMEM lanes)
constexpr int BK = 32;         // fp32 per k-block = 128 B = one swizzle row
constexpr int UMMA_K = 8;      // tf32
constexpr int MAX_STAGES = 8;
constexpr int A_BYTES = BM * BK * 4;   // 16 KB
constexpr int NTHREADS = 512;     // 16 warps, see the role table at the kernel
constexpr int NDRAIN = 256;       // drain/epilogue threads (warps 8..15)
constexpr int REGS_CTRL = 40, REGS_SPLIT = 64, REGS_DRAIN = 200;   // 128*40 + 128*64 + 256*200 <= 65536
constexpr int CHUNK_MMAS = 96;    // longest TMEM accumulation chain (RZ bias ~1.75e-8 per MMA)
constexpr uint32_t SMEM_LIMIT = 227 * 1024;

struct TcParams {
  dcae_epilogue e;
  int N, KB;                 // KB = K / 32 k-blocks
  int cblk_per_tap;          // (k0 + k1) / 32
  int col0, k0, col1;
  int taps;
  int B, h, w;
  TokenTiling tt;
  int BN, stages, tmem_cols;
  int n_tiles_n, total_tiles, chunk_kb;   // total_tiles: of CTAs, or of pairs (256 tokens x BN each)
  uint32_t stage_bytes, b_bytes;          // b_bytes: this CTA's weight rows (a pair's CTA holds BN/2) x 128 B
};

// Persistent kernel: grid = min(#tiles, #SMs) CTAs (or pairs); each walks its tiles in
// (token-tile major, n-tile minor) order so that CTAs running together share A tiles through L2.
//
// Accuracy: the tensor core's fp32 accumulator rounds toward zero, which biases a long accumulation
// chain by ~1.75e-8 per MMA (measured: 5.7e-5 at K = 8640).  Each TMEM chain is therefore limited to
// `chunk_kb` k-blocks (96 MMAs in the 3-pass mode); chains alternate between two TMEM buffers and the
// drain warps add the chunk partials into fp32 registers with round-to-nearest while the MMA warp is
// already filling the other buffer.  The same double buffering overlaps the epilogue of tile i with
// the mainloop of tile i+1.
//
// Warps: 0 = TMA producer, 1 = TMEM owner + MMA issuer, 2-3 idle, 4-7 = split warps (3-pass mode),
// 8-15 = drain/epilogue (two warps per TMEM lane quarter, half of the BN columns each).
// Registers are re-balanced with setmaxnreg: the drain warps hold BN/2 running sums per thread.
//
// PAIR: the MMA warp of the leader CTA issues for both CTAs.  Barriers (S stages): full[S] local (the CTA's own
// A tile landed; single CTA: its weights too), b_full[S] in the leader (weights of both CTAs), ready[S] in the
// leader (256 split threads of both CTAs), empty[S] and tmem_full[2] in both CTAs (multicast tcgen05.commit),
// tmem_empty[2] in the leader (512 drain threads).
template <bool PAIR, int PASSES>
__device__ __forceinline__ void gemm_tf32_body(const CUtensorMap& map_a, const CUtensorMap& map_bh, const CUtensorMap& map_bl,
                                               const TcParams& p) {
  static_assert(!PAIR || PASSES == 3, "the pair kernel runs the 3-pass mode only");
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], b_full[PAIR ? MAX_STAGES : 1], ready_bar[MAX_STAGES], empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp, rank: provably uniform
  const uint32_t rank = PAIR ? __shfl_sync(0xffffffffu, cluster_ctarank(), 0) : 0u;
  const bool leader = rank == 0;
  // a persistent worker (a CTA, or a pair) walks tiles first_tile(), + tile_stride(), ...  Both are re-read at every
  // use: held in registers across the kernel, they cost the single-CTA kernel 100 bytes of spill stores.
  auto first_tile = [] { return PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x; };
  auto tile_stride = [] { return PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x; };
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B atoms need 1024-B alignment

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      if (PAIR) mbar_init(smem_u32(&b_full[s]), 1);
      mbar_init(smem_u32(&ready_bar[s]), PAIR ? 256 : 128);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[b]), PAIR ? 2 * NDRAIN : NDRAIN);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bh) : "memory");
    if (PASSES == 3) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bl) : "memory");
  }
  if (warp == 1) tmem_alloc<PAIR ? 2 : 1>(smem_u32(&tmem_base_slot), p.tmem_cols);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (PAIR) cluster_sync_all();     // the peer's barriers exist before anything signals them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  // per-stage smem carve-up: [A | A_lo (x3) | B_hi | B_lo (x3)]
  const uint32_t off_al = A_BYTES;
  const uint32_t off_bh = (PASSES == 3) ? 2 * A_BYTES : A_BYTES;
  const uint32_t off_bl = off_bh + p.b_bytes;
  const int n_chunks = (p.KB + p.chunk_kb - 1) / p.chunk_kb;

  // tile -> this CTA's token tile (b, y0, x0) and the tile's first output column n0
  auto tile_coords = [&](int t, int& b, int& y0, int& x0, int& n0) {
    const int nt = t % p.n_tiles_n;
    int mt = PAIR ? (t / p.n_tiles_n) * 2 + (int)rank : t / p.n_tiles_n;   // b may reach B for a pair's odd tail tile:
    const int tile_x = mt % p.tt.tiles_x; mt /= p.tt.tiles_x;                 // TMA zero-fills, the epilogue skips it
    const int tile_y = mt % p.tt.tiles_y;
    b = mt / p.tt.tiles_y;
    x0 = tile_x * p.tt.TW; y0 = tile_y * p.tt.TH; n0 = nt * p.BN;
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
    if (warp == 0) {
      // ===================== TMA producer (warp-uniform; one elected lane issues, see elect_one) =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int t = first_tile(); t < p.total_tiles; t += tile_stride()) {
        int b, y0, x0, n0;
        tile_coords(t, b, y0, x0, n0);
        for (int kb = 0; kb < p.KB; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t sbase = smem0 + stage * p.stage_bytes;
          const uint32_t fb = smem_u32(&full_bar[stage]);
          const int tap = kb / p.cblk_per_tap;
          const int c = (kb - tap * p.cblk_per_tap) * BK;
          const int col = (c < p.k0) ? (p.col0 + c) : (p.col1 + (c - p.k0));
          int dy = 0, dx = 0;
          if (p.taps == 9) { dy = tap / 3 - 1; dx = tap % 3 - 1; }
          if (elect_one()) {
            if (PAIR) {
              const uint32_t bf = smem_u32(&b_full[stage]);
              const int nrow = n0 + (int)rank * (p.BN >> 1);
              mbar_expect_tx(fb, A_BYTES);
              tma_load_4d(sbase, &map_a, fb, col, x0 + dx, y0 + dy, b);
              if (leader) mbar_expect_tx(bf, 4 * p.b_bytes);            // hi + lo halves of both CTAs
              tma_load_2d_2sm(sbase + off_bh, &map_bh, bf, kb * BK, nrow);
              tma_load_2d_2sm(sbase + off_bl, &map_bl, bf, kb * BK, nrow);
            } else {
              mbar_expect_tx(fb, A_BYTES + (PASSES == 3 ? 2 : 1) * p.b_bytes);
              tma_load_4d(sbase, &map_a, fb, col, x0 + dx, y0 + dy, b);
              tma_load_2d(sbase + off_bh, &map_bh, fb, kb * BK, n0);
              if (PASSES == 3) tma_load_2d(sbase + off_bl, &map_bl, fb, kb * BK, n0);
            }
          }
          __syncwarp();
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    } else if (warp == 1 && leader) {
      // ===================== MMA issuer (the leader CTA of a pair; warp-uniform, one elected lane issues) =====================
      const uint32_t idesc = make_idesc_tf32((PAIR ? 2 : 1) * BM, p.BN);
      int stage = 0;
      uint32_t phase = 0, gchunk = 0;
      for (int t = first_tile(); t < p.total_tiles; t += tile_stride()) {
        for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
          const uint32_t buf = gchunk & 1;
          if (PAIR) mbar_wait_cluster(smem_u32(&tmem_empty_bar[buf]), ((gchunk >> 1) & 1) ^ 1);   // drained by the epilogue warps
          else mbar_wait(smem_u32(&tmem_empty_bar[buf]), ((gchunk >> 1) & 1) ^ 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tmem_acc = tmem_base + buf * (uint32_t)p.BN;
          const int kb_end = min(p.KB, (ck + 1) * p.chunk_kb);
          for (int kb = ck * p.chunk_kb; kb < kb_end; ++kb) {
            if (PAIR) {
              mbar_wait_cluster(smem_u32(&ready_bar[stage]), phase);
              mbar_wait_cluster(smem_u32(&b_full[stage]), phase);
            } else {
              mbar_wait(smem_u32(PASSES == 3 ? &ready_bar[stage] : &full_bar[stage]), phase);
            }
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sbase = smem0 + stage * p.stage_bytes;
            const uint32_t first = (kb == ck * p.chunk_kb) ? 0u : 1u;
            auto mma = [&](uint64_t a, uint64_t b, uint32_t accumulate) {
              if (PAIR) mma_tf32_2sm(tmem_acc, a, b, idesc, accumulate); else mma_tf32(tmem_acc, a, b, idesc, accumulate);
            };
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint32_t koff = k * UMMA_K * 4;
                const uint64_t a_hi = make_smem_desc(sbase + koff);
                const uint64_t b_hi = make_smem_desc(sbase + off_bh + koff);
                if (PASSES == 3) {
                  const uint64_t a_lo = make_smem_desc(sbase + off_al + koff);
                  const uint64_t b_lo = make_smem_desc(sbase + off_bl + koff);
                  mma(a_lo, b_hi, first | (uint32_t)(k != 0));
                  mma(a_hi, b_lo, 1);
                  mma(a_hi, b_hi, 1);
                } else {
                  mma(a_hi, b_hi, first | (uint32_t)(k != 0));
                }
              }
              // frees the smem slot (of both CTAs) once these MMAs retire
              if (PAIR) mma_commit_2sm(smem_u32(&empty_bar[stage])); else mma_commit(smem_u32(&empty_bar[stage]));
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          if (elect_one()) {        // this chain is complete (a pair: both CTAs drain their half)
            if (PAIR) mma_commit_2sm(smem_u32(&tmem_full_bar[buf])); else mma_commit(smem_u32(&tmem_full_bar[buf]));
          }
          __syncwarp();
        }
      }
    }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_SPLIT));
    if (PASSES == 3) {
      // ===================== split warps: own A tile -> (a_hi in place, a_lo) =====================
      const int st = threadIdx.x - 128;   // 0..127
      int stage = 0;
      uint32_t phase = 0;
      for (int t = first_tile(); t < p.total_tiles; t += tile_stride()) {
        for (int kb = 0; kb < p.KB; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          const uint32_t sbase = smem0 + stage * p.stage_bytes;
#pragma unroll
          for (int i = 0; i < A_BYTES / 16 / 128; ++i) {
            const uint32_t off = (uint32_t)(st + i * 128) * 16;
            float4 v;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(sbase + off));
            float4 hi, lo;
            hi.x = tf32_rna(v.x); hi.y = tf32_rna(v.y); hi.z = tf32_rna(v.z); hi.w = tf32_rna(v.w);
            lo.x = tf32_rna(v.x - hi.x); lo.y = tf32_rna(v.y - hi.y); lo.z = tf32_rna(v.z - hi.z); lo.w = tf32_rna(v.w - hi.w);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sbase + off), "f"(hi.x), "f"(hi.y), "f"(hi.z), "f"(hi.w) : "memory");
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sbase + off_al + off), "f"(lo.x), "f"(lo.y), "f"(lo.z), "f"(lo.w) : "memory");
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the MMA (async proxy)
          if (PAIR) mbar_arrive_cluster(smem_u32(&ready_bar[stage]), 0);      // the leader's barrier counts both CTAs
          else mbar_arrive(smem_u32(&ready_bar[stage]));
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_DRAIN));
    // ===================== drain + epilogue warps (own 128 rows) =====================
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may touch
    const int half = (warp - 8) >> 2;              // even / odd 32-column blocks
    uint32_t gchunk = 0;
    for (int t = first_tile(); t < p.total_tiles; t += tile_stride()) {
      EpiTile et;
      tile_coords(t, et.b, et.y0, et.x0, et.n0);
      et.B = p.B; et.h = p.h; et.w = p.w; et.tw_shift = p.tt.tw_shift; et.N = p.N; et.BN = p.BN;
      float acc[EPI_BLOCKS * 32];
      for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
        const uint32_t buf = gchunk & 1;
        mbar_wait(smem_u32(&tmem_full_bar[buf]), (gchunk >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        drain_chunk(acc, tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)p.BN, half, p.BN, ck == 0);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        // the MMA warp may start the next chain in this buffer
        if (PAIR) mbar_arrive_cluster(smem_u32(&tmem_empty_bar[buf]), 0); else mbar_arrive(smem_u32(&tmem_empty_bar[buf]));
      }
      // ---- epilogue of this tile (overlaps the next tile's mainloop) ----
      epilogue_store(acc, p.e, et, quarter, half, lane);
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (PAIR) cluster_sync_all();     // neither CTA may free TMEM / exit while the pair still uses its smem or TMEM
  if (warp == 1) tmem_dealloc<PAIR ? 2 : 1>(tmem_base, p.tmem_cols);
}

template <int PASSES>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_bh,
                    const __grid_constant__ CUtensorMap map_bl, const TcParams p) {
  gemm_tf32_body<false, PASSES>(map_a, map_bh, map_bl, p);
}

template <int PASSES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
gemm_tcgen05_2cta_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_bh,
                         const __grid_constant__ CUtensorMap map_bl, const TcParams p) {
  gemm_tf32_body<true, PASSES>(map_a, map_bh, map_bl, p);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int pick_bn(int N) {
  for (int bn = 256; bn >= 32; bn -= 32)
    if (N % bn == 0) return bn;
  return 0;
}

}  // namespace

int gemm_tcgen05(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int passes, cudaStream_t s) {
  DCAE_REQUIRE(w->w_hi != nullptr && (passes == 1 || w->w_lo != nullptr), "gemm(tcgen05): weight has no TF32 split (w_hi/w_lo)");
  DCAE_REQUIRE(aligned16(w->w_hi) && aligned16(w->w_lo), "gemm(tcgen05): split weights must be 16-byte aligned");
  DCAE_REQUIRE(e->act_cols <= 0 || e->act_cols >= w->N || e->act_cols % 32 == 0, "gemm(tcgen05): act_cols must be a multiple of 32");
  const int64_t T = (int64_t)a->B * a->h * a->w;
  if (T == 0) return DCAE_OK;
  TcParams p;
  p.e = *e;
  p.N = w->N;
  p.KB = w->K / BK;
  p.cblk_per_tap = (a->k0 + a->k1) / BK;
  p.col0 = a->col0; p.k0 = a->k0; p.col1 = a->col1;
  p.taps = a->taps;
  p.B = a->B; p.h = a->h; p.w = a->w;
  p.tt = token_tiling(a->h, a->w);
  p.BN = pick_bn(w->N);
  DCAE_REQUIRE(p.BN > 0, "gemm(tcgen05): N=%d must be a multiple of 32", w->N);
  const int m_tiles = p.tt.tiles_x * p.tt.tiles_y * a->B;
  // The thread-block pair needs two token tiles and BN/2 weight rows per CTA, a multiple of 16 (pick_bn returns a
  // multiple of 32).  Measured (profiles/r01/gemm_ab_v3.jsonl): it wins on long-K 3-pass layers (cc1: K = 8640..10944,
  // +8 %) and loses on short K, where the extra cross-CTA handshakes are not amortised.
  const bool pair = passes == 3 && w->K >= 4096 && p.BN % 32 == 0 && m_tiles >= 2;
  p.tmem_cols = 2 * p.BN <= 64 ? 64 : 2 * p.BN <= 128 ? 128 : 2 * p.BN <= 256 ? 256 : 512;   // two chain buffers
  p.n_tiles_n = w->N / p.BN;
  p.total_tiles = p.n_tiles_n * (pair ? (m_tiles + 1) / 2 : m_tiles);
  p.chunk_kb = (passes == 3) ? CHUNK_MMAS / 12 : p.KB;   // 3-pass: 12 MMAs per k-block; 1-pass: one chain
  p.b_bytes = (uint32_t)(pair ? p.BN / 2 : p.BN) * BK * 4;
  p.stage_bytes = (passes == 3) ? (2 * A_BYTES + 2 * p.b_bytes) : (A_BYTES + p.b_bytes);
  p.stages = (int)((SMEM_LIMIT - 2048) / p.stage_bytes);
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  if (p.stages > p.KB) p.stages = p.KB;
  DCAE_REQUIRE(p.stages >= 1, "gemm(tcgen05): tile does not fit in shared memory");
  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024;

  CUtensorMap map_a, map_bh, map_bl;
  {
    cuuint64_t dims[4] = {(cuuint64_t)a->ld, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->B};
    cuuint64_t str[3] = {(cuuint64_t)a->ld * 4, (cuuint64_t)a->ld * 4 * a->w, (cuuint64_t)a->ld * 4 * a->w * a->h};
    cuuint32_t box[4] = {BK, (cuuint32_t)p.tt.TW, (cuuint32_t)p.tt.TH, 1};
    DCAE_TRY(encode_map(&map_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a->base, 4, dims, str, box));
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)w->K, (cuuint64_t)w->N};
    cuuint64_t str[1] = {(cuuint64_t)w->K * 4};
    cuuint32_t box[2] = {BK, (cuuint32_t)(pair ? p.BN / 2 : p.BN)};
    DCAE_TRY(encode_map(&map_bh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w->w_hi, 2, dims, str, box));
    if (passes == 3) DCAE_TRY(encode_map(&map_bl, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w->w_lo, 2, dims, str, box));
    else map_bl = map_bh;
  }
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    const void* kernels[3] = {(const void*)gemm_tcgen05_kernel<1>, (const void*)gemm_tcgen05_kernel<3>,
                              (const void*)gemm_tcgen05_2cta_kernel<3>};
    for (int i = 0; i < 3 && attr_err == cudaSuccess; ++i)
      attr_err = cudaFuncSetAttribute(kernels[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT - 1024);
  });
  DCAE_CUDA(attr_err);
  if (pair) {       // the pair kernel's cluster shape is fixed at compile time (__cluster_dims__)
    const int max_pairs = num_sms() / 2;
    const int pairs = p.total_tiles < max_pairs ? p.total_tiles : max_pairs;
    gemm_tcgen05_2cta_kernel<3><<<dim3((unsigned)(2 * pairs)), NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
  } else {
    const int ctas = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
    if (passes == 3) gemm_tcgen05_kernel<3><<<dim3((unsigned)ctas), NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
    else gemm_tcgen05_kernel<1><<<dim3((unsigned)ctas), NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
  }
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae
