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
constexpr int MAX_GROUPS = 8;     // 16-column groups per drain thread: BN/2 <= 128
constexpr int REGS_CTRL = 40, REGS_SPLIT = 64, REGS_DRAIN = 200;   // 128*40 + 128*64 + 256*200 <= 65536
constexpr int CHUNK_MMAS = 96;    // longest TMEM accumulation chain (RZ bias ~1.75e-8 per MMA)
constexpr uint32_t SMEM_LIMIT = 227 * 1024;

struct TcParams {
  dcae_epilogue e;
  int N, KB;                 // KB = K / 32 k-blocks
  int cblk_per_tap;          // (k0 + k1) / 32
  int col0, k0, col1;
  int taps;
  int B, h, w, TH, TW, tw_shift, tiles_x, tiles_y;
  int BN, stages, tmem_cols;
  int n_tiles_n, total_tiles, chunk_kb;
  uint32_t stage_bytes, b_bytes;
};

// Persistent kernel: grid = min(#tiles, #SMs); each CTA walks tiles t = blockIdx.x + i * gridDim.x in
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
template <int PASSES>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_bh,
                    const __grid_constant__ CUtensorMap map_bl, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], ready_bar[MAX_STAGES], empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp: provably uniform
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B atoms need 1024-B alignment

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&ready_bar[s]), 128);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[b]), NDRAIN);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bh) : "memory");
    if (PASSES == 3) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bl) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  // per-stage smem carve-up: [A | A_lo (x3) | B_hi | B_lo (x3)]
  const uint32_t off_al = A_BYTES;
  const uint32_t off_bh = (PASSES == 3) ? 2 * A_BYTES : A_BYTES;
  const uint32_t off_bl = off_bh + p.b_bytes;
  const int n_chunks = (p.KB + p.chunk_kb - 1) / p.chunk_kb;

  auto tile_coords = [&](int t, int& b, int& y0, int& x0, int& n0) {
    const int nt = t % p.n_tiles_n;
    int mt = t / p.n_tiles_n;
    const int tile_x = mt % p.tiles_x; mt /= p.tiles_x;
    const int tile_y = mt % p.tiles_y;
    b = mt / p.tiles_y;
    x0 = tile_x * p.TW; y0 = tile_y * p.TH; n0 = nt * p.BN;
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
    if (warp == 0) {
      // ===================== TMA producer (warp-uniform; one elected lane issues, see elect_one) =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
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
            mbar_expect_tx(fb, A_BYTES + (PASSES == 3 ? 2 : 1) * p.b_bytes);
            tma_load_4d(sbase, &map_a, fb, col, x0 + dx, y0 + dy, b);
            tma_load_2d(sbase + off_bh, &map_bh, fb, kb * BK, n0);
            if (PASSES == 3) tma_load_2d(sbase + off_bl, &map_bl, fb, kb * BK, n0);
          }
          __syncwarp();
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    } else if (warp == 1) {
      // ===================== MMA issuer (warp-uniform; one elected lane issues) =====================
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0, gchunk = 0;
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
          const uint32_t buf = gchunk & 1;
          mbar_wait(smem_u32(&tmem_empty_bar[buf]), ((gchunk >> 1) & 1) ^ 1);   // drained by the epilogue warps
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tmem_acc = tmem_base + buf * (uint32_t)p.BN;
          const int kb_end = min(p.KB, (ck + 1) * p.chunk_kb);
          for (int kb = ck * p.chunk_kb; kb < kb_end; ++kb) {
            mbar_wait(smem_u32(PASSES == 3 ? &ready_bar[stage] : &full_bar[stage]), phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sbase = smem0 + stage * p.stage_bytes;
            const uint32_t first = (kb == ck * p.chunk_kb) ? 0u : 1u;
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint32_t koff = k * UMMA_K * 4;
                const uint64_t a_hi = make_smem_desc(sbase + koff);
                const uint64_t b_hi = make_smem_desc(sbase + off_bh + koff);
                if (PASSES == 3) {
                  const uint64_t a_lo = make_smem_desc(sbase + off_al + koff);
                  const uint64_t b_lo = make_smem_desc(sbase + off_bl + koff);
                  mma_tf32(tmem_acc, a_lo, b_hi, idesc, first | (uint32_t)(k != 0));
                  mma_tf32(tmem_acc, a_hi, b_lo, idesc, 1);
                  mma_tf32(tmem_acc, a_hi, b_hi, idesc, 1);
                } else {
                  mma_tf32(tmem_acc, a_hi, b_hi, idesc, first | (uint32_t)(k != 0));
                }
              }
              mma_commit(smem_u32(&empty_bar[stage]));       // frees the smem slot once these MMAs retire
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          if (elect_one()) mma_commit(smem_u32(&tmem_full_bar[buf]));       // this chain is complete
          __syncwarp();
        }
      }
    }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_SPLIT));
    if (PASSES == 3) {
      // ===================== split warps: a -> (a_hi in place, a_lo) =====================
      const int st = threadIdx.x - 128;   // 0..127
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
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
          mbar_arrive(smem_u32(&ready_bar[stage]));
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_DRAIN));
    // ===================== drain + epilogue warps =====================
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may touch
    const int half = (warp - 8) >> 2;              // even / odd 32-column blocks
    uint32_t gchunk = 0;
    for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
      EpiTile et;
      tile_coords(t, et.b, et.y0, et.x0, et.n0);
      et.B = p.B; et.h = p.h; et.w = p.w; et.tw_shift = p.tw_shift; et.N = p.N; et.BN = p.BN;
      float acc[EPI_BLOCKS * 32];
      for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
        const uint32_t buf = gchunk & 1;
        mbar_wait(smem_u32(&tmem_full_bar[buf]), (gchunk >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        drain_chunk(acc, tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)p.BN, half, p.BN, ck == 0);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        mbar_arrive(smem_u32(&tmem_empty_bar[buf]));   // the MMA warp may start the next chain in this buffer
      }
      // ---- epilogue of this tile (overlaps the next tile's mainloop) ----
      epilogue_store(acc, p.e, et, quarter, half, lane);
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
void pick_tile(int h, int w, int* TH, int* TW) {
  // 128 tokens per tile as a TH x TW box inside one image; minimise the number of tiles
  int best = 1 << 30;
  for (int tw = 128; tw >= 1; tw >>= 1) {
    const int th = 128 / tw;
    const int tiles = ((h + th - 1) / th) * ((w + tw - 1) / tw);
    // prefer wide-ish boxes (tw = 16) on ties: longer contiguous rows per TMA line group
    if (tiles < best || (tiles == best && tw == 16)) { best = tiles; *TH = th; *TW = tw; }
  }
}

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
  // thread-block-pair kernel (gemm_tcgen05_2cta.cu).  Measured (profiles/r01/gemm_ab_v3.jsonl): it wins on long-K
  // 3-pass layers (cc1: K = 8640..10944, +8 %) and loses on short K, where the extra cross-CTA handshakes are not amortised.
  if (passes == 3 && w->K >= 4096) {
    const int rc = gemm_tcgen05_2cta(a, w, e, passes, pick_bn(w->N), s);
    if (rc != 1) return rc;
  }
  TcParams p;
  p.e = *e;
  p.N = w->N;
  p.KB = w->K / BK;
  p.cblk_per_tap = (a->k0 + a->k1) / BK;
  p.col0 = a->col0; p.k0 = a->k0; p.col1 = a->col1;
  p.taps = a->taps;
  p.B = a->B; p.h = a->h; p.w = a->w;
  pick_tile(a->h, a->w, &p.TH, &p.TW);
  p.tw_shift = 0;
  while ((1 << p.tw_shift) < p.TW) ++p.tw_shift;
  p.tiles_x = (a->w + p.TW - 1) / p.TW;
  p.tiles_y = (a->h + p.TH - 1) / p.TH;
  p.BN = pick_bn(w->N);
  DCAE_REQUIRE(p.BN > 0, "gemm(tcgen05): N=%d must be a multiple of 32", w->N);
  p.tmem_cols = 2 * p.BN <= 64 ? 64 : 2 * p.BN <= 128 ? 128 : 2 * p.BN <= 256 ? 256 : 512;   // two chain buffers
  p.n_tiles_n = w->N / p.BN;
  p.total_tiles = p.n_tiles_n * p.tiles_x * p.tiles_y * a->B;
  p.chunk_kb = (passes == 3) ? CHUNK_MMAS / 12 : p.KB;   // 3-pass: 12 MMAs per k-block; 1-pass: one chain
  p.b_bytes = (uint32_t)p.BN * BK * 4;
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
    cuuint32_t box[4] = {BK, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1};
    DCAE_TRY(encode_map(&map_a, a->base, 4, dims, str, box));
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)w->K, (cuuint64_t)w->N};
    cuuint64_t str[1] = {(cuuint64_t)w->K * 4};
    cuuint32_t box[2] = {BK, (cuuint32_t)p.BN};
    DCAE_TRY(encode_map(&map_bh, w->w_hi, 2, dims, str, box));
    if (passes == 3) DCAE_TRY(encode_map(&map_bl, w->w_lo, 2, dims, str, box));
    else map_bl = map_bh;
  }
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    attr_err = cudaFuncSetAttribute(gemm_tcgen05_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT - 1024);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(gemm_tcgen05_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT - 1024);
  });
  DCAE_CUDA(attr_err);
  const int ctas = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
  dim3 grid((unsigned)ctas);
  if (passes == 3) gemm_tcgen05_kernel<3><<<grid, NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
  else gemm_tcgen05_kernel<1><<<grid, NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae
