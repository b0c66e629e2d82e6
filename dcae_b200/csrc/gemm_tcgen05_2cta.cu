// Thread-block-pair (tcgen05 cta_group::2) variant of the dense / implicit-conv GEMM of gemm_tcgen05.cu.
//
// Why: with one CTA per tile the 3-pass TF32 mainloop needs ~58 B/clk/SM from L2 (A + B_hi + B_lo per
// k-block) and only 2-3 stages fit in shared memory; the sweep in profiles/r01/gemm_knobs_v2.jsonl shows it
// starving.  Here two CTAs (one SM pair) compute a 256-token x BN tile with M = 256 MMAs issued by the
// leader CTA: each CTA loads its own 128-token A tile and only HALF of the weight tile (BN/2 rows), so the
// weight traffic and its shared-memory footprint are halved (x3, BN = 256: 64 KB per stage -> 3 stages,
// 31 B/clk/SM) while the MMA instruction does twice the work per issue.
//
// Everything else matches gemm_tcgen05.cu: TMA 4-D boxes (3x3 taps = shifted boxes with zero fill),
// in-place a_hi / a_lo split by 4 warps per CTA, chains of <= 96 MMAs alternating between two TMEM
// buffers and summed in fp32 registers by the drain warps (RZ-accumulator fix), persistent pairs.
//
// Barriers (S stages): a_full[S] local (x3: the CTA's own A tile landed), b_full[S] in the leader (weights of
// both CTAs; x1: A tiles too), ready[S] in the leader (256 split threads of both CTAs), empty[S] and
// tmem_full[2] in both CTAs (multicast tcgen05.commit), tmem_empty[2] in the leader (512 drain threads).
#include "common.cuh"
#include "tc_common.cuh"

namespace dcae {

namespace {

constexpr int BM = 128, BK = 32, UMMA_K = 8;
constexpr int A_BYTES = BM * BK * 4;
constexpr int MAX_STAGES = 8;
constexpr int NTHREADS = 512, NDRAIN = 256, MAX_GROUPS = 8;
constexpr int REGS_CTRL = 40, REGS_SPLIT = 64, REGS_DRAIN = 200;
constexpr int CHUNK_MMAS = 96;
constexpr uint32_t SMEM_LIMIT = 227 * 1024;

struct Tc2Params {
  dcae_epilogue e;
  int N, KB, cblk_per_tap, col0, k0, col1, taps;
  int B, h, w, TH, TW, tw_shift, tiles_x, tiles_y;
  int BN, stages, tmem_cols;
  int n_tiles_n, m_tiles, total_pair_tiles, chunk_kb;
  uint32_t stage_bytes, bh_bytes;   // bh_bytes = (BN/2) rows x 128 B: this CTA's half of a weight tile
};

// wait with cluster-scope acquire: the data guarded by the barrier was written by the peer CTA
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

template <int PASSES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
gemm_tcgen05_2cta_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_bh,
                         const __grid_constant__ CUtensorMap map_bl, const Tc2Params p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t a_full[MAX_STAGES], b_full[MAX_STAGES], ready_bar[MAX_STAGES], empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp, rank: provably uniform
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&a_full[s]), 1);
      mbar_init(smem_u32(&b_full[s]), 1);
      mbar_init(smem_u32(&ready_bar[s]), 256);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[b]), 2 * NDRAIN);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bh) : "memory");
    if (PASSES == 3) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bl) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();       // the peer's barriers exist before anything signals them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  // per-stage smem: [A | A_lo (x3) | B_hi half | B_lo half (x3)]
  const uint32_t off_al = A_BYTES;
  const uint32_t off_bh = (PASSES == 3) ? 2 * A_BYTES : A_BYTES;
  const uint32_t off_bl = off_bh + p.bh_bytes;
  const int n_chunks = (p.KB + p.chunk_kb - 1) / p.chunk_kb;
  const int half_n = p.BN >> 1;

  // pair tile -> this CTA's token tile (b, y0, x0) and the tile's first output column n0
  auto tile_coords = [&](int pt, int& b, int& y0, int& x0, int& n0) {
    const int nt = pt % p.n_tiles_n;
    int mt = (pt / p.n_tiles_n) * 2 + (int)rank;
    const int tile_x = mt % p.tiles_x; mt /= p.tiles_x;
    const int tile_y = mt % p.tiles_y;
    b = mt / p.tiles_y;                 // may be == B for the odd tail tile: TMA zero-fills, epilogue skips
    x0 = tile_x * p.TW; y0 = tile_y * p.TH; n0 = nt * p.BN;
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
    if (warp == 0) {
      // ===================== TMA producer (both CTAs; warp-uniform, one elected lane issues) =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = pair; pt < p.total_pair_tiles; pt += npairs) {
        int b, y0, x0, n0;
        tile_coords(pt, b, y0, x0, n0);
        for (int kb = 0; kb < p.KB; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t sbase = smem0 + stage * p.stage_bytes;
          const int tap = kb / p.cblk_per_tap;
          const int c = (kb - tap * p.cblk_per_tap) * BK;
          const int col = (c < p.k0) ? (p.col0 + c) : (p.col1 + (c - p.k0));
          int dy = 0, dx = 0;
          if (p.taps == 9) { dy = tap / 3 - 1; dx = tap % 3 - 1; }
          const uint32_t bf = smem_u32(&b_full[stage]);
          const uint32_t af = smem_u32(&a_full[stage]);
          if (elect_one()) {
            if (PASSES == 3) {
              mbar_expect_tx(af, A_BYTES);
              tma_load_4d(sbase, &map_a, af, col, x0 + dx, y0 + dy, b);
              if (leader) mbar_expect_tx(bf, 4 * p.bh_bytes);            // hi + lo halves of both CTAs
              tma_load_2d_2sm(sbase + off_bh, &map_bh, bf, kb * BK, n0 + (int)rank * half_n);
              tma_load_2d_2sm(sbase + off_bl, &map_bl, bf, kb * BK, n0 + (int)rank * half_n);
            } else {
              if (leader) mbar_expect_tx(bf, 2 * (A_BYTES + p.bh_bytes));
              tma_load_4d_2sm(sbase, &map_a, bf, col, x0 + dx, y0 + dy, b);
              tma_load_2d_2sm(sbase + off_bh, &map_bh, bf, kb * BK, n0 + (int)rank * half_n);
            }
          }
          __syncwarp();
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    } else if (warp == 1 && leader) {
      // ===================== MMA issuer (leader CTA only; warp-uniform, one elected lane issues): M = 256 across the pair =====================
      const uint32_t idesc = make_idesc_tf32(2 * BM, p.BN);
      int stage = 0;
      uint32_t phase = 0, gchunk = 0;
      for (int pt = pair; pt < p.total_pair_tiles; pt += npairs) {
        for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
          const uint32_t buf = gchunk & 1;
          mbar_wait_cluster(smem_u32(&tmem_empty_bar[buf]), ((gchunk >> 1) & 1) ^ 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tmem_acc = tmem_base + buf * (uint32_t)p.BN;
          const int kb_end = min(p.KB, (ck + 1) * p.chunk_kb);
          for (int kb = ck * p.chunk_kb; kb < kb_end; ++kb) {
            if (PASSES == 3) mbar_wait_cluster(smem_u32(&ready_bar[stage]), phase);
            mbar_wait_cluster(smem_u32(&b_full[stage]), phase);
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
                  mma_tf32_2sm(tmem_acc, a_lo, b_hi, idesc, first | (uint32_t)(k != 0));
                  mma_tf32_2sm(tmem_acc, a_hi, b_lo, idesc, 1);
                  mma_tf32_2sm(tmem_acc, a_hi, b_hi, idesc, 1);
                } else {
                  mma_tf32_2sm(tmem_acc, a_hi, b_hi, idesc, first | (uint32_t)(k != 0));
                }
              }
              mma_commit_2sm(smem_u32(&empty_bar[stage]));      // frees the slot in BOTH CTAs
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          if (elect_one()) mma_commit_2sm(smem_u32(&tmem_full_bar[buf]));      // chain complete: both CTAs drain their half
          __syncwarp();
        }
      }
    }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_SPLIT));
    if (PASSES == 3) {
      // ===================== split warps (both CTAs): own A tile -> (a_hi in place, a_lo) =====================
      const int st = threadIdx.x - 128;
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = pair; pt < p.total_pair_tiles; pt += npairs) {
        for (int kb = 0; kb < p.KB; ++kb) {
          mbar_wait(smem_u32(&a_full[stage]), phase);
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
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_arrive_cluster(smem_u32(&ready_bar[stage]), 0);      // the leader's barrier counts both CTAs
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_DRAIN));
    // ===================== drain + epilogue warps (both CTAs, own 128 rows) =====================
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may touch
    const int half = (warp - 8) >> 2;              // even / odd 32-column blocks
    uint32_t gchunk = 0;
    for (int pt = pair; pt < p.total_pair_tiles; pt += npairs) {
      EpiTile et;
      tile_coords(pt, et.b, et.y0, et.x0, et.n0);
      et.B = p.B; et.h = p.h; et.w = p.w; et.tw_shift = p.tw_shift; et.N = p.N; et.BN = p.BN;
      float acc[EPI_BLOCKS * 32];
      for (int ck = 0; ck < n_chunks; ++ck, ++gchunk) {
        const uint32_t buf = gchunk & 1;
        mbar_wait(smem_u32(&tmem_full_bar[buf]), (gchunk >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        drain_chunk(acc, tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)p.BN, half, p.BN, ck == 0);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        mbar_arrive_cluster(smem_u32(&tmem_empty_bar[buf]), 0);   // the MMA warp may start the next chain in this buffer
      }
      // ---- epilogue of this tile (overlaps the next tile's mainloop) ----
      epilogue_store(acc, p.e, et, quarter, half, lane);
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();       // neither CTA may free TMEM / exit while the pair still uses its smem or TMEM
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

void pick_tile2(int h, int w, int* TH, int* TW) {
  int best = 1 << 30;
  for (int tw = 128; tw >= 1; tw >>= 1) {
    const int th = 128 / tw;
    const int tiles = ((h + th - 1) / th) * ((w + tw - 1) / tw);
    if (tiles < best || (tiles == best && tw == 16)) { best = tiles; *TH = th; *TW = tw; }
  }
}

}  // namespace

// returns DCAE_OK, an error, or 1 if the pair kernel does not apply (caller falls back to the 1-CTA kernel)
int gemm_tcgen05_2cta(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int passes, int bn, cudaStream_t s) {
  if (bn % 32 != 0 || bn < 32) return 1;      // each CTA holds bn/2 weight rows (multiple of 16) and drains bn/2 columns
  Tc2Params p;
  p.e = *e;
  p.N = w->N;
  p.KB = w->K / BK;
  p.cblk_per_tap = (a->k0 + a->k1) / BK;
  p.col0 = a->col0; p.k0 = a->k0; p.col1 = a->col1;
  p.taps = a->taps;
  p.B = a->B; p.h = a->h; p.w = a->w;
  pick_tile2(a->h, a->w, &p.TH, &p.TW);
  p.tw_shift = 0;
  while ((1 << p.tw_shift) < p.TW) ++p.tw_shift;
  p.tiles_x = (a->w + p.TW - 1) / p.TW;
  p.tiles_y = (a->h + p.TH - 1) / p.TH;
  p.BN = bn;
  p.m_tiles = p.tiles_x * p.tiles_y * a->B;
  if (p.m_tiles < 2) return 1;
  p.tmem_cols = 2 * p.BN <= 64 ? 64 : 2 * p.BN <= 128 ? 128 : 2 * p.BN <= 256 ? 256 : 512;
  p.n_tiles_n = w->N / p.BN;
  p.total_pair_tiles = p.n_tiles_n * ((p.m_tiles + 1) / 2);
  p.chunk_kb = (passes == 3) ? CHUNK_MMAS / 12 : p.KB;
  p.bh_bytes = (uint32_t)(p.BN / 2) * BK * 4;
  p.stage_bytes = (passes == 3) ? (2 * A_BYTES + 2 * p.bh_bytes) : (A_BYTES + p.bh_bytes);
  p.stages = (int)((SMEM_LIMIT - 2048) / p.stage_bytes);
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  if (p.stages > p.KB) p.stages = p.KB;
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
    cuuint32_t box[2] = {BK, (cuuint32_t)(p.BN / 2)};
    DCAE_TRY(encode_map(&map_bh, w->w_hi, 2, dims, str, box));
    if (passes == 3) DCAE_TRY(encode_map(&map_bl, w->w_lo, 2, dims, str, box));
    else map_bl = map_bh;
  }
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    attr_err = cudaFuncSetAttribute(gemm_tcgen05_2cta_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT - 1024);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(gemm_tcgen05_2cta_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT - 1024);
  });
  DCAE_CUDA(attr_err);
  const int max_pairs = num_sms() / 2;
  const int pairs = p.total_pair_tiles < max_pairs ? p.total_pair_tiles : max_pairs;
  dim3 grid((unsigned)(2 * pairs));
  if (passes == 3) gemm_tcgen05_2cta_kernel<3><<<grid, NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
  else gemm_tcgen05_2cta_kernel<1><<<grid, NTHREADS, smem, s>>>(map_a, map_bh, map_bl, p);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

}  // namespace dcae
