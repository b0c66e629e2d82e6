// MS-SSIM (pytorch_msssim.ms_ssim v1.0 with its defaults, the distortion of the reference's ms-ssim rate-distortion
// loss) as per-level statistics, forward and backward, fp32 on the device.
//   window   1-D Gaussian, 11 taps, sigma 1.5, sum 1, applied W then H as a VALID correlation: map (h-10) x (w-10)
//   moments  mu_x = G*X, mu_y = G*Y, s_xx = G*(X^2) - mu_x^2, s_yy likewise, s_xy = G*(XY) - mu_x mu_y
//   maps     cs = (2 s_xy + C2) / (s_xx + s_yy + C2),  ssim = (2 mu_x mu_y + C1) / (mu_x^2 + mu_y^2 + C1) * cs
//   levels   5; X_{l+1} = avg_pool2d(X_l, 2, 2, padding = (h % 2, w % 2)), count_include_pad (border zeros count)
// The library produces the per-(level, image, channel) means of ssim and cs, [5, B, C]; the weighted product over the
// levels stays in torch (dcae_b200/msssim.py).
//
// Forward, one launch per level: a block owns a 32 x 32 tile of one plane's valid map, stages the 42 x 42 input tile
// of X and Y in shared memory, runs the horizontal pass of the five moments (4 outputs per thread, the 14 inputs and
// their products in registers), then the vertical pass (4 rows per thread), and forms ssim and cs in registers.  The
// block's two sums go to a per-(plane, tile) fp64 partial in a fixed butterfly order.  The same block writes the 2x2
// pooled X and Y of the next level for a 16 x 16 pooled tile (the last tile row / column also takes the remainder):
// every pooled pixel has exactly one writer.  A last launch sums each plane's partials in tile order in fp64.
//
// Backward, one launch per level, coarse to fine.  With a = dL/dmean(ssim) / n, b = dL/dmean(cs) / n per plane,
// L = N1 / D1, CS = N2 / D2:
//   gL = a CS,  gC = b + a L
//   G_mu = gL dL/dmu_x + gC (-2 mu_x dCS/ds_xx - mu_y dCS/ds_xy),  G_xx = gC dCS/ds_xx,  G_xy = gC dCS/ds_xy
//   dCS/ds_xx = -N2 / D2^2,  dCS/ds_xy = 2 / D2,  dL/dmu_x = (2 mu_y D1 - 2 mu_x N1) / D1^2
//   dX_l = full(G_mu) + 2 X_l full(G_xx) + Y_l full(G_xy) + 1/4 dX_{l+1}[(i + h%2) >> 1, (j + w%2) >> 1]
// full() is the transpose of the valid correlation: the zero-padded map correlated with the same (symmetric) window.
// A block owns a 32 x 32 tile of dX_l: it loads the 54 x 54 input tile around it, recomputes the moments on the
// 44 x 44 window of valid positions that reach the tile (zero outside the valid map), forms the three G maps there,
// runs the separable full correlation and combines it with X, Y and the coarser dX.  Nothing but the pooled pyramid is
// kept from the forward pass.
// No atomics anywhere: every output element and partial has one writer and a fixed summation order, and a plane's
// results depend on that plane alone.
#include "common.cuh"

namespace dcae {

constexpr int MS_LEVELS = 5;
constexpr int MS_TAPS = 11;
constexpr int MS_T = 32;                      // output tile side
constexpr int MS_THREADS = 256;
constexpr int MS_FIN = MS_T + MS_TAPS - 1;    // forward input tile side, 42
constexpr int MS_G = 44;                      // backward: valid positions that reach a tile (42, rounded to 4)
constexpr int MS_BIN = MS_G + MS_TAPS - 1;    // backward input tile side, 54
constexpr int MS_RED_THREADS = 128;

// exp(-(k-5)^2 / 4.5) normalised to sum 1, rounded to fp32
__device__ __forceinline__ float ms_win(int k) {
  constexpr float w[6] = {0.001028380123898387f, 0.0075987582094967365f, 0.036000773310661316f, 0.10936068743467331f,
                          0.21300554275512695f, 0.26601171493530273f};
  return w[k <= 5 ? k : 10 - k];
}

struct MsLevels {
  int h[MS_LEVELS], w[MS_LEVELS];
  int tiles[MS_LEVELS];                       // forward tiles of the valid map
  size_t px[MS_LEVELS], py[MS_LEVELS], dx[MS_LEVELS], part[MS_LEVELS];   // scratch offsets (levels >= 1 for px/py/dx)
  size_t bytes;
};

inline size_t ms_align(size_t v) { return (v + 255) & ~size_t(255); }
inline int ms_tiles(int n) { return (n + MS_T - 1) / MS_T; }

// level sizes and the scratch layout: pooled X, Y and dX of levels 1..4, then the fp64 partials of every level
MsLevels ms_layout(int64_t P, int H, int W) {
  MsLevels L;
  size_t off = 0;
  for (int l = 0; l < MS_LEVELS; ++l) {
    L.h[l] = l == 0 ? H : (L.h[l - 1] + 1) / 2;   // avg_pool2d(2, 2, padding = h % 2): ceil(h / 2)
    L.w[l] = l == 0 ? W : (L.w[l - 1] + 1) / 2;
    L.tiles[l] = ms_tiles(L.h[l] - 10) * ms_tiles(L.w[l] - 10);
    L.px[l] = L.py[l] = L.dx[l] = 0;
  }
  for (int l = 1; l < MS_LEVELS; ++l) {
    const size_t n = (size_t)P * L.h[l] * L.w[l] * sizeof(float);
    L.px[l] = off; off = ms_align(off + n);
    L.py[l] = off; off = ms_align(off + n);
    L.dx[l] = off; off = ms_align(off + n);
  }
  for (int l = 0; l < MS_LEVELS; ++l) {
    L.part[l] = off;
    off = ms_align(off + (size_t)P * L.tiles[l] * sizeof(double2));
  }
  L.bytes = off;
  return L;
}

struct MsFwdLevel {
  const float* x; const float* y;
  int h, w, hv, wv, tiles_x, tiles_y;
  float* px; float* py; int hp, wp;             // pooled outputs (nullptr at the last level)
  double2* part;                                // [P, tiles]
  int64_t planes;
  float c1, c2;
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// horizontal pass of the five moments: out[m][r][c0 .. c0+3] from in_x / in_y row r, columns c0 .. c0+13
template <int LDI, int ROWS, int LDO>
__device__ __forceinline__ void ms_hpass5(const float (*sx)[LDI], const float (*sy)[LDI], float (*sh)[ROWS][LDO], int r, int c0) {
  float xv[14], yv[14];
#pragma unroll
  for (int j = 0; j < 14; ++j) { xv[j] = sx[r][c0 + j]; yv[j] = sy[r][c0 + j]; }
  float acc[4][5];
#pragma unroll
  for (int o = 0; o < 4; ++o)
#pragma unroll
    for (int m = 0; m < 5; ++m) acc[o][m] = 0.f;
#pragma unroll
  for (int j = 0; j < 14; ++j) {
    const float x = xv[j], y = yv[j], xx = x * x, yy = y * y, xy = x * y;
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const int k = j - o;
      if (k < 0 || k >= MS_TAPS) continue;
      const float g = ms_win(k);
      acc[o][0] = fmaf(g, x, acc[o][0]);
      acc[o][1] = fmaf(g, y, acc[o][1]);
      acc[o][2] = fmaf(g, xx, acc[o][2]);
      acc[o][3] = fmaf(g, yy, acc[o][3]);
      acc[o][4] = fmaf(g, xy, acc[o][4]);
    }
  }
#pragma unroll
  for (int m = 0; m < 5; ++m)
#pragma unroll
    for (int o = 0; o < 4; ++o) sh[m][r][c0 + o] = acc[o][m];
}

// vertical pass of NM maps: acc[o][m] = sum_k g_k in[m][r0 + o + k][c], o < 4
template <int NM, int ROWS, int LD>
__device__ __forceinline__ void ms_vpass(const float (*sh)[ROWS][LD], int r0, int c, float (&acc)[4][NM]) {
#pragma unroll
  for (int o = 0; o < 4; ++o)
#pragma unroll
    for (int m = 0; m < NM; ++m) acc[o][m] = 0.f;
#pragma unroll
  for (int j = 0; j < 14; ++j) {
    float v[NM];
#pragma unroll
    for (int m = 0; m < NM; ++m) v[m] = sh[m][r0 + j][c];
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const int k = j - o;
      if (k < 0 || k >= MS_TAPS) continue;
      const float g = ms_win(k);
#pragma unroll
      for (int m = 0; m < NM; ++m) acc[o][m] = fmaf(g, v[m], acc[o][m]);
    }
  }
}

// numerators and denominators of L = N1 / D1 and CS = N2 / D2 from the five filtered moments.  The products are rounded
// on their own (no FMA contraction), so that for X == Y the numerators equal the denominators bit for bit and
// MS-SSIM is exactly 1.
struct MsTerms { float n1, d1, n2, d2; };
__device__ __forceinline__ MsTerms ms_terms(const float (&m)[5], float c1, float c2) {
  const float mxx = __fmul_rn(m[0], m[0]), myy = __fmul_rn(m[1], m[1]), mxy = __fmul_rn(m[0], m[1]);
  const float sxx = m[2] - mxx, syy = m[3] - myy, sxy = m[4] - mxy;
  return {2.f * mxy + c1, mxx + myy + c1, 2.f * sxy + c2, sxx + syy + c2};
}

__global__ void __launch_bounds__(MS_THREADS) msssim_forward_kernel(const MsFwdLevel a) {
  __shared__ float sx[MS_FIN][MS_FIN], sy[MS_FIN][MS_FIN];
  __shared__ float sh[5][MS_FIN][MS_T];
  __shared__ double2 red[MS_THREADS / 32];
  const int tid = threadIdx.x;
  const int tx = blockIdx.x % a.tiles_x, ty = blockIdx.x / a.tiles_x;
  const int r0 = ty * MS_T, c0 = tx * MS_T;
  for (int64_t p = blockIdx.y; p < a.planes; p += gridDim.y) {
    const float* x = a.x + p * a.h * a.w;
    const float* y = a.y + p * a.h * a.w;
    for (int i = tid; i < MS_FIN * MS_FIN; i += MS_THREADS) {
      const int r = i / MS_FIN, c = i % MS_FIN, gr = r0 + r, gc = c0 + c;
      const bool in = gr < a.h && gc < a.w;
      sx[r][c] = in ? __ldg(x + (int64_t)gr * a.w + gc) : 0.f;
      sy[r][c] = in ? __ldg(y + (int64_t)gr * a.w + gc) : 0.f;
    }
    __syncthreads();
    for (int i = tid; i < MS_FIN * (MS_T / 4); i += MS_THREADS) ms_hpass5<MS_FIN, MS_FIN, MS_T>(sx, sy, sh, i / (MS_T / 4), 4 * (i % (MS_T / 4)));
    __syncthreads();
    float acc[4][5];
    const int c = tid % MS_T, rg = 4 * (tid / MS_T);
    ms_vpass<5, MS_FIN, MS_T>(sh, rg, c, acc);
    float s_ssim = 0.f, s_cs = 0.f;
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      if (r0 + rg + o < a.hv && c0 + c < a.wv) {
        const MsTerms t = ms_terms(acc[o], a.c1, a.c2);
        const float cs = t.n2 / t.d2;
        const float ssim = t.n1 / t.d1 * cs;
        s_ssim += ssim;
        s_cs += cs;
      }
    }
    const double ds = warp_sum_d((double)s_ssim), dc = warp_sum_d((double)s_cs);
    if ((tid & 31) == 0) red[tid >> 5] = make_double2(ds, dc);
    // the next level's input: 2 x 2 means with the leading zero row / column of an odd size
    if (a.px) {
      const int pr0 = ty * (MS_T / 2), pc0 = tx * (MS_T / 2);
      const int pr1 = ty == a.tiles_y - 1 ? a.hp : pr0 + MS_T / 2, pc1 = tx == a.tiles_x - 1 ? a.wp : pc0 + MS_T / 2;
      const int ph = a.h & 1, pw = a.w & 1, nc = pc1 - pc0;
      float* px = a.px + p * a.hp * a.wp;
      float* py = a.py + p * a.hp * a.wp;
      for (int i = tid; i < (pr1 - pr0) * nc; i += MS_THREADS) {
        const int pi = pr0 + i / nc, pj = pc0 + i % nc;
        float sumx = 0.f, sumy = 0.f;
#pragma unroll
        for (int di = 0; di < 2; ++di)
#pragma unroll
          for (int dj = 0; dj < 2; ++dj) {
            const int r = 2 * pi - ph + di, cc = 2 * pj - pw + dj;
            if (r >= 0 && cc >= 0) {
              sumx += __ldg(x + (int64_t)r * a.w + cc);
              sumy += __ldg(y + (int64_t)r * a.w + cc);
            }
          }
        px[(int64_t)pi * a.wp + pj] = 0.25f * sumx;
        py[(int64_t)pi * a.wp + pj] = 0.25f * sumy;
      }
    }
    __syncthreads();
    if (tid == 0) {
      double2 t = red[0];
#pragma unroll
      for (int w = 1; w < MS_THREADS / 32; ++w) { t.x += red[w].x; t.y += red[w].y; }
      a.part[p * gridDim.x + blockIdx.x] = t;
    }
  }
}

// out_ssim[l, p], out_cs[l, p] = sum of the plane's tile partials in tile order / n_l
struct MsReduce {
  const double2* part[MS_LEVELS];
  int tiles[MS_LEVELS];
  double inv_n[MS_LEVELS];
  int64_t planes;
  float* ssim; float* cs;
};

__global__ void __launch_bounds__(MS_RED_THREADS) msssim_reduce_kernel(const __grid_constant__ MsReduce a) {
  __shared__ double2 red[MS_RED_THREADS / 32];
  const int l = blockIdx.x;
  const int nt = a.tiles[l];
  for (int64_t p = blockIdx.y; p < a.planes; p += gridDim.y) {
    const double2* part = a.part[l] + p * nt;
    double s = 0.0, c = 0.0;
    for (int i = threadIdx.x; i < nt; i += MS_RED_THREADS) { s += part[i].x; c += part[i].y; }
    s = warp_sum_d(s);
    c = warp_sum_d(c);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = make_double2(s, c);
    __syncthreads();
    if (threadIdx.x == 0) {
      double2 t = red[0];
#pragma unroll
      for (int w = 1; w < MS_RED_THREADS / 32; ++w) { t.x += red[w].x; t.y += red[w].y; }
      a.ssim[(int64_t)l * a.planes + p] = (float)(t.x * a.inv_n[l]);
      a.cs[(int64_t)l * a.planes + p] = (float)(t.y * a.inv_n[l]);
    }
    __syncthreads();
  }
}

struct MsBwdLevel {
  const float* x; const float* y;
  int h, w, hv, wv, tiles_x;
  const float* dnext; int hn, wn;               // dX of the next (coarser) level, nullptr at the last level
  float* dx;
  const float* g_ssim; const float* g_cs;       // [P] of this level
  float n;                                      // valid pixels of this level
  int64_t planes;
  float c1, c2;
};

struct MsBwdSmem {
  float sx[MS_BIN][MS_BIN], sy[MS_BIN][MS_BIN];
  union {
    float mom[5][MS_BIN][MS_G];                 // horizontal moments
    float fh[3][MS_G][MS_T];                    // horizontal full correlation of the G maps
  };
  float g[3][MS_G][MS_G];                       // G_mu, G_xx, G_xy on the valid positions reaching the tile
};

__global__ void __launch_bounds__(MS_THREADS, 2) msssim_backward_kernel(const MsBwdLevel a) {
  extern __shared__ __align__(16) unsigned char ms_smem[];
  MsBwdSmem& S = *reinterpret_cast<MsBwdSmem*>(ms_smem);
  const int tid = threadIdx.x;
  const int tx = blockIdx.x % a.tiles_x, ty = blockIdx.x / a.tiles_x;
  const int r0 = ty * MS_T, c0 = tx * MS_T;     // dX tile origin
  const int vr0 = r0 - (MS_TAPS - 1), vc0 = c0 - (MS_TAPS - 1);   // origin of the valid-position window (and input tile)
  for (int64_t p = blockIdx.y; p < a.planes; p += gridDim.y) {
    const float* x = a.x + p * a.h * a.w;
    const float* y = a.y + p * a.h * a.w;
    const float ga = a.g_ssim[p] / a.n, gb = a.g_cs[p] / a.n;
    for (int i = tid; i < MS_BIN * MS_BIN; i += MS_THREADS) {
      const int r = i / MS_BIN, c = i % MS_BIN, gr = vr0 + r, gc = vc0 + c;
      const bool in = gr >= 0 && gc >= 0 && gr < a.h && gc < a.w;
      S.sx[r][c] = in ? __ldg(x + (int64_t)gr * a.w + gc) : 0.f;
      S.sy[r][c] = in ? __ldg(y + (int64_t)gr * a.w + gc) : 0.f;
    }
    __syncthreads();
    for (int i = tid; i < MS_BIN * (MS_G / 4); i += MS_THREADS) ms_hpass5<MS_BIN, MS_BIN, MS_G>(S.sx, S.sy, S.mom, i / (MS_G / 4), 4 * (i % (MS_G / 4)));
    __syncthreads();
    for (int i = tid; i < MS_G * (MS_G / 4); i += MS_THREADS) {
      const int c = i % MS_G, rg = 4 * (i / MS_G);
      float acc[4][5];
      ms_vpass<5, MS_BIN, MS_G>(S.mom, rg, c, acc);
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        const int vr = vr0 + rg + o, vc = vc0 + c;
        float gmu = 0.f, gxx = 0.f, gxy = 0.f;
        if (vr >= 0 && vc >= 0 && vr < a.hv && vc < a.wv) {
          const MsTerms t = ms_terms(acc[o], a.c1, a.c2);
          const float mx = acc[o][0], my = acc[o][1];
          const float lum = t.n1 / t.d1, cs = t.n2 / t.d2;
          const float gl = ga * cs, gc = gb + ga * lum;
          const float dcs_xx = -cs / t.d2, dcs_xy = 2.f / t.d2;
          const float dl_mx = (2.f * my * t.d1 - 2.f * mx * t.n1) / (t.d1 * t.d1);
          gmu = gl * dl_mx + gc * (-2.f * mx * dcs_xx - my * dcs_xy);
          gxx = gc * dcs_xx;
          gxy = gc * dcs_xy;
        }
        S.g[0][rg + o][c] = gmu;
        S.g[1][rg + o][c] = gxx;
        S.g[2][rg + o][c] = gxy;
      }
    }
    __syncthreads();
    // horizontal full correlation: fh[m][r][c] = sum_k g_k G[m][r][c + k] (the window is symmetric)
    for (int i = tid; i < (MS_G - 2) * (MS_T / 4); i += MS_THREADS) {
      const int r = i / (MS_T / 4), cg = 4 * (i % (MS_T / 4));
      float acc[4][3];
#pragma unroll
      for (int o = 0; o < 4; ++o)
#pragma unroll
        for (int m = 0; m < 3; ++m) acc[o][m] = 0.f;
#pragma unroll
      for (int j = 0; j < 14; ++j) {
        float v[3];
#pragma unroll
        for (int m = 0; m < 3; ++m) v[m] = S.g[m][r][cg + j];
#pragma unroll
        for (int o = 0; o < 4; ++o) {
          const int k = j - o;
          if (k < 0 || k >= MS_TAPS) continue;
          const float g = ms_win(k);
#pragma unroll
          for (int m = 0; m < 3; ++m) acc[o][m] = fmaf(g, v[m], acc[o][m]);
        }
      }
#pragma unroll
      for (int m = 0; m < 3; ++m)
#pragma unroll
        for (int o = 0; o < 4; ++o) S.fh[m][r][cg + o] = acc[o][m];
    }
    __syncthreads();
    {
      const int c = tid % MS_T, rg = 4 * (tid / MS_T);
      float acc[4][3];
      ms_vpass<3, MS_G, MS_T>(S.fh, rg, c, acc);
      const int j = c0 + c;
      const int ph = a.h & 1, pw = a.w & 1;
      const float* dn = a.dnext ? a.dnext + p * a.hn * a.wn : nullptr;
      float* dx = a.dx + p * a.h * a.w;
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        const int i = r0 + rg + o;
        if (i < a.h && j < a.w) {
          const float xv = S.sx[rg + o + MS_TAPS - 1][c + MS_TAPS - 1], yv = S.sy[rg + o + MS_TAPS - 1][c + MS_TAPS - 1];
          float d = acc[o][0] + 2.f * xv * acc[o][1] + yv * acc[o][2];
          if (dn) d += 0.25f * __ldg(dn + (int64_t)((i + ph) >> 1) * a.wn + ((j + pw) >> 1));
          dx[(int64_t)i * a.w + j] = d;
        }
      }
    }
    __syncthreads();
  }
}

// C1 = (0.01 R)^2, C2 = (0.03 R)^2 in double, rounded once to fp32 (pytorch_msssim's Python floats)
inline double ms_sq(double v) { return v * v; }
inline unsigned ms_plane_blocks(int64_t planes) { return (unsigned)(planes < 65535 ? planes : 65535); }

// shared argument checks of both directions; *L gets the level layout
int ms_check(const char* fn, const float* x, const float* y, int32_t B, int32_t C, int32_t H, int32_t W, float data_range,
             const void* scratch, size_t scratch_bytes, MsLevels* L) {
  DCAE_REQUIRE(x && y, "%s: null input", fn);
  DCAE_REQUIRE(B >= 0 && C > 0, "%s: bad shape B=%d C=%d", fn, B, C);
  DCAE_REQUIRE(H > 160 && W > 160, "%s: min(H, W) must exceed 160 for 5 levels of an 11-tap window (H=%d W=%d)", fn, H, W);
  DCAE_REQUIRE((int64_t)H * W < (1ll << 31), "%s: bad shape H=%d W=%d", fn, H, W);
  DCAE_REQUIRE(data_range > 0.f && data_range < INFINITY, "%s: data_range must be positive and finite", fn);
  *L = ms_layout((int64_t)B * C, H, W);
  DCAE_REQUIRE(L->bytes == 0 || (scratch != nullptr && aligned16(scratch)), "%s: scratch null or not 16-byte aligned", fn);
  DCAE_REQUIRE(scratch_bytes >= L->bytes, "%s: scratch too small (%zu < %zu bytes)", fn, scratch_bytes, L->bytes);
  return DCAE_OK;
}

}  // namespace dcae

extern "C" size_t dcae_msssim_scratch_bytes(int32_t B, int32_t C, int32_t H, int32_t W) {
  if (B < 0 || C <= 0 || H <= 160 || W <= 160 || (int64_t)H * W >= (1ll << 31)) return 0;
  return dcae::ms_layout((int64_t)B * C, H, W).bytes;
}

extern "C" int dcae_msssim_forward(const dcae_msssim_args* a, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(a != nullptr, "dcae_msssim_forward: null arguments");
  MsLevels L;
  DCAE_TRY(ms_check("dcae_msssim_forward", a->x, a->y, a->B, a->C, a->H, a->W, a->data_range, a->scratch, a->scratch_bytes, &L));
  DCAE_REQUIRE(a->ssim && a->cs, "dcae_msssim_forward: null output");
  const int64_t P = (int64_t)a->B * a->C;
  if (P == 0) return DCAE_OK;
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const cudaStream_t s = (cudaStream_t)stream;
  char* base = static_cast<char*>(a->scratch);
  const float c1 = (float)ms_sq(0.01 * a->data_range), c2 = (float)ms_sq(0.03 * a->data_range);
  MsReduce red;
  for (int l = 0; l < MS_LEVELS; ++l) {
    MsFwdLevel f;
    f.x = l == 0 ? a->x : reinterpret_cast<const float*>(base + L.px[l]);
    f.y = l == 0 ? a->y : reinterpret_cast<const float*>(base + L.py[l]);
    f.h = L.h[l]; f.w = L.w[l]; f.hv = f.h - 10; f.wv = f.w - 10;
    f.tiles_x = ms_tiles(f.wv); f.tiles_y = ms_tiles(f.hv);
    const bool last = l == MS_LEVELS - 1;
    f.px = last ? nullptr : reinterpret_cast<float*>(base + L.px[l + 1]);
    f.py = last ? nullptr : reinterpret_cast<float*>(base + L.py[l + 1]);
    f.hp = last ? 0 : L.h[l + 1]; f.wp = last ? 0 : L.w[l + 1];
    f.part = reinterpret_cast<double2*>(base + L.part[l]);
    f.planes = P;
    f.c1 = c1; f.c2 = c2;
    msssim_forward_kernel<<<dim3((unsigned)L.tiles[l], ms_plane_blocks(P)), MS_THREADS, 0, s>>>(f);
    DCAE_LAUNCH_CHECK();
    red.part[l] = f.part;
    red.tiles[l] = L.tiles[l];
    red.inv_n[l] = 1.0 / ((double)f.hv * f.wv);
  }
  red.planes = P;
  red.ssim = a->ssim;
  red.cs = a->cs;
  msssim_reduce_kernel<<<dim3(MS_LEVELS, ms_plane_blocks(P)), MS_RED_THREADS, 0, s>>>(red);
  DCAE_LAUNCH_CHECK();
  return DCAE_OK;
}

extern "C" int dcae_msssim_backward(const dcae_msssim_bwd_args* a, void* stream) {
  using namespace dcae;
  DCAE_REQUIRE(a != nullptr, "dcae_msssim_backward: null arguments");
  MsLevels L;
  DCAE_TRY(ms_check("dcae_msssim_backward", a->x, a->y, a->B, a->C, a->H, a->W, a->data_range, a->scratch, a->scratch_bytes, &L));
  DCAE_REQUIRE(a->grad_ssim && a->grad_cs, "dcae_msssim_backward: null input");
  DCAE_REQUIRE(a->grad_x, "dcae_msssim_backward: null output");
  const int64_t P = (int64_t)a->B * a->C;
  if (P == 0) return DCAE_OK;
  // once per device, so that a call inside a stream capture makes no attribute call (the race is benign: same value)
  static bool smem_set[64] = {};
  int dev = 0;
  DCAE_CUDA(cudaGetDevice(&dev));
  if (dev >= 64 || !smem_set[dev]) {
    DCAE_CUDA(cudaFuncSetAttribute(msssim_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MsBwdSmem)));
    if (dev < 64) smem_set[dev] = true;
  }
  ProfileScope prof(DCAE_PROF_OTHER, 0.0, stream);
  const cudaStream_t s = (cudaStream_t)stream;
  char* base = static_cast<char*>(a->scratch);
  const float c1 = (float)ms_sq(0.01 * a->data_range), c2 = (float)ms_sq(0.03 * a->data_range);
  for (int l = MS_LEVELS - 1; l >= 0; --l) {
    MsBwdLevel b;
    b.x = l == 0 ? a->x : reinterpret_cast<const float*>(base + L.px[l]);
    b.y = l == 0 ? a->y : reinterpret_cast<const float*>(base + L.py[l]);
    b.h = L.h[l]; b.w = L.w[l]; b.hv = b.h - 10; b.wv = b.w - 10;
    b.tiles_x = ms_tiles(b.w);
    const bool last = l == MS_LEVELS - 1;
    b.dnext = last ? nullptr : reinterpret_cast<const float*>(base + L.dx[l + 1]);
    b.hn = last ? 0 : L.h[l + 1]; b.wn = last ? 0 : L.w[l + 1];
    b.dx = l == 0 ? a->grad_x : reinterpret_cast<float*>(base + L.dx[l]);
    b.g_ssim = a->grad_ssim + (int64_t)l * P;
    b.g_cs = a->grad_cs + (int64_t)l * P;
    b.n = (float)b.hv * (float)b.wv;
    b.planes = P;
    b.c1 = c1; b.c2 = c2;
    const unsigned tiles = (unsigned)(ms_tiles(b.h) * b.tiles_x);
    msssim_backward_kernel<<<dim3(tiles, ms_plane_blocks(P)), MS_THREADS, sizeof(MsBwdSmem), s>>>(b);
    DCAE_LAUNCH_CHECK();
  }
  return DCAE_OK;
}
