/*
 * dcae_b200.h -- C ABI of libdcae_b200.so: the B200 (sm_100a) implementation of the DCAE
 * entropy-model hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  The reference has no native code; its "FFI" for this
 * path is the Python operator interface of `/root/reference/models/dcae.py` plus compressai's
 * `GaussianConditional`.  Every entry point below names the reference call it replaces.
 *
 * Conventions
 *   - plain C types only; all pointers are DEVICE pointers unless named `*_host`;
 *   - the caller owns every buffer (inputs, outputs, workspace); nothing is allocated here except
 *     the small host-side plan object returned by dcae_slice_loop_create();
 *   - work is enqueued on the given CUDA stream (a `cudaStream_t`, passed as void*) and the call
 *     returns immediately; no host synchronisation inside;
 *   - return 0 on success, a negative DCAE_E_* code otherwise; dcae_last_error() returns a
 *     thread-local message;
 *   - results are deterministic (no atomics, fixed reduction order) and independent of B.
 *
 * Activations inside the library are TOKEN-MAJOR fp32: a matrix [T, C] with T = B*h*w tokens in
 * (b, y, x) order and an explicit leading dimension `ld` (elements).  NCHW tensors only appear at
 * the slice-loop entry/exit (dcae_slice_loop_*), where the reference's callers hold them.
 */
#ifndef DCAE_B200_H_
#define DCAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCAE_B200_VERSION 100 /* 0.1.0 */

enum {
  DCAE_OK = 0,
  DCAE_E_INVALID = -1,   /* bad argument (null pointer, misaligned, unsupported shape) */
  DCAE_E_CUDA = -2,      /* a CUDA runtime / driver call failed */
  DCAE_E_WORKSPACE = -3, /* workspace too small */
  DCAE_E_DEVICE = -4     /* not running on an sm_100 device */
};

/* GEMM arithmetic selection for the dense layers (A1-A3 of SURVEY section 8a). */
enum {
  DCAE_MATH_FP32_SIMT = 0, /* FFMA reference path: fp32 in, fp32 accumulate */
  DCAE_MATH_TF32X3 = 1,    /* tcgen05 kind::tf32, error-compensated 3-pass split: fp32-level accuracy */
  DCAE_MATH_TF32 = 2,      /* tcgen05 kind::tf32 single pass (like torch allow_tf32=True) */
  DCAE_MATH_F16X3 = 3,     /* tcgen05 kind::f16 on fp16 hi/lo operand planes, 3-pass: fp32-level accuracy (22-bit
                              operands) at twice the TF32 MMA rate and half the operand bytes per flop */
  DCAE_MATH_F16 = 4        /* the reduced-precision fast mode: same planes data flow, the dense layers multiply the hi
                              planes only (11-bit operands, fp32 accumulate), a third of the tensor work.  NOT a parity
                              mode: tolerance and symbol / index mismatch rates are measured and stated (DESIGN.md) */
};

/* fp16 hi/lo planes of a token-major matrix: value = float(hi[t, c]) + float(lo[t, c]) (22 significant bits).
 * Both planes are [T, ld] fp16; the pointers may be pre-offset to a column window (8-byte aligned, ld % 4 == 0).
 * Producers write them directly (out16 arguments below) so that DCAE_MATH_F16X3 GEMMs need no split pass. */
typedef struct { void* hi; void* lo; int64_t ld; } dcae_planes;

int dcae_version(void);
const char* dcae_last_error(void);
/* 0 if the current device is compute capability 10.x, DCAE_E_DEVICE otherwise. */
int dcae_device_check(void);

/* --------------------------------------------------------------------------------------------
 * Kernel 3: GaussianConditional in one HBM pass.
 * Replaces compressai GaussianConditional.forward / quantize / build_indexes / dequantize as
 * called at dcae.py:657-659 (forward), :738-740 (compress), :891-896 (decompress); math of
 * dcae.py:839-857 and dcae.py:57-58.
 *
 * The tensors are viewed as `rows` rows of `inner` contiguous fp32 (inner % 4 == 0, 16-byte aligned
 * rows), each tensor with its own row stride, so both NCHW slices (rows = B, inner = 64*h*w,
 * y row stride 320*h*w) and token-major slices (rows = T, inner = 64) are expressible.
 *
 * mode DCAE_GC_EVAL   : out = rint(y - mu) + mu
 * mode DCAE_GC_NOISE  : out = y + noise            (training; noise supplied by the caller)
 * mode DCAE_GC_DECODE : out = float(symbols_in) + mu   (y unused; lik not produced)
 * y_hat  <- rint(y - mu) + mu (EVAL/NOISE: the straight-through value of dcae.py:659) or out (DECODE)
 * lik    <- max(0.5 erfc(c (0.5-v)/s) - 0.5 erfc(c (-0.5-v)/s), lik_bound), v = |out - mu|,
 *           s = max(scale, scale_bound), c = -(2^-0.5)
 * sym    <- int32(rint(y - mu));   idx <- #{ j < n_table-1 : table[j] < s }
 * Any output pointer may be NULL.  log2_partials (nullable, >= dcae_gc_num_partials() floats)
 * receives per-block sums of log2(lik) in a fixed order (bpp numerator, train.py:82-85).
 * ------------------------------------------------------------------------------------------*/
enum { DCAE_GC_EVAL = 0, DCAE_GC_NOISE = 1, DCAE_GC_DECODE = 2 };
/* How the likelihood is evaluated.  Symbols, indexes and y_hat do not depend on it.
 * FAST (0, the default of a zero-initialised struct): erfc(x) = 2^P(x) with a divided-difference form of
 *   erfc(a) - erfc(b), no cancellation: <= 1e-5 relative to the EXACT value of the reference's formula everywhere above
 *   the 1e-9 floor (measured 6e-6; the reference's own fp32 evaluation is at 1.5e-4 at large scales).
 * REFERENCE (1): the reference's op order with libdevice erfcf and IEEE divisions: bit-identical to torch evaluating
 *   dcae.py:839-857 on the GPU; about twice the instructions (the test mode). */
enum { DCAE_GC_LIK_FAST = 0, DCAE_GC_LIK_REFERENCE = 1 };

typedef struct {
  const float* y;          int64_t y_ld;
  const float* mu;         int64_t mu_ld;
  const float* scale;      int64_t scale_ld;
  const float* noise;      int64_t noise_ld;      /* NOISE mode only */
  const int32_t* sym_in;   int64_t sym_in_ld;     /* DECODE mode only */
  const float* scale_table; int32_t n_table;      /* the module's scale_table buffer (64 entries) */
  float scale_bound;                              /* 0.11 */
  float lik_bound;                                /* 1e-9 */
  int32_t mode;
  int64_t rows; int64_t inner;
  float* y_hat;   int64_t y_hat_ld;
  dcae_planes y_hat16;                            /* optional: y_hat also as fp16 planes (LRP conv operand) */
  float* lik;     int64_t lik_ld;
  int32_t* sym;   int64_t sym_ld;
  int32_t* idx;   int64_t idx_ld;
  float* log2_partials;
  int32_t lik_math;                               /* DCAE_GC_LIK_FAST (default) or DCAE_GC_LIK_REFERENCE */
} dcae_gc_args;

int dcae_gc_fused(const dcae_gc_args* a, void* stream);
/* Backward of the likelihood for the training step (train.py:165-179 differentiates the rate term of :82-85 through
 * compressai's GaussianConditional.forward, called at dcae.py:657 with self.training).  Given dL/dlik it returns
 * dL/dy, dL/dmu (NOISE mode; zero in EVAL mode, where round() blocks them) and dL/dscale, with the LowerBound rule of
 * compressai for both bounds: the gradient passes where the input is above the bound or the gradient pushes it up.
 * Same row-strided tensor convention as dcae_gc_fused; any output may be NULL. */
typedef struct {
  const float* y;        int64_t y_ld;
  const float* mu;       int64_t mu_ld;
  const float* scale;    int64_t scale_ld;
  const float* noise;    int64_t noise_ld;       /* NOISE mode */
  const float* grad_lik; int64_t grad_lik_ld;
  float scale_bound; float lik_bound;
  int32_t mode;                                  /* DCAE_GC_EVAL or DCAE_GC_NOISE */
  int64_t rows; int64_t inner;
  float* grad_y;     int64_t grad_y_ld;
  float* grad_mu;    int64_t grad_mu_ld;
  float* grad_scale; int64_t grad_scale_ld;
} dcae_gc_bwd_args;
int dcae_gc_backward(const dcae_gc_bwd_args* a, void* stream);
/* number of per-block partial sums dcae_gc_fused writes for this problem size */
int64_t dcae_gc_num_partials(int64_t rows, int64_t inner);
/* out[0] = sum(partials[0..n)) in index order, one block (deterministic). */
int dcae_reduce_partials(const float* partials, int64_t n, float* out, void* stream);

/* --------------------------------------------------------------------------------------------
 * Hyper-latent entropy model (SURVEY 8f N3, first part): compressai EntropyBottleneck.forward / quantize / dequantize as
 * the reference calls them for z (dcae.py:629-633, :705-706, :861), one pass over NCHW z [B, C, h, w]:
 *   out = round(z - median_c) + median_c (EVAL) | z + noise (NOISE) | float(sym_in) + median_c (DECODE)
 *   lik = max(sigmoid(L_c(out + 1/2)) - sigmoid(L_c(out - 1/2)), lik_bound),  L_c = the channel's 1-3-3-3-3-1 network
 *   sym = int32(round(z - median_c)),  z_hat = round(z - median_c) + median_c
 * params: [C, 58] = per channel softplus(_matrix0..4) (3, 9, 9, 9, 3 row-major), _bias0..4 (3, 3, 3, 3, 1),
 * tanh(_factor0..3) (3 each), packed by the host once per weight load.  Any output may be NULL.
 * ------------------------------------------------------------------------------------------*/
typedef struct {
  const float* z; const float* noise; const int32_t* sym_in;
  const float* params; const float* medians;
  int32_t mode;            /* DCAE_GC_EVAL / DCAE_GC_NOISE / DCAE_GC_DECODE */
  int32_t B, C; int64_t HW;
  float lik_bound;
  float* z_hat; float* lik; int32_t* sym;
} dcae_eb_args;
int dcae_eb_fused(const dcae_eb_args* a, void* stream);
/* Backward of dcae_eb_fused's likelihood for the training step (train.py:165-179 differentiates the rate of z through
 * compressai's EntropyBottleneck.forward).  Given dL/dlik [B, C, HW] it overwrites
 *   grad_z [B, C, HW]    dL/dz through out = z + noise (NOISE); all zeros in EVAL mode, where round() passes no gradient
 *   grad_params [C, 58]  dL/d of the PACKED values softplus(_matrix*), _bias*, tanh(_factor*) in dcae_eb_fused's layout
 * with compressai's LowerBound rule for the likelihood floor (the gradient passes where lik >= lik_bound or where it is
 * negative).  The medians get no gradient (compressai detaches them).  mode: DCAE_GC_EVAL or DCAE_GC_NOISE.
 * Deterministic, no atomics: one block per channel sums the channel's B*HW elements in an order fixed by the shape, and
 * every grad_z element depends on its own element only (an image's rows do not depend on the rest of the batch). */
typedef struct {
  const float* z; const float* noise;
  const float* params; const float* medians;
  const float* grad_lik;
  int32_t mode;            /* DCAE_GC_EVAL / DCAE_GC_NOISE */
  int32_t B, C; int64_t HW;
  float lik_bound;
  float* grad_z; float* grad_params;
} dcae_eb_bwd_args;
int dcae_eb_backward(const dcae_eb_bwd_args* a, void* stream);

/* --------------------------------------------------------------------------------------------
 * MS-SSIM statistics (the distortion of the ms-ssim rate-distortion loss): pytorch_msssim.ms_ssim v1.0 with its
 * defaults -- 11-tap Gaussian window (sigma 1.5) as a valid separable correlation, C1 = (0.01 R)^2, C2 = (0.03 R)^2,
 * 5 levels joined by avg_pool2d(2, 2, padding = (h % 2, w % 2), count_include_pad).  x, y: fp32 NCHW [B, C, H, W],
 * min(H, W) > 160.  The forward writes the per-level means of the ssim and cs maps of each plane, ssim / cs [5, B, C]
 * (level-major); the weighted product over the levels is left to the caller.  The backward takes dL/dssim and dL/dcs
 * [5, B, C] and overwrites grad_x [B, C, H, W] = dL/dx (y gets no gradient).  Both take the same scratch, of at least
 * dcae_msssim_scratch_bytes(B, C, H, W) bytes, 16-byte aligned: the forward leaves the pooled pyramid of x and y there
 * and the backward reads it, so the backward must see the scratch of the forward on the same x and y.
 * Deterministic, no atomics; a plane's results do not depend on the other planes.  No host synchronisation.
 * ------------------------------------------------------------------------------------------*/
typedef struct {
  const float* x; const float* y;
  int32_t B, C, H, W;
  float data_range;                        /* R > 0 */
  void* scratch; size_t scratch_bytes;
  float* ssim; float* cs;                  /* [5, B, C] */
} dcae_msssim_args;
typedef struct {
  const float* x; const float* y;
  int32_t B, C, H, W;
  float data_range;
  void* scratch; size_t scratch_bytes;     /* as left by dcae_msssim_forward */
  const float* grad_ssim; const float* grad_cs;   /* [5, B, C] */
  float* grad_x;                           /* [B, C, H, W] */
} dcae_msssim_bwd_args;
/* scratch bytes for both directions; 0 for a shape they reject */
size_t dcae_msssim_scratch_bytes(int32_t B, int32_t C, int32_t H, int32_t W);
int dcae_msssim_forward(const dcae_msssim_args* a, void* stream);
int dcae_msssim_backward(const dcae_msssim_bwd_args* a, void* stream);

/* --------------------------------------------------------------------------------------------
 * Elementary token-major operators (each replaces one torch dispatch chain of dcae.py:300-509).
 * ------------------------------------------------------------------------------------------*/

/* A-operand of a GEMM: columns [col0, col0+k0) then [col1, col1+k1) of a token-major buffer,
 * optionally gathered over the 9 taps of a 3x3 / stride 1 / pad 1 window (taps = 9), in which case
 * K = 9*(k0+k1) ordered tap-major (tap = 3*(dy+1) + (dx+1)).  k0, k1 multiples of 32. */
typedef struct {
  const float* base; int64_t ld;
  int32_t col0, k0, col1, k1;
  int32_t taps;            /* 1 or 9 */
  int32_t B, h, w;         /* token grid */
  /* DCAE_MATH_F16X3 only: caller-owned scratch of dcae_planes_bytes(T, k0 + k1) bytes that receives the fp16
   * hi/lo planes of the operand window (the split runs as its own HBM-bound launch before the GEMM). */
  void* planes; int64_t planes_bytes;
  /* DCAE_MATH_F16X3: if src16.hi != NULL the window [col0, col0 + k0) is read from these planes directly
   * (k1 must be 0; base may be NULL; the window may be over-read up to the next multiple of 64 columns, which
   * must be allocated and finite -- the weight planes are zero there). */
  dcae_planes src16;
} dcae_operand;
int64_t dcae_planes_bytes(int64_t T, int32_t cols);

enum { DCAE_ACT_NONE = 0, DCAE_ACT_GELU = 1, DCAE_ACT_HALF_TANH = 2, DCAE_ACT_RELU = 3 /* dcae.py:135-140 */ };

/* out[t, n] = act_n( acc[t, n] + bias[n] + addend[t, n] ) + residual[t, n] * res_scale[n]
 * act applies to columns n < act_cols (all columns if act_cols <= 0 or >= N).
 * bias, addend, residual, res_scale nullable (res_scale NULL means 1). */
typedef struct {
  const float* bias;
  const float* addend;   int64_t addend_ld;
  const float* residual; int64_t residual_ld;
  const float* res_scale;
  int32_t act; int32_t act_cols;
  float* out; int64_t out_ld;          /* may be NULL when out16 is given */
  dcae_planes out16;                   /* tcgen05 paths only: also (or only) write the result as fp16 planes */
  dcae_planes out16_act;               /* DCAE_MATH_F16X3 only: planes of act2(result), e.g. the GELU prologue of the
                                          next dense layer (dcae.py:421-423) produced by this layer's epilogue */
  int32_t act2;
} dcae_epilogue;

/* Dense weight [N, K] row-major (K contiguous; nn.Linear layout).  `w` is the fp32 weight;
 * w_hi / w_lo are its TF32 split (w_hi = tf32(w), w_lo = tf32(w - w_hi)) made by dcae_split_tf32,
 * required by the tcgen05 paths. */
typedef struct {
  const float* w; const float* w_hi; const float* w_lo;
  int32_t N; int32_t K;
  /* DCAE_MATH_F16X3: fp16 hi/lo planes of w * 2^e, [N, K16] with each tap's channel run padded to a multiple
   * of 64 (K16 = taps * pad64(K / taps)); descale = 2^-e is applied to the accumulator (exact).  Made by
   * dcae_split_f16_weight. */
  const void* w16_hi; const void* w16_lo;
  int32_t K16; float descale;
} dcae_weight;
/* w: [N, taps * kc] fp32 -> hi/lo: [N, taps * pad64(kc)] fp16 of w * scale (scale a power of two). */
int dcae_split_f16_weight(const float* w, int32_t N, int32_t taps, int32_t kc, float scale, void* hi, void* lo, void* stream);

/* nn.Linear / 1x1 conv / 3x3 conv as one GEMM: acc[T, N] = A[T, K] * W[N, K]^T.
 * Replaces F.linear / F.conv2d dispatches of dcae.py:482-507 and :584-611. */
int dcae_op_gemm(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int math, void* stream);
int dcae_split_tf32(const float* w, float* w_hi, float* w_lo, int64_t n, void* stream);

/* LayerNorm over C channels per token, eps 1e-5 (dcae.py:461,465,467,471; the Swin blocks' ln1 / ln2, :349,352).
 * C: any multiple of 4 up to 1024. */
int dcae_op_layernorm(const float* x, int64_t x_ld, const float* gamma, const float* beta, int32_t C,
                      int64_t T, float* out, int64_t out_ld, const dcae_planes* out16, void* stream);
/* out = gelu(x) (exact erf form), [T, C] (dcae.py:421-423 prologue GELU of the dense block). */
int dcae_op_gelu(const float* x, int64_t x_ld, int32_t C, int64_t T, float* out, int64_t out_ld,
                 const dcae_planes* out16, void* stream);
/* In every operator below `out` may be NULL when `out16` (fp16 planes of the same result) is given. */
/* Depthwise 3x3, stride 1, pad 1 on a token grid (dcae.py:303,404): wt is [9, C] tap-major.
 * out = act(dw(x) + bias) * gate   (gate nullable: ConvolutionalGLU, dcae.py:325-326). */
int dcae_op_dwconv3x3(const float* x, int64_t x_ld, const float* wt, const float* bias, int32_t C,
                      int32_t B, int32_t h, int32_t w, int32_t act, const float* gate, int64_t gate_ld,
                      float* out, int64_t out_ld, const dcae_planes* out16, void* stream);
/* SpatialAttentionModule + residual (dcae.py:386-397, 446, 484):
 * out = s_out * sigmoid(conv7x7([mean_c s_out, max_c s_out])) + res_scale * x0.
 * stats: scratch [T, 2].  w7: [2, 7, 7]. */
int dcae_op_spatial_gate(const float* s_out, int64_t s_ld, const float* x0, int64_t x0_ld,
                         const float* res_scale, const float* w7, int32_t C, int32_t B, int32_t h, int32_t w,
                         float* stats, float* out, int64_t out_ld, void* stream);
/* The same with the LayerNorm that follows it in the module (lnx, dcae.py:487) fused in: the warp that produces a token's
 * row also normalises it and writes LN(out) * gamma + beta as fp16 planes (ln_out16; NULL = no LayerNorm). */
int dcae_op_spatial_gate_ln(const float* s_out, int64_t s_ld, const float* x0, int64_t x0_ld,
                            const float* res_scale, const float* w7, int32_t C, int32_t B, int32_t h, int32_t w,
                            float* stats, float* out, int64_t out_ld, const float* ln_gamma, const float* ln_beta,
                            const dcae_planes* ln_out16, void* stream);
/* Dictionary attention core (dcae.py:489-501): per head e (20 heads of 32):
 * out[t, e, :] = softmax_j( q[t, e, :] . K[e, j, :] * head_scale[e] ) V[e, j, :], j < 128.
 * The dictionary side is batch invariant (dcae.py:492-495) and prepared once per weight load:
 *   Kh, Vh            [20, 128, 32] fp32  (K = k(LN(dt)) and V = LN(dt), split per head)
 *   Kh_hi, Kh_lo      TF32 split of Kh                      (tcgen05 paths)
 *   Vt_hi, Vt_lo      TF32 split of Vh transposed per head, [20, 32, 128]
 *   K16_hi, K16_lo    fp16 planes of K * 2^e as the [128, 640] matrix k(LN(dt)) itself (columns = (head, dim)),
 *                     k_descale = 2^-e                       (DCAE_MATH_F16X3)
 *   Vt16_hi, Vt16_lo  fp16 planes of LN(dt)^T * 2^e', [640, 128], v_descale = 2^-e'
 * math FP32_SIMT = FFMA kernel; TF32X3 / TF32 = kernel 1 (tcgen05 + TMEM, softmax in registers) on the fp32 query;
 * F16X3 = kernel 1 on fp16 planes: the query is read from q16 (q may be NULL), e.g. the q_trans GEMM's out16. */
typedef struct {
  const float* Kh; const float* Vh;
  const float* Kh_hi; const float* Kh_lo;
  const float* Vt_hi; const float* Vt_lo;
  const float* head_scale;     /* [20] learned per-head scale (dcae.py:457,498) */
  const void* K16_hi; const void* K16_lo;
  const void* Vt16_hi; const void* Vt16_lo;
  float k_descale, v_descale;
} dcae_dict_kv;
int dcae_op_dict_attention(const float* q, int64_t q_ld, const dcae_planes* q16, const dcae_dict_kv* kv, int64_t T, float* out,
                           int64_t out_ld, const dcae_planes* out16, int math, void* stream);
/* 'b c h w -> (b h w) c' and back, for a channel window of the token-major buffer. */
int dcae_op_nchw_to_tokens(const float* src, int32_t B, int32_t C, int64_t HW, float* dst, int64_t dst_ld,
                           const dcae_planes* dst16, void* stream);
int dcae_op_tokens_to_nchw(const float* src, int64_t src_ld, int32_t B, int32_t C, int64_t HW, float* dst, void* stream);
int dcae_op_tokens_to_nchw_i32(const int32_t* src, int64_t src_ld, int32_t B, int32_t C, int64_t HW, int32_t* dst, void* stream);
int dcae_op_nchw_to_tokens_i32(const int32_t* src, int32_t B, int32_t C, int64_t HW, int32_t* dst, int64_t dst_ld, void* stream);

/* --------------------------------------------------------------------------------------------
 * Operators of the transform stacks around the entropy model (SURVEY 8f N3 / N4: h_a, h_z_s1, h_z_s2, g_a, g_s;
 * dcae.py:152-383, 541-582).  dcae_b200/transforms.py composes them with dcae_op_gemm / layernorm / dwconv3x3.
 * ------------------------------------------------------------------------------------------*/

/* WMSA core (dcae.py:262-291) on a token grid, windows of `window` x `window` tokens (4 or 8), heads of head_dim
 * (8, 16 or 32) channels:
 *   out[t, e*hd : (e+1)*hd] = softmax_j( q_e[t] . k_e[j] / sqrt(hd) + rel_bias[e, dy, dx] (+ SW mask) ) v_e[j]
 * over the tokens j of t's window.  q / k / v of head e are the columns q_col / k_col / v_col + e*hd of `qkv`
 * (the '(threeh c)' order of embedding_layer, :275-276).  shift = 0: W windows; shift = window / 2: SW windows,
 * i.e. the cyclic roll of :270 / :289 and generate_mask (:244-260) folded into the indexing.  rel_bias is
 * relative_position_params as the state dict holds it, [n_heads, 2*window-1, 2*window-1] contiguous (:240, 293-296).
 * h and w must be multiples of window. */
int dcae_op_window_attention(const float* qkv, int64_t ld, int32_t q_col, int32_t k_col, int32_t v_col, int32_t C,
                             int32_t head_dim, int32_t window, int32_t shift, const float* rel_bias, int32_t B, int32_t h,
                             int32_t w, float* out, int64_t out_ld, const dcae_planes* out16, void* stream);
/* Backward of dcae_op_window_attention, same qkv / window / head_dim / shift / rel_bias arguments, plus the output
 * cotangent dout [T, dout_ld] (columns e*hd.. of head e).  Per window and head, s = 1/sqrt(hd), with S and P recomputed
 * exactly as the forward computes them:
 *   dP = dO V^T;  D_i = sum_j P_ij dP_ij;  dS = P o (dP - D);  dQ = s dS K;  dK = s dS^T Q;  dV = P^T dO
 *   drel[e, dy, dx] = sum of dS over every (query, key) pair at that offset, in every window and image (masked pairs add 0)
 * dq / dk / dv are written into the q_col / k_col / v_col column windows of dqkv [T, dqkv_ld] (the three windows must not
 * overlap; other columns are left untouched); drel [n_heads, 2*window-1, 2*window-1] is overwritten.  dqkv must not alias
 * qkv or dout.  scratch: device memory of at least dcae_window_attention_backward_scratch_bytes() bytes (16-byte aligned),
 * per-block partial sums of drel; its size does not grow with the image beyond a fixed number of blocks.  Deterministic, no
 * atomics: every dqkv element has one writer, drel is summed in a fixed order that depends on the shape only, and the dqkv
 * rows of an image do not depend on the rest of the batch.  8x8 windows run on warp-level TF32 MMAs with the 3-pass split,
 * 4x4 windows on FFMA.  Work booked: 10 T window^2 C flop. */
size_t dcae_window_attention_backward_scratch_bytes(int32_t B, int32_t h, int32_t w, int32_t C, int32_t head_dim, int32_t window);
int dcae_op_window_attention_backward(const float* qkv, int64_t ld, int32_t q_col, int32_t k_col, int32_t v_col, int32_t C,
                                      int32_t head_dim, int32_t window, int32_t shift, const float* rel_bias,
                                      int32_t B, int32_t h, int32_t w, const float* dout, int64_t dout_ld,
                                      float* dqkv, int64_t dqkv_ld, float* drel, void* scratch, size_t scratch_bytes, void* stream);
/* out[(b, y', x'), (sy*2 + sx)*Cs + c] = x[(b, 2y' + sy, 2x' + sx), c] for c < C, 0 elsewhere (c >= C, odd edge);
 * output grid ceil(h/2) x ceil(w/2), 4*Cs columns.  With the weights re-indexed at pack time a stride-2 k x k
 * convolution (conv(), dcae.py:35-42) becomes a stride-1 3x3 convolution over this image (dcae_op_gemm, taps = 9). */
int dcae_op_space_to_depth(const float* x, int64_t ld, int32_t C, int32_t Cs, int32_t B, int32_t h, int32_t w, float* out,
                           int64_t out_ld, const dcae_planes* out16, void* stream);
/* out[(b, 2y + py, 2x + px), c] = x[(b, y, x), (py*2 + px)*Cs + c] for c < C, 0 for C <= c < Cpad; output grid
 * 2h x 2w.  A stride-2 transposed convolution (deconv(), dcae.py:44-52) is a stride-1 3x3 convolution producing
 * the four output phases as 4*Cs channels, then this rearrangement. */
int dcae_op_depth_to_space(const float* x, int64_t ld, int32_t Cs, int32_t C, int32_t Cpad, int32_t B, int32_t h, int32_t w,
                           float* out, int64_t out_ld, const dcae_planes* out16, void* stream);

/* Coder hand-off (SURVEY 8f N1; replaces the per-slice `.tolist()` of dcae.py:742-743 on the device side): the int32
 * symbols / indexes of a compress() call, in coder order, packed to int16 / uint8 for one small D2H copy.  Symbols
 * outside int16 saturate and are counted in *overflow_count (device scalar): when it is not zero the caller must
 * use the int32 tensor (the coder's bypass path needs the exact value).  n must be a multiple of 4. */
int dcae_pack_symbols(const int32_t* symbols, const int32_t* indexes, int64_t n, int16_t* symbols16, uint8_t* indexes8,
                      unsigned long long* overflow_count, void* stream);

/* --------------------------------------------------------------------------------------------
 * The y range coder on the GPU, in the opt-in interleaved format ilv1 (include/dcae_rans.h describes it; the default
 * reference format stays with the host coder).  One string per image; the bytes equal dcae_rans_ilv_encode's.
 * The coder tables are device copies of GaussianConditional's quantized_cdf [n_cdfs, cdf_stride], cdf_length and
 * offset (int32), uploaded once per table version.
 * ------------------------------------------------------------------------------------------*/
typedef struct {
  const int32_t* cdfs; int32_t cdf_stride;
  const int32_t* cdf_sizes;
  const int32_t* offsets;
  int32_t n_cdfs;
} dcae_coder_tables;
/* per-image status words written by the coder kernels: 0 = ok */
enum { DCAE_ILV_OK = 0, DCAE_ILV_E_HEADER = 1, DCAE_ILV_E_CORRUPT = 2, DCAE_ILV_E_INDEX = 3, DCAE_ILV_E_TABLE = 4 };
/* Encode: one warp per (image, slice), two phases (count the words, then code and store them at their final place), no
 * atomics.  symbols / indexes: int32 [5, B, 64, h, w], the coder order of dcae_slice_loop_store.  Outputs:
 * sizes [B, 5] (u32 bytes of each segment; image b's string is 24 + the sum of its five), the B strings back to back
 * from out[0], and status [B] (DCAE_ILV_E_INDEX / _TABLE for an index or table row the coder cannot use).
 * out: 4-byte aligned, out_capacity >= dcae_ilv_encode_max_bytes; scratch: 8-byte aligned, >= _scratch_bytes. */
typedef struct {
  const int32_t* symbols; const int32_t* indexes;
  int32_t B, h, w, lanes;                 /* lanes: 1, 2, 4, 8, 16 or 32 */
  dcae_coder_tables tables;
  void* scratch; size_t scratch_bytes;
  uint32_t* sizes;
  uint8_t* out; int64_t out_capacity;
  int32_t* status;
} dcae_ilv_enc_args;
size_t dcae_ilv_encode_scratch_bytes(int32_t B, int32_t h, int32_t w, int32_t lanes);
int64_t dcae_ilv_encode_max_bytes(int32_t B, int32_t h, int32_t w, int32_t lanes);
int dcae_ilv_encode(const dcae_ilv_enc_args* a, void* stream);
/* Decode slice `slice` of B images: one warp per image.  Image b's string is strings[bounds[2b] .. bounds[2b + 1])
 * (start 4-byte aligned); indexes: int32 [B, 64, h, w] (dcae_slice_loop_indexes), symbols: int32 [B, 64, h, w] out
 * (dcae_slice_loop_decode's input).  Every read is checked against the string and its segment.  A malformed or corrupt
 * string sets status[b] (DCAE_ILV_E_HEADER / _CORRUPT / _INDEX / _TABLE), writes 0 for the image's symbols and skips the
 * image in later slices; status must be zero before slice 0 and is read by the host once, after the last slice. */
typedef struct {
  const uint8_t* strings; const int64_t* bounds;
  const int32_t* indexes;
  int32_t slice, B, h, w;
  dcae_coder_tables tables;
  int32_t* symbols;
  int32_t* status;
} dcae_ilv_dec_args;
int dcae_ilv_decode(const dcae_ilv_dec_args* a, void* stream);

/* --------------------------------------------------------------------------------------------
 * The channel-slice loop (dcae.py:638-670 forward, :713-753 compress, :878-906 decompress).
 * Packed weights of one slice i.  Dense weights are dcae_weight (row-major [N, K]); packing rules
 * (done by dcae_b200/weights.py from a reference state dict):
 *   - 3x3 conv weights [N, C, 3, 3] -> [N, 9, C'] (tap-major K), with the input channels permuted
 *     from the reference's `support = [latent_scales, latent_means, y_hat_0.., dict_info]` order to
 *     this library's support-buffer order `[dict_info, latent_scales, latent_means, y_hat_0..]`;
 *   - cc1 = rows [cc_mean.0 (224) | cc_scale.0 (224) | lrp.0 restricted to the support channels (224)];
 *     lrp1y = lrp.0 restricted to its last 64 input channels (the current y_hat slice);
 *   - depthwise weights [C, 1, 3, 3] -> [9, C];
 *   - Kh = per-head split of k(LN_dict(dt)), Vh = per-head split of LN_dict(dt)   [20, 128, 32]
 *     (batch invariant, dcae.py:492-495; computed once per weight load).
 * ------------------------------------------------------------------------------------------*/
typedef struct {
  dcae_weight x_trans;  const float* x_trans_b;
  const float* ln_scale_g; const float* ln_scale_b;
  dcae_weight msa_s;    const float* msa_s_b;
  dcae_weight dense_in[3];  const float* dense_in_b[3];
  const float* dense_dw[3]; const float* dense_dw_b[3];
  dcae_weight dense_out[3]; const float* dense_out_b[3];
  dcae_weight dense_proj;   const float* dense_proj_b;
  const float* spatial_w7;
  const float* res_scale_1; const float* res_scale_2; const float* res_scale_3;
  const float* lnx_g; const float* lnx_b;
  dcae_weight q_trans;  const float* q_trans_b;
  dcae_dict_kv kv;
  dcae_weight linear;   const float* linear_b;
  const float* ln_mlp_g; const float* ln_mlp_b;
  dcae_weight fc1;      const float* fc1_b;
  const float* mlp_dw;  const float* mlp_dw_b;
  dcae_weight fc2;      const float* fc2_b;
  dcae_weight output_trans; const float* output_trans_b;
  dcae_weight cc1;      const float* cc1_b;          /* N = 672, bias = [mean.0.b | scale.0.b | 0] */
  dcae_weight mean2;    const float* mean2_b;        /* [128, 9*224] */
  dcae_weight scale2;   const float* scale2_b;
  dcae_weight mean3;    const float* mean3_b;        /* [64, 9*128] */
  dcae_weight scale3;   const float* scale3_b;
  dcae_weight lrp1y;    const float* lrp1_b;         /* [224, 9*64], bias of lrp.0 */
  dcae_weight lrp2;     const float* lrp2_b;
  dcae_weight lrp3;     const float* lrp3_b;
} dcae_slice_weights;

typedef struct dcae_slice_loop dcae_slice_loop;

size_t dcae_slice_loop_workspace_bytes(int32_t B, int32_t h, int32_t w);
/* weights: array of 5; scale_table: device [n_table] (the module's buffer, dcae.py:616-621; 2..256 entries, NULL if
 * update() has not run: indexes are then unavailable); workspace: device, 256-byte aligned. */
int dcae_slice_loop_create(dcae_slice_loop** out, int32_t B, int32_t h, int32_t w,
                           const dcae_slice_weights* weights, const float* scale_table, int32_t n_table,
                           void* workspace, size_t workspace_bytes, int math);
void dcae_slice_loop_destroy(dcae_slice_loop* p);
/* Plan options.  DCAE_OPT_LIK_MATH: DCAE_GC_LIK_FAST (default) or DCAE_GC_LIK_REFERENCE for kernel 3's likelihood.
 * DCAE_OPT_WANT_SYMBOLS (default 1): dcae_slice_loop_encode also writes the int32 symbols / indexes (28 B/element);
 * 0 = DCAE.forward only needs y_hat and likelihoods (20 B/element).  dcae_slice_loop_forward sets it per call from its
 * symbols / indexes arguments. */
enum { DCAE_OPT_LIK_MATH = 0, DCAE_OPT_WANT_SYMBOLS = 1 };
int dcae_slice_loop_set_option(dcae_slice_loop* p, int32_t option, int32_t value);

/* NCHW fp32 [B,320,h,w] -> token-major workspace.  y may be NULL (decompress). */
int dcae_slice_loop_load(dcae_slice_loop* p, const float* y, const float* latent_scales,
                         const float* latent_means, void* stream);
/* slice i: dict_info, mu, scale (dcae.py:644-655); idx if `want_indexes`. */
int dcae_slice_loop_params(dcae_slice_loop* p, int32_t i, void* stream);
/* slice i: quantise + likelihood + indexes (kernel 3) then LRP (dcae.py:657-664 / :738-750).
 * gc_mode DCAE_GC_EVAL or DCAE_GC_NOISE (noise: NCHW [B,64,h,w] for this slice, or NULL). */
int dcae_slice_loop_encode(dcae_slice_loop* p, int32_t i, int32_t gc_mode, const float* noise, void* stream);
/* slice i of decompress: indexes for the coder are available after _params (dcae_slice_loop_indexes);
 * then y_hat = symbols + mu and LRP (dcae.py:891-904).  symbols: NCHW int32 [B,64,h,w]. */
int dcae_slice_loop_indexes(dcae_slice_loop* p, int32_t i, int32_t* indexes_nchw, void* stream);
int dcae_slice_loop_decode(dcae_slice_loop* p, int32_t i, const int32_t* symbols_nchw, void* stream);
/* Token-major workspace -> the caller's NCHW tensors; any pointer may be NULL.
 * y_hat/means/scales/lik: fp32 [B,320,h,w]; symbols/indexes: int32 [5,B,64,h,w] (the reference's
 * coder order, dcae.py:742-743).  log2_lik_sum: 1 float = sum log2(lik) (deterministic). */
int dcae_slice_loop_store(dcae_slice_loop* p, float* y_hat, float* means, float* scales, float* lik,
                          int32_t* symbols, int32_t* indexes, float* log2_lik_sum, void* stream);
/* DCAE_MATH_F16X3 range validation.  Activations travel as fp16 hi/lo planes written with a saturating convert, so a
 * magnitude above 65504 would be clamped silently.  With `enable` != 0 every later call on this plan counts, behind
 * each producer, the plane elements that sit at the clamp; the call itself returns the count accumulated so far in
 * *clamped_host (nullable; reading synchronises the device) and resets it.  Meant for validating a checkpoint once
 * (dcae_b200.EntropySliceLoop.check_f16_range), not for the hot path: it adds one small launch per producer. */
int dcae_slice_loop_check_f16_range(dcae_slice_loop* p, int32_t enable, unsigned long long* clamped_host);
/* elements of the [T, cols] window of `planes` whose hi half is at the fp16 clamp or not finite, added to *counter (device). */
int dcae_count_f16_clamped(const dcae_planes* planes, int64_t T, int32_t cols, unsigned long long* counter, void* stream);

/* Module-level calls, for callers that keep the reference's loop text and swap single modules (SURVEY 8b): one
 * module of slice i on the caller's NCHW fp32 tensors, through the plan's buffers -- do not interleave with a slice
 * loop in flight on the same plan.
 *   _module_dca : net.dt_cross_attention[i](x, dt)            dcae.py:479-509, called at :646, :730, :881
 *                 x [B, 640 + 64 i, h, w] = cat(latent_scales, latent_means, y_hat_0..) -> out [B, 320, h, w];
 *                 the dictionary is the one packed into the plan's weights (K = k(LN(dt)), V = LN(dt)).
 *   _module_conv: which 0 = cc_mean_transforms[i], 1 = cc_scale_transforms[i]   (dcae.py:649-655; x [B, 960 + 64 i, h, w])
 *                 which 2 = lrp_transforms[i]                  (dcae.py:661-662; x [B, 1024 + 64 i, h, w]); the RAW conv
 *                 stack, the caller applies 0.5 tanh (dcae.py:663)            -> out [B, 64, h, w] */
int dcae_slice_loop_module_dca(dcae_slice_loop* p, int32_t i, const float* x, float* out, void* stream);
int dcae_slice_loop_module_conv(dcae_slice_loop* p, int32_t i, int32_t which, const float* x, float* out, void* stream);
/* load + 5 x (params, encode) + store. */
int dcae_slice_loop_forward(dcae_slice_loop* p, const float* y, const float* latent_scales,
                            const float* latent_means, float* y_hat, float* means, float* scales,
                            float* lik, int32_t* symbols, int32_t* indexes, float* log2_lik_sum, void* stream);
/* Debug/test access to a named token-major intermediate of the last call ("x0","x1","q","attn","x2",
 * "x3","support","h1"...): returns pointer, columns and ld; 0 on success. */
int dcae_slice_loop_tap(dcae_slice_loop* p, const char* name, const float** ptr, int32_t* cols, int64_t* ld);
/* Same for intermediates that only exist as fp16 planes in DCAE_MATH_F16X3 mode ("support", "ln", "gelu", "dw",
 * "dense", "attn", "glu", "x3", "h1", "h2", "l1", "l2"). */
int dcae_slice_loop_tap16(dcae_slice_loop* p, const char* name, dcae_planes* planes, int32_t* cols);
/* Number of kernels the last dcae_slice_loop_* call enqueued (bench `gpu_launches`). */
int64_t dcae_launch_count(void);

/* Optional per-kernel-family timing with CUDA events on the launching stream (bench.py roofline).
 * Families: 0 = dense GEMM (work = 2*T*N*K flop), 1 = dictionary attention core (work = 327680 flop per
 * token), 2 = kernel 3 (work = algorithmic bytes: 4 B per tensor touched per element), 3 = other
 * elementwise kernels (work = 0).  dcae_profile_stop synchronises the device and fills 4-entry arrays. */
enum { DCAE_PROF_GEMM = 0, DCAE_PROF_ATTN = 1, DCAE_PROF_GC = 2, DCAE_PROF_OTHER = 3, DCAE_PROF_FAMILIES = 4 };
int dcae_profile_start(void);
int dcae_profile_stop(double* ms, double* work, int64_t* launches);
/* Like dcae_profile_stop, but also writes one CSV line per recorded op (index, family, work, ms) to `path`. */
int dcae_profile_dump(const char* path, double* ms, double* work, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* DCAE_B200_H_ */
