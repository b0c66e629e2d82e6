// C ABI glue + the host-side plan of the channel-slice loop
// (/root/reference/models/dcae.py:638-670 forward, :713-753 compress, :878-906 decompress).
#include <stdarg.h>
#include <string.h>

#include <new>
#include <vector>

#include "common.cuh"

namespace dcae {

thread_local int64_t g_launches = 0;
static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

// ---- event-based per-family timing ----------------------------------------------------------------
namespace {
struct ProfRec { int family; double work; cudaEvent_t a, b; };
std::vector<ProfRec> g_prof;
std::vector<cudaEvent_t> g_event_pool;
bool g_prof_on = false;
size_t g_prof_used = 0;
cudaEvent_t take_event() {
  if (g_prof_used < g_event_pool.size()) return g_event_pool[g_prof_used++];
  cudaEvent_t e;
  cudaEventCreate(&e);
  g_event_pool.push_back(e);
  ++g_prof_used;
  return e;
}
}  // namespace

ProfileScope::ProfileScope(int family, double work, void* s) : slot(-1), stream(s) {
  if (!g_prof_on) return;
  ProfRec r{family, work, take_event(), take_event()};
  cudaEventRecord(r.a, (cudaStream_t)stream);
  slot = (int)g_prof.size();
  g_prof.push_back(r);
}
ProfileScope::~ProfileScope() {
  if (slot >= 0) cudaEventRecord(g_prof[slot].b, (cudaStream_t)stream);
}
bool profiling_on() { return g_prof_on; }

}  // namespace dcae

using namespace dcae;

extern "C" int dcae_profile_start(void) {
  g_prof.clear();
  g_prof_used = 0;
  g_prof_on = true;
  return DCAE_OK;
}

extern "C" int dcae_profile_dump(const char* path, double* ms, double* work, int64_t* launches) {
  DCAE_REQUIRE(ms && work && launches, "dcae_profile_stop: null output");
  g_prof_on = false;
  DCAE_CUDA(cudaDeviceSynchronize());
  FILE* f = path ? fopen(path, "w") : nullptr;
  if (f) fprintf(f, "index,family,work,ms,start_ms\n");
  for (int k = 0; k < DCAE_PROF_FAMILIES; ++k) { ms[k] = 0; work[k] = 0; launches[k] = 0; }
  int i = 0;
  for (const ProfRec& r : g_prof) {
    float t = 0.f;
    DCAE_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    ms[r.family] += t;
    work[r.family] += r.work;
    launches[r.family] += 1;
    if (f) {
      float t0 = 0.f;                                  // start of this op relative to the first recorded one
      DCAE_CUDA(cudaEventElapsedTime(&t0, g_prof.front().a, r.a));
      fprintf(f, "%d,%d,%.6g,%.6f,%.6f\n", i, r.family, r.work, t, t0);
    }
    ++i;
  }
  if (f) fclose(f);
  g_prof.clear();
  g_prof_used = 0;
  return DCAE_OK;
}

extern "C" int dcae_profile_stop(double* ms, double* work, int64_t* launches) { return dcae_profile_dump(nullptr, ms, work, launches); }

extern "C" int dcae_version(void) { return DCAE_B200_VERSION; }
extern "C" const char* dcae_last_error(void) { return g_error; }
extern "C" int64_t dcae_launch_count(void) { return g_launches; }

extern "C" int dcae_device_check(void) {
  int dev = 0, major = 0;
  DCAE_CUDA(cudaGetDevice(&dev));
  DCAE_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) {
    set_error("libdcae_b200 is built for sm_100a only; device %d has compute capability major %d", dev, major);
    return DCAE_E_DEVICE;
  }
  return DCAE_OK;
}

static int check_gemm_args(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e) {
  DCAE_REQUIRE(a && w && e, "dcae_op_gemm: null argument struct");
  DCAE_REQUIRE((a->base || a->src16.hi) && (e->out || e->out16.hi || e->out16_act.hi), "dcae_op_gemm: null operand/output pointer");
  DCAE_REQUIRE(planes_ok(&e->out16) && planes_ok(&e->out16_act) && planes_ok(&a->src16), "dcae_op_gemm: fp16 planes must be 8-byte aligned with ld %% 4 == 0");
  DCAE_REQUIRE(a->taps == 1 || a->taps == 9, "dcae_op_gemm: taps must be 1 or 9 (got %d)", a->taps);
  DCAE_REQUIRE(a->k0 > 0 && a->k0 % 32 == 0 && a->k1 >= 0 && a->k1 % 32 == 0 && a->col0 % 4 == 0 && a->col1 % 4 == 0,
               "dcae_op_gemm: operand segments must be multiples of 32 columns (k0=%d k1=%d)", a->k0, a->k1);
  DCAE_REQUIRE(w->K == a->taps * (a->k0 + a->k1), "dcae_op_gemm: weight K=%d != taps*(k0+k1)=%d", w->K, a->taps * (a->k0 + a->k1));
  DCAE_REQUIRE(w->N > 0 && w->N % 16 == 0, "dcae_op_gemm: N=%d must be a positive multiple of 16", w->N);
  DCAE_REQUIRE(a->B >= 0 && a->h >= 0 && a->w >= 0 && (int64_t)a->B * a->h * a->w < (1ll << 31), "dcae_op_gemm: bad token grid");
  DCAE_REQUIRE(a->ld % 4 == 0 && e->out_ld % 4 == 0 && aligned16(a->base) && aligned16(e->out), "dcae_op_gemm: operand/output must be 16-byte aligned, ld %% 4 == 0");
  DCAE_REQUIRE(a->col0 + a->k0 <= a->ld && (a->k1 == 0 || a->col1 + a->k1 <= a->ld), "dcae_op_gemm: operand columns exceed ld");
  DCAE_REQUIRE(e->act >= DCAE_ACT_NONE && e->act <= DCAE_ACT_RELU, "dcae_op_gemm: bad activation %d", e->act);
  DCAE_REQUIRE(e->act_cols % 4 == 0, "dcae_op_gemm: act_cols must be a multiple of 4");
  DCAE_REQUIRE((!e->addend || (aligned16(e->addend) && e->addend_ld % 4 == 0)) && (!e->residual || (aligned16(e->residual) && e->residual_ld % 4 == 0)) &&
                   aligned16(e->bias) && aligned16(e->res_scale),
               "dcae_op_gemm: epilogue tensors must be 16-byte aligned");
  return DCAE_OK;
}

extern "C" int dcae_op_gemm(const dcae_operand* a, const dcae_weight* w, const dcae_epilogue* e, int math, void* stream) {
  DCAE_TRY(check_gemm_args(a, w, e));
  DCAE_REQUIRE(math == DCAE_MATH_F16X3 || math == DCAE_MATH_F16 || !e->out16_act.hi, "dcae_op_gemm: out16_act is a DCAE_MATH_F16X3 / F16 feature");
  ProfileScope prof(DCAE_PROF_GEMM, 2.0 * a->B * a->h * a->w * (double)w->N * (double)w->K, stream);
  switch (math) {
    case DCAE_MATH_FP32_SIMT:
      DCAE_REQUIRE(a->base && e->out && !e->out16.hi, "dcae_op_gemm(fp32): fp16 planes are a tcgen05-path feature");
      return gemm_simt(a, w, e, (cudaStream_t)stream);
    case DCAE_MATH_TF32X3:
      DCAE_REQUIRE(a->base, "dcae_op_gemm(tf32x3): needs the fp32 operand");
      return gemm_tcgen05(a, w, e, 3, (cudaStream_t)stream);
    case DCAE_MATH_TF32:
      DCAE_REQUIRE(a->base, "dcae_op_gemm(tf32): needs the fp32 operand");
      return gemm_tcgen05(a, w, e, 1, (cudaStream_t)stream);
    case DCAE_MATH_F16X3: return gemm_tcgen05_f16x3(a, w, e, 3, (cudaStream_t)stream);
    case DCAE_MATH_F16: return gemm_tcgen05_f16x3(a, w, e, 1, (cudaStream_t)stream);
  }
  set_error("dcae_op_gemm: unknown math mode %d", math);
  return DCAE_E_INVALID;
}

extern "C" int dcae_op_dict_attention(const float* q, int64_t q_ld, const dcae_planes* q16, const dcae_dict_kv* kv, int64_t T,
                                      float* out, int64_t out_ld, const dcae_planes* out16, int math, void* stream) {
  const dcae_planes o16 = planes_or_null(out16);
  const bool f16 = math == DCAE_MATH_F16X3 || math == DCAE_MATH_F16;
  DCAE_REQUIRE((f16 || q) && kv && kv->Kh && kv->Vh && kv->head_scale && (out || o16.hi) && planes_ok(out16) && planes_ok(q16),
               "dcae_op_dict_attention: null pointer / bad planes");
  DCAE_REQUIRE(math != DCAE_MATH_FP32_SIMT || (out && !o16.hi), "dcae_op_dict_attention(fp32): fp16 planes are a tcgen05-path feature");
  DCAE_REQUIRE(aligned16(q) && aligned16(out) && aligned16(kv->Kh) && aligned16(kv->Vh) && (f16 || (q_ld % 4 == 0 && q_ld >= 640)) &&
                   out_ld % 4 == 0 && (!out || out_ld >= 640),
               "dcae_op_dict_attention: 16-byte alignment and ld >= 640 required");
  DCAE_REQUIRE(T >= 0 && T < (1ll << 31), "dcae_op_dict_attention: bad token count");
  ProfileScope prof(DCAE_PROF_ATTN, 327680.0 * (double)T, stream);
  switch (math) {
    case DCAE_MATH_FP32_SIMT:
      return dict_attention_simt(q, q_ld, kv->Kh, kv->Vh, kv->head_scale, T, out, out_ld, (cudaStream_t)stream);
    case DCAE_MATH_F16X3:
    case DCAE_MATH_F16:   // the attention core stays 3-pass in the fast mode too (3 % of the step)
      return dict_attention_tcgen05_f16(q16, kv, T, out, out_ld, o16, (cudaStream_t)stream);
    case DCAE_MATH_TF32X3: return dict_attention_tcgen05(q, q_ld, kv, T, out, out_ld, o16, 3, (cudaStream_t)stream);
    case DCAE_MATH_TF32: return dict_attention_tcgen05(q, q_ld, kv, T, out, out_ld, o16, 1, (cudaStream_t)stream);
  }
  set_error("dcae_op_dict_attention: unknown math mode %d", math);
  return DCAE_E_INVALID;
}

// =============================================================================================
// Slice-loop plan
// =============================================================================================
namespace {

constexpr int NS = 5, M = 320, SL = 64, D = 640;
constexpr int SUP_LD = 1344;   // [dict_info 320 | latent_scales 320 | latent_means 320 | y_hat 5x64 | y_hat_pre 64]
constexpr int SUP_DICT = 0, SUP_LS = 320, SUP_LM = 640, SUP_YHAT = 960, SUP_PRE = 1280;
constexpr int GC_PARTIALS_MAX = 148 * 8;

struct Buf {
  float* p = nullptr;
  int cols = 0;
};

}  // namespace

// fp16 hi/lo planes buffer [T, ld] (DCAE_MATH_F16X3 data flow: producers write planes, GEMMs read them)
struct PBuf {
  __half* hi = nullptr;
  __half* lo = nullptr;
  int ld = 0;
};

struct dcae_slice_loop {
  int B, h, w, math;
  bool pm;          // planes mode: math == DCAE_MATH_F16X3
  int64_t T, HW;
  dcae_slice_weights wt[NS];
  const float* scale_table;
  // token-major fp32 workspace
  Buf sup, y, means, scales, lik, x0, x1, x2, x3, ln, q, ao, so, dc, ga, t1, t2, f, g, h1, h2, l1, l2, stats, part, stage;
  // fp16 planes (planes mode)
  PBuf supp, lnp, gap, t2p, dcp, aop, gp, x3p, h1p, h2p, l1p, l2p;
  char* planes_begin; size_t planes_total;
  int32_t *sym, *idx, *istage;
  void* planes;     // scratch for the split pass of operands that have no producer-written planes
  int64_t planes_bytes;
  int64_t n_part;   // partial sums per slice
  // planes mode: the cc_scale chain (scale2 -> scale3) runs on a side stream beside the cc_mean chain -- each is
  // 192 tiles on 148 SMs (a 30%-full second wave); side by side the second kernel's CTAs take the SMs the first frees
  cudaStream_t side;
  cudaEvent_t ev_fork, ev_join;
  int n_table;                       // entries of scale_table (2..256)
  int lik_math;                      // DCAE_GC_LIK_FAST (default) / DCAE_GC_LIK_REFERENCE
  bool want_sym;                     // encode also emits int32 symbols / indexes (DCAE_OPT_WANT_SYMBOLS; forward sets it per call)
  bool check_range;                  // DCAE_MATH_F16X3: count operand-plane elements that hit the fp16 clamp (see dcae_slice_loop_check_f16_range)
  unsigned long long* sat_count;     // device counter, part of the workspace
};

static void free_slice_loop(dcae_slice_loop* p) {
  if (!p) return;
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_join) cudaEventDestroy(p->ev_join);
  if (p->side) cudaStreamDestroy(p->side);
  delete p;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static size_t carve(dcae_slice_loop* p, char* base) {
  // Returns total bytes; assigns pointers when base != nullptr.
  size_t off = 0;
  const size_t T = (size_t)p->T;
  auto take = [&](Buf& b, int cols) {
    b.cols = cols;
    b.p = base ? reinterpret_cast<float*>(base + off) : nullptr;
    off = align_up(off + T * cols * sizeof(float), 256);
  };
  take(p->sup, SUP_LD); take(p->y, M); take(p->means, M); take(p->scales, M); take(p->lik, M);
  take(p->x0, D); take(p->x1, D); take(p->x2, D); take(p->x3, D); take(p->ln, D); take(p->q, D);
  take(p->ao, D); take(p->so, D); take(p->dc, 4 * D); take(p->ga, D); take(p->t1, D); take(p->t2, D);
  take(p->f, 4 * D); take(p->g, 2 * D); take(p->h1, 672); take(p->h2, 256); take(p->l1, 224); take(p->l2, 128);
  take(p->stats, 4); take(p->stage, SL);
  p->sym = base ? reinterpret_cast<int32_t*>(base + off) : nullptr; off = align_up(off + T * M * 4, 256);
  p->idx = base ? reinterpret_cast<int32_t*>(base + off) : nullptr; off = align_up(off + T * M * 4, 256);
  p->istage = base ? reinterpret_cast<int32_t*>(base + off) : nullptr; off = align_up(off + T * SL * 4, 256);
  p->part.cols = 0;
  p->part.p = base ? reinterpret_cast<float*>(base + off) : nullptr;
  off = align_up(off + (size_t)NS * GC_PARTIALS_MAX * sizeof(float), 256);
  p->planes_bytes = dcae_planes_bytes((int64_t)T, 4 * D);        // widest operand window: the dense concat
  p->planes = base ? static_cast<void*>(base + off) : nullptr;
  off = align_up(off + (size_t)p->planes_bytes, 256);
  // planes buffers; widths are multiples of 64 so that a padded K window never leaves the allocation
  p->planes_begin = base ? base + off : nullptr;
  const size_t off0 = off;
  auto takep = [&](PBuf& b, int cols) {
    b.ld = cols;
    b.hi = base ? reinterpret_cast<__half*>(base + off) : nullptr;
    off = align_up(off + T * cols * sizeof(__half), 256);
    b.lo = base ? reinterpret_cast<__half*>(base + off) : nullptr;
    off = align_up(off + T * cols * sizeof(__half), 256);
  };
  takep(p->supp, SUP_LD); takep(p->lnp, D); takep(p->gap, D); takep(p->t2p, D); takep(p->dcp, 4 * D); takep(p->aop, D);
  takep(p->gp, 2 * D); takep(p->x3p, D); takep(p->h1p, 704); takep(p->h2p, 256); takep(p->l1p, 256); takep(p->l2p, 128);
  p->planes_total = off - off0;
  p->sat_count = base ? reinterpret_cast<unsigned long long*>(base + off) : nullptr;
  off = align_up(off + sizeof(unsigned long long), 256);
  return off;
}

extern "C" size_t dcae_slice_loop_workspace_bytes(int32_t B, int32_t h, int32_t w) {
  if (B < 0 || h < 0 || w < 0) return 0;
  dcae_slice_loop tmp;
  memset(&tmp, 0, sizeof(tmp));
  tmp.T = (int64_t)B * h * w;
  return carve(&tmp, nullptr) + 256;
}

extern "C" int dcae_slice_loop_create(dcae_slice_loop** out, int32_t B, int32_t h, int32_t w,
                                      const dcae_slice_weights* weights, const float* scale_table, int32_t n_table, void* workspace,
                                      size_t workspace_bytes, int math) {
  DCAE_REQUIRE(out && weights && workspace, "dcae_slice_loop_create: null argument");
  DCAE_REQUIRE(B > 0 && h > 0 && w > 0 && (int64_t)B * h * w < (1ll << 31) / 4, "dcae_slice_loop_create: bad shape B=%d h=%d w=%d", B, h, w);
  DCAE_REQUIRE(math >= DCAE_MATH_FP32_SIMT && math <= DCAE_MATH_F16, "dcae_slice_loop_create: bad math mode %d", math);
  DCAE_REQUIRE(scale_table == nullptr || (n_table >= 2 && n_table <= 256), "dcae_slice_loop_create: scale table of %d entries (2..256 supported: indexes travel as uint8)", n_table);
  DCAE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "dcae_slice_loop_create: workspace must be 256-byte aligned");
  DCAE_TRY(dcae_device_check());
  dcae_slice_loop* p = new (std::nothrow) dcae_slice_loop;
  DCAE_REQUIRE(p != nullptr, "dcae_slice_loop_create: out of host memory");
  memset(static_cast<void*>(p), 0, sizeof(*p));
  p->B = B; p->h = h; p->w = w; p->math = math;
  p->pm = math == DCAE_MATH_F16X3 || math == DCAE_MATH_F16;
  p->HW = (int64_t)h * w;
  p->T = (int64_t)B * h * w;
  const size_t need = carve(p, nullptr);
  if (need > workspace_bytes) {
    set_error("dcae_slice_loop_create: workspace too small (%zu < %zu)", workspace_bytes, need);
    free_slice_loop(p);
    return DCAE_E_WORKSPACE;
  }
  carve(p, static_cast<char*>(workspace));
  memcpy(p->wt, weights, sizeof(dcae_slice_weights) * NS);
  p->scale_table = scale_table;
  p->n_table = scale_table ? n_table : 0;
  p->want_sym = true;
  p->n_part = dcae_gc_num_partials(p->T, SL);
  if (p->pm) {
    // padded K windows over-read a few never-written plane columns (their weight planes are zero): make them finite
    // (the memset runs on the legacy stream; the plan may be used on any non-blocking stream right after create)
    cudaError_t e = cudaMemset(p->planes_begin, 0, p->planes_total);
    if (e == cudaSuccess) e = cudaMemset(p->sat_count, 0, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->side, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      set_error("dcae_slice_loop_create: planes-mode setup failed: %s", cudaGetErrorString(e));
      free_slice_loop(p);
      return DCAE_E_CUDA;
    }
  }
  *out = p;
  return DCAE_OK;
}

extern "C" void dcae_slice_loop_destroy(dcae_slice_loop* p) { free_slice_loop(p); }

extern "C" int dcae_slice_loop_set_option(dcae_slice_loop* p, int32_t option, int32_t value) {
  DCAE_REQUIRE(p, "dcae_slice_loop_set_option: null plan");
  switch (option) {
    case DCAE_OPT_WANT_SYMBOLS:
      p->want_sym = value != 0;
      return DCAE_OK;
    case DCAE_OPT_LIK_MATH:
      DCAE_REQUIRE(value == DCAE_GC_LIK_FAST || value == DCAE_GC_LIK_REFERENCE, "dcae_slice_loop_set_option: bad lik_math %d", value);
      p->lik_math = value;
      return DCAE_OK;
  }
  set_error("dcae_slice_loop_set_option: unknown option %d", option);
  return DCAE_E_INVALID;
}

// ---- small builders --------------------------------------------------------------------------
static dcae_planes pl(const PBuf& b, int col = 0) {
  dcae_planes r;
  r.hi = b.hi ? b.hi + col : nullptr;
  r.lo = b.lo ? b.lo + col : nullptr;
  r.ld = b.ld;
  return r;
}
static dcae_planes no_planes() {
  dcae_planes r;
  r.hi = nullptr; r.lo = nullptr; r.ld = 0;
  return r;
}
// fp32 operand window (split by the GEMM itself if the mode needs planes)
static dcae_operand opnd(const dcae_slice_loop* p, const float* base, int64_t ld, int col0, int k0, int taps, int col1 = 0, int k1 = 0) {
  dcae_operand a;
  memset(&a, 0, sizeof(a));
  a.base = base; a.ld = ld; a.col0 = col0; a.k0 = k0; a.col1 = col1; a.k1 = k1; a.taps = taps;
  a.B = p->B; a.h = p->h; a.w = p->w;
  a.planes = p->planes; a.planes_bytes = p->planes_bytes;
  return a;
}
// operand = planes window in planes mode, the fp32 window otherwise
static dcae_operand opnd2(const dcae_slice_loop* p, const Buf& f32, int64_t ld, const PBuf& f16, int col0, int k0, int taps) {
  dcae_operand a = opnd(p, f32.p, ld, col0, k0, taps);
  if (p->pm) { a.src16 = pl(f16); a.base = nullptr; }
  return a;
}
static dcae_epilogue epi(const float* bias, float* out, int64_t out_ld, int act = DCAE_ACT_NONE) {
  dcae_epilogue e;
  memset(&e, 0, sizeof(e));
  e.bias = bias; e.out = out; e.out_ld = out_ld; e.act = act;
  return e;
}
// output = planes window only (planes mode) or the fp32 buffer (other modes)
static dcae_epilogue epi2(const dcae_slice_loop* p, const float* bias, float* out, int64_t out_ld, const PBuf& f16, int col16, int act = DCAE_ACT_NONE) {
  dcae_epilogue e = epi(bias, out, out_ld, act);
  if (p->pm) { e.out = nullptr; e.out16 = pl(f16, col16); }
  return e;
}
// range check (validation mode): count clamped elements of a freshly written planes window
static int chk(const dcae_slice_loop* p, const dcae_planes& pl16, int cols, void* s) {
  if (!p->check_range || !pl16.hi) return DCAE_OK;
  return dcae_count_f16_clamped(&pl16, p->T, cols, p->sat_count, s);
}
static int gemm(const dcae_slice_loop* p, const dcae_operand& a, const dcae_weight& w, const dcae_epilogue& e, void* s) {
  DCAE_TRY(dcae_op_gemm(&a, &w, &e, p->math, s));
  DCAE_TRY(chk(p, e.out16, w.N, s));
  return chk(p, e.out16_act, w.N, s);
}

extern "C" int dcae_slice_loop_load(dcae_slice_loop* p, const float* y, const float* latent_scales,
                                    const float* latent_means, void* stream) {
  DCAE_REQUIRE(p && latent_scales && latent_means, "dcae_slice_loop_load: null argument");
  g_launches = 0;
  if (y) DCAE_TRY(dcae_op_nchw_to_tokens(y, p->B, M, p->HW, p->y.p, M, nullptr, stream));
  if (p->pm) {   // the latents are only ever GEMM operands: straight to fp16 planes
    const dcae_planes ls = pl(p->supp, SUP_LS), lm = pl(p->supp, SUP_LM);
    DCAE_TRY(dcae_op_nchw_to_tokens(latent_scales, p->B, M, p->HW, nullptr, 0, &ls, stream));
    DCAE_TRY(dcae_op_nchw_to_tokens(latent_means, p->B, M, p->HW, nullptr, 0, &lm, stream));
    DCAE_TRY(chk(p, ls, M, stream));
    DCAE_TRY(chk(p, lm, M, stream));
  } else {
    DCAE_TRY(dcae_op_nchw_to_tokens(latent_scales, p->B, M, p->HW, p->sup.p + SUP_LS, SUP_LD, nullptr, stream));
    DCAE_TRY(dcae_op_nchw_to_tokens(latent_means, p->B, M, p->HW, p->sup.p + SUP_LM, SUP_LD, nullptr, stream));
  }
  return DCAE_OK;
}

// dictionary cross-attention module of slice i (dcae.py:479-509) -> support columns [0, 320)
static int run_dca(dcae_slice_loop* p, int i, void* s, bool dict_f32 = false) {   // dict_f32: also keep dict_info in fp32 (module-level call)
  const dcae_slice_weights& W = p->wt[i];
  const int64_t T = p->T;
  const bool pm = p->pm;
  const int cq = 2 * M + SL * i;
  const dcae_planes none = no_planes();
  const dcae_planes lnp = pm ? pl(p->lnp) : none;
  float* ln32 = pm ? nullptr : p->ln.p;
  // x = x_trans(query)                                                       dcae.py:481-482
  DCAE_TRY(gemm(p, opnd2(p, p->sup, SUP_LD, p->supp, SUP_LS, cq, 1), W.x_trans, epi(W.x_trans_b, p->x0.p, D), s));
  // msa(ln_scale(x))                                                         dcae.py:484, 435-448
  DCAE_TRY(dcae_op_layernorm(p->x0.p, D, W.ln_scale_g, W.ln_scale_b, D, T, ln32, D, &lnp, s));
  DCAE_TRY(chk(p, lnp, D, s));
  {
    dcae_epilogue e = epi(W.msa_s_b, p->dc.p, 4 * D);
    if (pm) {   // planes for proj + planes of GELU(.) = the prologue of dense layer 0; no fp32 copy at all
      e.out = nullptr; e.out16 = pl(p->dcp, 0); e.out16_act = pl(p->gap); e.act2 = DCAE_ACT_GELU;
    }
    DCAE_TRY(gemm(p, opnd2(p, p->ln, D, p->lnp, 0, D, 1), W.msa_s, e, s));
  }
  for (int j = 0; j < 3; ++j) {                                            // DenseBlock dcae.py:416-433
    const dcae_planes t2p = pm ? pl(p->t2p) : none;
    if (!pm) DCAE_TRY(dcae_op_gelu(p->dc.p + D * j, 4 * D, D, T, p->ga.p, D, nullptr, s));
    DCAE_TRY(gemm(p, opnd2(p, p->ga, D, p->gap, 0, D, 1), W.dense_in[j], epi(W.dense_in_b[j], p->t1.p, D, DCAE_ACT_GELU), s));
    DCAE_TRY(dcae_op_dwconv3x3(p->t1.p, D, W.dense_dw[j], W.dense_dw_b[j], D, p->B, p->h, p->w, DCAE_ACT_GELU, nullptr, 0,
                               pm ? nullptr : p->t2.p, D, &t2p, s));
    DCAE_TRY(chk(p, t2p, D, s));
    dcae_epilogue e = epi(W.dense_out_b[j], p->dc.p + D * (j + 1), 4 * D);
    if (pm) {
      e.out = nullptr;
      e.out16 = pl(p->dcp, D * (j + 1));
      if (j < 2) { e.out16_act = pl(p->gap); e.act2 = DCAE_ACT_GELU; }   // GELU prologue of the next dense layer
    }
    DCAE_TRY(gemm(p, opnd2(p, p->t2, D, p->t2p, 0, D, 1), W.dense_out[j], e, s));
  }
  DCAE_TRY(gemm(p, opnd2(p, p->dc, 4 * D, p->dcp, 0, 4 * D, 1), W.dense_proj, epi(W.dense_proj_b, p->so.p, D), s));
  // x = s_out * spatial_atte(s_out) + res_scale_1(x)                         dcae.py:446, 484
  // planes mode: the gate kernel also writes lnx(x) (the row is in its registers): one launch less per slice
  if (pm) {
    DCAE_TRY(dcae_op_spatial_gate_ln(p->so.p, D, p->x0.p, D, W.res_scale_1, W.spatial_w7, D, p->B, p->h, p->w, p->stats.p, p->x1.p, D,
                                     W.lnx_g, W.lnx_b, &lnp, s));
  } else {
    DCAE_TRY(dcae_op_spatial_gate(p->so.p, D, p->x0.p, D, W.res_scale_1, W.spatial_w7, D, p->B, p->h, p->w, p->stats.p, p->x1.p, D, s));
    // q = q_trans(lnx(x)); attention against the dictionary                    dcae.py:486-501
    DCAE_TRY(dcae_op_layernorm(p->x1.p, D, W.lnx_g, W.lnx_b, D, T, ln32, D, &lnp, s));
  }
  DCAE_TRY(chk(p, lnp, D, s));
  {
    dcae_epilogue e = epi(W.q_trans_b, p->q.p, D);
    if (pm) { e.out = nullptr; e.out16 = pl(p->gap); }     // planes mode: q as fp16 planes in the (idle) GELU buffer
    DCAE_TRY(gemm(p, opnd2(p, p->ln, D, p->lnp, 0, D, 1), W.q_trans, e, s));
  }
  {
    const dcae_planes aop = pm ? pl(p->aop) : none;
    const dcae_planes qp = pm ? pl(p->gap) : none;
    DCAE_TRY(dcae_op_dict_attention(pm ? nullptr : p->q.p, D, &qp, &W.kv, T, pm ? nullptr : p->ao.p, D, &aop, p->math, s));
    DCAE_TRY(chk(p, aop, D, s));
  }
  // output = linear(output) + res_scale_2(shortcut)                          dcae.py:503
  {
    dcae_epilogue e = epi(W.linear_b, p->x2.p, D);
    e.residual = p->x1.p; e.residual_ld = D; e.res_scale = W.res_scale_2;
    DCAE_TRY(gemm(p, opnd2(p, p->ao, D, p->aop, 0, D, 1), W.linear, e, s));
  }
  // output = mlp(ln_mlp(output)) + res_scale_3(output)                       dcae.py:505, 312-328
  DCAE_TRY(dcae_op_layernorm(p->x2.p, D, W.ln_mlp_g, W.ln_mlp_b, D, T, ln32, D, &lnp, s));
  DCAE_TRY(chk(p, lnp, D, s));
  DCAE_TRY(gemm(p, opnd2(p, p->ln, D, p->lnp, 0, D, 1), W.fc1, epi(W.fc1_b, p->f.p, 4 * D), s));
  {
    const dcae_planes gp = pm ? pl(p->gp) : none;
    DCAE_TRY(dcae_op_dwconv3x3(p->f.p, 4 * D, W.mlp_dw, W.mlp_dw_b, 2 * D, p->B, p->h, p->w, DCAE_ACT_GELU, p->f.p + 2 * D, 4 * D,
                               pm ? nullptr : p->g.p, 2 * D, &gp, s));
    DCAE_TRY(chk(p, gp, 2 * D, s));
  }
  {
    dcae_epilogue e = epi2(p, W.fc2_b, p->x3.p, D, p->x3p, 0);
    e.residual = p->x2.p; e.residual_ld = D; e.res_scale = W.res_scale_3;
    DCAE_TRY(gemm(p, opnd2(p, p->g, 2 * D, p->gp, 0, 2 * D, 1), W.fc2, e, s));
  }
  // dict_info = output_trans(output)                                         dcae.py:507
  {
    dcae_epilogue e = epi2(p, W.output_trans_b, p->sup.p + SUP_DICT, SUP_LD, p->supp, SUP_DICT);
    if (dict_f32) { e.out = p->sup.p + SUP_DICT; e.out_ld = SUP_LD; }
    DCAE_TRY(gemm(p, opnd2(p, p->x3, D, p->x3p, 0, D, 1), W.output_trans, e, s));
  }
  return DCAE_OK;
}

extern "C" int dcae_slice_loop_params(dcae_slice_loop* p, int32_t i, void* s) {
  DCAE_REQUIRE(p && i >= 0 && i < NS, "dcae_slice_loop_params: bad slice index");
  const dcae_slice_weights& W = p->wt[i];
  DCAE_TRY(run_dca(p, i, s));
  const int cs = 3 * M + SL * i;   // support channels of slice i (dcae.py:647)
  // layer 1 of cc_mean | cc_scale | lrp(support part) share the A operand: N = 672       dcae.py:649-655, 661-662
  {
    dcae_epilogue e = epi(W.cc1_b, p->h1.p, 672, DCAE_ACT_GELU);       // fp32 kept: columns 448.. are the LRP addend
    e.act_cols = 448;
    if (p->pm) e.out16 = pl(p->h1p, 0);
    DCAE_TRY(gemm(p, opnd2(p, p->sup, SUP_LD, p->supp, 0, cs, 9), W.cc1, e, s));
  }
  // The two chains are independent (dcae.py:649-655) and write disjoint columns / buffers.  In planes mode no split
  // scratch is shared either, so the scale chain forks onto the side stream and joins before the caller continues.
  void* s2 = s;
  if (p->pm && p->side && !profiling_on()) {     // an instrumented step times every kernel ALONE (dcae_profile_start)
    s2 = p->side;
    DCAE_CUDA(cudaEventRecord(p->ev_fork, (cudaStream_t)s));
    DCAE_CUDA(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
  }
  DCAE_TRY(gemm(p, opnd2(p, p->h1, 672, p->h1p, 0, 224, 9), W.mean2, epi2(p, W.mean2_b, p->h2.p, 256, p->h2p, 0, DCAE_ACT_GELU), s));
  DCAE_TRY(gemm(p, opnd2(p, p->h1, 672, p->h1p, 224, 224, 9), W.scale2, epi2(p, W.scale2_b, p->h2.p + 128, 256, p->h2p, 128, DCAE_ACT_GELU), s2));
  DCAE_TRY(gemm(p, opnd2(p, p->h2, 256, p->h2p, 0, 128, 9), W.mean3, epi(W.mean3_b, p->means.p + SL * i, M), s));
  DCAE_TRY(gemm(p, opnd2(p, p->h2, 256, p->h2p, 128, 128, 9), W.scale3, epi(W.scale3_b, p->scales.p + SL * i, M), s2));
  if (s2 != s) {
    DCAE_CUDA(cudaEventRecord(p->ev_join, (cudaStream_t)s2));
    DCAE_CUDA(cudaStreamWaitEvent((cudaStream_t)s, p->ev_join, 0));
  }
  return DCAE_OK;
}

// ---- module-level entry points (SURVEY 8b: the reference's own nn.Module surfaces) -------------------------
// One module of slice i on the caller's NCHW tensor, through the plan's buffers (do not interleave with a slice
// loop in flight on the same plan).  The reference channel order of the inputs is the support-buffer order
// [latent_scales | latent_means | y_hat_0.. | (dict_info) | (y_hat_slice)], so windows land by column.
static int load_window(dcae_slice_loop* p, const float* x, int64_t x_channels, int c0, int C, int sup_col, void* s) {
  for (int b = 0; b < p->B; ++b) {                       // per image: the window's batch stride is the caller's
    const float* src = x + ((int64_t)b * x_channels + c0) * p->HW;
    const int64_t row0 = (int64_t)b * p->HW;
    if (p->pm) {
      dcae_planes w = pl(p->supp, sup_col);
      w.hi = static_cast<__half*>(w.hi) + row0 * w.ld;
      w.lo = static_cast<__half*>(w.lo) + row0 * w.ld;
      DCAE_TRY(dcae_op_nchw_to_tokens(src, 1, C, p->HW, p->sup.p + row0 * SUP_LD + sup_col, SUP_LD, &w, s));
      if (p->check_range) DCAE_TRY(dcae_count_f16_clamped(&w, p->HW, C, p->sat_count, s));
    } else {
      DCAE_TRY(dcae_op_nchw_to_tokens(src, 1, C, p->HW, p->sup.p + row0 * SUP_LD + sup_col, SUP_LD, nullptr, s));
    }
  }
  return DCAE_OK;
}

extern "C" int dcae_slice_loop_module_dca(dcae_slice_loop* p, int32_t i, const float* x, float* out, void* s) {
  DCAE_REQUIRE(p && x && out && i >= 0 && i < NS, "dcae_slice_loop_module_dca: bad argument");
  const int cq = 2 * M + SL * i;
  DCAE_TRY(load_window(p, x, cq, 0, cq, SUP_LS, s));
  DCAE_TRY(run_dca(p, i, s, true));
  return dcae_op_tokens_to_nchw(p->sup.p + SUP_DICT, SUP_LD, p->B, M, p->HW, out, s);
}

// which: 0 = cc_mean_transforms[i], 1 = cc_scale_transforms[i] (x: [B, 960 + 64 i, h, w]), 2 = lrp_transforms[i]
// (x: [B, 1024 + 64 i, h, w], the RAW conv stack: the caller applies 0.5 tanh as dcae.py:663 does).
extern "C" int dcae_slice_loop_module_conv(dcae_slice_loop* p, int32_t i, int32_t which, const float* x, float* out, void* s) {
  DCAE_REQUIRE(p && x && out && i >= 0 && i < NS && which >= 0 && which <= 2, "dcae_slice_loop_module_conv: bad argument");
  const dcae_slice_weights& W = p->wt[i];
  const int cq = 2 * M + SL * i, cs = 3 * M + SL * i, cx = cs + (which == 2 ? SL : 0);
  DCAE_TRY(load_window(p, x, cx, 0, cq, SUP_LS, s));
  DCAE_TRY(load_window(p, x, cx, cq, M, SUP_DICT, s));
  if (which == 2) DCAE_TRY(load_window(p, x, cx, cs, SL, SUP_PRE, s));
  {
    dcae_epilogue e = epi(W.cc1_b, p->h1.p, 672, DCAE_ACT_GELU);       // the fused first layer of all three stacks
    e.act_cols = 448;
    if (p->pm) e.out16 = pl(p->h1p, 0);
    DCAE_TRY(gemm(p, opnd2(p, p->sup, SUP_LD, p->supp, 0, cs, 9), W.cc1, e, s));
  }
  float* res = nullptr;
  if (which == 0) {
    DCAE_TRY(gemm(p, opnd2(p, p->h1, 672, p->h1p, 0, 224, 9), W.mean2, epi2(p, W.mean2_b, p->h2.p, 256, p->h2p, 0, DCAE_ACT_GELU), s));
    res = p->means.p + SL * i;
    DCAE_TRY(gemm(p, opnd2(p, p->h2, 256, p->h2p, 0, 128, 9), W.mean3, epi(W.mean3_b, res, M), s));
  } else if (which == 1) {
    DCAE_TRY(gemm(p, opnd2(p, p->h1, 672, p->h1p, 224, 224, 9), W.scale2, epi2(p, W.scale2_b, p->h2.p + 128, 256, p->h2p, 128, DCAE_ACT_GELU), s));
    res = p->scales.p + SL * i;
    DCAE_TRY(gemm(p, opnd2(p, p->h2, 256, p->h2p, 128, 128, 9), W.scale3, epi(W.scale3_b, res, M), s));
  } else {
    dcae_epilogue e = epi2(p, W.lrp1_b, p->l1.p, 224, p->l1p, 0, DCAE_ACT_GELU);
    e.addend = p->h1.p + 448; e.addend_ld = 672;
    DCAE_TRY(gemm(p, opnd2(p, p->sup, SUP_LD, p->supp, SUP_PRE, SL, 9), W.lrp1y, e, s));
    DCAE_TRY(gemm(p, opnd2(p, p->l1, 224, p->l1p, 0, 224, 9), W.lrp2, epi2(p, W.lrp2_b, p->l2.p, 128, p->l2p, 0, DCAE_ACT_GELU), s));
    res = p->lik.p + SL * i;                                           // scratch window: raw lrp stack output
    DCAE_TRY(gemm(p, opnd2(p, p->l2, 128, p->l2p, 0, 128, 9), W.lrp3, epi(W.lrp3_b, res, M), s));
  }
  return dcae_op_tokens_to_nchw(res, M, p->B, SL, p->HW, out, s);
}

// LRP of slice i (dcae.py:661-664): y_hat_i = y_hat_pre + 0.5 tanh(lrp(cat(support, y_hat_pre)))
static int run_lrp(dcae_slice_loop* p, int i, void* s) {
  const dcae_slice_weights& W = p->wt[i];
  {
    dcae_epilogue e = epi2(p, W.lrp1_b, p->l1.p, 224, p->l1p, 0, DCAE_ACT_GELU);
    e.addend = p->h1.p + 448; e.addend_ld = 672;     // support part of lrp layer 1, accumulated with cc1
    DCAE_TRY(gemm(p, opnd2(p, p->sup, SUP_LD, p->supp, SUP_PRE, SL, 9), W.lrp1y, e, s));
  }
  DCAE_TRY(gemm(p, opnd2(p, p->l1, 224, p->l1p, 0, 224, 9), W.lrp2, epi2(p, W.lrp2_b, p->l2.p, 128, p->l2p, 0, DCAE_ACT_GELU), s));
  {
    dcae_epilogue e = epi(W.lrp3_b, p->sup.p + SUP_YHAT + SL * i, SUP_LD, DCAE_ACT_HALF_TANH);   // fp32: the loop's output
    e.residual = p->sup.p + SUP_PRE; e.residual_ld = SUP_LD;
    if (p->pm) e.out16 = pl(p->supp, SUP_YHAT + SL * i);                                        // planes: later slices' operand
    DCAE_TRY(gemm(p, opnd2(p, p->l2, 128, p->l2p, 0, 128, 9), W.lrp3, e, s));
  }
  return DCAE_OK;
}

static dcae_gc_args gc_base(dcae_slice_loop* p, int i) {
  dcae_gc_args a;
  memset(&a, 0, sizeof(a));
  a.mu = p->means.p + SL * i; a.mu_ld = M;
  a.scale = p->scales.p + SL * i; a.scale_ld = M;
  a.scale_table = p->scale_table; a.n_table = p->n_table;
  a.scale_bound = 0.11f; a.lik_bound = 1e-9f;
  a.rows = p->T; a.inner = SL;
  a.lik_math = p->lik_math;
  return a;
}

extern "C" int dcae_slice_loop_encode(dcae_slice_loop* p, int32_t i, int32_t gc_mode, const float* noise, void* s) {
  DCAE_REQUIRE(p && i >= 0 && i < NS, "dcae_slice_loop_encode: bad slice index");
  DCAE_REQUIRE(gc_mode == DCAE_GC_EVAL || (gc_mode == DCAE_GC_NOISE && noise), "dcae_slice_loop_encode: bad mode / missing noise");
  dcae_gc_args a = gc_base(p, i);
  a.mode = gc_mode;
  a.y = p->y.p + SL * i; a.y_ld = M;
  if (gc_mode == DCAE_GC_NOISE) {
    DCAE_TRY(dcae_op_nchw_to_tokens(noise, p->B, SL, p->HW, p->stage.p, SL, nullptr, s));
    a.noise = p->stage.p; a.noise_ld = SL;
  }
  a.y_hat = p->sup.p + SUP_PRE; a.y_hat_ld = SUP_LD;
  if (p->pm) a.y_hat16 = pl(p->supp, SUP_PRE);
  a.lik = p->lik.p + SL * i; a.lik_ld = M;
  if (p->want_sym) {                 // forward without symbols: the 20 B/element variant (no int32 stores)
    a.sym = p->sym + SL * i; a.sym_ld = M;
    if (p->scale_table) { a.idx = p->idx + SL * i; a.idx_ld = M; }
  }
  a.log2_partials = p->part.p + (int64_t)i * p->n_part;
  DCAE_TRY(dcae_gc_fused(&a, s));
  DCAE_TRY(chk(p, a.y_hat16, SL, s));
  return run_lrp(p, i, s);
}

extern "C" int dcae_slice_loop_indexes(dcae_slice_loop* p, int32_t i, int32_t* indexes_nchw, void* s) {
  DCAE_REQUIRE(p && i >= 0 && i < NS && indexes_nchw, "dcae_slice_loop_indexes: bad arguments");
  DCAE_REQUIRE(p->scale_table, "dcae_slice_loop_indexes: no scale table (update_scale_table not called)");
  dcae_gc_args a = gc_base(p, i);
  a.mode = DCAE_GC_EVAL;
  a.idx = p->idx + SL * i; a.idx_ld = M;
  DCAE_TRY(dcae_gc_fused(&a, s));
  return dcae_op_tokens_to_nchw_i32(p->idx + SL * i, M, p->B, SL, p->HW, indexes_nchw, s);
}

extern "C" int dcae_slice_loop_decode(dcae_slice_loop* p, int32_t i, const int32_t* symbols_nchw, void* s) {
  DCAE_REQUIRE(p && i >= 0 && i < NS && symbols_nchw, "dcae_slice_loop_decode: bad arguments");
  DCAE_TRY(dcae_op_nchw_to_tokens_i32(symbols_nchw, p->B, SL, p->HW, p->istage, SL, s));
  dcae_gc_args a = gc_base(p, i);
  a.mode = DCAE_GC_DECODE;
  a.scale = nullptr;
  a.sym_in = p->istage; a.sym_in_ld = SL;
  a.y_hat = p->sup.p + SUP_PRE; a.y_hat_ld = SUP_LD;
  if (p->pm) a.y_hat16 = pl(p->supp, SUP_PRE);
  DCAE_TRY(dcae_gc_fused(&a, s));
  DCAE_TRY(chk(p, a.y_hat16, SL, s));
  return run_lrp(p, i, s);
}

extern "C" int dcae_slice_loop_check_f16_range(dcae_slice_loop* p, int32_t enable, unsigned long long* clamped_host) {
  DCAE_REQUIRE(p, "dcae_slice_loop_check_f16_range: null plan");
  if (clamped_host) {                                  // read (synchronises the device) and reset
    DCAE_CUDA(cudaDeviceSynchronize());
    DCAE_CUDA(cudaMemcpy(clamped_host, p->sat_count, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  }
  DCAE_CUDA(cudaMemset(p->sat_count, 0, sizeof(unsigned long long)));
  p->check_range = enable != 0 && p->pm;
  return DCAE_OK;
}

extern "C" int dcae_slice_loop_store(dcae_slice_loop* p, float* y_hat, float* means, float* scales, float* lik,
                                     int32_t* symbols, int32_t* indexes, float* log2_lik_sum, void* s) {
  DCAE_REQUIRE(p, "dcae_slice_loop_store: null plan");
  if (y_hat) DCAE_TRY(dcae_op_tokens_to_nchw(p->sup.p + SUP_YHAT, SUP_LD, p->B, M, p->HW, y_hat, s));
  if (means) DCAE_TRY(dcae_op_tokens_to_nchw(p->means.p, M, p->B, M, p->HW, means, s));
  if (scales) DCAE_TRY(dcae_op_tokens_to_nchw(p->scales.p, M, p->B, M, p->HW, scales, s));
  if (lik) DCAE_TRY(dcae_op_tokens_to_nchw(p->lik.p, M, p->B, M, p->HW, lik, s));
  const int64_t per_slice = (int64_t)p->B * SL * p->HW;
  DCAE_REQUIRE(!(symbols || indexes) || p->want_sym, "dcae_slice_loop_store: symbols / indexes requested but DCAE_OPT_WANT_SYMBOLS was off during encode");
  for (int i = 0; i < NS; ++i) {
    if (symbols) DCAE_TRY(dcae_op_tokens_to_nchw_i32(p->sym + SL * i, M, p->B, SL, p->HW, symbols + i * per_slice, s));
    if (indexes) {
      DCAE_REQUIRE(p->scale_table, "dcae_slice_loop_store: indexes requested but no scale table");
      DCAE_TRY(dcae_op_tokens_to_nchw_i32(p->idx + SL * i, M, p->B, SL, p->HW, indexes + i * per_slice, s));
    }
  }
  if (log2_lik_sum) DCAE_TRY(dcae_reduce_partials(p->part.p, NS * p->n_part, log2_lik_sum, s));
  return DCAE_OK;
}

extern "C" int dcae_slice_loop_forward(dcae_slice_loop* p, const float* y, const float* latent_scales,
                                       const float* latent_means, float* y_hat, float* means, float* scales, float* lik,
                                       int32_t* symbols, int32_t* indexes, float* log2_lik_sum, void* s) {
  DCAE_REQUIRE(p && y, "dcae_slice_loop_forward: null argument");
  p->want_sym = symbols != nullptr || indexes != nullptr;
  DCAE_TRY(dcae_slice_loop_load(p, y, latent_scales, latent_means, s));
  for (int i = 0; i < NS; ++i) {
    DCAE_TRY(dcae_slice_loop_params(p, i, s));
    DCAE_TRY(dcae_slice_loop_encode(p, i, DCAE_GC_EVAL, nullptr, s));
  }
  return dcae_slice_loop_store(p, y_hat, means, scales, lik, symbols, indexes, log2_lik_sum, s);
}

extern "C" int dcae_slice_loop_tap(dcae_slice_loop* p, const char* name, const float** ptr, int32_t* cols, int64_t* ld) {
  DCAE_REQUIRE(p && name && ptr && cols && ld, "dcae_slice_loop_tap: null argument");
  struct { const char* n; Buf* b; } tbl[] = {
      {"support", &p->sup}, {"y", &p->y}, {"means", &p->means}, {"scales", &p->scales}, {"lik", &p->lik},
      {"x0", &p->x0}, {"x1", &p->x1}, {"x2", &p->x2}, {"x3", &p->x3}, {"q", &p->q}, {"attn", &p->ao},
      {"s_out", &p->so}, {"dense", &p->dc}, {"fc1", &p->f}, {"glu", &p->g}, {"h1", &p->h1}, {"h2", &p->h2},
      {"l1", &p->l1}, {"l2", &p->l2}};
  for (auto& t : tbl)
    if (strcmp(t.n, name) == 0) {
      *ptr = t.b->p; *cols = t.b->cols; *ld = t.b->cols;
      return DCAE_OK;
    }
  set_error("dcae_slice_loop_tap: unknown buffer '%s'", name);
  return DCAE_E_INVALID;
}

extern "C" int dcae_slice_loop_tap16(dcae_slice_loop* p, const char* name, dcae_planes* planes, int32_t* cols) {
  DCAE_REQUIRE(p && name && planes && cols, "dcae_slice_loop_tap16: null argument");
  DCAE_REQUIRE(p->pm, "dcae_slice_loop_tap16: the plan is not in DCAE_MATH_F16X3 mode");
  struct { const char* n; PBuf* b; } tbl[] = {
      {"support", &p->supp}, {"ln", &p->lnp}, {"gelu", &p->gap}, {"dw", &p->t2p}, {"dense", &p->dcp}, {"attn", &p->aop},
      {"glu", &p->gp}, {"x3", &p->x3p}, {"h1", &p->h1p}, {"h2", &p->h2p}, {"l1", &p->l1p}, {"l2", &p->l2p}};
  for (auto& t : tbl)
    if (strcmp(t.n, name) == 0) {
      planes->hi = t.b->hi; planes->lo = t.b->lo; planes->ld = t.b->ld;
      *cols = t.b->ld;
      return DCAE_OK;
    }
  set_error("dcae_slice_loop_tap16: unknown planes buffer '%s'", name);
  return DCAE_E_INVALID;
}
