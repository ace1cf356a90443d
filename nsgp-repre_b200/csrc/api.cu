// C ABI (include/nsgp_repre_b200.h) over the kernels of this directory.
#include <cstdarg>
#include <mutex>
#include <vector>

#include "../../include/nsgp_repre_b200.h"
#include "common.cuh"
#include "geometry.h"
#include "repre.h"
#include "sgd.h"

namespace nsgp {

static thread_local char g_err[512] = "";
unsigned long long g_launches = 0;
#ifdef NSGP_BRINGUP
int g_engine = 0;
#endif

int g_profile = 0;
namespace {
struct ProfRec { cudaEvent_t a, b; };
std::vector<ProfRec> g_prof[kProfKinds];
cudaEvent_t g_prof_open[kProfKinds];
}
namespace {
constexpr int kTlSlots = 512;
unsigned long long* g_tl_dev = nullptr;
int g_tl_n = 0;
int g_tl_kind[kTlSlots];
}
unsigned long long* timeline_slot(int kind) {
  static const bool on = nsgp_env("NSGP_TIMELINE") != nullptr;
  if (!on || g_tl_n >= kTlSlots) return nullptr;
  if (g_tl_dev == nullptr) {
    if (cudaMalloc(&g_tl_dev, kTlSlots * 2 * sizeof(unsigned long long)) != cudaSuccess) return nullptr;
    std::vector<unsigned long long> init(kTlSlots * 2);
    for (int i = 0; i < kTlSlots; ++i) { init[2 * i] = ~0ull; init[2 * i + 1] = 0; }
    cudaMemcpy(g_tl_dev, init.data(), init.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice);
  }
  g_tl_kind[g_tl_n] = kind;
  return g_tl_dev + 2 * (g_tl_n++);
}
void profile_begin(int kind, cudaStream_t s) {
  cudaEvent_t e;
  cudaEventCreate(&e);
  cudaEventRecord(e, s);
  g_prof_open[kind] = e;
}
void profile_end(int kind, cudaStream_t s) {
  cudaEvent_t e;
  cudaEventCreate(&e);
  cudaEventRecord(e, s);
  g_prof[kind].push_back({g_prof_open[kind], e});
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int contraction(const ContractionArgs& a, cudaStream_t stream) {
#ifdef NSGP_BRINGUP
  if (g_engine == 1) return contraction_simt(a, stream);
#endif
  return contraction_tc(a, stream);
}

static int pick_splits(int tiles, int nkb) {
  // enough CTAs for ~3 waves over 148 SMs, at least 8 K-blocks per CTA
  int want = ceil_div(148 * 3, tiles);
  int cap = nkb / 8;
  if (cap < 1) cap = 1;
  if (want > cap) want = cap;
  return want < 1 ? 1 : want;
}

static inline char* align_up(char* p, size_t a) {
  return reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(p) + a - 1) / a * a);
}

}  // namespace nsgp

using namespace nsgp;

extern "C" {

int nsgp_abi_version(void) { return NSGP_ABI_VERSION; }
const char* nsgp_last_error(void) { return g_err; }
unsigned long long nsgp_launch_count(void) { return g_launches; }
#ifdef NSGP_BRINGUP
int nsgp_set_engine(int engine) {
  int prev = g_engine;
  if (engine == 0 || engine == 1) g_engine = engine;
  return prev;
}
int nsgp_get_engine(void) { return g_engine; }
#endif

int nsgp_profile_enable(int on) {
  int prev = g_profile;
  g_profile = on ? 1 : 0;
  return prev;
}

int nsgp_profile_read(int kind, double* ms_total, unsigned long long* launches) {
  NSGP_REQUIRE(kind >= 0 && kind < kProfKinds && ms_total && launches, "profile_read: bad arguments");
  double total = 0.0;
  for (auto& r : g_prof[kind]) {
    NSGP_CHECK_CUDA(cudaEventSynchronize(r.b));
    float ms = 0.f;
    NSGP_CHECK_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    total += ms;
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  *ms_total = total;
  *launches = g_prof[kind].size();
  g_prof[kind].clear();
  return 0;
}

// ---------------------------------------------------------------- covariance
// Per-layer group table (autocorrelation layout: 29 problems -> one launch) kept behind
// the staged operand in the same workspace.
static size_t layer_table_bytes(const ConvGeom& g) {
  if (g.mode != kModeAutocorr) return 0;
  ContractionArgs probs[kMaxConvProblems];
  int n = 0;
  conv_problems(g, nullptr, nullptr, probs, &n);
  return group_table_bytes(probs, n) + 1024 + autocorr_table_bytes(&g, 1) + 256;
}

int nsgp_cov_conv2d_layout(int C, int H, int W, int kh, int kw, int sh, int sw, int ph, int pw,
                           nsgp_cov_layout_t* out) {
  NSGP_REQUIRE(out != nullptr, "layout: out is null");
  ConvGeom g;
  NSGP_REQUIRE(make_conv_geom(C, H, W, kh, kw, sh, sw, ph, pw, &g) == 0,
               "layout: invalid conv geometry C=%d H=%d W=%d k=%dx%d s=%dx%d p=%dx%d", C, H, W,
               kh, kw, sh, sw, ph, pw);
  out->d = g.d;
  out->d_int = g.d_int;
  out->taps = g.T;
  if (g.mode == kModeAutocorr) {
    out->kind = 1;
    out->ld = (int)round_up(g.C, 4);
    out->acc_bytes = (size_t)kAcMats * g.C * out->ld * sizeof(float);
  } else {
    out->kind = 0;
    out->ld = (int)round_up(g.d_int, 4);
    out->acc_bytes = (size_t)out->ld * g.d_int * sizeof(float);
  }
  out->workspace_bytes = stage_bytes(g) + 1024 + layer_table_bytes(g) +
                         mean_scratch_elems(g) * sizeof(float) + 256;
  return 0;
}

int nsgp_cov_linear_layout(int d, nsgp_cov_layout_t* out) {
  NSGP_REQUIRE(out != nullptr && d > 0, "linear layout: bad arguments");
  out->d = d;
  out->d_int = d;
  out->taps = 1;
  out->kind = 0;
  out->ld = (int)round_up(d, 4);
  out->acc_bytes = (size_t)out->ld * d * sizeof(float);
  out->workspace_bytes = (size_t)round_up(d, 4) * sizeof(float) + 256;
  return 0;
}

// Group table of a set of staged layers: generic problems (single-CTA / pair kernel) and,
// for the autocorrelation layers, the 13 R blocks through the sliding-window kernel.
static int cov_layers_group_build(const ConvGeom* geoms, float* const* stages, float* const* accs,
                                  int n, void* table_dev, size_t table_bytes, GroupInfo* gi,
                                  cudaStream_t stream) {
  std::vector<ContractionArgs> probs;
  std::vector<ConvGeom> ac_g;
  std::vector<const float*> ac_s;
  std::vector<float*> ac_a;
  for (int i = 0; i < n; ++i) {
    ContractionArgs p[kMaxConvProblems];
    int np = 0;
    conv_problems(geoms[i], stages[i], accs[i], p, &np, i + 1);
    if (geoms[i].mode == kModeAutocorr && geoms[i].tiled) {
      ac_g.push_back(geoms[i]);             // R blocks go to the sliding-window kernel
      ac_s.push_back(stages[i]);
      ac_a.push_back(accs[i]);
    }
    probs.insert(probs.end(), p, p + np);
  }
  int rc = group_table_build(probs.data(), (int)probs.size(), kProfGram, table_dev, table_bytes,
                             gi, stream);
  if (rc) return rc;
  if (!ac_g.empty()) {
    const size_t off = (size_t)round_up((long long)gi->bytes, 256);
    NSGP_REQUIRE(off <= table_bytes, "cov group: table too small");
    SubGroup sg{};
    rc = autocorr_table_build(ac_g.data(), ac_s.data(), ac_a.data(), (int)ac_g.size(),
                              (char*)table_dev + off, table_bytes - off, &sg, stream);
    if (rc) return rc;
    sg.off_probs += off;
    sg.off_items += off;
    gi->sub[2] = sg;
    gi->bytes = sg.off_items + (size_t)sg.n_items * 32 + 64;     // + the scheduler's counters
  }
  return 0;
}

static size_t cov_layers_group_bytes(const ConvGeom* geoms, int n) {
  std::vector<ContractionArgs> probs;
  std::vector<ConvGeom> ac_g;
  for (int i = 0; i < n; ++i) {
    ContractionArgs p[kMaxConvProblems];
    int np = 0;
    conv_problems(geoms[i], nullptr, nullptr, p, &np, i + 1);
    probs.insert(probs.end(), p, p + np);
    if (geoms[i].mode == kModeAutocorr && geoms[i].tiled) ac_g.push_back(geoms[i]);
  }
  return group_table_bytes(probs.data(), (int)probs.size()) + 1024 +
         autocorr_table_bytes(ac_g.data(), (int)ac_g.size());
}

static int cov_conv2d_setup(int C, int H, int W, int kh, int kw, int sh, int sw, int ph, int pw,
                            void* workspace, size_t workspace_bytes, ConvGeom* g, float** stage) {
  NSGP_REQUIRE(make_conv_geom(C, H, W, kh, kw, sh, sw, ph, pw, g) == 0,
               "cov_conv2d: invalid conv geometry");
  char* ws = align_up((char*)workspace, 1024);
  NSGP_REQUIRE(ws + stage_bytes(*g) <= (char*)workspace + workspace_bytes,
               "cov_conv2d: workspace too small (%zu < %zu)", workspace_bytes,
               stage_bytes(*g) + 1024);
  *stage = reinterpret_cast<float*>(ws);
  return 0;
}

int nsgp_cov_conv2d_stage(const float* x, int B, int C, int H, int W, int kh, int kw, int sh,
                          int sw, int ph, int pw, void* workspace, size_t workspace_bytes,
                          void* stream_) {
  NSGP_REQUIRE(x && workspace, "cov_conv2d_stage: null pointer");
  NSGP_REQUIRE(B > 0, "cov_conv2d: empty batch");
  ConvGeom g;
  float* stage;
  int rc = cov_conv2d_setup(C, H, W, kh, kw, sh, sw, ph, pw, workspace, workspace_bytes, &g, &stage);
  if (rc) return rc;
  // [staged operand | per-layer group table | batch-mean scratch]
  float* mean = nullptr;
  if (mean_scratch_elems(g) > 0) {
    char* m = align_up((char*)stage + stage_bytes(g) + layer_table_bytes(g), 256);
    if (m + mean_scratch_elems(g) * sizeof(float) <= (char*)workspace + workspace_bytes)
      mean = reinterpret_cast<float*>(m);
  }
  return launch_stage_conv(x, stage, g, B, mean, (cudaStream_t)stream_);
}

int nsgp_cov_conv2d_contract(int C, int H, int W, int kh, int kw, int sh, int sw, int ph, int pw,
                             float* acc, const void* workspace, size_t workspace_bytes,
                             void* stream_) {
  NSGP_REQUIRE(acc && workspace, "cov_conv2d_contract: null pointer");
  ConvGeom g;
  float* stage;
  int rc = cov_conv2d_setup(C, H, W, kh, kw, sh, sw, ph, pw, const_cast<void*>(workspace),
                            workspace_bytes, &g, &stage);
  if (rc) return rc;
  ContractionArgs probs[kMaxConvProblems];
  int n = 0;
  conv_problems(g, stage, acc, probs, &n);
  if (n > 1 && g_engine == 0) {
    // one or two persistent launches for all problems of the layer
    char* table = align_up((char*)stage + stage_bytes(g), 256);
    const size_t room = (size_t)(((const char*)workspace + workspace_bytes) - table);
    GroupInfo gi{};
    float* stage_p = stage;
    rc = cov_layers_group_build(&g, &stage_p, &acc, 1, table, room, &gi, (cudaStream_t)stream_);
    if (rc) return rc;
    return group_launch(table, gi, (cudaStream_t)stream_);
  }
  for (int i = 0; i < n; ++i) {
    if (probs[i].epi == kEpiGramAtomic) {
      int tiles_1d = ceil_div(probs[i].A.rows, 128);
      probs[i].splits = pick_splits(tiles_1d * (tiles_1d + 1) / 2, k_blocks(probs[i].A));
    }
    rc = contraction(probs[i], (cudaStream_t)stream_);
    if (rc) return rc;
  }
  return 0;
}

int nsgp_cov_conv2d_accumulate(const float* x, int B, int C, int H, int W, int kh, int kw,
                               int sh, int sw, int ph, int pw, float* acc, void* workspace,
                               size_t workspace_bytes, void* stream_) {
  NSGP_REQUIRE(x && acc && workspace, "cov_conv2d: null pointer");
  int rc = nsgp_cov_conv2d_stage(x, B, C, H, W, kh, kw, sh, sw, ph, pw, workspace,
                                 workspace_bytes, stream_);
  if (rc) return rc;
  return nsgp_cov_conv2d_contract(C, H, W, kh, kw, sh, sw, ph, pw, acc, workspace,
                                  workspace_bytes, stream_);
}

int nsgp_cov_linear_accumulate(const float* x, int R, int d, float* acc, void* workspace,
                               size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(x && acc && workspace, "cov_linear: null pointer");
  NSGP_REQUIRE(R > 0 && d > 0, "cov_linear: empty input");
  char* ws = align_up((char*)workspace, 256);
  NSGP_REQUIRE(ws + (size_t)d * 4 <= (char*)workspace + workspace_bytes,
               "cov_linear: workspace too small");
  return launch_linear_cov(x, R, d, acc, (int)round_up(d, 4), reinterpret_cast<float*>(ws),
                           stream);
}

int nsgp_cov_finalize(const float* acc, const nsgp_cov_layout_t* L, float* cov_out,
                      int accumulate, void* stream_) {
  NSGP_REQUIRE(acc && L && cov_out, "cov_finalize: null pointer");
  NSGP_REQUIRE(L->taps >= 1 && L->d % L->taps == 0, "cov_finalize: bad layout");
  if (L->kind == 1) {
    NSGP_REQUIRE(L->taps == 9, "cov_finalize: autocorrelation layout needs 9 taps");
    return launch_cov_finalize_autocorr(acc, cov_out, L->d / 9, accumulate, (cudaStream_t)stream_);
  }
  return launch_cov_finalize(acc, L->ld, cov_out, L->d / L->taps, L->taps, accumulate,
                             (cudaStream_t)stream_);
}

// ---------------------------------------------------------------- projection
int nsgp_projector_prepare_lowrank(const float* U, int d, int r, float* ut_hi, float* ut_lo,
                                   float* un_hi, float* un_lo, void* stream_) {
  NSGP_REQUIRE(U && ut_hi && ut_lo && un_hi && un_lo && d > 0 && r > 0,
               "projector_prepare_lowrank: bad arguments");
  cudaStream_t stream = (cudaStream_t)stream_;
  // U^T (r x pitch(d)): transpose + split;  U (d x pitch(r)): split with padded pitch
  int rc = launch_transpose_split_rect(U, ut_hi, ut_lo, d, r, (int)round_up(d, 4), stream);
  if (rc) return rc;
  return launch_split_pitched(U, un_hi, un_lo, d, r, (int)round_up(r, 4), stream);
}

int nsgp_projector_prepare(const float* P, int d, float* pt_hi, float* pt_lo, void* stream_) {
  NSGP_REQUIRE(P && pt_hi && pt_lo && d > 0, "projector_prepare: bad arguments");
  return launch_transpose_split(P, pt_hi, pt_lo, d, (int)round_up(d, 4), (cudaStream_t)stream_);
}

static int sgd_tables(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                      const nsgp_proj_layer_t* layers, int n_layers, double momentum_hint,
                      std::vector<SgdTensorDev>* host, std::vector<int>* chunk_start) {
  host->resize(n_tensors);
  chunk_start->resize(n_tensors + 1);
  int total = 0;
  for (int i = 0; i < n_tensors; ++i) {
    const nsgp_sgd_tensor_t& t = tensors[i];
    NSGP_REQUIRE(t.w && t.g, "sgd_step: tensor %d has a null weight/grad pointer", i);
    NSGP_REQUIRE(momentum_hint == 0.0 || t.buf, "sgd_step: tensor %d needs a momentum buffer", i);
    SgdTensorDev d{};
    d.w = t.w; d.g = t.g; d.buf = t.buf; d.numel = t.numel; d.first = t.first_step;
    if (t.layer >= 0) {
      NSGP_REQUIRE(t.layer < n_layers && layers, "sgd_step: tensor %d: bad layer index", i);
      const nsgp_proj_layer_t& L = layers[t.layer];
      NSGP_REQUIRE((long long)L.cout * L.d == t.numel,
                   "sgd_step: tensor %d: cout*d != numel", i);
      d.u_hi = L.u_hi; d.u_lo = L.u_lo;
      d.d = L.d; d.ldu = (int)round_up(L.d, 4);
      d.apply = L.r > 0 ? L.scale : 0.f;
      if (L.r > 0)
        NSGP_REQUIRE(L.ut_hi && L.ut_lo && L.un_hi && L.un_lo && L.t && L.t_hi && L.t_lo,
                     "sgd_step: tensor %d: low-rank projection needs U, U^T and T buffers", i);
      else
        NSGP_REQUIRE(L.pt_hi && L.pt_lo, "sgd_step: tensor %d: dense projection needs P^T", i);
    }
    (*host)[i] = d;
    (*chunk_start)[i] = total;
    total += sgd_chunks(t.numel);
  }
  (*chunk_start)[n_tensors] = total;
  return 0;
}

// slot [3] of nsgp_group_t is reserved and always zero
static void group_to_abi(const GroupInfo& gi, nsgp_group_t* g) {
  *g = nsgp_group_t{};
  g->kind = gi.kind;
  for (int k = 0; k < 3; ++k) {
    g->n_problems[k] = gi.sub[k].n_problems;
    g->n_items[k] = gi.sub[k].n_items;
    g->off_probs[k] = gi.sub[k].off_probs;
    g->off_items[k] = gi.sub[k].off_items;
  }
  g->bytes = gi.bytes;
}
static GroupInfo group_from_abi(const nsgp_group_t& g) {
  GroupInfo gi{};
  gi.kind = g.kind;
  for (int k = 0; k < 3; ++k)
    gi.sub[k] = SubGroup{g.n_problems[k], g.n_items[k], g.off_probs[k], g.off_items[k]};
  gi.bytes = g.bytes;
  return gi;
}

// first GEMM of a protected layer: dense  W += update @ P,  low-rank  T += update @ U
static ContractionArgs proj_args(const nsgp_proj_layer_t& L, float* w) {
  ContractionArgs a{};
  const int ldk = (int)round_up(L.d, 4);
  a.A = matrix_operand(L.u_hi, L.u_lo, L.cout, L.d, ldk);
  a.alpha = 1.f;
  a.epi = kEpiGemmRmw;
  a.splits = 1;
  if (L.r > 0) {
    a.B = matrix_operand(L.ut_hi, L.ut_lo, L.r, L.d, ldk);
    a.out = L.t;
    a.ld = (int)round_up(L.r, 4);
    a.n_cols = L.r;
    // T is a tall, narrow product (N = r, tens of columns) with K = d: one K chain per tile
    // leaves ~170 latency-bound items for 148 SMs (0.23 ms measured).  T is zeroed before
    // the launch and the epilogue is a red.add, so the chain is cut into 16-block pieces -
    // ~5x the items, each a fifth as long; the fp32 partial sums meet in L2.
    a.chain = 16;
  } else {
    a.B = matrix_operand(L.pt_hi, L.pt_lo, L.d, L.d, ldk);
    a.out = w;
    a.ld = L.d;
    a.n_cols = L.d;
  }
  return a;
}
// second GEMM of a low-rank layer:  W += -scale * T @ U^T
static ContractionArgs proj_args2(const nsgp_proj_layer_t& L, float* w) {
  ContractionArgs a{};
  const int ldr = (int)round_up(L.r, 4);
  a.A = matrix_operand(L.t_hi, L.t_lo, L.cout, L.r, ldr);
  a.B = matrix_operand(L.un_hi, L.un_lo, L.d, L.r, ldr);
  a.out = w;
  a.ld = L.d;
  a.n_cols = L.d;
  a.alpha = -L.scale;
  a.epi = kEpiGemmRmw;
  a.splits = 1;
  return a;
}

size_t nsgp_sgd_step_workspace_bytes(int n_tensors, int n_layers) {
  (void)n_layers;
  return (size_t)n_tensors * sizeof(SgdTensorDev) + (size_t)(n_tensors + 1) * sizeof(int) + 512;
}

int nsgp_sgd_nscl_step(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                       const nsgp_proj_layer_t* layers, int n_layers, double lr,
                       double momentum, double dampening, double weight_decay, int nesterov,
                       void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(n_tensors >= 0 && n_layers >= 0, "sgd_step: negative counts");
  if (n_tensors == 0) return 0;
  NSGP_REQUIRE(tensors && workspace, "sgd_step: null pointer");
  NSGP_REQUIRE(workspace_bytes >= nsgp_sgd_step_workspace_bytes(n_tensors, n_layers),
               "sgd_step: workspace too small");
  std::vector<SgdTensorDev> host;
  std::vector<int> chunk_start;
  int rc = sgd_tables(tensors, n_tensors, layers, n_layers, momentum, &host, &chunk_start);
  if (rc) return rc;
  const int total = chunk_start[n_tensors];
  char* ws = align_up((char*)workspace, 256);
  SgdTensorDev* dev_t = reinterpret_cast<SgdTensorDev*>(ws);
  int* dev_c = reinterpret_cast<int*>(ws + (size_t)n_tensors * sizeof(SgdTensorDev));
  NSGP_CHECK_CUDA(cudaMemcpyAsync(dev_t, host.data(), host.size() * sizeof(SgdTensorDev),
                                  cudaMemcpyHostToDevice, stream));
  NSGP_CHECK_CUDA(cudaMemcpyAsync(dev_c, chunk_start.data(), chunk_start.size() * sizeof(int),
                                  cudaMemcpyHostToDevice, stream));
  rc = launch_sgd_prologue(dev_t, dev_c, n_tensors, total, (float)lr, (float)momentum,
                           (float)(1.0 - dampening), (float)weight_decay, nesterov, stream);
  if (rc) return rc;
  for (int i = 0; i < n_tensors; ++i) {
    if (tensors[i].layer < 0) continue;
    const nsgp_proj_layer_t& L = layers[tensors[i].layer];
    if (L.r > 0) {
      const size_t te = (size_t)L.cout * round_up(L.r, 4);
      NSGP_CHECK_CUDA(cudaMemsetAsync(L.t, 0, te * sizeof(float), stream));
    }
    rc = contraction(proj_args(L, tensors[i].w), stream);
    if (rc) return rc;
    if (L.r > 0) {
      const size_t te = (size_t)L.cout * round_up(L.r, 4);
      rc = launch_split(L.t, L.t_hi, L.t_lo, (long long)te, stream);
      if (rc) return rc;
      rc = contraction(proj_args2(L, tensors[i].w), stream);
      if (rc) return rc;
    }
  }
  return 0;
}

// ---- prepared plan: tables uploaded once, two launches per step ---------------
static void proj_problems(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                          const nsgp_proj_layer_t* layers, std::vector<ContractionArgs>* out,
                          std::vector<ContractionArgs>* out2) {
  for (int i = 0; i < n_tensors; ++i) {
    if (tensors[i].layer < 0) continue;
    const nsgp_proj_layer_t& L = layers[tensors[i].layer];
    out->push_back(proj_args(L, tensors[i].w));
    if (L.r > 0) out2->push_back(proj_args2(L, tensors[i].w));
  }
}

size_t nsgp_sgd_plan_bytes(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                           const nsgp_proj_layer_t* layers, int n_layers) {
  if (!tensors || n_tensors <= 0) return 1024;
  std::vector<ContractionArgs> probs, probs2;
  for (int i = 0; i < n_tensors; ++i)
    if (tensors[i].layer >= 0 && tensors[i].layer < n_layers && layers) {
      const nsgp_proj_layer_t& L = layers[tensors[i].layer];
      probs.push_back(proj_args(L, tensors[i].w));
      if (L.r > 0) probs2.push_back(proj_args2(L, tensors[i].w));
    }
  return nsgp_sgd_step_workspace_bytes(n_tensors, n_layers) + 2048 +
         group_table_bytes(probs.data(), (int)probs.size()) +
         group_table_bytes(probs2.data(), (int)probs2.size());
}

int nsgp_sgd_plan_build(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                        const nsgp_proj_layer_t* layers, int n_layers, float* t_arena,
                        size_t t_elems, void* plan_dev, size_t plan_bytes,
                        nsgp_sgd_plan_t* plan, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(tensors && plan_dev && plan && n_tensors > 0, "sgd_plan_build: bad arguments");
  NSGP_REQUIRE((reinterpret_cast<uintptr_t>(plan_dev) & 255) == 0,
               "sgd_plan_build: plan buffer must be 256-byte aligned");
  NSGP_REQUIRE(g_engine == 0, "sgd_plan_build: plans need the tcgen05 engine");
  for (int i = 0; i < n_tensors; ++i)
    NSGP_REQUIRE(tensors[i].layer < n_layers && (tensors[i].layer < 0 || layers),
                 "sgd_plan_build: tensor %d: bad layer index", i);
  const size_t off_chunks = round_up((long long)((size_t)n_tensors * sizeof(SgdTensorDev)), 256);
  const size_t off_group =
      round_up((long long)(off_chunks + (size_t)(n_tensors + 1) * sizeof(int)), 256);
  NSGP_REQUIRE(off_group <= plan_bytes, "sgd_plan_build: plan buffer too small");
  std::vector<ContractionArgs> probs, probs2;
  proj_problems(tensors, n_tensors, layers, &probs, &probs2);
  for (int i = 0; i < n_layers; ++i)
    if (layers[i].r > 0)
      NSGP_REQUIRE(t_arena && layers[i].t >= t_arena &&
                       layers[i].t + (size_t)layers[i].cout * round_up(layers[i].r, 4) <=
                           t_arena + t_elems,
                   "sgd_plan_build: layer %d: T must live inside the T arena", i);
  GroupInfo gi{}, gi2{};
  int rc = group_table_build(probs.data(), (int)probs.size(), kProfGemm,
                             (char*)plan_dev + off_group, plan_bytes - off_group, &gi, stream);
  if (rc) return rc;
  const size_t off_group2 = round_up((long long)(off_group + gi.bytes), 256);
  NSGP_REQUIRE(off_group2 <= plan_bytes, "sgd_plan_build: plan buffer too small");
  rc = group_table_build(probs2.data(), (int)probs2.size(), kProfGemm,
                         (char*)plan_dev + off_group2, plan_bytes - off_group2, &gi2, stream);
  if (rc) return rc;
  plan->n_tensors = n_tensors;
  plan->total_chunks = 0;
  for (int i = 0; i < n_tensors; ++i) plan->total_chunks += sgd_chunks(tensors[i].numel);
  plan->all_have_buf = 0;
  plan->off_chunks = off_chunks;
  plan->off_group = off_group;
  plan->off_group2 = off_group2;
  group_to_abi(gi, &plan->group);
  group_to_abi(gi2, &plan->group2);
  plan->t_arena = t_arena;
  plan->t_elems = t_elems;
  plan->bytes = off_group2 + gi2.bytes;
  return 0;
}

int nsgp_sgd_plan_step(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                       const nsgp_proj_layer_t* layers, int n_layers, void* plan_dev,
                       const nsgp_sgd_plan_t* plan, double lr, double momentum, double dampening,
                       double weight_decay, int nesterov, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(plan_dev && plan, "sgd_plan_step: null pointer");
  NSGP_REQUIRE(n_tensors == plan->n_tensors, "sgd_plan_step: plan was built for %d tensors",
               plan->n_tensors);
  // The tensor table (weights, gradients, momentum buffers, first-step flags) is uploaded
  // when the caller passes it; tensors == NULL means "the table uploaded by the previous
  // step is still valid" (same gradient / momentum pointers, same first-step flags).  The
  // grouped GEMM table (staged updates, projectors, weights) is always reused.
  SgdTensorDev* dev_t = reinterpret_cast<SgdTensorDev*>(plan_dev);
  int* dev_c = reinterpret_cast<int*>((char*)plan_dev + plan->off_chunks);
  int rc = 0;
  if (tensors != nullptr) {
    std::vector<SgdTensorDev> host;
    std::vector<int> chunk_start;
    rc = sgd_tables(tensors, n_tensors, layers, n_layers, momentum, &host, &chunk_start);
    if (rc) return rc;
    NSGP_REQUIRE(chunk_start[n_tensors] == plan->total_chunks,
                 "sgd_plan_step: tensor sizes differ from the plan");
    NSGP_CHECK_CUDA(cudaMemcpyAsync(dev_t, host.data(), host.size() * sizeof(SgdTensorDev),
                                    cudaMemcpyHostToDevice, stream));
    NSGP_CHECK_CUDA(cudaMemcpyAsync(dev_c, chunk_start.data(), chunk_start.size() * sizeof(int),
                                    cudaMemcpyHostToDevice, stream));
  }
  rc = launch_sgd_prologue(dev_t, dev_c, n_tensors, plan->total_chunks, (float)lr,
                           (float)momentum, (float)(1.0 - dampening), (float)weight_decay,
                           nesterov, stream);
  if (rc) return rc;
  const bool lowrank = plan->group2.n_items[0] + plan->group2.n_items[1] > 0;
  if (lowrank)
    NSGP_CHECK_CUDA(cudaMemsetAsync(plan->t_arena, 0, plan->t_elems * sizeof(float), stream));
  rc = group_launch((const char*)plan_dev + plan->off_group, group_from_abi(plan->group), stream);
  if (rc || !lowrank) return rc;
  rc = launch_split(plan->t_arena, plan->t_arena + plan->t_elems,
                    plan->t_arena + 2 * plan->t_elems, (long long)plan->t_elems, stream);
  if (rc) return rc;
  return group_launch((const char*)plan_dev + plan->off_group2, group_from_abi(plan->group2),
                      stream);
}

// ---- grouped covariance contraction (deferred mode of the hooks) ----------------
static int cov_jobs_setup(const nsgp_cov_job_t* jobs, int n_jobs, std::vector<ConvGeom>* geoms,
                          std::vector<float*>* stages, std::vector<float*>* accs) {
  for (int i = 0; i < n_jobs; ++i) {
    const nsgp_cov_job_t& j = jobs[i];
    ConvGeom g;
    float* stage;
    int rc = cov_conv2d_setup(j.Cin, j.H, j.W, j.kh, j.kw, j.sh, j.sw, j.ph, j.pw,
                              const_cast<void*>(j.workspace), j.workspace_bytes, &g, &stage);
    if (rc) return rc;
    NSGP_REQUIRE(j.acc != nullptr, "cov_group: null accumulator");
    geoms->push_back(g);
    stages->push_back(stage);
    accs->push_back(j.acc);
  }
  return 0;
}

size_t nsgp_cov_group_bytes(const nsgp_cov_job_t* jobs, int n_jobs) {
  if (!jobs || n_jobs <= 0) return 1024;
  std::vector<ConvGeom> geoms;
  std::vector<float*> stages, accs;
  if (cov_jobs_setup(jobs, n_jobs, &geoms, &stages, &accs)) return 0;
  return cov_layers_group_bytes(geoms.data(), n_jobs) + 256;
}

int nsgp_cov_group_build(const nsgp_cov_job_t* jobs, int n_jobs, void* table_dev,
                         size_t table_bytes, nsgp_group_t* group, void* stream_) {
  NSGP_REQUIRE(jobs && table_dev && group && n_jobs > 0, "cov_group_build: bad arguments");
  NSGP_REQUIRE(g_engine == 0, "cov_group_build: groups need the tcgen05 engine");
  std::vector<ConvGeom> geoms;
  std::vector<float*> stages, accs;
  int rc = cov_jobs_setup(jobs, n_jobs, &geoms, &stages, &accs);
  if (rc) return rc;
  GroupInfo gi{};
  rc = cov_layers_group_build(geoms.data(), stages.data(), accs.data(), n_jobs, table_dev,
                              table_bytes, &gi, (cudaStream_t)stream_);
  if (rc) return rc;
  group_to_abi(gi, group);
  return 0;
}

int nsgp_group_launch(const void* table_dev, const nsgp_group_t* group, void* stream_) {
  NSGP_REQUIRE(table_dev && group, "group_launch: null pointer");
  return group_launch(table_dev, group_from_abi(*group), (cudaStream_t)stream_);
}

// ---- grouped staging: all layer inputs of a forward in one (two) launches ----------
static float* job_mean_scratch(const nsgp_cov_job_t& j, const ConvGeom& g, float* stage) {
  if (mean_scratch_elems(g) == 0) return nullptr;
  char* m = align_up((char*)stage + stage_bytes(g) + layer_table_bytes(g), 256);
  if (m + mean_scratch_elems(g) * sizeof(float) <= (const char*)j.workspace + j.workspace_bytes)
    return reinterpret_cast<float*>(m);
  return nullptr;
}

size_t nsgp_cov_stage_group_bytes(const nsgp_cov_job_t* jobs, int n_jobs, int B) {
  if (!jobs || n_jobs <= 0 || B <= 0) return 1024;
  std::vector<ConvGeom> geoms;
  std::vector<float*> stages, accs;
  if (cov_jobs_setup(jobs, n_jobs, &geoms, &stages, &accs)) return 0;
  return stage_group_bytes(geoms.data(), n_jobs, B) + 256;
}

int nsgp_cov_stage_group_build(const nsgp_cov_job_t* jobs, int n_jobs, int B,
                               const int* same_input, void* table_dev, size_t table_bytes,
                               nsgp_stage_group_t* out, void* stream_) {
  NSGP_REQUIRE(jobs && table_dev && out && n_jobs > 0 && B > 0,
               "cov_stage_group_build: bad arguments");
  std::vector<ConvGeom> geoms;
  std::vector<float*> stages, accs, means;
  int rc = cov_jobs_setup(jobs, n_jobs, &geoms, &stages, &accs);
  if (rc) return rc;
  for (int i = 0; i < n_jobs; ++i) means.push_back(job_mean_scratch(jobs[i], geoms[i], stages[i]));
  StageGroupInfo gi{};
  rc = stage_group_build(geoms.data(), stages.data(), means.data(), n_jobs, B, same_input,
                         table_dev, table_bytes, &gi, (cudaStream_t)stream_);
  if (rc) return rc;
  out->n_jobs = gi.n_jobs; out->B = gi.B;
  out->n_items[0] = gi.n_items[0]; out->n_items[1] = gi.n_items[1];
  out->off_jobs = gi.off_jobs;
  out->off_items[0] = gi.off_items[0]; out->off_items[1] = gi.off_items[1];
  out->off_xs = gi.off_xs; out->bytes = gi.bytes;
  out->n_items_tma = gi.n_items_tma; out->pad = 0; out->off_items_tma = gi.off_items_tma;
  out->off_maps = gi.off_maps;
  return 0;
}

static StageGroupInfo stage_from_abi(const nsgp_stage_group_t* sg) {
  StageGroupInfo gi{};
  gi.n_jobs = sg->n_jobs; gi.B = sg->B;
  gi.n_items[0] = sg->n_items[0]; gi.n_items[1] = sg->n_items[1];
  gi.off_jobs = sg->off_jobs;
  gi.off_items[0] = sg->off_items[0]; gi.off_items[1] = sg->off_items[1];
  gi.off_xs = sg->off_xs; gi.bytes = sg->bytes;
  gi.n_items_tma = sg->n_items_tma; gi.off_items_tma = sg->off_items_tma;
  gi.off_maps = sg->off_maps;
  return gi;
}

// geometries of the jobs a staging table was built for (the TMA kernel's tensor maps are
// re-encoded per launch from them and the current input pointers)
static int stage_job_geoms(const nsgp_cov_job_t* jobs, int n, std::vector<ConvGeom>* geoms) {
  geoms->resize(n);
  for (int i = 0; i < n; ++i)
    NSGP_REQUIRE(make_conv_geom(jobs[i].Cin, jobs[i].H, jobs[i].W, jobs[i].kh, jobs[i].kw,
                                jobs[i].sh, jobs[i].sw, jobs[i].ph, jobs[i].pw,
                                &(*geoms)[i]) == 0, "stage group: invalid conv geometry");
  return 0;
}

int nsgp_cov_stage_group_launch(void* table_dev, const nsgp_stage_group_t* sg,
                                const nsgp_cov_job_t* jobs, const void* const* xs,
                                void* stream_) {
  NSGP_REQUIRE(table_dev && sg && xs && jobs, "cov_stage_group_launch: null pointer");
  std::vector<ConvGeom> geoms;
  int rc = stage_job_geoms(jobs, sg->n_jobs, &geoms);
  if (rc) return rc;
  return stage_group_launch(table_dev, stage_from_abi(sg), xs, (cudaStream_t)stream_,
                            geoms.data());
}

// ---- pipelined covariance pass: contraction of forward i-1 || staging of forward i ----
int nsgp_cov_pipeline_launch(const void* prev_table, const nsgp_group_t* prev_group,
                             void* stage_table, const nsgp_stage_group_t* sg,
                             const nsgp_cov_job_t* stage_jobs, const void* const* xs,
                             int stage_sms, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const bool have_prev = prev_table && prev_group;
  const bool have_stage = stage_table && sg && xs && stage_jobs;
  NSGP_REQUIRE(have_prev || have_stage, "cov_pipeline_launch: nothing to launch");
  StageGroupInfo si{};
  int rc = 0;
  if (have_stage) {
    si = stage_from_abi(sg);
    // the pointer table travels BEFORE the kernels: a copy between two kernels would break
    // their programmatic pairing
    std::vector<ConvGeom> geoms;
    rc = stage_job_geoms(stage_jobs, si.n_jobs, &geoms);
    if (rc) return rc;
    rc = stage_group_upload(stage_table, si, xs, stream, geoms.data());
    if (rc) return rc;
  }
  const int sms = tc::sm_count();
  const bool overlap = have_prev && have_stage && stage_sms > 0 && stage_sms <= sms - 16 &&
                       (si.n_items[0] > 0 || si.n_items_tma > 0);
  if (!overlap) {
    if (have_prev) {
      rc = group_launch(prev_table, group_from_abi(*prev_group), stream);
      if (rc) return rc;
    }
    if (have_stage) {
      rc = stage_group_launch_tma(stage_table, si, 0, 0, stream);
      if (rc) return rc;
      for (int ph = 0; ph < 2; ++ph) {
        rc = stage_group_launch_phase(stage_table, si, ph, 0, 0, stream);
        if (rc) return rc;
      }
    }
    return 0;
  }
  // Partitioned: the sliding-window kernel (MMA-issue bound, barely affected by HBM traffic
  // next to it: +6 % measured) takes sms - stage_sms SMs, the HBM-bound first staging phase
  // the other stage_sms, started by programmatic dependent launch as soon as every
  // contraction CTA is resident.  The generic kernel is bound by operand delivery and
  // measured 2x slower next to the staging traffic, so it runs alone on the whole GPU:
  //   sliding-window(i-1) || staging phase 0 (i)  ->  generic(i-1)  ->  staging phase 1 (i)
  const GroupInfo gi = group_from_abi(*prev_group);
  const int ctas = sms - stage_sms;
  const bool have_ac = gi.sub[2].n_items > 0, have_gen = gi.sub[0].n_items > 0;
  NSGP_REQUIRE(gi.sub[1].n_items == 0,
               "cov_pipeline_launch: bring-up sub-tables are not pipelined");
  // the staging half: the TMA kernel when the table has TMA items (the heavy routines), else
  // the register kernel's phase 0; whatever is left of phase 0 follows as an ordinary launch
  const bool tma = si.n_items_tma > 0;
  if (have_ac) {
    rc = group_launch_sub(prev_table, gi, 2, ctas, 0, stream);
    if (rc) return rc;
    rc = tma ? stage_group_launch_tma(stage_table, si, 1, stage_sms, stream)
             : stage_group_launch_phase(stage_table, si, 0, 1, stage_sms, stream);
    if (rc) return rc;
    if (tma) rc = stage_group_launch_phase(stage_table, si, 0, 0, 0, stream);
    if (rc) return rc;
    if (have_gen) rc = group_launch_sub(prev_table, gi, 0, 0, 0, stream);
  } else {
    if (have_gen) rc = group_launch_sub(prev_table, gi, 0, 0, 0, stream);
    if (rc) return rc;
    rc = stage_group_launch_tma(stage_table, si, 0, 0, stream);
    if (rc) return rc;
    rc = stage_group_launch_phase(stage_table, si, 0, 0, 0, stream);
  }
  if (rc) return rc;
  return stage_group_launch_phase(stage_table, si, 1, 0, 0, stream);
}

// ---------------------------------------------------------------- RePRE
int repre_class_index(const int64_t* labels, int M, int C, int32_t* counts, int32_t* offsets,
                      int32_t* rows, void* stream_) {
  NSGP_REQUIRE(labels && counts && offsets && rows, "class_index: null pointer");
  NSGP_REQUIRE(M >= 0 && C > 0, "class_index: bad sizes");
  return launch_class_index_fused((const long long*)labels, M, C, counts, offsets, rows,
                                  (cudaStream_t)stream_);
}

int repre_segment_mean(const float* F, int D, const int32_t* seg_offsets, const int32_t* rows,
                       int n_segments, int max_seg_rows, float* out, void* stream_) {
  NSGP_REQUIRE(F && seg_offsets && rows && out, "segment_mean: null pointer");
  return launch_segment_mean(F, D, seg_offsets, rows, n_segments, max_seg_rows, nullptr, 0,
                             out, (cudaStream_t)stream_);
}

int repre_segment_var(const float* F, int D, const int32_t* seg_offsets, const int32_t* rows,
                      int n_segments, int max_seg_rows, const float* mu, float* out,
                      void* stream_) {
  NSGP_REQUIRE(F && seg_offsets && rows && out && mu, "segment_var: null pointer");
  return launch_segment_mean(F, D, seg_offsets, rows, n_segments, max_seg_rows, mu, 1, out,
                             (cudaStream_t)stream_);
}

size_t repre_cosine_count_workspace_bytes(int n, int D) {
  size_t n8 = (size_t)round_up(n, 8);
  return 2 * n8 * (size_t)D * 4 + n8 * (size_t)round_up(n, 4) * 4 + 2048;
}

int repre_cosine_count(const float* F, int D, const int32_t* rows, int n, float thresh,
                       uint8_t* mask, int32_t* counts, float* sim_out, void* workspace,
                       size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(F && rows && mask && counts && workspace, "cosine_count: null pointer");
  NSGP_REQUIRE(n >= 0 && D > 0 && D % 4 == 0, "cosine_count: bad sizes");
  if (n == 0) return 0;
  NSGP_REQUIRE(workspace_bytes >= repre_cosine_count_workspace_bytes(n, D),
               "cosine_count: workspace too small");
  size_t n8 = (size_t)round_up(n, 8);
  char* ws = align_up((char*)workspace, 1024);
  float* hi = reinterpret_cast<float*>(ws);
  float* lo = hi + n8 * D;
  float* S = lo + n8 * D;
  int ld = (int)round_up(n, 4);
  int rc = launch_normalize_split(F, D, rows, n, hi, lo, stream);
  if (rc) return rc;
  NSGP_CHECK_CUDA(cudaMemsetAsync(S, 0, (size_t)n * ld * 4, stream));
  ContractionArgs a{};
  a.A = matrix_operand(hi, lo, n, D, D);
  a.B = a.A;
  a.out = S;
  a.ld = ld;
  a.n_cols = n;
  a.alpha = 1.f;
  a.epi = kEpiGramAtomic;
  int t1 = ceil_div(n, 128);
  a.splits = pick_splits(t1 * (t1 + 1) / 2, k_blocks(a.A));
  rc = contraction(a, stream);
  if (rc) return rc;
  return launch_threshold_count(S, n, ld, thresh, mask, counts, sim_out, stream);
}

// ---- density ordering + greedy cover + segment table on the device (:421-448) -------
size_t repre_greedy_segments_workspace_bytes(const int32_t* sizes, int n_classes, int max_picks) {
  if (!sizes || n_classes <= 0 || max_picks < 0) return 1024;
  size_t n = 0;
  for (int c = 0; c < n_classes; ++c) n += (size_t)sizes[c];
  return (size_t)n_classes * sizeof(GreedyClass) + n * 4 + n + 64 +
         (size_t)n_classes * (max_picks + 2) * 4 + 2048;
}

int repre_greedy_segments(const uint8_t* masks, const int32_t* counts, const int32_t* rows_sel,
                          const int32_t* sizes, const int32_t* class_ids, int n_classes,
                          int max_picks, const uint8_t* saved, const int32_t* n_saved,
                          int32_t* seg_off, int32_t* seg_rows, int32_t* seg_label,
                          int32_t* info, void* workspace, size_t workspace_bytes,
                          void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(masks && counts && rows_sel && sizes && class_ids && seg_off && seg_rows &&
                   seg_label && info && workspace,
               "greedy_segments: null pointer");
  NSGP_REQUIRE(n_classes > 0 && max_picks >= 0, "greedy_segments: bad sizes");
  NSGP_REQUIRE(workspace_bytes >= repre_greedy_segments_workspace_bytes(sizes, n_classes, max_picks),
               "greedy_segments: workspace too small");
  std::vector<GreedyClass> h(n_classes);
  long long moff = 0, soff = 0;
  int roff = 0, max_n = 0;
  for (int c = 0; c < n_classes; ++c) {
    NSGP_REQUIRE(sizes[c] > 0, "greedy_segments: class %d has no rows", class_ids[c]);
    GreedyClass& g = h[c];
    g.mask_off = moff; g.saved_off = soff; g.row_off = roff; g.n = sizes[c];
    g.n_saved = (saved && n_saved) ? n_saved[c] : 0;
    NSGP_REQUIRE(g.n_saved >= 0 && g.n_saved <= max_picks, "greedy_segments: bad n_saved");
    g.class_id = class_ids[c];
    moff += (long long)sizes[c] * sizes[c];
    soff += (long long)g.n_saved * sizes[c];
    roff += sizes[c];
    if (sizes[c] > max_n) max_n = sizes[c];
  }
  char* ws = align_up((char*)workspace, 256);
  GreedyClass* cls_dev = reinterpret_cast<GreedyClass*>(ws);
  int* order_ws = reinterpret_cast<int*>(align_up(ws + (size_t)n_classes * sizeof(GreedyClass), 16));
  int* seg_sizes = order_ws + roff;
  int* seg_base = seg_sizes + (size_t)n_classes * (max_picks + 1);
  unsigned char* covered_ws = reinterpret_cast<unsigned char*>(seg_base + n_classes);
  NSGP_CHECK_CUDA(cudaMemcpyAsync(cls_dev, h.data(), (size_t)n_classes * sizeof(GreedyClass),
                                  cudaMemcpyHostToDevice, stream));
  // info: [0] = number of segments, [1 .. n_classes] = picks per class, then the picks
  int* nseg = info;
  int* npicks = info + 1;
  int* picks = info + 1 + n_classes;
  return launch_greedy_segments(cls_dev, n_classes, max_n, masks, counts, saved, rows_sel,
                                max_picks, order_ws, covered_ws, seg_sizes, seg_base, picks,
                                npicks, seg_off, seg_rows, seg_label, nseg, stream);
}

int repre_segment_mean_dev(const float* F, int D, const int32_t* seg_offsets, const int32_t* rows,
                           int max_segments, const int32_t* n_segments_dev, int max_seg_rows,
                           float* out, void* stream_) {
  NSGP_REQUIRE(F && seg_offsets && rows && out && n_segments_dev, "segment_mean_dev: null pointer");
  return launch_segment_mean(F, D, seg_offsets, rows, max_segments, max_seg_rows, nullptr, 0, out,
                             (cudaStream_t)stream_, n_segments_dev);
}

// ---- all classes at once: 1 normalise launch, 1 memset, 1 grouped Gram, 1 threshold launch
static void batched_layout(const int32_t* sizes, int n_classes, int D, size_t* n_total,
                           size_t* s_elems, size_t* table_bytes) {
  size_t n = 0, s = 0;
  // the tcgen05 engine wants >= 8 operand rows: a smaller class is contracted as 8 rows
  // (the extra rows are the next class's or padding; only its own n x n block is read back)
  for (int c = 0; c < n_classes; ++c) {
    const size_t ne = sizes[c] > 0 && sizes[c] < 8 ? 8 : (size_t)sizes[c];
    n += (size_t)sizes[c];
    s += ne * (size_t)round_up((long long)ne, 4);
  }
  *n_total = n;
  *s_elems = s;
  std::vector<ContractionArgs> probs;
  for (int c = 0; c < n_classes; ++c) {
    if (sizes[c] <= 0) continue;
    const int ne = sizes[c] < 8 ? 8 : sizes[c];
    ContractionArgs a{};
    a.A = matrix_operand(nullptr, nullptr, ne, D, D);
    a.B = a.A;
    a.n_cols = ne;
    a.epi = kEpiGramAtomic;
    probs.push_back(a);
  }
  *table_bytes = group_table_bytes(probs.data(), (int)probs.size()) + 1024;
}

size_t repre_cosine_count_batched_workspace_bytes(const int32_t* sizes, int n_classes, int D) {
  if (!sizes || n_classes <= 0) return 1024;
  size_t n, s, tb;
  batched_layout(sizes, n_classes, D, &n, &s, &tb);
  return 2 * ((size_t)round_up((long long)n, 8) + 8) * D * 4 + s * 4 + tb +
         (size_t)n_classes * sizeof(ClassExtent) + 4096;
}

int repre_cosine_count_batched(const float* F, int D, const int32_t* rows, const int32_t* sizes,
                               int n_classes, float thresh, uint8_t* mask, int32_t* counts,
                               void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(F && rows && sizes && mask && counts && workspace, "cosine_count_batched: null pointer");
  NSGP_REQUIRE(n_classes >= 0 && D > 0 && D % 4 == 0, "cosine_count_batched: bad sizes");
  if (n_classes == 0) return 0;
  NSGP_REQUIRE(g_engine == 0, "cosine_count_batched needs the tcgen05 engine");
  NSGP_REQUIRE(workspace_bytes >= repre_cosine_count_batched_workspace_bytes(sizes, n_classes, D),
               "cosine_count_batched: workspace too small");
  size_t n_total, s_elems, table_bytes;
  batched_layout(sizes, n_classes, D, &n_total, &s_elems, &table_bytes);
  if (n_total == 0) return 0;
  char* ws = align_up((char*)workspace, 1024);
  float* hi = reinterpret_cast<float*>(ws);
  const size_t rows_alloc = (size_t)round_up((long long)n_total, 8) + 8;
  float* lo = hi + rows_alloc * D;
  float* S = lo + rows_alloc * D;
  char* table = align_up(reinterpret_cast<char*>(S + s_elems), 256);
  ClassExtent* ext_dev = reinterpret_cast<ClassExtent*>(align_up(table + table_bytes, 256));
  NSGP_REQUIRE((char*)(ext_dev + n_classes) <= (char*)workspace + workspace_bytes,
               "cosine_count_batched: workspace layout overflow");
  int rc = launch_normalize_split(F, D, rows, (int)n_total, hi, lo, stream);
  if (rc) return rc;
  // rows past the last class that an 8-row operand may touch
  NSGP_CHECK_CUDA(cudaMemsetAsync(hi + n_total * D, 0, (rows_alloc - n_total) * D * 4, stream));
  NSGP_CHECK_CUDA(cudaMemsetAsync(lo + n_total * D, 0, (rows_alloc - n_total) * D * 4, stream));
  NSGP_CHECK_CUDA(cudaMemsetAsync(S, 0, s_elems * 4, stream));
  std::vector<ContractionArgs> probs;
  std::vector<ClassExtent> ext(n_classes);
  size_t row_off = 0, s_off = 0, mask_off = 0;
  int max_n = 0;
  for (int c = 0; c < n_classes; ++c) {
    const int n = sizes[c], ne = (n > 0 && n < 8) ? 8 : n, ld = (int)round_up(ne, 4);
    ext[c] = ClassExtent{(long long)s_off, (long long)mask_off, (int)row_off, n, ld, 0};
    if (n > 0) {
      ContractionArgs a{};
      a.A = matrix_operand(hi + row_off * D, lo + row_off * D, ne, D, D);
      a.B = a.A;
      a.out = S + s_off;
      a.ld = ld;
      a.n_cols = ne;
      a.alpha = 1.f;
      a.epi = kEpiGramAtomic;
      a.splits = 1;
      probs.push_back(a);
    }
    if (n > max_n) max_n = n;
    row_off += n;
    s_off += (size_t)ne * ld;
    mask_off += (size_t)n * n;
  }
  GroupInfo gi{};
  rc = group_table_build(probs.data(), (int)probs.size(), kProfRepre, table, table_bytes, &gi,
                         stream);
  if (rc) return rc;
  NSGP_CHECK_CUDA(cudaMemcpyAsync(ext_dev, ext.data(), ext.size() * sizeof(ClassExtent),
                                  cudaMemcpyHostToDevice, stream));
  rc = group_launch(table, gi, stream);
  if (rc) return rc;
  return launch_threshold_count_batched(S, ext_dev, n_classes, max_n, thresh, mask, counts,
                                        stream);
}

// ---- device-sized prototype build: fixed launch sequence, no host read in the middle ----
namespace {
struct ReBuildLayout {
  size_t off_hi, off_lo, off_S, off_prob, off_items, off_pairs, off_ext, off_cls, off_hdr,
      off_nsaved, off_savedlen, off_greedy, bytes;
  int ld_s, max_items, max_pairs;
};
ReBuildLayout rebuild_layout(int M, int D, int n_classes, int max_picks) {
  ReBuildLayout L{};
  const size_t Mp = (size_t)round_up(M, 128);
  L.ld_s = (int)Mp;
  const size_t tiles = Mp / 128;
  L.max_pairs = (int)(tiles * (tiles + 1) / 2);
  // items: pairs x splits, capped (the plan lowers the split count to fit)
  L.max_items = L.max_pairs * 8 > 4096 ? L.max_pairs * 8 : 4096;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (size_t)round_up((long long)(off + bytes), 1024); return o; };
  L.off_hi = take(Mp * D * 4);
  L.off_lo = take(Mp * D * 4);
  L.off_S = take(Mp * Mp * 4);
  L.off_prob = take(contraction_problem_bytes());
  L.off_items = take((size_t)L.max_items * contraction_item_bytes());
  L.off_pairs = take((size_t)L.max_pairs * 8);
  L.off_ext = take((size_t)n_classes * sizeof(ClassExtent));
  L.off_cls = take((size_t)n_classes * sizeof(GreedyClass));
  L.off_hdr = take(64);
  L.off_nsaved = take((size_t)n_classes * 4);
  L.off_savedlen = take((size_t)n_classes * 4);
  // greedy scratch: order (M ints), segment sizes / bases, covered flags (M bytes)
  L.off_greedy = take((size_t)M * 4 + (size_t)n_classes * (max_picks + 2) * 4 + (size_t)M + 256);
  L.bytes = off + 1024;
  return L;
}
}  // namespace

size_t repre_build_prototypes_workspace_bytes(int M, int D, int n_classes, int max_picks) {
  if (M <= 0 || D <= 0 || n_classes <= 0 || max_picks < 0) return 1024;
  return rebuild_layout(M, D, n_classes, max_picks).bytes;
}

int repre_build_prototypes(const float* F, int D, int M, const int32_t* rows,
                           const int32_t* offsets, int class_first, int n_classes, float thresh,
                           int max_picks, const uint8_t* saved, const int32_t* n_saved,
                           const int32_t* saved_len, uint8_t* masks, int32_t* counts,
                           int32_t* seg_off, int32_t* seg_rows, int32_t* seg_label, int32_t* info,
                           float* protos, void* workspace, size_t workspace_bytes, int flags,
                           void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const bool tables_resident = (flags & 1) != 0;
  NSGP_REQUIRE(!(tables_resident && saved), "build_prototypes: replayed masks are uploaded per "
               "call (flags & 1 needs saved == NULL)");
  NSGP_REQUIRE(F && rows && offsets && masks && counts && seg_off && seg_rows && seg_label &&
                   info && protos && workspace,
               "build_prototypes: null pointer");
  NSGP_REQUIRE(M > 0 && D > 0 && D % 4 == 0 && n_classes > 0 && class_first >= 0 && max_picks >= 0,
               "build_prototypes: bad sizes");
  NSGP_REQUIRE(g_engine == 0, "build_prototypes needs the tcgen05 engine");
  const ReBuildLayout L = rebuild_layout(M, D, n_classes, max_picks);
  char* ws = align_up((char*)workspace, 1024);
  NSGP_REQUIRE(ws + L.bytes - 1024 <= (char*)workspace + workspace_bytes,
               "build_prototypes: workspace too small (%zu < %zu)", workspace_bytes, L.bytes);
  float* hi = reinterpret_cast<float*>(ws + L.off_hi);
  float* lo = reinterpret_cast<float*>(ws + L.off_lo);
  float* S = reinterpret_cast<float*>(ws + L.off_S);
  ClassExtent* ext = reinterpret_cast<ClassExtent*>(ws + L.off_ext);
  GreedyClass* cls = reinterpret_cast<GreedyClass*>(ws + L.off_cls);
  int* hdr = reinterpret_cast<int*>(ws + L.off_hdr);
  int* nsaved_dev = nullptr;
  int* savedlen_dev = nullptr;
  if (saved && n_saved && saved_len) {
    nsaved_dev = reinterpret_cast<int*>(ws + L.off_nsaved);
    savedlen_dev = reinterpret_cast<int*>(ws + L.off_savedlen);
    for (int c = 0; c < n_classes; ++c)
      NSGP_REQUIRE(n_saved[c] >= 0 && n_saved[c] <= max_picks, "build_prototypes: bad n_saved");
    NSGP_CHECK_CUDA(cudaMemcpyAsync(nsaved_dev, n_saved, (size_t)n_classes * 4,
                                    cudaMemcpyHostToDevice, stream));
    NSGP_CHECK_CUDA(cudaMemcpyAsync(savedlen_dev, saved_len, (size_t)n_classes * 4,
                                    cudaMemcpyHostToDevice, stream));
  }
  // the ONE Gram problem: all foreground rows (class-sorted, at most round_up(M,128) of them)
  const int Mp = L.ld_s;
  ContractionArgs a{};
  a.A = matrix_operand(hi, lo, Mp, D, D);
  a.B = a.A;
  a.out = S;
  a.ld = L.ld_s;
  a.n_cols = Mp;
  a.alpha = 1.f;
  a.epi = kEpiGramAtomic;
  a.splits = 1;
  int rc = 0;
  if (!tables_resident) {
    std::vector<char> prob_host(contraction_problem_bytes());
    rc = contraction_build_problem(a, prob_host.data());
    if (rc) return rc;
    NSGP_CHECK_CUDA(cudaMemcpyAsync(ws + L.off_prob, prob_host.data(), prob_host.size(),
                                    cudaMemcpyHostToDevice, stream));
  }
  const int nkb = ceil_div(D, 32);
  rc = launch_repre_plan(offsets, class_first, n_classes, L.ld_s, nsaved_dev, savedlen_dev, nkb,
                         L.max_items, ext, cls, ws + L.off_pairs, ws + L.off_items,
                         ws + L.off_prob, hdr, stream);
  if (rc) return rc;
  rc = launch_repre_prepare(F, D, M, rows, offsets, class_first, hdr, hi, lo, ws + L.off_pairs, S,
                            L.ld_s, stream);
  if (rc) return rc;
  rc = contraction_launch_dev_items(ws + L.off_prob, ws + L.off_items, L.max_items, hdr + 2,
                                    kProfRepre, stream);
  if (rc) return rc;
  rc = launch_threshold_count_dev(S, ext, n_classes, M, hdr, thresh, masks, counts, stream);
  if (rc) return rc;
  // density ordering + greedy cover + segment table + segment rows (one CTA per class)
  int* order_ws = reinterpret_cast<int*>(ws + L.off_greedy);
  int* seg_sizes = order_ws + M;
  int* seg_base = seg_sizes + (size_t)n_classes * (max_picks + 1);
  unsigned char* covered_ws = reinterpret_cast<unsigned char*>(seg_base + n_classes);
  int* nseg = info;
  int* npicks = info + 1;
  int* picks = info + 1 + n_classes;
  rc = launch_greedy_segments(cls, n_classes, M, masks, counts, saved,
                              rows, max_picks, order_ws, covered_ws, seg_sizes,
                              seg_base, picks, npicks, seg_off, seg_rows, seg_label, nseg, stream,
                              offsets + class_first);
  if (rc) return rc;
  // plan status behind the picks: info[1 + n_classes + n_classes * max_picks + {0, 1}]
  NSGP_CHECK_CUDA(cudaMemcpyAsync(info + 1 + n_classes + (size_t)n_classes * max_picks, hdr + 3,
                                  4, cudaMemcpyDeviceToDevice, stream));
  NSGP_CHECK_CUDA(cudaMemcpyAsync(info + 2 + n_classes + (size_t)n_classes * max_picks, hdr, 4,
                                  cudaMemcpyDeviceToDevice, stream));
  return launch_segment_mean(F, D, seg_off, seg_rows, n_classes * (max_picks + 1), M, nullptr, 0,
                             protos, stream, nseg);
}

int repre_replay_gather(const float* protos, const float* sigma, const int64_t* idx, int P,
                        int D, uint64_t seed, float* out, void* stream_) {
  NSGP_REQUIRE(protos && out, "replay_gather: null pointer");
  return launch_replay_gather(protos, sigma, (const long long*)idx, P, D, seed, out,
                              (cudaStream_t)stream_);
}

int repre_replay_gather_rois(const float* feats, const int64_t* cls_targets,
                             const float* cls_weights, const float* bbox_targets,
                             const float* bbox_weights, const float* rois, const int64_t* idx,
                             int P, int D, float* out_feats, int64_t* out_cls_targets,
                             float* out_cls_weights, float* out_bbox_targets,
                             float* out_bbox_weights, float* out_rois, void* stream_) {
  NSGP_REQUIRE(feats && cls_targets && cls_weights && bbox_targets && bbox_weights && rois &&
                   idx && out_feats && out_cls_targets && out_cls_weights && out_bbox_targets &&
                   out_bbox_weights && out_rois,
               "replay_gather_rois: null pointer");
  NSGP_REQUIRE(P >= 0 && D > 0, "replay_gather_rois: bad sizes");
  return launch_replay_gather_rois(feats, (const long long*)cls_targets, cls_weights,
                                   bbox_targets, bbox_weights, rois, (const long long*)idx, P, D,
                                   out_feats, (long long*)out_cls_targets, out_cls_weights,
                                   out_bbox_targets, out_bbox_weights, out_rois,
                                   (cudaStream_t)stream_);
}

size_t repre_kmeans_assign_workspace_bytes(int n, int k, int D) {
  size_t n8 = (size_t)round_up(n, 8), k8 = (size_t)round_up(k, 8);
  return 2 * (n8 + k8) * (size_t)D * 4 + n8 * (size_t)round_up(k, 4) * 4 + k8 * 4 + 4096;
}

int repre_kmeans_assign(const float* X, int n, int D, const float* centres, int k,
                        int64_t* labels, void* workspace, size_t workspace_bytes,
                        void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(X && centres && labels && workspace, "kmeans_assign: null pointer");
  NSGP_REQUIRE(n >= 0 && k > 0 && D > 0 && D % 4 == 0, "kmeans_assign: bad sizes");
  if (n == 0) return 0;
  NSGP_REQUIRE(workspace_bytes >= repre_kmeans_assign_workspace_bytes(n, k, D),
               "kmeans_assign: workspace too small");
  size_t n8 = (size_t)round_up(n, 8), k8 = (size_t)round_up(k, 8);
  char* ws = align_up((char*)workspace, 1024);
  float* xh = reinterpret_cast<float*>(ws);
  float* xl = xh + n8 * D;
  float* ch = xl + n8 * D;
  float* cl = ch + k8 * D;
  float* dots = cl + k8 * D;
  int ld = (int)round_up(k, 4);
  float* cn = dots + n8 * ld;
  int rc = launch_split(X, xh, xl, (long long)n * D, stream);
  if (rc) return rc;
  rc = launch_split(centres, ch, cl, (long long)k * D, stream);
  if (rc) return rc;
  rc = launch_row_sqnorm(centres, k, D, D, cn, stream);
  if (rc) return rc;
  NSGP_CHECK_CUDA(cudaMemsetAsync(dots, 0, (size_t)n * ld * 4, stream));
  ContractionArgs a{};
  a.A = matrix_operand(xh, xl, n, D, D);
  a.B = matrix_operand(ch, cl, k, D, D);
  a.out = dots;
  a.ld = ld;
  a.n_cols = k;
  a.alpha = 1.f;
  a.epi = kEpiGemmRmw;
  a.splits = 1;
  rc = contraction(a, stream);
  if (rc) return rc;
  return launch_kmeans_argmin(dots, n, k, ld, cn, (long long*)labels, stream);
}

#ifdef NSGP_BRINGUP
int nsgp_debug_read_counters(unsigned long long* out, int n) {
  NSGP_REQUIRE(out && n != 0 && n <= 160 * 8 && n >= -160 * 8, "debug_read_counters: bad arguments");
  if (n < 0) return debug_read_ac_counters(out, -n);     // autocorrelation kernel's counters
  return debug_read_counters(out, n);
}

int nsgp_debug_mma_rate(int mode, int iters, unsigned long long* out_dev, int n_ctas,
                        void* stream_) {
  NSGP_REQUIRE(out_dev && iters > 0 && n_ctas > 0, "debug_mma_rate: bad arguments");
  return debug_mma_rate(mode, iters, out_dev, n_ctas, (cudaStream_t)stream_);
}

int nsgp_debug_timeline_read(unsigned long long* out, int* kinds, int max_slots) {
  NSGP_REQUIRE(out && kinds && max_slots > 0, "timeline_read: bad arguments");
  NSGP_CHECK_CUDA(cudaDeviceSynchronize());
  const int n = g_tl_n < max_slots ? g_tl_n : max_slots;
  if (n > 0) {
    NSGP_CHECK_CUDA(cudaMemcpy(out, g_tl_dev, (size_t)n * 2 * sizeof(unsigned long long),
                               cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) kinds[i] = g_tl_kind[i];
    std::vector<unsigned long long> init(kTlSlots * 2);
    for (int i = 0; i < kTlSlots; ++i) { init[2 * i] = ~0ull; init[2 * i + 1] = 0; }
    cudaMemcpy(g_tl_dev, init.data(), init.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice);
  }
  g_tl_n = 0;
  return n;
}

int nsgp_debug_occupy(int threads, size_t smem, long long cycles, int n_ctas, void* stream_) {
  NSGP_REQUIRE(threads > 0 && threads <= 1024 && n_ctas > 0 && smem <= 227 * 1024,
               "debug_occupy: bad arguments");
  return debug_occupy(threads, smem, cycles, n_ctas, (cudaStream_t)stream_);
}

int nsgp_debug_tma3d_probe(const float* base, long long img_elems, int B, int box_rows,
                           int boxes_per_cta, int depth, unsigned long long* out_dev, int n_ctas,
                           void* stream_) {
  NSGP_REQUIRE(base && out_dev && n_ctas > 0, "tma3d_probe: bad arguments");
  return debug_tma3d_probe(base, img_elems, B, box_rows, boxes_per_cta, depth, out_dev, n_ctas,
                           (cudaStream_t)stream_);
}

int nsgp_debug_bulk_probe(const void* src, long long bytes_per_cta, int chunk, int depth,
                          unsigned long long* out_dev, int n_ctas, void* stream_) {
  NSGP_REQUIRE(src && out_dev && n_ctas > 0, "bulk_probe: bad arguments");
  return debug_bulk_probe(src, bytes_per_cta, chunk, depth, out_dev, n_ctas, (cudaStream_t)stream_);
}

int nsgp_debug_tma_probe(const float* base, long long pitch_elems, int K, int rows, int iters,
                         int depth, unsigned long long* out_dev, int n_ctas, void* stream_) {
  NSGP_REQUIRE(base && out_dev, "tma_probe: null pointer");
  return debug_tma_probe(base, pitch_elems, K, rows, iters, depth, out_dev, n_ctas,
                         (cudaStream_t)stream_);
}

#endif  // NSGP_BRINGUP

int nsgp_split_tf32(const float* src, float* hi, float* lo, size_t n, void* stream_) {
  NSGP_REQUIRE(src && hi && lo, "split: null pointer");
  return launch_split(src, hi, lo, (long long)n, (cudaStream_t)stream_);
}

int nsgp_gemm_nt(const float* a_hi, const float* a_lo, const float* b_hi,
                       const float* b_lo, int M, int N, int K, float* C, int ldc,
                       void* stream_) {
  NSGP_REQUIRE(a_hi && a_lo && b_hi && b_lo && C, "gemm_nt: null pointer");
  ContractionArgs a{};
  a.A = matrix_operand(a_hi, a_lo, M, K, K);
  a.B = matrix_operand(b_hi, b_lo, N, K, K);
  a.out = C;
  a.ld = ldc;
  a.n_cols = N;
  a.alpha = 1.f;
  a.epi = kEpiGemmRmw;
  a.splits = 1;
  return contraction(a, (cudaStream_t)stream_);
}

}  // extern "C"
