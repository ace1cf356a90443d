// Host-side geometry of one hooked Conv2d input and how it is staged in HBM.
// See DESIGN.md "Data layout" for the derivation.
#pragma once
#include "common.cuh"

namespace nsgp {

enum StageMode : int {
  kModeImplicit = 0,  // kw column-shifted copies per row phase; row taps are TMA y offsets
  kModeFlat = 1,      // 1x1, pad 0: K = Hout*Wout flattened, no halo, no waste
  kModeExplicit = 2,  // explicit im2col rows in reference order (fallback)
  kModeAutocorr = 3,  // 3x3 s1 p1: spatial autocorrelation blocks + edge corrections
};

// Autocorrelation layout (3x3, stride 1, pad 1).  With m the batch-averaged map and
// zero padding, the covariance block of taps (i,j),(i',j') is
//     G = R_D - [i=i'=0] RowE(bottom, dx) - [i=i'=2] RowE(top, dx)
//             - [j=j'=0] ColE(right, dy)  - [j=j'=2] ColE(left, dy)  + [corner tap, same tap] Corner
// with D = (dy,dx) = (i'-i, j'-j),  R_D[c,c'] = sum_{u,v} m[c][u][v] m[c'][u+dy][v+dx]  the
// spatial autocorrelation at displacement D, and RowE / ColE / Corner the same sums
// restricted to one edge row / edge column / corner pixel (derivation in DESIGN.md; a
// numpy check is tests/test_oracle_golden.py::test_autocorrelation_identity).  Only 13
// displacements occur in the upper triangle, so a layer costs 12.5 C x C x K GEMM blocks
// instead of the 40.5 of the tap-pair Gram: 3.2x fewer tensor FLOPs for the same result.
// Accumulator = 29 running C x C matrices; nsgp_cov_finalize assembles the d x d matrix.
constexpr int kAcR = 13, kAcMats = 29;
constexpr int kAcRowBottom = 13, kAcRowTop = 16, kAcColRight = 19, kAcColLeft = 22,
              kAcCorner = 25;
// index of R_(dy,dx) for dy in {0,1,2}: (0,0) (0,1) (0,2) (1,-2..2) (2,-2..2)
static inline __host__ __device__ int ac_ridx(int dy, int dx) {
  return dy == 0 ? dx : 3 + (dy - 1) * 5 + (dx + 2);
}

// Implicit layout.  TMA needs the innermost (column) coordinate 16-byte aligned, so
// a +-1 column tap shift cannot be a coordinate.  Instead every kernel column j gets
// its own copy of the (batch-averaged) map, already shifted and stride-sampled:
//     copy(p, j)[c][r][x] = mean_b in[c][sh*(r - Ht) + py_p][sw*x - pw + j]   (0 outside)
// for x < Wout; p enumerates the distinct row phases py = (i - ph) mod sh.  Tap (i, j)
// at output position (oy, ox) then reads copy(p(i), j)[c][oy + yoff_i][ox]: the row
// tap is a plain TMA y offset (zero halo rows are staged), the K tail ox >= Wout is
// out of bounds of the tensor map and reads as zero.
struct ConvGeom {
  int C, H, W, kh, kw, sh, sw, ph, pw;
  int Hout, Wout;
  int mode;
  int T;        // taps that index Gram rows (implicit: kh*kw, else 1)
  int Cs;       // staged rows per tap (implicit/flat: C; explicit: round_up(d, 8))
  int ncopy;    // implicit: (#row phases) * kw, else 1
  int nrowphase;
  int rowphase_py[kMaxTaps];   // py of row-phase slot p
  int Hs, Ws;   // staged plane height / pitch
  int Ht;       // top halo in plane rows
  int tiled;    // autocorr: copies stored tile-major (128 channels x 32 columns = 16 KB
                // contiguous per (copy, channel block, row, column strip)) for the
                // sliding-window kernel; TMA of contiguous tiles sustains > 2x the bytes/cycle
                // of 128 scattered 128-byte rows (scripts/tma_probe.py)
  int d;        // true covariance dimension C*kh*kw
  int d_int;    // internal accumulator dimension (T*Cs)
};

static inline int floor_div(int a, int b) {
  int q = a / b, r = a % b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}
static inline int pos_mod(int a, int b) { return a - floor_div(a, b) * b; }

// returns 0 on success
static inline int make_conv_geom(int C, int H, int W, int kh, int kw, int sh, int sw, int ph,
                                 int pw, ConvGeom* out) {
  ConvGeom g{};
  g.C = C; g.H = H; g.W = W; g.kh = kh; g.kw = kw; g.sh = sh; g.sw = sw; g.ph = ph; g.pw = pw;
  if (C <= 0 || H <= 0 || W <= 0 || kh <= 0 || kw <= 0 || sh <= 0 || sw <= 0 || ph < 0 || pw < 0)
    return -1;
  g.Hout = (H + 2 * ph - kh) / sh + 1;
  g.Wout = (W + 2 * pw - kw) / sw + 1;
  if (g.Hout <= 0 || g.Wout <= 0) return -1;
  g.d = C * kh * kw;
  g.ncopy = 1; g.nrowphase = 1;
  const bool one_by_one = (kh == 1 && kw == 1 && ph == 0 && pw == 0);
  static const bool no_autocorr = nsgp_env("NSGP_NO_AUTOCORR") != nullptr;   // bring-up switch
  if (!no_autocorr && kh == 3 && kw == 3 && sh == 1 && sw == 1 && ph == 1 && pw == 1 &&
      C % 8 == 0 && H >= 3 && W >= 3) {
    g.mode = kModeAutocorr;
    g.T = 9; g.Cs = C; g.ncopy = 3;
    g.Hs = H + 2;                                  // two zero rows below
    g.Ws = (int)round_up(W + 2, 4);                // >= two zero columns on the right
    g.Ht = 0;
    g.d_int = kAcMats * C;
    g.tiled = (g_engine == 0 && autocorr_kernel_enabled()) ? 1 : 0;
    *out = g;
    return 0;
  }
  if (one_by_one && C % 8 == 0) {
    g.mode = kModeFlat;
    g.T = 1; g.Cs = C;
    g.Hs = 1; g.Ws = (int)round_up((long long)g.Hout * g.Wout, 4);
    g.Ht = 0;
  } else if (kh * kw <= kMaxTaps && C % 8 == 0) {
    g.mode = kModeImplicit;
    g.T = kh * kw; g.Cs = C;
    g.nrowphase = 0;
    for (int i = 0; i < kh; ++i) {
      int py = pos_mod(i - ph, sh), p = 0;
      while (p < g.nrowphase && g.rowphase_py[p] != py) ++p;
      if (p == g.nrowphase) g.rowphase_py[g.nrowphase++] = py;
    }
    g.ncopy = g.nrowphase * kw;
    g.Ht = ceil_div(ph, sh);
    int qy_max = floor_div(kh - 1 - ph, sh);
    g.Hs = g.Hout + qy_max + g.Ht;
    g.Ws = (int)round_up(g.Wout, 4);
  } else {
    g.mode = kModeExplicit;
    g.T = 1; g.Cs = (int)round_up(g.d, 8);
    g.Hs = 1; g.Ws = (int)round_up((long long)g.Hout * g.Wout, 4);
    g.Ht = 0;
  }
  g.d_int = g.T * g.Cs;
  *out = g;
  return 0;
}

// autocorr extras: edge columns (2 sides x 3 row shifts, pitch Hc) and corner pixels
static inline int ac_col_pitch(const ConvGeom& g) { return (int)round_up(g.H + 2, 4); }
static inline int ac_cblocks(const ConvGeom& g) { return ceil_div(g.C, 128); }
static inline int ac_strips(const ConvGeom& g) { return ceil_div(g.W, 32); }
static inline int ac_row_pitch(const ConvGeom& g) { return (int)round_up(g.W, 4); }
// tiled: [3 copies x cblocks x Hs rows x strips] tiles of 4096 floats, then the two edge
// rows of the three copies in plain layout (for the edge-row GEMMs)
static inline long long ac_main_elems(const ConvGeom& g) {
  return g.tiled ? 3LL * ac_cblocks(g) * g.Hs * ac_strips(g) * 4096 : 3LL * g.C * g.Hs * g.Ws;
}
static inline long long ac_rowbuf_off(const ConvGeom& g) { return ac_main_elems(g); }
static inline long long ac_colbuf_off(const ConvGeom& g) {
  return ac_main_elems(g) + (g.tiled ? 6LL * g.C * ac_row_pitch(g) : 0);
}
static inline long long ac_cornerbuf_off(const ConvGeom& g) {
  return ac_colbuf_off(g) + 6LL * g.C * ac_col_pitch(g);
}
static inline long long stage_hl_stride(const ConvGeom& g) {
  if (g.mode == kModeAutocorr) return round_up(ac_cornerbuf_off(g) + 16LL * g.C, 4);
  return (long long)g.Cs * g.Hs * g.Ws * g.ncopy;
}
static inline size_t stage_bytes(const ConvGeom& g) {
  return (size_t)stage_hl_stride(g) * 2 * sizeof(float);
}

// Virtual K-major operand over the staged planes.  Implicit mode: K is the FLAT
// index oy * Ws + x over the staged rows (the < 4 padding columns per row are staged
// as zeros), so tap (i, j) is simply the copy's plane shifted by yoff_i rows.
static inline Operand conv_operand(const ConvGeom& g, const float* stage) {
  Operand o{};
  o.base = stage;
  o.hl_stride = stage_hl_stride(g);
  o.T = g.T; o.Cs = g.Cs;
  if (g.mode == kModeImplicit) {
    const long long plane = (long long)g.Cs * g.Hs * g.Ws;
    o.row_pitch = (long long)g.Hs * g.Ws;
    o.K = g.Hout * g.Ws;
    o.rows = g.T * g.Cs;
    for (int i = 0; i < g.kh; ++i) {
      int ay = i - g.ph;
      int qy = floor_div(ay, g.sh), py = pos_mod(ay, g.sh), p = 0;
      while (g.rowphase_py[p] != py) ++p;
      for (int j = 0; j < g.kw; ++j)
        o.tap_off[i * g.kw + j] = (long long)(p * g.kw + j) * plane + (long long)(qy + g.Ht) * g.Ws;
    }
  } else {
    o.row_pitch = g.Ws;
    o.K = g.Hout * g.Wout;
    o.rows = (g.mode == kModeExplicit) ? g.d : g.Cs;
    o.tap_off[0] = 0;
  }
  return o;
}

// Plain row-major matrix (rows x K, pitch ld) with separate hi / lo copies.
static inline Operand matrix_operand(const float* hi, const float* lo, int rows, int K, int ld) {
  Operand o{};
  o.base = hi;
  o.hl_stride = (long long)(lo - hi);
  o.row_pitch = ld;
  o.T = 1; o.Cs = rows; o.K = K; o.rows = rows;
  o.tap_off[0] = 0;
  return o;
}

// The contraction problems of one staged conv input: one Gram for the tap-pair layouts,
// 29 small-N GEMMs for the autocorrelation layout.  acc: the layer's accumulator.
static inline void conv_problems(const ConvGeom& g, const float* stage, float* acc,
                                 ContractionArgs* out, int* n_out, int l2_group = 1) {
  if (g.mode != kModeAutocorr) {
    ContractionArgs a{};
    a.A = conv_operand(g, stage);
    a.B = a.A;
    a.out = acc;
    a.ld = (int)round_up(g.d_int, 4);
    a.n_cols = a.A.rows;
    a.alpha = 1.f;
    a.epi = kEpiGramAtomic;
    a.splits = 1;
    out[0] = a;
    *n_out = 1;
    return;
  }
  const int C = g.C, ldc = (int)round_up(C, 4);
  const long long hl = stage_hl_stride(g), plane = (long long)C * g.Hs * g.Ws;
  const int pitch = g.Hs * g.Ws, Kmain = g.H * g.Ws;
  const int Hc = ac_col_pitch(g);
  int n = 0;
  auto mat = [&](int idx) { return acc + (long long)idx * C * ldc; };
  auto add = [&](const float* a_base, const float* b_base, int K, int ld, float* dst, bool gram) {
    ContractionArgs a{};
    a.A = matrix_operand(a_base, a_base + hl, C, K, ld);
    a.B = matrix_operand(b_base, b_base + hl, C, K, ld);
    a.out = dst;
    a.ld = ldc;
    a.n_cols = C;
    a.alpha = 1.f;
    a.epi = gram ? kEpiGramAtomic : kEpiGemmRmw;
    a.splits = 1;
    a.chain = 64;
    a.l2_group = l2_group;
    out[n++] = a;
  };
  // R_(dy,dx): generic GEMM problems over the plane layout; with the tiled layout they
  // are computed by the sliding-window kernel instead (contraction_ac.cu)
  for (int dy = 0; dy <= 2 && !g.tiled; ++dy)
    for (int dx = (dy == 0 ? 0 : -2); dx <= 2; ++dx) {
      const float* a_base = stage + (dx < 0 ? -dx : 0) * plane;
      const float* b_base = stage + (dx > 0 ? dx : 0) * plane + (long long)dy * g.Ws;
      add(a_base, b_base, Kmain, pitch, mat(ac_ridx(dy, dx)), dy == 0 && dx == 0);
    }
  // edge rows: bottom (u = H-1) and top (u = 0), dx = 0..2
  for (int e = 0; e < 2; ++e) {
    if (g.tiled) {
      const int Wr = ac_row_pitch(g);
      const float* rb = stage + ac_rowbuf_off(g) + (long long)e * 3 * g.C * Wr;
      for (int dx = 0; dx <= 2; ++dx)
        add(rb, rb + (long long)dx * g.C * Wr, g.W, Wr,
            mat((e == 0 ? kAcRowBottom : kAcRowTop) + dx), false);
      continue;
    }
    const long long row = (long long)(e == 0 ? g.H - 1 : 0) * g.Ws;
    for (int dx = 0; dx <= 2; ++dx)
      add(stage + row, stage + dx * plane + row, g.Ws, pitch,
          mat((e == 0 ? kAcRowBottom : kAcRowTop) + dx), false);
  }
  // edge columns: right (v = W-1) and left (v = 0), dy = 0..2
  const float* cb = stage + ac_colbuf_off(g);
  for (int e = 0; e < 2; ++e)
    for (int dy = 0; dy <= 2; ++dy)
      add(cb + (long long)(e * 3) * C * Hc, cb + (long long)(e * 3 + dy) * C * Hc, Hc, Hc,
          mat((e == 0 ? kAcColRight : kAcColLeft) + dy), false);
  // corner pixels of the four corner taps
  const float* kb = stage + ac_cornerbuf_off(g);
  for (int q = 0; q < 4; ++q)
    add(kb + (long long)q * C * 4, kb + (long long)q * C * 4, 4, 4, mat(kAcCorner + q), false);
  *n_out = n;
}
constexpr int kMaxConvProblems = kAcMats;

int launch_stage_conv(const float* x, float* stage, const ConvGeom& g, int B,
                      float* mean_scratch, cudaStream_t s);
// scratch (floats) for the batch mean of the gather layouts' two-pass staging
static inline size_t mean_scratch_elems(const ConvGeom& g) {
  const bool vec_flat = g.mode == kModeFlat && g.sh == 1 && g.sw == 1 && (g.H * g.W) % 4 == 0;
  const bool vec_ac = g.mode == kModeAutocorr && g.W % 4 == 0 && (g.tiled || g.Ws == g.W + 4);
  if (vec_flat || vec_ac) return 0;
  return (size_t)round_up((long long)g.C * g.H * g.W, 4);
}
// grouped staging (stage.cu): all layer inputs of a forward in one or two launches
enum StageKind : int {
  kStFlatVec = 0, kStAcVec, kStAcEdges, kStMean, kStConv, kStExplicit, kStAcScalar, kSt3x3Vec,
  kStFlatSub,    // kStFlatVec that also writes the stride-2 subsample of a 1x1 s2 job on the same input
  kStS2x3        // 3x3 stride-2 pad-1 tap copies straight from the input (TMA kernel only)
};
struct alignas(16) StageJobDev {
  ConvGeom g;
  float* stage;
  float* mean;                 // batch-mean scratch of the two-pass layouts (or null)
  long long hl;
  long long rowbuf_off, colbuf_off, cornerbuf_off;
  int Hc, pad;
  // kStFlatSub: staged operand of the 1x1 stride-2 job that reads the same tensor (row pitch
  // sub_pitch, sub_wout = W / 2 output columns per output row)
  float* sub_stage;
  long long sub_hl;
  int sub_pitch, sub_wout;
};
struct alignas(16) StageItem {
  int job;
  short kind, from_mean;
  long long lo, hi;
  long long pad;
};
struct StageGroupInfo {
  int n_jobs, B;
  int n_items[2];
  size_t off_jobs, off_items[2], off_xs, bytes;
  // TMA-fed phase 0 (stage_tma_kernel): its items and one 3-D tensor map per job (re-encoded
  // for the current input pointers at every launch)
  int n_items_tma, pad;
  size_t off_items_tma, off_maps;
};
size_t stage_group_bytes(const ConvGeom* geoms, int n, int B);
// same_input (n entries or null): same_input[i] = k >= 0 when job i is given the same tensor as
// job k at every launch
int stage_group_build(const ConvGeom* geoms, float* const* stages, float* const* means, int n,
                      int B, const int* same_input, void* table_dev, size_t table_bytes,
                      StageGroupInfo* info, cudaStream_t stream);
int stage_group_launch(const void* table_dev, const StageGroupInfo& info, const void* const* xs,
                       cudaStream_t stream, const ConvGeom* geoms = nullptr);
int stage_group_upload(const void* table_dev, const StageGroupInfo& info, const void* const* xs,
                       cudaStream_t stream, const ConvGeom* geoms = nullptr);
int stage_group_launch_tma(const void* table_dev, const StageGroupInfo& info, int pdl, int sms,
                           cudaStream_t stream);
int stage_group_launch_phase(const void* table_dev, const StageGroupInfo& info, int ph, int pdl,
                             int sms, cudaStream_t stream);
int launch_cov_finalize_autocorr(const float* acc, float* out, int C, int accumulate,
                                 cudaStream_t s);
int launch_linear_cov(const float* x, int R, int d, float* acc, int ld, float* mean_ws,
                      cudaStream_t s);
int launch_cov_finalize(const float* acc, int ld, float* out, int C, int T, int accumulate,
                        cudaStream_t s);
int launch_split(const float* src, float* hi, float* lo, long long n, cudaStream_t s);
int launch_transpose_split(const float* src, float* hi, float* lo, int d, int ld_dst,
                           cudaStream_t s);
// src (rows x cols) row-major -> hi/lo of its transpose (cols rows of pitch ld_dst)
int launch_transpose_split_rect(const float* src, float* hi, float* lo, int rows, int cols,
                                int ld_dst, cudaStream_t s);
// src (rows x cols) row-major -> hi/lo with row pitch ld_dst (pad columns zeroed)
int launch_split_pitched(const float* src, float* hi, float* lo, int rows, int cols, int ld_dst,
                         cudaStream_t s);

}  // namespace nsgp
