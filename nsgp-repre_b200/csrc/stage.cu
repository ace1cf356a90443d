// Staging kernels: batch-mean + tf32 hi/lo split + layout for the contraction
// engines.  All are HBM-bound element-wise/reduction kernels.
#include <vector>

#include <algorithm>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "geometry.h"
#include "tc_common.cuh"

namespace nsgp {

// ---------------------------------------------------------------------------
// Conv2d input -> staged planes (implicit-im2col or flat layout).
// One thread per staged element (plane, c, r, xs); it averages the B input
// values that land there (nsrunner_roi_replay.py:908 takes the batch mean BEFORE
// unfolding), splits into tf32 hi/lo and writes both copies.  Halo / padding
// elements are written as zeros, so the workspace needs no memset.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
  float4 v;
  asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
      : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void split_store4(float* hi, float* lo, float a, float b, float c,
                                             float d) {
  float4 h, l;
  tf32_split(a, h.x, l.x);
  tf32_split(b, h.y, l.y);
  tf32_split(c, h.z, l.z);
  tf32_split(d, h.w, l.w);
  *reinterpret_cast<float4*>(hi) = h;
  *reinterpret_cast<float4*>(lo) = l;
}

// Every staging routine is a __device__ body over an index span (first, step, end) so that
// the same code runs as a stand-alone grid-stride kernel (per-layer entry points) and as
// one work item of the grouped staging kernel (stage_group_kernel, end of this file).
// I = index type: 32-bit arithmetic for the decode whenever the index space allows (a 64-bit
// division is ~5x the instructions, and the gather routines are instruction-bound)
template <typename I>
__device__ __forceinline__ void
stage_conv_body_t(const float* __restrict__ x, float* __restrict__ stage, const ConvGeom& g,
                  int B, long long hl_stride, long long first, long long step, long long end) {
  // one thread per aligned group of 4 staged columns (Ws % 4 == 0): the row decode is
  // paid once per float4 and both planes are written with 128-bit stores
  const int W4 = g.Ws >> 2;
  const long long total = (long long)g.Cs * g.Hs * g.ncopy * W4;
  const long long img = (long long)g.C * g.H * g.W;
  const float fb = (float)B;
  const int HWout = g.Hout * g.Wout;
  if (end > total) end = total;
  // (x4, r, c, copy) of the thread's first index by division, then advanced by `step` as a
  // mixed-radix number: the gather routines are instruction-bound and the divisions were most
  // of their instructions
  int x4 = 0, r = 0, c = 0, copy = 0;
  if ((I)first < (I)end) {
    x4 = (int)((I)first % W4);
    I rest = (I)first / W4;
    r = (int)(rest % g.Hs);
    rest /= g.Hs;
    c = (int)(rest % g.Cs);
    copy = (int)(rest / g.Cs);
  }
  const int dx = (int)(step % W4);
  const long long srest = step / W4;
  const int dr = (int)(srest % g.Hs);
  const long long srest2 = srest / g.Hs;
  const int dc = (int)(srest2 % g.Cs), dcopy = (int)(srest2 / g.Cs);
  for (I idx = (I)first; idx < (I)end; idx += (I)step,
         x4 += dx, r += dr + (x4 >= W4), x4 -= (x4 >= W4) ? W4 : 0,
         c += dc + (r >= g.Hs), r -= (r >= g.Hs) ? g.Hs : 0,
         copy += dcopy + (c >= g.Cs), c -= (c >= g.Cs) ? g.Cs : 0) {
    int p = 0, j = 0, y = 0;
    bool row_ok = true;
    if (g.mode != kModeFlat) {
      p = copy / g.kw; j = copy - p * g.kw;
      y = g.sh * (r - g.Ht) + g.rowphase_py[p];
      row_ok = (y >= 0) && (y < g.H);
    }
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int xs = x4 * 4 + e;
      int yy, xx;
      bool valid;
      if (g.mode == kModeFlat) {
        valid = xs < HWout;
        const int oy = xs / g.Wout, ox = xs - oy * g.Wout;
        yy = oy * g.sh;
        xx = ox * g.sw;
      } else {
        yy = y;
        xx = g.sw * xs - g.pw + j;
        valid = row_ok && (xs < g.Wout) && (xx >= 0) && (xx < g.W);
      }
      float acc = 0.f;
      if (valid) {
        const float* q = x + ((long long)c * g.H + yy) * g.W + xx;
        for (int b = 0; b < B; ++b) acc += __ldg(q + (long long)b * img);
        acc /= fb;
      }
      v[e] = acc;
    }
    float* o = stage + (((long long)copy * g.Cs + c) * g.Hs + r) * g.Ws + x4 * 4;
    split_store4(o, o + hl_stride, v[0], v[1], v[2], v[3]);
  }
}

constexpr long long kIdx32Max = 0x7fffffffLL - (1LL << 24);   // room for one stride past the end
__device__ __forceinline__ void
stage_conv_body(const float* __restrict__ x, float* __restrict__ stage, const ConvGeom& g,
                int B, long long hl_stride, long long first, long long step, long long end) {
  const long long total = (long long)g.Cs * g.Hs * g.ncopy * (g.Ws >> 2);
  if (total < kIdx32Max && step < (1LL << 24))
    stage_conv_body_t<int>(x, stage, g, B, hl_stride, first, step, end);
  else
    stage_conv_body_t<long long>(x, stage, g, B, hl_stride, first, step, end);
}

__global__ void __launch_bounds__(256)
stage_conv_kernel(const float* __restrict__ x, float* __restrict__ stage, ConvGeom g,
                  int B, long long hl_stride) {
  stage_conv_body(x, stage, g, B, hl_stride, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, 1LL << 62);
}

// ---------------------------------------------------------------------------
// Fast paths (same staged layout as stage_conv_kernel, 128-bit loads and stores).
// ---------------------------------------------------------------------------
// 1x1 stride-1 conv input with H*W % 4 == 0: the staged plane is the batch mean of
// x itself.  One thread per float4.
template <int B_UNROLL>
__device__ __forceinline__ void
stage_flat_vec_body(const float* __restrict__ x, float* __restrict__ stage, long long n4,
                    int B, long long img, long long hl_stride, long long first, long long step,
                    long long end) {
  const float inv_div = (float)B;
  if (end > n4) end = n4;
  for (long long i = first; i < end; i += step) {
    const float* p = x + i * 4;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int b = 0;
    for (; b + B_UNROLL <= B; b += B_UNROLL) {
      float4 v[B_UNROLL];
#pragma unroll
      for (int u = 0; u < B_UNROLL; ++u) v[u] = ldg_stream4(p + (long long)(b + u) * img);
#pragma unroll
      for (int u = 0; u < B_UNROLL; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
    for (; b < B; ++b) {
      float4 v = ldg_stream4(p + (long long)b * img);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    split_store4(stage + i * 4, stage + i * 4 + hl_stride, s.x / inv_div, s.y / inv_div,
                 s.z / inv_div, s.w / inv_div);
  }
}

template <int B_UNROLL>
__global__ void __launch_bounds__(256)
stage_flat_vec_kernel(const float* __restrict__ x, float* __restrict__ stage, long long n4,
                      int B, long long img, long long hl_stride) {
  stage_flat_vec_body<B_UNROLL>(x, stage, n4, B, img, hl_stride, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, n4);
}

// Batch mean of x (B, n) -> out (n), n % 4 == 0, 16-byte aligned: first pass of the
// two-pass staging used by the layouts whose second pass is a gather (stride-2 tap
// copies, odd widths, the explicit stem): the gather then reads 1/B of the data.
template <int B_UNROLL>
__device__ __forceinline__ void
batch_mean_vec_body(const float* __restrict__ x, float* __restrict__ out, long long n4, int B,
                    long long img, long long first, long long step, long long end) {
  const float fb = (float)B;
  if (end > n4) end = n4;
  for (long long i = first; i < end; i += step) {
    const float* p = x + i * 4;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int b = 0;
    for (; b + B_UNROLL <= B; b += B_UNROLL) {
      float4 v[B_UNROLL];
#pragma unroll
      for (int u = 0; u < B_UNROLL; ++u) v[u] = ldg_stream4(p + (long long)(b + u) * img);
#pragma unroll
      for (int u = 0; u < B_UNROLL; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
    for (; b < B; ++b) {
      float4 v = ldg_stream4(p + (long long)b * img);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    *reinterpret_cast<float4*>(out + i * 4) =
        make_float4(s.x / fb, s.y / fb, s.z / fb, s.w / fb);
  }
}

template <int B_UNROLL>
__global__ void __launch_bounds__(256)
batch_mean_vec_kernel(const float* __restrict__ x, float* __restrict__ out, long long n4, int B,
                      long long img) {
  batch_mean_vec_body<B_UNROLL>(x, out, n4, B, img, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, n4);
}

// 3x3 stride-1 pad-1 conv input with W % 4 == 0: each thread averages one aligned
// float4 of the input row and writes it to the three column-shifted copies; the
// +-1 neighbours come from the adjacent lanes (or one extra scalar load at the
// warp / row edges).  Halo rows (r = 0, Hs-1) are written as zeros.
template <int B_UNROLL>
__device__ __forceinline__ void
stage_3x3s1_vec_body(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                     int W, int B, long long hl_stride, long long first, long long step,
                     long long end) {
  const int W4 = W >> 2, Hs = H + 2;
  const long long total = (long long)C * Hs * W4;
  const long long img = (long long)C * H * W;
  const long long copy_stride = (long long)C * Hs * W;
  const float fb = (float)B;
  const int lane = threadIdx.x & 31;
  // every lane of a warp runs the same number of iterations (shuffles below)
  const long long total_r = (total + 31) / 32 * 32;
  if (end > total_r) end = total_r;
  for (long long idx = first; idx < end; idx += step) {
    const bool live = idx < total;
    int x4 = 0, r = 0, c = 0;
    if (live) {
      x4 = (int)(idx % W4);
      long long rest = idx / W4;
      r = (int)(rest % Hs);
      c = (int)(rest / Hs);
    }
    const int y = r - 1;
    const bool row_ok = live && y >= 0 && y < H;
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* p = x + ((long long)c * H + y) * W + x4 * 4;
    if (row_ok) {
      int b = 0;
      for (; b + B_UNROLL <= B; b += B_UNROLL) {
        float4 v[B_UNROLL];
#pragma unroll
        for (int u = 0; u < B_UNROLL; ++u) v[u] = ldg_stream4(p + (long long)(b + u) * img);
#pragma unroll
        for (int u = 0; u < B_UNROLL; ++u) { m.x += v[u].x; m.y += v[u].y; m.z += v[u].z; m.w += v[u].w; }
      }
      for (; b < B; ++b) {
        float4 v = ldg_stream4(p + (long long)b * img);
        m.x += v.x; m.y += v.y; m.z += v.z; m.w += v.w;
      }
      m.x /= fb; m.y /= fb; m.z /= fb; m.w /= fb;
    }
    // neighbours: left = mean at x-1, right = mean at x+4 (same row)
    float left = __shfl_up_sync(0xffffffffu, m.w, 1);
    float right = __shfl_down_sync(0xffffffffu, m.x, 1);
    if (row_ok) {
      if (x4 == 0) left = 0.f;
      else if (lane == 0) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s += __ldg(p - 1 + (long long)b * img);
        left = s / fb;
      }
      if (x4 == W4 - 1) right = 0.f;
      else if (lane == 31) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s += __ldg(p + 4 + (long long)b * img);
        right = s / fb;
      }
    } else {
      left = right = 0.f;
    }
    if (live) {
      float* o = stage + ((long long)c * Hs + r) * W + x4 * 4;
      split_store4(o, o + hl_stride, left, m.x, m.y, m.z);                                  // j = 0
      split_store4(o + copy_stride, o + copy_stride + hl_stride, m.x, m.y, m.z, m.w);      // j = 1
      split_store4(o + 2 * copy_stride, o + 2 * copy_stride + hl_stride, m.y, m.z, m.w, right);  // j = 2
    }
  }
}

template <int B_UNROLL>
__global__ void __launch_bounds__(256)
stage_3x3s1_vec_kernel(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                       int W, int B, long long hl_stride) {
  stage_3x3s1_vec_body<B_UNROLL>(x, stage, C, H, W, B, hl_stride, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, 1LL << 62);
}

// ---------------------------------------------------------------------------
// Autocorrelation layout (3x3 s1 p1, geometry.h): three column-shifted copies of the
// zero-extended batch mean, copy_s[c][r][x] = m~[c][r][x+s], r < H+2, x < Ws, plus the
// edge-column and corner-pixel buffers of the boundary corrections.
// ---------------------------------------------------------------------------
// tiled: destination of element (copy s, channel c, row r, column xs) in the tile-major
// layout: tile ((s*CB + c/128)*Hs + r)*NS + xs/32, 128 channels x 32 columns per tile
__device__ __forceinline__ long long ac_tiled_off(int s, int c, int r, int xs, int CB, int Hs,
                                                  int NS) {
  const long long tile = ((long long)(s * CB + (c >> 7)) * Hs + r) * NS + (xs >> 5);
  return tile * 4096 + (long long)(c & 127) * 32 + (xs & 31);
}

template <typename I>
__device__ __forceinline__ void
stage_autocorr_body_t(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                      int W, int Hs, int Ws, int B, long long hl_stride, int tiled,
                      float* __restrict__ rowbuf, long long first, long long step,
                      long long end) {
  // plane layout: [3][C][Hs][Ws];  tiled layout: [3][CB*128][Hs][NS*32] tile-major, plus the
  // two edge rows of every copy in plain layout rowbuf[e][s][c][Wr]
  const int CB = (C + 127) >> 7, NS = (W + 31) >> 5, Wr = (W + 3) & ~3;
  const int Cc = tiled ? CB * 128 : C, Wc = tiled ? NS * 32 : Ws;
  const long long total = 3LL * Cc * Hs * Wc;
  const long long img = (long long)C * H * W;
  const float fb = (float)B;
  if (end > total) end = total;
  for (I idx = (I)first; idx < (I)end; idx += (I)step) {
    int xs = (int)(idx % Wc);
    I rest = idx / Wc;
    int r = (int)(rest % Hs);
    rest /= Hs;
    int c = (int)(rest % Cc);
    int s = (int)(rest / Cc);
    int xx = xs + s;
    float v = 0.f;
    if (c < C && r < H && xx < W) {
      const float* p = x + ((long long)c * H + r) * W + xx;
      float acc = 0.f;
#pragma unroll 4
      for (int b = 0; b < B; ++b) acc += __ldg(p + (long long)b * img);
      v = acc / fb;
    }
    float hi, lo;
    tf32_split(v, hi, lo);
    const long long o = tiled ? ac_tiled_off(s, c, r, xs, CB, Hs, NS) : idx;
    stage[o] = hi;
    stage[o + hl_stride] = lo;
    if (tiled && c < C && xs < Wr && (r == 0 || r == H - 1)) {
      if (r == H - 1) {
        const long long q = ((long long)(0 * 3 + s) * C + c) * Wr + xs;
        rowbuf[q] = hi; rowbuf[q + hl_stride] = lo;
      }
      if (r == 0) {
        const long long q = ((long long)(1 * 3 + s) * C + c) * Wr + xs;
        rowbuf[q] = hi; rowbuf[q + hl_stride] = lo;
      }
    }
  }
}

__device__ __forceinline__ void
stage_autocorr_body(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                    int W, int Hs, int Ws, int B, long long hl_stride, int tiled,
                    float* __restrict__ rowbuf, long long first, long long step,
                    long long end) {
  const int CB = (C + 127) >> 7, NS = (W + 31) >> 5;
  const long long total = 3LL * (tiled ? CB * 128 : C) * Hs * (tiled ? NS * 32 : Ws);
  if (total < kIdx32Max && step < (1LL << 24))
    stage_autocorr_body_t<int>(x, stage, C, H, W, Hs, Ws, B, hl_stride, tiled, rowbuf, first, step, end);
  else
    stage_autocorr_body_t<long long>(x, stage, C, H, W, Hs, Ws, B, hl_stride, tiled, rowbuf, first, step, end);
}

__global__ void __launch_bounds__(256)
stage_autocorr_kernel(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                      int W, int Hs, int Ws, int B, long long hl_stride, int tiled,
                      float* __restrict__ rowbuf) {
  stage_autocorr_body(x, stage, C, H, W, Hs, Ws, B, hl_stride, tiled, rowbuf, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, 1LL << 62);
}

// W % 4 == 0, 16-byte aligned input: one thread per aligned float4 of a staged row.
template <int B_UNROLL>
__device__ __forceinline__ void
stage_autocorr_vec_body(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                        int W, int B, long long hl_stride, int tiled,
                        float* __restrict__ rowbuf, long long first, long long step,
                        long long end) {
  const int CB = (C + 127) >> 7, NS = (W + 31) >> 5, Wr = W;      // W % 4 == 0 here
  const int Hs = H + 2, Ws = tiled ? NS * 32 : W + 4, W4 = Ws >> 2;
  const int Cc = tiled ? CB * 128 : C;
  const long long total = (long long)Cc * Hs * W4;
  const long long img = (long long)C * H * W;
  const long long plane = (long long)C * Hs * Ws;
  const float fb = (float)B;
  const int lane = threadIdx.x & 31;
  const long long total_r = (total + 31) / 32 * 32;
  if (end > total_r) end = total_r;
  for (long long idx = first; idx < end; idx += step) {
    const bool live = idx < total;
    int x4 = 0, r = 0, c = 0;
    if (live) {
      x4 = (int)(idx % W4);
      long long rest = idx / W4;
      r = (int)(rest % Hs);
      c = (int)(rest / Hs);
    }
    const bool data = live && c < C && r < H && x4 * 4 < W;
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* p = x + ((long long)c * H + r) * W + x4 * 4;
    if (data) {
      int b = 0;
      for (; b + B_UNROLL <= B; b += B_UNROLL) {
        float4 v[B_UNROLL];
#pragma unroll
        for (int u = 0; u < B_UNROLL; ++u) v[u] = ldg_stream4(p + (long long)(b + u) * img);
#pragma unroll
        for (int u = 0; u < B_UNROLL; ++u) { m.x += v[u].x; m.y += v[u].y; m.z += v[u].z; m.w += v[u].w; }
      }
      for (; b < B; ++b) {
        float4 v = ldg_stream4(p + (long long)b * img);
        m.x += v.x; m.y += v.y; m.z += v.z; m.w += v.w;
      }
      m.x /= fb; m.y /= fb; m.z /= fb; m.w /= fb;
    }
    // the next two means of the same row come from the next lane (or an extra load at
    // the warp edge; zero past the row end)
    float n0 = __shfl_down_sync(0xffffffffu, m.x, 1);
    float n1 = __shfl_down_sync(0xffffffffu, m.y, 1);
    const bool next_data = data && (x4 + 1) * 4 < W;
    if (!next_data) {
      n0 = n1 = 0.f;
    } else if (lane == 31) {
      float s0 = 0.f, s1 = 0.f;
      for (int b = 0; b < B; ++b) {
        s0 += __ldg(p + 4 + (long long)b * img);
        s1 += __ldg(p + 5 + (long long)b * img);
      }
      n0 = s0 / fb; n1 = s1 / fb;
    }
    if (live && !tiled) {
      float* o = stage + ((long long)c * Hs + r) * Ws + x4 * 4;
      split_store4(o, o + hl_stride, m.x, m.y, m.z, m.w);                          // shift 0
      split_store4(o + plane, o + plane + hl_stride, m.y, m.z, m.w, n0);          // shift 1
      split_store4(o + 2 * plane, o + 2 * plane + hl_stride, m.z, m.w, n0, n1);   // shift 2
    } else if (live) {
      float* o0 = stage + ac_tiled_off(0, c, r, x4 * 4, CB, Hs, NS);
      float* o1 = stage + ac_tiled_off(1, c, r, x4 * 4, CB, Hs, NS);
      float* o2 = stage + ac_tiled_off(2, c, r, x4 * 4, CB, Hs, NS);
      split_store4(o0, o0 + hl_stride, m.x, m.y, m.z, m.w);
      split_store4(o1, o1 + hl_stride, m.y, m.z, m.w, n0);
      split_store4(o2, o2 + hl_stride, m.z, m.w, n0, n1);
      if (c < C && x4 * 4 < Wr && (r == 0 || r == H - 1)) {
        // edge rows of the three copies, plain layout (pitch Wr)
        for (int e = 0; e < 2; ++e) {
          if (r != (e == 0 ? H - 1 : 0)) continue;
          float* q = rowbuf + ((long long)(e * 3) * C + c) * Wr + x4 * 4;
          const long long cs = (long long)C * Wr;
          split_store4(q, q + hl_stride, m.x, m.y, m.z, m.w);
          split_store4(q + cs, q + cs + hl_stride, m.y, m.z, m.w, n0);
          split_store4(q + 2 * cs, q + 2 * cs + hl_stride, m.z, m.w, n0, n1);
        }
      }
    }
  }
}

template <int B_UNROLL>
__global__ void __launch_bounds__(256)
stage_autocorr_vec_kernel(const float* __restrict__ x, float* __restrict__ stage, int C, int H,
                          int W, int B, long long hl_stride, int tiled,
                          float* __restrict__ rowbuf) {
  stage_autocorr_vec_body<B_UNROLL>(x, stage, C, H, W, B, hl_stride, tiled, rowbuf, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x,
                                    1LL << 62);
}

// edge columns colbuf[side][shift][c][u] = m~[c][u+shift][side ? 0 : W-1] (pitch Hc) and
// corner pixels cornerbuf[q][c][0] (pitch 4): q = 0 (H-1,W-1), 1 (H-1,0), 2 (0,W-1), 3 (0,0)
__device__ __forceinline__ void
stage_autocorr_edges_body(const float* __restrict__ x, float* __restrict__ colbuf,
                          float* __restrict__ cornerbuf, int C, int H, int W, int Hc, int B,
                          long long hl_stride, long long first, long long step, long long end) {
  const long long n_col = 6LL * C * Hc, n_cor = 16LL * C;
  const long long img = (long long)C * H * W;
  const float fb = (float)B;
  if (end > n_col + n_cor) end = n_col + n_cor;
  for (long long idx = first; idx < end; idx += step) {
    int c, y, xx;
    bool valid;
    float* dst;
    if (idx < n_col) {
      int u = (int)(idx % Hc);
      long long rest = idx / Hc;
      c = (int)(rest % C);
      int ss = (int)(rest / C);
      int side = ss / 3, shift = ss - side * 3;
      y = u + shift;
      xx = side ? 0 : W - 1;
      valid = y < H;
      dst = colbuf + idx;
    } else {
      long long j = idx - n_col;
      int e = (int)(j & 3);
      c = (int)((j >> 2) % C);
      int q = (int)((j >> 2) / C);
      y = (q < 2) ? H - 1 : 0;
      xx = (q & 1) ? 0 : W - 1;
      valid = e == 0;
      dst = cornerbuf + j;
    }
    float v = 0.f;
    if (valid) {
      const float* p = x + ((long long)c * H + y) * W + xx;
      float acc = 0.f;
      for (int b = 0; b < B; ++b) acc += __ldg(p + (long long)b * img);
      v = acc / fb;
    }
    float hi, lo;
    tf32_split(v, hi, lo);
    dst[0] = hi;
    dst[hl_stride] = lo;
  }
}

__global__ void __launch_bounds__(256)
stage_autocorr_edges_kernel(const float* __restrict__ x, float* __restrict__ colbuf,
                            float* __restrict__ cornerbuf, int C, int H, int W, int Hc, int B,
                            long long hl_stride) {
  stage_autocorr_edges_body(x, colbuf, cornerbuf, C, H, W, Hc, B, hl_stride, blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, 1LL << 62);
}

// ---------------------------------------------------------------------------
// Explicit im2col fallback (any kernel size / dilation-free conv whose channel
// count does not fit the implicit path, e.g. the 7x7 stem with Cin = 3).
// Rows are written directly in the reference's (Cin, kh, kw) order.
// stage[hl][row][k],  row < d, k < Hout*Wout, pitch Ws.
// ---------------------------------------------------------------------------
template <typename I>
__device__ __forceinline__ void
stage_conv_explicit_body_t(const float* __restrict__ x, float* __restrict__ stage,
                           const ConvGeom& g, int B, long long hl_stride, long long first,
                           long long step, long long end) {
  // index = (im2col row (c, i, j), group of 4 K columns)
  const long long img = (long long)g.C * g.H * g.W;
  const int taps = g.kh * g.kw;
  const int d = g.C * taps;
  const int K = g.Hout * g.Wout;
  const float fb = (float)B;
  const int W4 = g.Ws >> 2;
  const long long total = (long long)g.Cs * W4;
  if (end > total) end = total;
  // (row, k4) of the thread's first index by division, then advanced by `step`
  int row = 0, k4 = 0;
  if ((I)first < (I)end) {
    row = (int)((I)first / W4);
    k4 = (int)((I)first - (I)row * W4);
  }
  const int drow = (int)(step / W4), dk4 = (int)(step - (long long)drow * W4);
  for (I idx = (I)first; idx < (I)end; idx += (I)step,
         k4 += dk4, row += drow + (k4 >= W4), k4 -= (k4 >= W4) ? W4 : 0) {
    const int c = row / taps, t = row - c * taps;
    const int i = t / g.kw, j = t - i * g.kw;
    const bool row_ok = row < d;
    float v[4];
    int k = k4 * 4;
    int oy = k / g.Wout, ox = k - oy * g.Wout;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float acc = 0.f;
      if (row_ok && k + e < K) {
        const int y = oy * g.sh - g.ph + i, xx = ox * g.sw - g.pw + j;
        if (y >= 0 && y < g.H && xx >= 0 && xx < g.W) {
          const float* q = x + ((long long)c * g.H + y) * g.W + xx;
          for (int b = 0; b < B; ++b) acc += __ldg(q + (long long)b * img);
          acc /= fb;
        }
      }
      v[e] = acc;
      if (++ox == g.Wout) { ox = 0; ++oy; }
    }
    float* o = stage + (long long)row * g.Ws + k;
    split_store4(o, o + hl_stride, v[0], v[1], v[2], v[3]);
  }
}

// One im2col row per work item (the grouped kernel's items never cross a row; Wout % 4 == 0,
// plain layout): the (c, i, j) decode is paid once per item, (oy, ox) advance incrementally
// and the four columns of a float4 share their input row - the general routine above spends
// most of its instructions on three divisions and four bounds checks per float4.
__device__ __forceinline__ void
stage_conv_explicit_row_body(const float* __restrict__ x, float* __restrict__ stage,
                             const ConvGeom& g, int B, long long hl_stride, long long first,
                             int tid, int step, long long end) {
  const int W4 = g.Ws >> 2;
  const int row = (int)(first / W4);
  const int k4_lo = (int)(first - (long long)row * W4), k4_hi = (int)(end - (long long)row * W4);
  const int taps = g.kh * g.kw;
  const int c = row / taps, t = row - c * taps;
  const int i = t / g.kw, jj = t - i * g.kw;
  const bool row_ok = row < g.C * taps;
  const long long img = (long long)g.C * g.H * g.W;
  const float fb = (float)B;
  int k4 = k4_lo + tid;
  int oy = (k4 * 4) / g.Wout, ox = k4 * 4 - oy * g.Wout;
  const int d_oy = (step * 4) / g.Wout, d_ox = step * 4 - d_oy * g.Wout;
  float* out = stage + (long long)row * g.Ws;
  const float* plane = x + (long long)c * g.H * g.W;
  for (; k4 < k4_hi; k4 += step) {
    const int y = oy * g.sh - g.ph + i;
    const int xx0 = ox * g.sw - g.pw + jj;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (row_ok && y >= 0 && y < g.H) {
      const float* src = plane + (long long)y * g.W + xx0;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int xx = xx0 + e * g.sw;
        if (xx >= 0 && xx < g.W) {
          float acc = 0.f;
          for (int b = 0; b < B; ++b) acc += __ldg(src + e * g.sw + (long long)b * img);
          v[e] = acc / fb;
        }
      }
    }
    float* o = out + k4 * 4;
    split_store4(o, o + hl_stride, v[0], v[1], v[2], v[3]);
    ox += d_ox;
    oy += d_oy + (ox >= g.Wout);
    ox -= (ox >= g.Wout) ? g.Wout : 0;
  }
}

__device__ __forceinline__ void
stage_conv_explicit_body(const float* __restrict__ x, float* __restrict__ stage,
                         const ConvGeom& g, int B, long long hl_stride, long long first,
                         long long step, long long end) {
  const long long total = (long long)g.Cs * (g.Ws >> 2);
  if (total < kIdx32Max && step < (1LL << 24))
    stage_conv_explicit_body_t<int>(x, stage, g, B, hl_stride, first, step, end);
  else
    stage_conv_explicit_body_t<long long>(x, stage, g, B, hl_stride, first, step, end);
}

__global__ void __launch_bounds__(256)
stage_conv_explicit_kernel(const float* __restrict__ x, float* __restrict__ stage,
                           ConvGeom g, int B, long long hl_stride) {
  stage_conv_explicit_body(x, stage, g, B, hl_stride,
                           blockIdx.x * (long long)blockDim.x + threadIdx.x,
                           (long long)gridDim.x * blockDim.x, 1LL << 62);
}

int launch_stage_conv(const float* x, float* stage, const ConvGeom& g, int B,
                      float* mean_scratch, cudaStream_t stream) {
  long long total = (g.mode == kModeExplicit) ? (long long)g.Cs * g.Ws
                                              : (long long)g.Cs * g.Hs * g.Ws * g.ncopy;
  long long hl = stage_hl_stride(g);
  const long long img = (long long)g.C * g.H * g.W;
  const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && img % 4 == 0;
  ProfScope prof(kProfStage, stream);
  if (g.mode == kModeAutocorr) {
    float* rowbuf = stage + ac_rowbuf_off(g);
    if (aligned && g.W % 4 == 0 && (g.tiled || g.Ws == g.W + 4)) {
      long long n = g.tiled ? (long long)ac_cblocks(g) * 128 * g.Hs * (ac_strips(g) * 8)
                            : (long long)g.C * g.Hs * (g.Ws / 4);
      int blocks = (int)((n + 255) / 256);
      if (blocks > 148 * 16) blocks = 148 * 16;
      stage_autocorr_vec_kernel<8><<<blocks, 256, 0, stream>>>(x, stage, g.C, g.H, g.W, B, hl,
                                                              g.tiled, rowbuf);
    } else {
      const float* src = x;
      int Bg = B;
      if (B > 1 && aligned && mean_scratch != nullptr) {
        long long n4 = img / 4;
        int mb = (int)((n4 + 255) / 256);
        if (mb > 148 * 16) mb = 148 * 16;
        batch_mean_vec_kernel<8><<<mb, 256, 0, stream>>>(x, mean_scratch, n4, B, img);
        NSGP_LAUNCHED();
        src = mean_scratch;
        Bg = 1;
      }
      long long n = g.tiled ? 3LL * ac_cblocks(g) * 128 * g.Hs * ac_strips(g) * 32
                            : (long long)g.C * g.Hs * g.Ws * 3;
      int blocks = (int)((n + 255) / 256);
      if (blocks > 148 * 32) blocks = 148 * 32;
      stage_autocorr_kernel<<<blocks, 256, 0, stream>>>(src, stage, g.C, g.H, g.W, g.Hs, g.Ws, Bg,
                                                       hl, g.tiled, rowbuf);
    }
    NSGP_LAUNCHED();
    const int Hc = ac_col_pitch(g);
    long long ne = 6LL * g.C * Hc + 16LL * g.C;
    int eb = (int)((ne + 255) / 256);
    if (eb > 148 * 8) eb = 148 * 8;
    stage_autocorr_edges_kernel<<<eb, 256, 0, stream>>>(x, stage + ac_colbuf_off(g),
                                                        stage + ac_cornerbuf_off(g), g.C, g.H,
                                                        g.W, Hc, B, hl);
    NSGP_LAUNCHED();
    return 0;
  }
  if (g.mode == kModeFlat && g.sh == 1 && g.sw == 1 && aligned && (g.H * g.W) % 4 == 0) {
    long long n4 = (long long)g.C * g.H * g.W / 4;
    int blocks = (int)((n4 + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    stage_flat_vec_kernel<8><<<blocks, 256, 0, stream>>>(x, stage, n4, B, img, hl);
  } else if (g.mode == kModeImplicit && g.kh == 3 && g.kw == 3 && g.sh == 1 && g.sw == 1 &&
             g.ph == 1 && g.pw == 1 && aligned && g.W % 4 == 0) {
    long long n = (long long)g.C * g.Hs * (g.W / 4);
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    stage_3x3s1_vec_kernel<8><<<blocks, 256, 0, stream>>>(x, stage, g.C, g.H, g.W, B, hl);
  } else {
    // gather layouts: average the batch first (vectorised), then gather from the mean -
    // unless the gather touches only a fraction of the input (strided 1x1)
    const float* src = x;
    int Bg = B;
    const bool sparse = g.mode == kModeFlat && g.sh * g.sw > 1;
    if (B > 1 && aligned && mean_scratch != nullptr && !sparse) {
      long long n4 = img / 4;
      int mb = (int)((n4 + 255) / 256);
      if (mb > 148 * 16) mb = 148 * 16;
      batch_mean_vec_kernel<8><<<mb, 256, 0, stream>>>(x, mean_scratch, n4, B, img);
      NSGP_LAUNCHED();
      src = mean_scratch;
      Bg = 1;
    }
    if (g.mode == kModeExplicit) {
      long long ne = (long long)g.Cs * (g.Ws / 4);
      int grid = (int)((ne + 255) / 256);
      if (grid > 148 * 32) grid = 148 * 32;
      stage_conv_explicit_kernel<<<grid, 256, 0, stream>>>(src, stage, g, Bg, hl);
    } else {
      int blocks = (int)((total / 4 + 255) / 256);
      if (blocks > 148 * 32) blocks = 148 * 32;
      if (blocks < 1) blocks = 1;
      stage_conv_kernel<<<blocks, 256, 0, stream>>>(src, stage, g, Bg, hl);
    }
  }
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Grouped staging: the layer inputs of a whole forward staged by ONE launch (two when a
// gather layout reads the batch mean written by the first).  A layer's staging kernels
// are short (34 MB of input takes ~10 us, of which half is launch ramp and tail) and
// there are ~90 of them per forward; as work items of one persistent launch they stream
// back to back.  Item = (job, routine, index range); phase 0 reads the layer inputs,
// phase 1 reads the batch means phase 0 wrote.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 4)
stage_group_kernel(const StageJobDev* __restrict__ jobs, const StageItem* __restrict__ items,
                   int n_items, const float* const* __restrict__ xs, int B,
                   unsigned long long* tl) {
  // programmatic dependent launch: a kernel queued behind this one with the programmatic
  // stream-serialization attribute may start as soon as every block of this grid is running
  // (the pipelined covariance pass puts a contraction kernel there, on the other SMs)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  tl_begin(tl);
  for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
    const StageItem it = items[w];
    const StageJobDev& j = jobs[it.job];
    const ConvGeom& g = j.g;
    const float* x = it.from_mean ? j.mean : xs[it.job];
    const int Bx = it.from_mean ? 1 : B;
    const long long first = it.lo + threadIdx.x, step = blockDim.x, end = it.hi;
    const long long img = (long long)g.C * g.H * g.W;
    switch (it.kind) {
      case kStFlatVec:
        stage_flat_vec_body<8>(x, j.stage, img / 4, Bx, img, j.hl, first, step, end);
        break;
      case kStAcVec:
        stage_autocorr_vec_body<8>(x, j.stage, g.C, g.H, g.W, Bx, j.hl, g.tiled,
                                   j.stage + j.rowbuf_off, first, step, end);
        break;
      case kStAcEdges:
        stage_autocorr_edges_body(x, j.stage + j.colbuf_off, j.stage + j.cornerbuf_off, g.C,
                                  g.H, g.W, j.Hc, Bx, j.hl, first, step, end);
        break;
      case kStMean:
        batch_mean_vec_body<8>(x, j.mean, img / 4, Bx, img, first, step, end);
        break;
      case kStConv:
        stage_conv_body(x, j.stage, g, Bx, j.hl, first, step, end);
        break;
      case kStExplicit:
        if (g.Wout % 4 == 0)                        // items are row-aligned (plan_stage_job)
          stage_conv_explicit_row_body(x, j.stage, g, Bx, j.hl, it.lo, threadIdx.x, blockDim.x,
                                       end);
        else
          stage_conv_explicit_body(x, j.stage, g, Bx, j.hl, first, step, end);
        break;
      case kStAcScalar:
        stage_autocorr_body(x, j.stage, g.C, g.H, g.W, g.Hs, g.Ws, Bx, j.hl, g.tiled,
                            j.stage + j.rowbuf_off, first, step, end);
        break;
      case kSt3x3Vec:
        stage_3x3s1_vec_body<8>(x, j.stage, g.C, g.H, g.W, Bx, j.hl, first, step, end);
        break;
      default:
        break;
    }
  }
  tl_end(tl);
}

// ---------------------------------------------------------------------------
// TMA-fed phase 0 (batch mean, flat 1x1 staging, vectorised autocorrelation staging).
// The register routines keep their loads in flight in registers - ~128 KB per SM at most,
// fine when all 148 SMs stage, not when the staging only gets a slice of the GPU next to the
// sliding-window contraction.  Here ONE 3-D tensor-map box (256 floats x rows x B images,
// <= 32 KB) brings the same chunk of all B images into shared memory and six or seven of
// them are in flight per SM (scripts/tma3d_probe.py: the loads alone reach 149 GB/s per SM).
//   warp 0        producer: cp.async.bulk.tensor.3d into a 6- or 7-stage ring, mbarrier tx
//   warps 1..16   kTmaGroups consumer groups; group g takes the chunks g, g + G, ... of the
//                 CTA's chunk sequence: batch mean out of shared memory, tf32 split, layout
//                 stores.  A group does not see every lap of a ring slot, so before the
//                 parity wait on full[slot] it checks on empty[slot] that the slot's previous
//                 lap was consumed - otherwise it could be two mbarrier phases ahead and pass
//                 the parity wait early (measured: "unspecified launch failure").  Two groups
//                 of 8 warps and four of 4 perform alike (profiles/pipeline_r02.txt): next to
//                 the sliding-window kernel the phase is HBM-bound from ~56 SMs on.
// Index space = float4s of the per-image tensor (every routine's input is contiguous).
// Autocorrelation layout: the two column-shifted copies need the NEXT float4's first two
// means; inside a stage they come from the next lane (compile-time batch <= 8) or through a
// double-buffered, per-group shared array; at a stage end the owner writes only the words it knows and the
// first thread of the next stage (maybe in another CTA) writes the rest - disjoint words, no
// ordering needed.  The threads that hold the first / last float4 of an image row also write
// the edge-column and corner-pixel buffers of the boundary corrections.  Padding of the tiled
// layout (rows H, H+1, columns >= W, channels >= C) and of those buffers is zeroed once at
// table build.
// ---------------------------------------------------------------------------
constexpr int kTmaStages = 12;                     // at most
constexpr int kTmaRingBytes = 192 * 1024;
constexpr int kTmaMaxRows = 8;                     // <= 512 float4s of means per stage
constexpr int kTmaGroups = 2;
constexpr int kTmaGroupThreads = 256;
constexpr int kTmaThreads = 32 + kTmaGroups * kTmaGroupThreads;
// rows of 1 KB per box: 8 / 4 rows (every thread of a group busy) while the stage stays
// <= 32 KB, else as many as fit 48 KB (B = 16: 3 rows, 192 of the 256 threads busy)
static inline int tma_box_rows(int B) {
  if (B < 1 || B > 32) return 0;
  if (8 * B <= 32) return 8;
  if (4 * B <= 48) return 4;
  return 48 / B > 0 ? 48 / B : 1;
}
constexpr int kTmaMeanBytes = kTmaMaxRows * 1024;    // one buffer of means
constexpr int kTmaMeansBytes = 2 * kTmaGroups * kTmaMeanBytes;
// The sliding-window routine needs the next float4's means.  Template instances with a
// compile-time batch <= 8 take them from the next lane (lane 31 recomputes them from the raw
// chunk): no mean buffers, the ring gets their 32 KB (7 x 32 KB stages at B = 8).  Larger or
// run-time batches exchange the means through shared memory (lane 31's serial recompute of
// B loads costs more than the group barrier there: configs[4] 5.58 vs 5.75 ms per step).
static inline bool tma_shuffle_variant(int B) { return B == 8 || B == 4 || B == 2 || B == 1; }
// ring slots: as many stages as fit the ring (<= kTmaStages)
static inline int tma_ring_stages(int B) {
  const int ring = kTmaRingBytes + (tma_shuffle_variant(B) ? kTmaMeansBytes : 0);
  const int n = ring / (B * tma_box_rows(B) * 1024);
  return n >= kTmaStages ? kTmaStages : n;
}
static inline size_t stage_tma_smem_bytes() {
  return (size_t)kTmaRingBytes + kTmaMeansBytes + 128 /* alignment slack */;
}

// cvt.rna.tf32.f32 is lowered to integer add + mask + an inf / NaN guard on sm_100a; the
// staging consumers are instruction-bound, so they use the two instructions without the guard
// (finite inputs: bit-identical; an inf stays inf, a NaN stays non-finite)
__device__ __forceinline__ float tf32_rna_finite(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void tf32_split_finite(float x, float& hi, float& lo) {
  hi = tf32_rna_finite(x);
  lo = tf32_rna_finite(x - hi);
}
__device__ __forceinline__ void store_hl4(float* p, long long hl, const float* h, const float* l,
                                          int i) {
  *reinterpret_cast<float4*>(p) = make_float4(h[i], h[i + 1], h[i + 2], h[i + 3]);
  *reinterpret_cast<float4*>(p + hl) = make_float4(l[i], l[i + 1], l[i + 2], l[i + 3]);
}
// (c, r, x) += (dc, dr, dx) as a mixed-radix number with radices (-, R, X)
__device__ __forceinline__ void radix_add(int& c, int& r, int& x, int dc, int dr, int dx, int R,
                                          int X) {
  x += dx;
  const int cx = x >= X;
  x -= cx ? X : 0;
  r += dr + cx;
  const int cr = r >= R;
  r -= cr ? R : 0;
  c += dc + cr;
}

// KB / KROWS > 0: batch size and box rows known at compile time (the loads get immediate
// offsets and the batch loop is unrolled); 0: run-time values
template <int KB, int KROWS>
__global__ void __launch_bounds__(kTmaThreads, 1)
stage_tma_kernel(const StageJobDev* __restrict__ jobs, const StageItem* __restrict__ items,
                 int n_items, const CUtensorMap* __restrict__ maps, int B_rt, int rows_rt,
                 int n_stages, unsigned long long* tl) {
  using namespace tc;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  extern __shared__ __align__(128) uint8_t tma_smem_raw[];
  // 128-byte aligned start of the ring (pointer arithmetic on the shared array itself, so
  // that the accesses stay LDS / STS instead of generic loads)
  uint8_t* const smem = tma_smem_raw + ((128u - (smem_u32(tma_smem_raw) & 127u)) & 127u);
  __shared__ uint64_t full[kTmaStages], empty[kTmaStages];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = KB > 0 ? KB : B_rt, rows = KROWS > 0 ? KROWS : rows_rt;
  tl_begin(tl);
  if (threadIdx.x == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], kTmaGroupThreads / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int E4 = rows * 64;                        // float4s of one image per stage
  const uint32_t stage_tx = (uint32_t)B * rows * 1024u;      // = bytes of one ring slot
  if (warp == 0) {
    // ============================ producer ============================
    uint32_t st = 0, ph = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const StageItem it = items[w];
      const CUtensorMap* map = &maps[it.job];
      for (long long q0 = it.lo; q0 < it.hi; q0 += E4) {
        mbar_wait_warp(&empty[st], ph ^ 1, lane);
        mbar_expect_tx_elect(&full[st], stage_tx);
        if (lane == 0)
          asm volatile(
              "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
              "[%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem + st * stage_tx)),
              "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(&full[st])), "r"(0),
              "r"((int)(q0 >> 6)), "r"(0)
              : "memory");
        __syncwarp();
        if (++st == (uint32_t)n_stages) { st = 0; ph ^= 1; }
      }
    }
  } else {
    // ============================ consumers ============================
    const int gid = (threadIdx.x - 32) / kTmaGroupThreads;
    const int tid = (threadIdx.x - 32) % kTmaGroupThreads;
    const float fb = (float)B, inv = 1.f / fb;
    const bool pow2 = (B & (B - 1)) == 0;          // then x * (1/B) == x / B exactly
    // ring slot / lap of the group's next chunk (chunk gid of the CTA's chunk sequence)
    uint32_t st = gid % n_stages, lap = gid / n_stages;
    uint32_t n = 0;                                // chunks of the CTA before the current item
    auto wait_chunk = [&]() {
      if (lap > 0) mbar_wait_warp(&empty[st], (lap - 1) & 1, lane);   // previous lap consumed
      mbar_wait_warp(&full[st], lap & 1, lane);
    };
    auto next_chunk = [&]() {
      st += kTmaGroups;
      while (st >= (uint32_t)n_stages) { st -= n_stages; ++lap; }
    };
    constexpr bool kShuffle = KB == 8 || KB == 4 || KB == 2 || KB == 1;   // tma_shuffle_variant
    float4* const mean_s = reinterpret_cast<float4*>(smem + kTmaRingBytes +
                                                     gid * 2 * kTmaMeanBytes);
    int mbuf = 0;
    // batch mean of float4 f of the chunk in `raw`
    auto mean4 = [&](const float4* raw, int f) {
      float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (KB > 0) {
#pragma unroll
        for (int b = 0; b < (KB > 0 ? KB : 1); ++b) {
          const float4 v = raw[b * E4 + f];
          s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
        }
      } else {
        const float4* p = raw + f;
#pragma unroll 4
        for (int b = 0; b < B; ++b, p += E4) {
          const float4 v = *p;
          s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
        }
      }
      if (pow2) { s4.x *= inv; s4.y *= inv; s4.z *= inv; s4.w *= inv; }
      else { s4.x /= fb; s4.y /= fb; s4.z /= fb; s4.w /= fb; }
      return s4;
    };
    // first two elements of the batch mean of float4 f (same summation order as mean4)
    auto mean2 = [&](const float4* raw, int f) {
      float2 s2 = make_float2(0.f, 0.f);
#pragma unroll
      for (int b = 0; b < (KB > 0 ? KB : 1); ++b) {
        const float2 v = *reinterpret_cast<const float2*>(raw + b * E4 + f);
        s2.x += v.x; s2.y += v.y;
      }
      if (pow2) { s2.x *= inv; s2.y *= inv; }
      else { s2.x /= fb; s2.y /= fb; }
      return s2;
    };
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const StageItem it = items[w];
      const StageJobDev& j = jobs[it.job];
      const int kind = it.kind;
      const long long hl = j.hl;
      float* const stage = j.stage;
      const int n_chunks = (int)((it.hi - it.lo + E4 - 1) / E4);
      static_assert((kTmaGroups & (kTmaGroups - 1)) == 0 && kTmaGroups <= 4, "2 or 4 groups");
      const int k0 = (int)((gid - n) & (kTmaGroups - 1));   // first chunk of the item that is ours
      n += n_chunks;
      if (kind == kStFlatSub) {
        // flat 1x1 staging + the stride-2 subsample for the 1x1 s2 job on the same tensor:
        // even rows, elements .x / .z of every float4 (W % 4 == 0)
        const int H = j.g.H, W4 = j.g.W >> 2, HW4 = H * W4;
        float* const sub = j.sub_stage;
        const long long sub_hl = j.sub_hl;
        const int sub_pitch = j.sub_pitch, sub_wout = j.sub_wout;
        int c0, r0, x0, dcC, drC, dxC, dcU, drU, dxU;
        {
          const long long q = it.lo + (long long)k0 * E4 + tid;
          c0 = (int)(q / HW4);
          int rem = (int)(q - (long long)c0 * HW4);
          r0 = rem / W4; x0 = rem - r0 * W4;
          const int dC = kTmaGroups * E4;
          dcC = dC / HW4; rem = dC - dcC * HW4; drC = rem / W4; dxC = rem - drC * W4;
          const int dU = kTmaGroupThreads;
          dcU = dU / HW4; rem = dU - dcU * HW4; drU = rem / W4; dxU = rem - drU * W4;
        }
        for (int k = k0; k < n_chunks; k += kTmaGroups) {
          const long long q0 = it.lo + (long long)k * E4;
          wait_chunk();
          const float4* raw = reinterpret_cast<const float4*>(smem + st * stage_tx);
          int c = c0, r = r0, x4 = x0;
          for (int f = tid; f < E4;
               f += kTmaGroupThreads, radix_add(c, r, x4, dcU, drU, dxU, H, W4)) {
            const float4 m = mean4(raw, f);
            const long long q = q0 + f;
            if (q >= it.hi) continue;
            float4 h, l;
            tf32_split_finite(m.x, h.x, l.x); tf32_split_finite(m.y, h.y, l.y);
            tf32_split_finite(m.z, h.z, l.z); tf32_split_finite(m.w, h.w, l.w);
            *reinterpret_cast<float4*>(stage + q * 4) = h;
            *reinterpret_cast<float4*>(stage + q * 4 + hl) = l;
            if ((r & 1) == 0) {
              float* o = sub + (long long)c * sub_pitch + (r >> 1) * sub_wout + 2 * x4;
              *reinterpret_cast<float2*>(o) = make_float2(h.x, h.z);
              *reinterpret_cast<float2*>(o + sub_hl) = make_float2(l.x, l.z);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
          next_chunk();
          radix_add(c0, r0, x0, dcC, drC, dxC, H, W4);
        }
        continue;
      }
      if (kind == kStS2x3) {
        // 3x3 stride-2 pad-1: copy(p, jj)[c][r][x] = m[c][2(r-1) + py_p][2x - 1 + jj] with
        // py = (1, 0): input row y lands in row phase p = 1 - (y & 1) at r = (y >> 1) + 1, its
        // even columns in tap column 1, its odd columns in tap columns 0 (one to the right)
        // and 2; every input element is read once, halo / padding words stay zero
        const int H = j.g.H, W4 = j.g.W >> 2, HW4 = H * W4;
        const int Hs = j.g.Hs, Ws = j.g.Ws, Wout = j.g.Wout, Cs = j.g.Cs;
        const long long plane = (long long)Cs * Hs * Ws;     // one copy
        int c0, r0, x0, dcC, drC, dxC, dcU, drU, dxU;
        {
          const long long q = it.lo + (long long)k0 * E4 + tid;
          c0 = (int)(q / HW4);
          int rem = (int)(q - (long long)c0 * HW4);
          r0 = rem / W4; x0 = rem - r0 * W4;
          const int dC = kTmaGroups * E4;
          dcC = dC / HW4; rem = dC - dcC * HW4; drC = rem / W4; dxC = rem - drC * W4;
          const int dU = kTmaGroupThreads;
          dcU = dU / HW4; rem = dU - dcU * HW4; drU = rem / W4; dxU = rem - drU * W4;
        }
        for (int k = k0; k < n_chunks; k += kTmaGroups) {
          const long long q0 = it.lo + (long long)k * E4;
          wait_chunk();
          const float4* raw = reinterpret_cast<const float4*>(smem + st * stage_tx);
          int c = c0, y = r0, x4 = x0;
          for (int f = tid; f < E4;
               f += kTmaGroupThreads, radix_add(c, y, x4, dcU, drU, dxU, H, W4)) {
            const float4 m = mean4(raw, f);
            if (q0 + f >= it.hi) continue;
            float4 h, l;
            tf32_split_finite(m.x, h.x, l.x); tf32_split_finite(m.y, h.y, l.y);
            tf32_split_finite(m.z, h.z, l.z); tf32_split_finite(m.w, h.w, l.w);
            const int p = 1 - (y & 1);
            float* o = stage + (long long)(p * 3) * plane +
                       ((long long)c * Hs + (y >> 1) + 1) * Ws + 2 * x4;
            float* o1 = o + plane;                   // tap column 1: even input columns
            float* o2 = o1 + plane;                  // tap column 2: odd input columns
            *reinterpret_cast<float2*>(o1) = make_float2(h.x, h.z);
            *reinterpret_cast<float2*>(o1 + hl) = make_float2(l.x, l.z);
            *reinterpret_cast<float2*>(o2) = make_float2(h.y, h.w);
            *reinterpret_cast<float2*>(o2 + hl) = make_float2(l.y, l.w);
            o[1] = h.y; o[1 + hl] = l.y;             // tap column 0: x = (xx + 1) / 2
            if (2 * x4 + 2 < Wout) { o[2] = h.w; o[2 + hl] = l.w; }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
          next_chunk();
          radix_add(c0, r0, x0, dcC, drC, dxC, H, W4);
        }
        continue;
      }
      if (kind != kStAcVec) {
        float* const dst = kind == kStMean ? j.mean : stage;
        for (int k = k0; k < n_chunks; k += kTmaGroups) {
          const long long q0 = it.lo + (long long)k * E4;
          wait_chunk();
          const float4* raw = reinterpret_cast<const float4*>(smem + st * stage_tx);
          for (int f = tid; f < E4; f += kTmaGroupThreads) {
            const float4 m = mean4(raw, f);
            const long long q = q0 + f;
            if (q >= it.hi) continue;
            if (kind == kStMean) {
              *reinterpret_cast<float4*>(dst + q * 4) = m;
            } else {
              float4 h, l;
              tf32_split_finite(m.x, h.x, l.x); tf32_split_finite(m.y, h.y, l.y);
              tf32_split_finite(m.z, h.z, l.z); tf32_split_finite(m.w, h.w, l.w);
              *reinterpret_cast<float4*>(dst + q * 4) = h;
              *reinterpret_cast<float4*>(dst + q * 4 + hl) = l;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
          next_chunk();
        }
        continue;
      }
      // ---- autocorrelation layout (tiled; W % 4 == 0)
      const int H = j.g.H, W = j.g.W, C = j.g.C;
      const int W4 = W >> 2, HW4 = H * W4;
      const int CB = (C + 127) >> 7, NS = (W + 31) >> 5, Hs = H + 2;
      const long long copy_stride = (long long)CB * Hs * NS * 4096;
      float* const rowbuf = stage + j.rowbuf_off;
      float* const colbuf = stage + j.colbuf_off;
      float* const cornerbuf = stage + j.cornerbuf_off;
      const int Hc = j.Hc;
      // coordinates (c, r, x4) of this thread's first float4 of the group's first chunk of
      // the item, by division; afterwards advanced as a mixed-radix number (the divisions
      // would be a third of the consumer's instructions)
      int c0, r0, x0, dcC, drC, dxC, dcU, drU, dxU;
      {
        const long long q = it.lo + (long long)k0 * E4 + tid;
        c0 = (int)(q / HW4);
        int rem = (int)(q - (long long)c0 * HW4);
        r0 = rem / W4; x0 = rem - r0 * W4;
        const int dC = kTmaGroups * E4;            // from one of our chunks to the next
        dcC = dC / HW4; rem = dC - dcC * HW4; drC = rem / W4; dxC = rem - drC * W4;
        const int dU = kTmaGroupThreads;           // from one float4 of a chunk to the next
        dcU = dU / HW4; rem = dU - dcU * HW4; drU = rem / W4; dxU = rem - drU * W4;
      }
      for (int k = k0; k < n_chunks; k += kTmaGroups) {
        const long long q0 = it.lo + (long long)k * E4;
        wait_chunk();
        const float4* raw = reinterpret_cast<const float4*>(smem + st * stage_tx);
        float4* ms = mean_s + mbuf * (kTmaMeanBytes / 16);
        if (!kShuffle) {
          // means into shared memory (the raw chunk is then consumed), then the stores
          mbuf ^= 1;
          for (int f = tid; f < E4; f += kTmaGroupThreads) ms[f] = mean4(raw, f);
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
          switch (gid) {                             // the group's own named barrier
            case 0: asm volatile("bar.sync 1, %0;" ::"n"(kTmaGroupThreads) : "memory"); break;
            case 1: asm volatile("bar.sync 2, %0;" ::"n"(kTmaGroupThreads) : "memory"); break;
            case 2: asm volatile("bar.sync 3, %0;" ::"n"(kTmaGroupThreads) : "memory"); break;
            default: asm volatile("bar.sync 4, %0;" ::"n"(kTmaGroupThreads) : "memory"); break;
          }
        }
        int c = c0, r = r0, x4 = x0;
        for (int f = tid; f < E4; f += kTmaGroupThreads, radix_add(c, r, x4, dcU, drU, dxU, H, W4)) {
          if (q0 + f >= it.hi) break;                // warp-uniform: hi is a multiple of 64
          const bool next_data = x4 + 1 < W4;
          const bool in_stage = f + 1 < E4;          // the next float4 belongs to this chunk
          float4 mm;
          float2 nx = make_float2(0.f, 0.f);
          if (kShuffle) {
            // the next float4's two means from the next lane; lane 31 recomputes them
            mm = mean4(raw, f);
            const float sx = __shfl_down_sync(0xffffffffu, mm.x, 1);
            const float sy = __shfl_down_sync(0xffffffffu, mm.y, 1);
            if (next_data && in_stage) nx = lane == 31 ? mean2(raw, f + 1) : make_float2(sx, sy);
          } else {
            mm = ms[f];
            if (next_data && in_stage) nx = *reinterpret_cast<const float2*>(ms + f + 1);
          }
          const bool defer = next_data && !in_stage;
          float h[6], l[6];
          tf32_split_finite(mm.x, h[0], l[0]); tf32_split_finite(mm.y, h[1], l[1]);
          tf32_split_finite(mm.z, h[2], l[2]); tf32_split_finite(mm.w, h[3], l[3]);
          tf32_split_finite(nx.x, h[4], l[4]); tf32_split_finite(nx.y, h[5], l[5]);
          float* o0 = stage + ((long long)(((c >> 7) * Hs + r) * NS + (x4 >> 3)) * 4096 +
                               (c & 127) * 32 + (x4 & 7) * 4);
          float* o1 = o0 + copy_stride;
          float* o2 = o1 + copy_stride;
          store_hl4(o0, hl, h, l, 0);
          if (!defer) {
            store_hl4(o1, hl, h, l, 1);
            store_hl4(o2, hl, h, l, 2);
          } else {
            o1[0] = h[1]; o1[1] = h[2]; o1[2] = h[3];
            o1[hl] = l[1]; o1[hl + 1] = l[2]; o1[hl + 2] = l[3];
            o2[0] = h[2]; o2[1] = h[3];
            o2[hl] = l[2]; o2[hl + 1] = l[3];
          }
          // the previous float4 of this row ended a stage: complete its shifted copies
          const bool fix_prev = f == 0 && x4 > 0;
          if (fix_prev) {
            // one float4 to the left inside the same 32-column strip, or the last one of the
            // previous strip
            const long long back = (x4 & 7) ? 4 : 4096 - 28;
            float* p1 = o1 - back;
            float* p2 = o2 - back;
            p1[3] = h[0]; p1[hl + 3] = l[0];
            p2[2] = h[0]; p2[hl + 2] = l[0];
            p2[3] = h[1]; p2[hl + 3] = l[1];
          }
          const bool first_x = x4 == 0, last_x = x4 == W4 - 1;
          const bool edge_row = r == 0 || r == H - 1;
          if (!(first_x || last_x || edge_row)) continue;
          if (first_x || last_x) {
            // edge columns (x = W-1: side 0, x = 0: side 1) of the three row shifts and the
            // corner pixels (layouts: stage_autocorr_edges_body); their padding is zeroed at
            // table build like the rest of the workspace
            for (int side = 0; side < 2; ++side) {
              if (side == 0 ? !last_x : !first_x) continue;
              const float vh = side == 0 ? h[3] : h[0], vl = side == 0 ? l[3] : l[0];
              float* cb = colbuf + ((long long)(side * 3) * C + c) * Hc + r;
              const long long ss = (long long)C * Hc;
              cb[0] = vh; cb[hl] = vl;
              if (r >= 1) { cb[ss - 1] = vh; cb[ss - 1 + hl] = vl; }
              if (r >= 2) { cb[2 * ss - 2] = vh; cb[2 * ss - 2 + hl] = vl; }
              if (edge_row) {
                const int q = (r == 0 ? 2 : 0) + side;
                float* kb = cornerbuf + ((long long)q * C + c) * 4;
                kb[0] = vh; kb[hl] = vl;
              }
            }
          }
          if (edge_row) {
            // edge rows of the three copies, plain layout (pitch W)
            const long long cs = (long long)C * W;
            for (int e = 0; e < 2; ++e) {
              if (r != (e == 0 ? H - 1 : 0)) continue;
              float* qb = rowbuf + ((long long)(e * 3) * C + c) * W + x4 * 4;
              store_hl4(qb, hl, h, l, 0);
              if (!defer) {
                store_hl4(qb + cs, hl, h, l, 1);
                store_hl4(qb + 2 * cs, hl, h, l, 2);
              } else {
                float* q1 = qb + cs;
                float* q2 = qb + 2 * cs;
                q1[0] = h[1]; q1[1] = h[2]; q1[2] = h[3];
                q1[hl] = l[1]; q1[hl + 1] = l[2]; q1[hl + 2] = l[3];
                q2[0] = h[2]; q2[1] = h[3];
                q2[hl] = l[2]; q2[hl + 1] = l[3];
              }
              if (fix_prev) {
                float* q1 = qb + cs - 4;
                float* q2 = qb + 2 * cs - 4;
                q1[3] = h[0]; q1[hl + 3] = l[0];
                q2[2] = h[0]; q2[hl + 2] = l[0];
                q2[3] = h[1]; q2[hl + 3] = l[1];
              }
            }
          }
        }
        radix_add(c0, r0, x0, dcC, drC, dxC, H, W4);
        if (kShuffle) {                              // the raw chunk was read until here
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
        }
        next_chunk();
      }
    }
  }
  __syncthreads();
  tl_end(tl);
}

// Plans one layer: the same routine choice as launch_stage_conv (x assumed 16-byte aligned;
// the caller checks).  Appends to items[list] when items != nullptr, always counts.
// lists: [0] phase 0, register kernel; [1] phase 1 (after the batch means; also the light
// phase-0 routines when the TMA kernel takes the heavy ones); [2] phase 0, TMA kernel
static bool stage_tma_enabled(int B) {
  return tma_box_rows(B) > 0 && tma_ring_stages(B) >= kTmaGroups;
}

// role: 0 = plain; 1 = this flat 1x1 job also writes the stride-2 subsample of a sibling job
// (kStFlatSub); 2 = this job is that sibling (no items of its own)
static bool stage_sub_pair_ok(const ConvGeom& sub, const ConvGeom& full, int B);
static void plan_stage_job(const ConvGeom& g, int job, int B, bool have_mean,
                           std::vector<StageItem>* items /* [3] or null */, size_t* counts,
                           int role = 0) {
  if (role == 2) return;
  const long long img = (long long)g.C * g.H * g.W;
  const bool aligned = img % 4 == 0;
  const bool tma = stage_tma_enabled(B);
  const bool tma_job = tma && img % 256 == 0;
  auto add = [&](int list, int kind, int from_mean, long long total, long long chunk) {
    for (long long lo = 0; lo < total; lo += chunk) {
      ++counts[list];
      if (items) {
        StageItem it{};
        it.job = job; it.kind = (short)kind; it.from_mean = (short)from_mean;
        it.lo = lo; it.hi = lo + chunk < total ? lo + chunk : total;
        items[list].push_back(it);
      }
    }
  };
  const long long kVec = 2048, kScalar = 8192;
  const long long kTma = 32LL * 64 * (tma ? tma_box_rows(B) : 1);    // 32 stages per item
  const int light = tma ? 1 : 0;       // light phase-0 routines ride with phase 1 under TMA
  const bool two_pass_ok = B > 1 && aligned && have_mean;
  if (g.mode == kModeAutocorr) {
    if (aligned && g.W % 4 == 0 && (g.tiled || g.Ws == g.W + 4)) {
      if (tma_job && g.tiled) {
        add(2, kStAcVec, 0, img / 4, kTma);      // writes the edge columns and corners too
        return;
      } else {
        const long long n = g.tiled ? (long long)ac_cblocks(g) * 128 * g.Hs * (ac_strips(g) * 8)
                                    : (long long)g.C * g.Hs * (g.Ws / 4);
        add(0, kStAcVec, 0, round_up(n, 32), kVec);
      }
    } else {
      const long long n = g.tiled ? 3LL * ac_cblocks(g) * 128 * g.Hs * ac_strips(g) * 32
                                  : (long long)g.C * g.Hs * g.Ws * 3;
      if (two_pass_ok) {
        if (tma_job) add(2, kStMean, 0, img / 4, kTma); else add(0, kStMean, 0, img / 4, kVec);
        add(1, kStAcScalar, 1, n, kScalar);
      } else {
        add(light, kStAcScalar, 0, n, kScalar);
      }
    }
    add(light, kStAcEdges, 0, 6LL * g.C * ac_col_pitch(g) + 16LL * g.C, kVec);
    return;
  }
  if (g.mode == kModeFlat && g.sh == 1 && g.sw == 1 && aligned && (g.H * g.W) % 4 == 0) {
    if (tma_job) add(2, role == 1 ? kStFlatSub : kStFlatVec, 0, img / 4, kTma);
    else add(0, kStFlatVec, 0, img / 4, kVec);
    return;
  }
  if (g.mode == kModeImplicit && g.kh == 3 && g.kw == 3 && g.sh == 1 && g.sw == 1 && g.ph == 1 &&
      g.pw == 1 && aligned && g.W % 4 == 0) {
    add(0, kSt3x3Vec, 0, round_up((long long)g.C * g.Hs * (g.W / 4), 32), kVec);
    return;
  }
  if (tma_job && g.mode == kModeImplicit && g.kh == 3 && g.kw == 3 && g.sh == 2 && g.sw == 2 &&
      g.ph == 1 && g.pw == 1 && g.W % 4 == 0 && g.nrowphase == 2 && g.rowphase_py[0] == 1 &&
      g.rowphase_py[1] == 0 && g.Ht == 1) {
    add(2, kStS2x3, 0, img / 4, kTma);              // no batch-mean pass, no gather
    return;
  }
  const bool sparse = g.mode == kModeFlat && g.sh * g.sw > 1;
  const bool two = two_pass_ok && !sparse;
  if (two) {
    if (tma_job) add(2, kStMean, 0, img / 4, kTma); else add(0, kStMean, 0, img / 4, kVec);
  }
  if (g.mode == kModeExplicit) {
    // one item never crosses an im2col row (stage_conv_explicit_row_body)
    const long long w4 = g.Ws / 4;
    for (int row = 0; row < g.Cs; ++row)
      for (long long lo = 0; lo < w4; lo += kVec) {
        ++counts[two ? 1 : light];
        if (items) {
          StageItem it{};
          it.job = job; it.kind = (short)kStExplicit; it.from_mean = (short)(two ? 1 : 0);
          it.lo = row * w4 + lo;
          it.hi = row * w4 + (lo + kVec < w4 ? lo + kVec : w4);
          items[two ? 1 : light].push_back(it);
        }
      }
  } else
    add(two ? 1 : light, kStConv, two ? 1 : 0, (long long)g.Cs * g.Hs * g.ncopy * (g.Ws / 4), kVec);
}

namespace tc { int sm_count(); }
using tc::sm_count;

// a 1x1 stride-2 conv (`sub`) and a 1x1 stride-1 conv (`full`) on the same tensor: the staged
// operand of the first is every other row / column of the staged operand of the second, so
// the TMA consumer that stages `full` writes it along (no second read of the input)
static bool stage_sub_pair_ok(const ConvGeom& sub, const ConvGeom& full, int B) {
  const long long img = (long long)full.C * full.H * full.W;
  return stage_tma_enabled(B) && img % 256 == 0 && full.W % 4 == 0 && full.mode == kModeFlat &&
         sub.mode == kModeFlat && full.sh == 1 && full.sw == 1 && sub.sh == 2 && sub.sw == 2 &&
         sub.C == full.C && sub.H == full.H && sub.W == full.W && sub.Wout * 2 == full.W;
}

size_t stage_group_bytes(const ConvGeom* geoms, int n, int B) {
  size_t counts[3] = {0, 0, 0};
  for (int i = 0; i < n; ++i) plan_stage_job(geoms[i], i, B, true, nullptr, counts);
  return (size_t)n * sizeof(StageJobDev) + (counts[0] + counts[1] + counts[2]) * sizeof(StageItem) +
         (size_t)n * sizeof(void*) + (size_t)n * sizeof(CUtensorMap) + 2048;
}

// input pointers last uploaded into a staging table (the upload and the tensor-map encodes
// are skipped when a launch sees the same pointers again)
static std::mutex g_upload_mu;
static std::unordered_map<const void*, std::vector<const void*>> g_uploaded;

int stage_group_build(const ConvGeom* geoms, float* const* stages, float* const* means, int n,
                      int B, const int* same_input, void* table_dev, size_t table_bytes,
                      StageGroupInfo* info, cudaStream_t stream) {
  NSGP_REQUIRE((reinterpret_cast<uintptr_t>(table_dev) & 127) == 0,
               "stage group table must be 128-byte aligned");
  {
    std::lock_guard<std::mutex> lk(g_upload_mu);
    g_uploaded.erase(table_dev);
  }
  std::vector<StageJobDev> jobs(n);
  std::vector<StageItem> items[3];
  size_t counts[3] = {0, 0, 0};
  // pairs (1x1 s2 job, 1x1 s1 job on the same tensor): role[i] = 2, role[k] = 1, sub_of[k] = i
  std::vector<int> role(n, 0), sub_of(n, -1);
  for (int i = 0; i < n && same_input; ++i) {
    const int k = same_input[i];
    if (k < 0 || k >= n || k == i || role[i] || role[k]) continue;
    if (stage_sub_pair_ok(geoms[i], geoms[k], B)) { role[i] = 2; role[k] = 1; sub_of[k] = i; }
  }
  for (int i = 0; i < n; ++i) {
    const ConvGeom& g = geoms[i];
    StageJobDev& j = jobs[i];
    memset(&j, 0, sizeof(j));
    j.g = g;
    j.stage = stages[i];
    j.mean = means[i];
    j.hl = stage_hl_stride(g);
    if (g.mode == kModeAutocorr) {
      j.rowbuf_off = ac_rowbuf_off(g);
      j.colbuf_off = ac_colbuf_off(g);
      j.cornerbuf_off = ac_cornerbuf_off(g);
      j.Hc = ac_col_pitch(g);
    }
    if (role[i] == 1) {
      const ConvGeom& sg = geoms[sub_of[i]];
      j.sub_stage = stages[sub_of[i]];
      j.sub_hl = stage_hl_stride(sg);
      j.sub_pitch = sg.Ws;
      j.sub_wout = sg.Wout;
      // the zero tail of the rows (Hout * Wout .. Ws) is written here, once per table
      NSGP_CHECK_CUDA(cudaMemsetAsync(stages[sub_of[i]], 0, stage_bytes(sg), stream));
    }
    const size_t before = items[2].size();
    plan_stage_job(g, i, B, means[i] != nullptr, items, counts, role[i]);
    // the TMA autocorrelation / stride-2 routines write the data words only: the padding of
    // the layouts (halo rows, columns past the row end, channels >= C) is zeroed here, once
    // per table
    if (items[2].size() > before &&
        (items[2][before].kind == kStAcVec || items[2][before].kind == kStS2x3))
      NSGP_CHECK_CUDA(cudaMemsetAsync(stages[i], 0, stage_bytes(g), stream));
  }
  info->n_jobs = n;
  info->B = B;
  info->off_jobs = 0;
  size_t off = round_up((long long)((size_t)n * sizeof(StageJobDev)), 64);
  for (int ph = 0; ph < 2; ++ph) {
    info->n_items[ph] = (int)items[ph].size();
    info->off_items[ph] = off;
    off = round_up((long long)(off + items[ph].size() * sizeof(StageItem)), 64);
  }
  info->n_items_tma = (int)items[2].size();
  info->pad = 0;
  info->off_items_tma = off;
  off = round_up((long long)(off + items[2].size() * sizeof(StageItem)), 64);
  info->off_xs = off;
  off = round_up((long long)(off + (size_t)n * sizeof(void*)), 128);
  info->off_maps = off;
  off += (size_t)n * sizeof(CUtensorMap);
  info->bytes = off;
  NSGP_REQUIRE(off <= table_bytes, "stage group table too small (%zu < %zu)", table_bytes, off);
  char* t = (char*)table_dev;
  NSGP_CHECK_CUDA(cudaMemcpyAsync(t, jobs.data(), (size_t)n * sizeof(StageJobDev),
                                  cudaMemcpyHostToDevice, stream));
  for (int ph = 0; ph < 3; ++ph) {
    const size_t o = ph < 2 ? info->off_items[ph] : info->off_items_tma;
    if (!items[ph].empty())
      NSGP_CHECK_CUDA(cudaMemcpyAsync(t + o, items[ph].data(),
                                      items[ph].size() * sizeof(StageItem),
                                      cudaMemcpyHostToDevice, stream));
  }
  return 0;
}

// Per launch: the current input pointers and, for the TMA kernel, one 3-D tensor map per job
// over that input (geoms: the geometries the table was built for; null: no TMA items).
int stage_group_upload(const void* table_dev, const StageGroupInfo& info, const void* const* xs,
                       cudaStream_t stream, const ConvGeom* geoms) {
  if (info.n_jobs == 0) return 0;
  const char* t = (const char*)table_dev;
  for (int i = 0; i < info.n_jobs; ++i)
    NSGP_REQUIRE(xs[i] && (reinterpret_cast<uintptr_t>(xs[i]) & 15) == 0,
                 "stage group: input %d must be a 16-byte aligned device pointer", i);
  {
    std::lock_guard<std::mutex> lk(g_upload_mu);
    std::vector<const void*>& last = g_uploaded[table_dev];
    if ((int)last.size() == info.n_jobs && std::equal(last.begin(), last.end(), xs)) return 0;
    last.assign(xs, xs + info.n_jobs);
  }
  NSGP_CHECK_CUDA(cudaMemcpyAsync((void*)(t + info.off_xs), xs,
                                  (size_t)info.n_jobs * sizeof(void*), cudaMemcpyHostToDevice,
                                  stream));
  if (info.n_items_tma > 0) {
    NSGP_REQUIRE(geoms != nullptr, "stage group: the TMA staging needs the job geometries");
    std::vector<CUtensorMap> maps(info.n_jobs);
    memset(maps.data(), 0, maps.size() * sizeof(CUtensorMap));
    const int rows = tma_box_rows(info.B);
    for (int i = 0; i < info.n_jobs; ++i) {
      const long long img = (long long)geoms[i].C * geoms[i].H * geoms[i].W;
      if (img % 256 != 0) continue;               // this job has no TMA items
      int rc = encode_batch_rows_map(&maps[i], (const float*)xs[i], img, info.B, rows);
      if (rc) return rc;
    }
    NSGP_CHECK_CUDA(cudaMemcpyAsync((void*)(t + info.off_maps), maps.data(),
                                    maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice,
                                    stream));
  }
  return 0;
}

// TMA-fed phase 0: one CTA per SM (its 32 KB stages fill the SM's shared memory, so no other
// block joins it); sms > 0 confines it to that many SMs, pdl as for the other phases
int stage_group_launch_tma(const void* table_dev, const StageGroupInfo& info, int pdl, int sms,
                           cudaStream_t stream) {
  if (info.n_items_tma == 0) return 0;
  const char* t = (const char*)table_dev;
  const size_t smem = stage_tma_smem_bytes();
  const int B = info.B, rows = tma_box_rows(B);
  using Kernel = void (*)(const StageJobDev*, const StageItem*, int, const CUtensorMap*, int, int,
                          int, unsigned long long*);
  Kernel kernel = stage_tma_kernel<0, 0>;
  if (B == 8 && rows == 4) kernel = stage_tma_kernel<8, 4>;
  else if (B == 16 && rows == 3) kernel = stage_tma_kernel<16, 3>;
  else if (B == 4 && rows == 8) kernel = stage_tma_kernel<4, 8>;
  else if (B == 2 && rows == 8) kernel = stage_tma_kernel<2, 8>;
  else if (B == 1 && rows == 8) kernel = stage_tma_kernel<1, 8>;
  static const bool configured = [smem] {
    bool ok = true;
    for (Kernel k : {(Kernel)stage_tma_kernel<0, 0>, (Kernel)stage_tma_kernel<8, 4>,
                     (Kernel)stage_tma_kernel<16, 3>, (Kernel)stage_tma_kernel<4, 8>,
                     (Kernel)stage_tma_kernel<2, 8>, (Kernel)stage_tma_kernel<1, 8>})
      ok = ok && cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem) == cudaSuccess;
    return ok;
  }();
  NSGP_REQUIRE(configured, "stage_tma_kernel: %zu bytes of shared memory refused", smem);
  ProfScope prof(kProfStage, stream);
  int cap = sms > 0 ? sms : sm_count();
  int grid = info.n_items_tma < cap ? info.n_items_tma : cap;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kTmaThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  NSGP_CHECK_CUDA(cudaLaunchKernelEx(
      &cfg, kernel, reinterpret_cast<const StageJobDev*>(t + info.off_jobs),
      reinterpret_cast<const StageItem*>(t + info.off_items_tma), info.n_items_tma,
      reinterpret_cast<const CUtensorMap*>(t + info.off_maps), B, rows,
      tma_ring_stages(B), timeline_slot(2)));
  NSGP_LAUNCHED();
  return 0;
}

// One phase of the grouped staging (register kernel).  sms > 0: the launch is confined to
// `sms` SMs - every block asks for kStagePartSmem bytes of (unused) dynamic shared memory,
// which does not fit next to a resident contraction CTA (>= 225 KB), so the blocks only land
// on the SMs the contraction grid left free; pdl: launched with the programmatic
// stream-serialization attribute, i.e. it starts while the kernel queued before it is still
// running.
// Blocks per SM: 4 x 256 threads x 64 registers fill the register file (the gather routines
// are latency-bound: phase 1 0.58 -> 0.53 ms from 3 to 4 blocks; issuing the loads of two
// positions per iteration was measured too: spills, 0.58 ms).
constexpr int kStageBlocksPerSm = 4;
constexpr size_t kStagePartSmem = 8 * 1024;
int stage_group_launch_phase(const void* table_dev, const StageGroupInfo& info, int ph, int pdl,
                             int sms, cudaStream_t stream) {
  if (info.n_jobs == 0 || info.n_items[ph] == 0) return 0;
  const char* t = (const char*)table_dev;
  ProfScope prof(kProfStage, stream);
  int cap = (sms > 0 ? sms : sm_count()) * kStageBlocksPerSm;
  int grid = info.n_items[ph] < cap ? info.n_items[ph] : cap;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(256);
  cfg.dynamicSmemBytes = sms > 0 ? kStagePartSmem : 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  NSGP_CHECK_CUDA(cudaLaunchKernelEx(
      &cfg, stage_group_kernel, reinterpret_cast<const StageJobDev*>(t + info.off_jobs),
      reinterpret_cast<const StageItem*>(t + info.off_items[ph]), info.n_items[ph],
      reinterpret_cast<const float* const*>(t + info.off_xs), info.B, timeline_slot(2)));
  NSGP_LAUNCHED();
  return 0;
}

int stage_group_launch(const void* table_dev, const StageGroupInfo& info, const void* const* xs,
                       cudaStream_t stream, const ConvGeom* geoms) {
  int rc = stage_group_upload(table_dev, info, xs, stream, geoms);
  if (rc) return rc;
  rc = stage_group_launch_tma(table_dev, info, 0, 0, stream);
  if (rc) return rc;
  for (int ph = 0; ph < 2; ++ph) {
    rc = stage_group_launch_phase(table_dev, info, ph, 0, 0, stream);
    if (rc) return rc;
  }
  return 0;
}

// ---------------------------------------------------------------------------
// Linear input (R, d) -> batch-mean row m (d)  [nsrunner_roi_replay.py:901],
// then the rank-1 update acc += m m^T on the upper block-triangle.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
row_mean_kernel(const float* __restrict__ x, float* __restrict__ m, int R, int d) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d) return;
  float s = 0.f;
  for (int r = 0; r < R; ++r) s += __ldg(x + (long long)r * d + j);
  m[j] = s / (float)R;
}

__global__ void __launch_bounds__(256)
rank1_update_kernel(const float* __restrict__ m, float* __restrict__ acc, int d, int ld) {
  // 2D grid: blockIdx.y = row, threads over columns in float4 groups (ld % 4 == 0).
  int i = blockIdx.y;
  int j4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (j4 >= d) return;
  // only the upper block-triangle (128-row blocks) is maintained
  if (j4 + 3 < (i / 128) * 128) return;
  float mi = __ldg(m + i);
  float4* p = reinterpret_cast<float4*>(acc + (long long)i * ld + j4);
  float4 a = *p;
  a.x += mi * __ldg(m + j4);
  if (j4 + 1 < d) a.y += mi * __ldg(m + j4 + 1);
  if (j4 + 2 < d) a.z += mi * __ldg(m + j4 + 2);
  if (j4 + 3 < d) a.w += mi * __ldg(m + j4 + 3);
  *p = a;
}

int launch_linear_cov(const float* x, int R, int d, float* acc, int ld, float* mean_ws,
                      cudaStream_t stream) {
  row_mean_kernel<<<ceil_div(d, 256), 256, 0, stream>>>(x, mean_ws, R, d);
  NSGP_LAUNCHED();
  dim3 grid(ceil_div(ceil_div(d, 4), 256), d);
  rank1_update_kernel<<<grid, 256, 0, stream>>>(mean_ws, acc, d, ld);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Finalize: tap-major upper block-triangle accumulator -> reference-order dense
// symmetric covariance.  out[c*T+t][c'*T+t'] (+)= acc[min][max] with
// row' = t*C + c.  32x32 smem-tiled so both sides stay coalesced.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cov_finalize_kernel(const float* __restrict__ acc, int ld, float* __restrict__ out, int C,
                    int T, int d, int accumulate) {
  // one thread per output element, output-coalesced; the accumulator read is a
  // gather (stride T) that stays inside L2 - this runs once per task.
  long long total = (long long)d * d;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int col = (int)(idx % d), row = (int)(idx / d);
    int ri = (row % T) * C + row / T;   // reference (c,t) -> internal (t,c)
    int ci = (col % T) * C + col / T;
    int lo_i = ri < ci ? ri : ci, hi_i = ri < ci ? ci : ri;
    float v = acc[(long long)lo_i * ld + hi_i];
    if (accumulate) v += out[idx];
    out[idx] = v;
  }
}

// Autocorrelation layout -> reference-order dense symmetric covariance (geometry.h).
__global__ void __launch_bounds__(256)
cov_finalize_autocorr_kernel(const float* __restrict__ acc, float* __restrict__ out, int C,
                             int ldc, int accumulate) {
  const int d = C * 9;
  const long long total = (long long)d * d;
  const long long mat = (long long)C * ldc;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(idx % d), row = (int)(idx / d);
    int a = row / 9, ta = row - a * 9, b = col / 9, tb = col - b * 9;
    if (ta > tb) { int t = ta; ta = tb; tb = t; t = a; a = b; b = t; }   // transpose
    const int i = ta / 3, j = ta - i * 3, i2 = tb / 3, j2 = tb - i2 * 3;
    const int dy = i2 - i, dx = j2 - j;
    const long long e = (long long)a * ldc + b;
    float v;
    if (dy == 0 && dx == 0) {            // R_0 is a Gram: only its upper block tiles exist
      const int lo_i = a < b ? a : b, hi_i = a < b ? b : a;
      v = acc[(long long)lo_i * ldc + hi_i];
    } else {
      v = acc[ac_ridx(dy, dx) * mat + e];
    }
    if (i == i2 && i == 0) v -= acc[(kAcRowBottom + dx) * mat + e];
    if (i == i2 && i == 2) v -= acc[(kAcRowTop + dx) * mat + e];
    if (j == j2 && j == 0) v -= acc[(kAcColRight + dy) * mat + e];
    if (j == j2 && j == 2) v -= acc[(kAcColLeft + dy) * mat + e];
    if (ta == tb && i != 1 && j != 1)
      v += acc[(kAcCorner + (i == 0 ? 0 : 2) + (j == 0 ? 0 : 1)) * mat + e];
    if (accumulate) v += out[idx];
    out[idx] = v;
  }
}

int launch_cov_finalize_autocorr(const float* acc, float* out, int C, int accumulate,
                                 cudaStream_t stream) {
  const long long total = 81LL * C * C;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  cov_finalize_autocorr_kernel<<<blocks, 256, 0, stream>>>(acc, out, C, (int)round_up(C, 4),
                                                          accumulate);
  NSGP_LAUNCHED();
  return 0;
}

int launch_cov_finalize(const float* acc, int ld, float* out, int C, int T, int accumulate,
                        cudaStream_t stream) {
  int d = C * T;
  long long total = (long long)d * d;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  cov_finalize_kernel<<<blocks, 256, 0, stream>>>(acc, ld, out, C, T, d, accumulate);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// tf32 split helpers for persistent operands (projector P, updates).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
split_kernel(const float* __restrict__ src, float* __restrict__ hi, float* __restrict__ lo,
             long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    float h, l;
    tf32_split(src[i], h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// dst(hi/lo)[n][k] = src[k][n]  (d x d), so that B = P^T is K-major for D = U * P.
__global__ void __launch_bounds__(256)
transpose_split_kernel(const float* __restrict__ src, float* __restrict__ hi,
                       float* __restrict__ lo, int d, int ld_dst) {
  __shared__ float tile[32][33];
  int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    int row = by + r, col = bx + tx;
    tile[r][tx] = (row < d && col < d) ? src[(long long)row * d + col] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    int row = bx + r, col = by + tx;   // transposed
    if (row < d && col < d) {
      float h, l;
      tf32_split(tile[tx][r], h, l);
      hi[(long long)row * ld_dst + col] = h;
      lo[(long long)row * ld_dst + col] = l;
    }
  }
}

__global__ void __launch_bounds__(256)
transpose_split_rect_kernel(const float* __restrict__ src, float* __restrict__ hi,
                            float* __restrict__ lo, int rows, int cols, int ld_dst) {
  __shared__ float tile[32][33];
  int bx = blockIdx.x * 32, by = blockIdx.y * 32;       // bx over cols, by over rows
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    int row = by + r, col = bx + tx;
    tile[r][tx] = (row < rows && col < cols) ? src[(long long)row * cols + col] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    int orow = bx + r, ocol = by + tx;                   // transposed: (col, row)
    if (orow < cols && ocol < rows) {
      float h, l;
      tf32_split(tile[tx][r], h, l);
      hi[(long long)orow * ld_dst + ocol] = h;
      lo[(long long)orow * ld_dst + ocol] = l;
    }
  }
}

__global__ void __launch_bounds__(256)
split_pitched_kernel(const float* __restrict__ src, float* __restrict__ hi,
                     float* __restrict__ lo, int rows, int cols, int ld_dst) {
  long long total = (long long)rows * ld_dst;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % ld_dst);
    long long r = i / ld_dst;
    float h = 0.f, l = 0.f;
    if (c < cols) tf32_split(src[r * cols + c], h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

int launch_transpose_split_rect(const float* src, float* hi, float* lo, int rows, int cols,
                                int ld_dst, cudaStream_t stream) {
  dim3 grid(ceil_div(cols, 32), ceil_div(rows, 32));
  transpose_split_rect_kernel<<<grid, 256, 0, stream>>>(src, hi, lo, rows, cols, ld_dst);
  NSGP_LAUNCHED();
  return 0;
}

int launch_split_pitched(const float* src, float* hi, float* lo, int rows, int cols, int ld_dst,
                         cudaStream_t stream) {
  long long total = (long long)rows * ld_dst;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  split_pitched_kernel<<<blocks, 256, 0, stream>>>(src, hi, lo, rows, cols, ld_dst);
  NSGP_LAUNCHED();
  return 0;
}

int launch_split(const float* src, float* hi, float* lo, long long n, cudaStream_t stream) {
  int blocks = (int)((n + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  split_kernel<<<blocks, 256, 0, stream>>>(src, hi, lo, n);
  NSGP_LAUNCHED();
  return 0;
}

int launch_transpose_split(const float* src, float* hi, float* lo, int d, int ld_dst,
                           cudaStream_t stream) {
  dim3 grid(ceil_div(d, 32), ceil_div(d, 32));
  transpose_split_kernel<<<grid, 256, 0, stream>>>(src, hi, lo, d, ld_dst);
  NSGP_LAUNCHED();
  return 0;
}

}  // namespace nsgp
