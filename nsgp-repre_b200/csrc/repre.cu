// RePRE prototype statistics: HBM-bound kernels (128-bit coalesced loads, warp
// shuffles, shared-memory staging).  Reference: StandardMultiPrototypeReplayHead
// (mmdet/models/roi_heads/standard_roi_replay_head.py:404-463).
#include "common.cuh"
#include "repre.h"
#include "tc_common.cuh"

namespace nsgp {

// ---------------------------------------------------------------------------
// Class index (stable): rows of class c in ascending row order, like the boolean
// mask gather feats[cls_targets == c] of the reference (:412-413).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
class_count_kernel(const long long* __restrict__ labels, int M, int* __restrict__ counts) {
  const int c = blockIdx.x;
  int n = 0;
  for (int i = threadIdx.x; i < M; i += 256) n += (labels[i] == c);
  __shared__ int red[8];
  for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < 8; ++w) s += red[w];
    counts[c] = s;
  }
}

__global__ void __launch_bounds__(256)
class_compact_kernel(const long long* __restrict__ labels, int M, int C,
                     const int* __restrict__ counts, int* __restrict__ offsets,
                     int* __restrict__ rows) {
  const int c = blockIdx.x;
  __shared__ int warp_sums[8];
  __shared__ int base;
  if (threadIdx.x == 0) {
    int off = 0;
    for (int k = 0; k < c; ++k) off += counts[k];
    base = off;
    offsets[c] = off;
    if (c == C - 1) offsets[C] = off + counts[c];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int start = 0; start < M; start += 256) {
    int i = start + threadIdx.x;
    bool hit = (i < M) && (labels[i] == c);
    unsigned ballot = __ballot_sync(0xffffffffu, hit);
    int in_warp = __popc(ballot & ((1u << lane) - 1));
    if (lane == 0) warp_sums[warp] = __popc(ballot);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < 8; ++w) {
      int s = warp_sums[w];
      if (w < warp) before += s;
      total += s;
    }
    if (hit) rows[base + before + in_warp] = i;
    __syncthreads();
    if (threadIdx.x == 0) base += total;
    __syncthreads();
  }
}

int launch_class_index(const long long* labels, int M, int C, int* counts, int* offsets,
                       int* rows, cudaStream_t stream) {
  class_count_kernel<<<C, 256, 0, stream>>>(labels, M, counts);
  NSGP_LAUNCHED();
  class_compact_kernel<<<C, 256, 0, stream>>>(labels, M, C, counts, offsets, rows);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Segmented mean over gathered rows: out[s][:] = mean(F[rows[off[s]:off[s+1]]]).
// Used for the coarse class means (:412-414) and the masked fine-grained
// prototype means (:443).  mode 1: mean of squared deviations from mu[s]
// (extension: per-class diagonal covariance).
// grid = (column chunks of 64 threads x float4, segments, row splits).
// ---------------------------------------------------------------------------
constexpr int kSegThreads = 64;

template <int MODE>
__global__ void __launch_bounds__(kSegThreads)
segment_mean_kernel(const float* __restrict__ F, int D, const int* __restrict__ seg_off,
                    const int* __restrict__ rows, const float* __restrict__ mu,
                    float* __restrict__ out, const int* __restrict__ nseg_dev) {
  const int s = blockIdx.y;
  if (nseg_dev != nullptr && s >= *nseg_dev) return;   // grid sized for the maximum
  const int col = (blockIdx.x * kSegThreads + threadIdx.x) * 4;
  if (col >= D) return;
  const int beg = seg_off[s], end = seg_off[s + 1];
  const int n = end - beg;
  // row split: contiguous slices so that S == 1 keeps the plain sequential order
  const int per = (n + gridDim.z - 1) / gridDim.z;
  const int r0 = beg + blockIdx.z * per;
  const int r1 = min(end, r0 + per);
  float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (MODE == 1) m4 = *reinterpret_cast<const float4*>(mu + (long long)s * D + col);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int r = r0;
  for (; r + 8 <= r1; r += 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u)
      v[u] = __ldg(reinterpret_cast<const float4*>(F + (long long)rows[r + u] * D + col));
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (MODE == 1) {
        float a = v[u].x - m4.x, b = v[u].y - m4.y, c = v[u].z - m4.z, d = v[u].w - m4.w;
        acc.x += a * a; acc.y += b * b; acc.z += c * c; acc.w += d * d;
      } else {
        acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
      }
    }
  }
  for (; r < r1; ++r) {
    float4 v = __ldg(reinterpret_cast<const float4*>(F + (long long)rows[r] * D + col));
    if (MODE == 1) {
      float a = v.x - m4.x, b = v.y - m4.y, c = v.z - m4.z, d = v.w - m4.w;
      acc.x += a * a; acc.y += b * b; acc.z += c * c; acc.w += d * d;
    } else {
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  const float fn = (float)n;   // n == 0 -> NaN like torch.mean of an empty slice
  float* o = out + (long long)s * D + col;
  if (gridDim.z == 1) {
    *reinterpret_cast<float4*>(o) = make_float4(acc.x / fn, acc.y / fn, acc.z / fn, acc.w / fn);
  } else if (r1 > r0 || (n == 0 && blockIdx.z == 0)) {
    atomicAdd(o + 0, acc.x / fn);
    atomicAdd(o + 1, acc.y / fn);
    atomicAdd(o + 2, acc.z / fn);
    atomicAdd(o + 3, acc.w / fn);
  }
}

// zero the rows the row-split means add into: the live ones only when the segment count is
// read on the device, so that the rows past it keep whatever the caller left there
__global__ void __launch_bounds__(256)
zero_live_rows_kernel(float* __restrict__ out, int D, int nseg, const int* __restrict__ nseg_dev) {
  const long long n4 = (long long)min(*nseg_dev, nseg) * (D / 4);
  float4* o = reinterpret_cast<float4*>(out);
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256)
    o[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

int launch_segment_mean(const float* F, int D, const int* seg_off, const int* rows, int nseg,
                        int max_seg_rows, const float* mu, int mode, float* out,
                        cudaStream_t stream, const int* nseg_dev) {
  NSGP_REQUIRE(D % 4 == 0, "segment_mean: D must be a multiple of 4");
  if (nseg == 0) return 0;
  int chunks = ceil_div(D, kSegThreads * 4);
  int splits = 1;
  // fill the 148 SMs a few times over when there are few / long segments (row-split partial
  // means meet by atomicAdd, so deterministic mode keeps one sequential pass per segment)
  while (!g_deterministic && splits < 32 && (long long)chunks * nseg * splits < 148 * 8 &&
         max_seg_rows / (splits * 2) >= 16)
    splits *= 2;
  if (splits > 1 && nseg_dev == nullptr) {
    NSGP_CHECK_CUDA(cudaMemsetAsync(out, 0, (size_t)nseg * D * sizeof(float), stream));
  } else if (splits > 1) {
    const int blocks = (int)std::min<long long>(ceil_div((long long)nseg * (D / 4), 256), 148 * 4);
    zero_live_rows_kernel<<<blocks, 256, 0, stream>>>(out, D, nseg, nseg_dev);
    NSGP_LAUNCHED();
  }
  dim3 grid(chunks, nseg, splits);
  ProfScope prof(kProfRepre, stream);
  if (mode == 1)
    segment_mean_kernel<1><<<grid, kSegThreads, 0, stream>>>(F, D, seg_off, rows, mu, out,
                                                             nseg_dev);
  else
    segment_mean_kernel<0><<<grid, kSegThreads, 0, stream>>>(F, D, seg_off, rows, mu, out,
                                                             nseg_dev);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// L2-normalise gathered rows and split into tf32 hi/lo (:417): one CTA per row,
// the row (<= 50 KB) is re-read from L1/L2 for the second pass.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
normalize_split_kernel(const float* __restrict__ F, int D, const int* __restrict__ rows,
                       float* __restrict__ hi, float* __restrict__ lo) {
  const int i = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(F + (long long)rows[i] * D);
  const int n4 = D >> 2;
  float ss = 0.f;
  for (int j = threadIdx.x; j < n4; j += 256) {
    float4 v = __ldg(src + j);
    ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  __shared__ float red[8];
  __shared__ float norm_s;
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    norm_s = sqrtf(t);
  }
  __syncthreads();
  const float nrm = norm_s;
  float4* dh = reinterpret_cast<float4*>(hi + (long long)i * D);
  float4* dl = reinterpret_cast<float4*>(lo + (long long)i * D);
  for (int j = threadIdx.x; j < n4; j += 256) {
    float4 v = __ldg(src + j), h, l;
    tf32_split(v.x / nrm, h.x, l.x);
    tf32_split(v.y / nrm, h.y, l.y);
    tf32_split(v.z / nrm, h.z, l.z);
    tf32_split(v.w / nrm, h.w, l.w);
    dh[j] = h;
    dl[j] = l;
  }
}

int launch_normalize_split(const float* F, int D, const int* rows, int n, float* hi, float* lo,
                           cudaStream_t stream) {
  NSGP_REQUIRE(D % 4 == 0, "normalize: D must be a multiple of 4");
  if (n == 0) return 0;
  normalize_split_kernel<<<n, 256, 0, stream>>>(F, D, rows, hi, lo);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Threshold + neighbour count (:420-421) on the upper block-triangular Gram
// produced by the contraction engine: one warp per row.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
threshold_count_kernel(const float* __restrict__ S, int n, int ld, float thresh,
                       unsigned char* __restrict__ mask, int* __restrict__ counts,
                       float* __restrict__ sim_out) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  int cnt = 0;
  for (int j = lane; j < n; j += 32) {
    float v = (i <= j) ? S[(long long)i * ld + j] : S[(long long)j * ld + i];
    bool m = v >= thresh;
    mask[(long long)i * n + j] = m ? 1 : 0;
    if (sim_out) sim_out[(long long)i * n + j] = v;
    cnt += m;
  }
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) counts[i] = cnt;
}

// batched over classes: blockIdx.y = class, per-class extents from a small device table
__global__ void __launch_bounds__(256)
threshold_count_batched_kernel(const float* __restrict__ S_all,
                               const ClassExtent* __restrict__ ext, float thresh,
                               unsigned char* __restrict__ mask_all,
                               int* __restrict__ counts_all) {
  const ClassExtent e = ext[blockIdx.y];
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= e.n) return;
  const float* S = S_all + e.s_off;
  unsigned char* mask = mask_all + e.mask_off;
  int cnt = 0;
  for (int j = lane; j < e.n; j += 32) {
    float v = (i <= j) ? S[(long long)i * e.ld + j] : S[(long long)j * e.ld + i];
    bool m = v >= thresh;
    mask[(long long)i * e.n + j] = m ? 1 : 0;
    cnt += m;
  }
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) counts_all[e.row_off + i] = cnt;
}

int launch_threshold_count_batched(const float* S_all, const ClassExtent* ext_dev, int n_classes,
                                   int max_n, float thresh, unsigned char* mask_all,
                                   int* counts_all, cudaStream_t stream) {
  if (n_classes == 0 || max_n == 0) return 0;
  dim3 grid(ceil_div(max_n, 8), n_classes);
  threshold_count_batched_kernel<<<grid, 256, 0, stream>>>(S_all, ext_dev, thresh, mask_all,
                                                           counts_all);
  NSGP_LAUNCHED();
  return 0;
}

int launch_threshold_count(const float* S, int n, int ld, float thresh, unsigned char* mask,
                           int* counts, float* sim_out, cudaStream_t stream) {
  if (n == 0) return 0;
  threshold_count_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(S, n, ld, thresh, mask, counts,
                                                             sim_out);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Density ordering + greedy cover (:421-448) on the device: one CTA per class.
//   order  = stable descending sort of the neighbour counts (torch's CPU sort is stable:
//            equal counts keep ascending row order), rank by counting - n is hundreds
//   thr    = sorted[-n // 3]  (python floor division: index n - ceil(n/3))
//   covered= count <= thr;  then up to max_picks times: the first not-covered row in
//            density order becomes a prototype seed, its neighbour mask is OR-ed into
//            covered (:430-448).  Masks replayed from mask.pth come first (:425-433).
// Outputs per class: picks (row within the class, -2 = replayed mask), npicks, and the
// segment sizes [n, popcount(mask_0), ...] that the segment table is built from.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
greedy_cover_kernel(const GreedyClass* __restrict__ cls, const unsigned char* __restrict__ masks,
                    const int* __restrict__ counts, const unsigned char* __restrict__ saved,
                    int max_picks, int* __restrict__ order_ws,
                    unsigned char* __restrict__ covered_ws, int* __restrict__ picks,
                    int* __restrict__ npicks, int* __restrict__ seg_sizes) {
  const int ci = blockIdx.x;
  const GreedyClass e = cls[ci];
  const int n = e.n, tid = threadIdx.x;
  const int* cnt = counts + e.row_off;
  const unsigned char* mask = masks + e.mask_off;
  int* order = order_ws + e.row_off;
  unsigned char* cov = covered_ws + e.row_off;
  __shared__ int s_best, s_red[8];
  if (n == 0) {                       // empty class: reported through the plan's status word
    if (tid == 0) { npicks[ci] = 0; seg_sizes[ci * (max_picks + 1)] = 0; }
    return;
  }
  for (int i = tid; i < n; i += 256) {
    const int ci_cnt = cnt[i];
    int r = 0;
    for (int j = 0; j < n; ++j) {
      const int cj = cnt[j];
      r += (cj > ci_cnt) || (cj == ci_cnt && j < i);
    }
    order[r] = i;
  }
  __syncthreads();
  const int thr = cnt[order[n - (n + 2) / 3]];
  for (int i = tid; i < n; i += 256) cov[i] = cnt[i] <= thr ? 1 : 0;
  if (tid == 0) seg_sizes[ci * (max_picks + 1)] = n;
  __syncthreads();
  int np = 0;
  for (int p = 0; p < max_picks; ++p) {
    const unsigned char* m;
    int pick;
    if (p < e.n_saved) {
      m = saved + e.saved_off + (long long)p * n;
      pick = -2;
    } else {
      if (tid == 0) s_best = 0x7fffffff;
      __syncthreads();
      for (int r = tid; r < n; r += 256)
        if (!cov[order[r]]) { atomicMin(&s_best, r); break; }
      __syncthreads();
      const int best = s_best;
      __syncthreads();
      if (best == 0x7fffffff) break;              // nothing left to cover (uniform)
      pick = order[best];
      m = mask + (long long)pick * n;
    }
    int local = 0;
    for (int i = tid; i < n; i += 256)
      if (m[i]) { cov[i] = 1; ++local; }
    for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((tid & 31) == 0) s_red[tid >> 5] = local;
    __syncthreads();
    if (tid == 0) {
      int t = 0;
      for (int w = 0; w < 8; ++w) t += s_red[w];
      picks[ci * max_picks + np] = pick;
      seg_sizes[ci * (max_picks + 1) + 1 + np] = t;
    }
    ++np;
    __syncthreads();
  }
  if (tid == 0) npicks[ci] = np;
}

// segment numbering and row offsets over all classes (one block; classes are few)
__global__ void __launch_bounds__(256)
segment_table_kernel(const GreedyClass* __restrict__ cls, int n_classes, int max_picks,
                     const int* __restrict__ npicks, const int* __restrict__ seg_sizes,
                     int* __restrict__ seg_base, int* __restrict__ seg_off,
                     int* __restrict__ seg_label, int* __restrict__ nseg_out) {
  __shared__ int s_nseg;
  if (threadIdx.x == 0) {
    int sb = 0;
    for (int ci = 0; ci < n_classes; ++ci) { seg_base[ci] = sb; sb += 1 + npicks[ci]; }
    s_nseg = sb;
    *nseg_out = sb;
  }
  __syncthreads();
  // row offset of a class = rows of all earlier classes' segments
  for (int ci = threadIdx.x; ci < n_classes; ci += blockDim.x) {
    int off = 0;
    for (int cj = 0; cj < ci; ++cj) {
      const int k = 1 + npicks[cj];
      for (int q = 0; q < k; ++q) off += seg_sizes[cj * (max_picks + 1) + q];
    }
    const int k = 1 + npicks[ci], b = seg_base[ci];
    for (int q = 0; q < k; ++q) {
      seg_off[b + q] = off;
      seg_label[b + q] = cls[ci].class_id;
      off += seg_sizes[ci * (max_picks + 1) + q];
    }
    if (ci == n_classes - 1) seg_off[s_nseg] = off;
  }
}

// rows of segment (class, slot): slot 0 = every row of the class, slot q > 0 = the rows
// under the q-th mask, ascending (the boolean-mask gather of :443)
__global__ void __launch_bounds__(256)
segment_rows_kernel(const GreedyClass* __restrict__ cls, const unsigned char* __restrict__ masks,
                    const unsigned char* __restrict__ saved, const int* __restrict__ rows_sel,
                    int max_picks, const int* __restrict__ picks, const int* __restrict__ npicks,
                    const int* __restrict__ seg_base, const int* __restrict__ seg_off,
                    int* __restrict__ seg_rows, const int* __restrict__ rows_base) {
  const int q = blockIdx.x, ci = blockIdx.y;
  if (q > npicks[ci]) return;
  const GreedyClass e = cls[ci];
  const int n = e.n;
  // rows_base: device offset of the first selected class in the row list (device-sized build)
  const int* src = rows_sel + (rows_base ? *rows_base : 0) + e.row_off;
  int* dst = seg_rows + seg_off[seg_base[ci] + q];
  if (q == 0) {
    for (int i = threadIdx.x; i < n; i += 256) dst[i] = src[i];
    return;
  }
  const int pick = picks[ci * max_picks + q - 1];
  const unsigned char* m = pick == -2 ? saved + e.saved_off + (long long)(q - 1) * n
                                      : masks + e.mask_off + (long long)pick * n;
  __shared__ int warp_sums[8];
  __shared__ int base;
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int start = 0; start < n; start += 256) {
    const int i = start + threadIdx.x;
    const bool hit = (i < n) && m[i];
    const unsigned ballot = __ballot_sync(0xffffffffu, hit);
    const int in_warp = __popc(ballot & ((1u << lane) - 1));
    if (lane == 0) warp_sums[warp] = __popc(ballot);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < 8; ++w) {
      const int sw = warp_sums[w];
      if (w < warp) before += sw;
      total += sw;
    }
    if (hit) dst[base + before + in_warp] = src[i];
    __syncthreads();
    if (threadIdx.x == 0) base += total;
    __syncthreads();
  }
}

int launch_greedy_segments(const GreedyClass* cls_dev, int n_classes, int max_n,
                           const unsigned char* masks, const int* counts,
                           const unsigned char* saved, const int* rows_sel, int max_picks,
                           int* order_ws, unsigned char* covered_ws, int* seg_sizes,
                           int* seg_base, int* picks, int* npicks, int* seg_off, int* seg_rows,
                           int* seg_label, int* nseg_out, cudaStream_t stream,
                           const int* rows_base) {
  if (n_classes == 0) return 0;
  ProfScope prof(kProfRepre, stream);
  greedy_cover_kernel<<<n_classes, 256, 0, stream>>>(cls_dev, masks, counts, saved, max_picks,
                                                     order_ws, covered_ws, picks, npicks,
                                                     seg_sizes);
  NSGP_LAUNCHED();
  segment_table_kernel<<<1, 256, 0, stream>>>(cls_dev, n_classes, max_picks, npicks, seg_sizes,
                                              seg_base, seg_off, seg_label, nseg_out);
  NSGP_LAUNCHED();
  dim3 grid(max_picks + 1, n_classes);
  segment_rows_kernel<<<grid, 256, 0, stream>>>(cls_dev, masks, saved, rows_sel, max_picks, picks,
                                                npicks, seg_base, seg_off, seg_rows, rows_base);
  NSGP_LAUNCHED();
  (void)max_n;
  return 0;
}

// ---------------------------------------------------------------------------
// Device-sized prototype build (repre_build_prototypes): nothing on the host ever learns a
// class size, so the build is a fixed sequence of launches with no read-back in the middle.
// ---------------------------------------------------------------------------
// Stable class index in ONE launch (a single CTA of 32 warps): warp w owns classes w, w+32,
// ...; it scans the labels 32 at a time - a ballot gives the class's rows of the chunk in
// ascending order - once to count, once (after the offsets are known) to compact.
constexpr int kCiTile = 8192;                 // labels per tile: 8 chunks of 32 per warp
constexpr int kCiMaxC = 256;                  // classes of the single-launch index
__global__ void __launch_bounds__(1024)
class_index_fused_kernel(const long long* __restrict__ labels, int M, int C,
                         int* __restrict__ counts, int* __restrict__ offsets,
                         int* __restrict__ rows) {
  // Warp w owns the labels [256 w, 256 w + 256) of every tile of 8192, in order.  For a chunk
  // of 32 labels __match_any_sync gives every lane the lanes holding the same class: its rank
  // among them is its position inside the chunk, the group's lowest lane adds the group size
  // to the (warp, class) counter.  A scan over the 32 warps per class turns the counters
  // into write positions, so rows of one class come out in ascending order (stable).
  extern __shared__ int ci_smem[];            // [C] running position, [32][C] per-warp counts
  int* s_run = ci_smem;
  int* s_wc = ci_smem + C;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1;
  for (int c = threadIdx.x; c < C; c += 1024) s_run[c] = 0;
  for (int pass = 0; pass < 2; ++pass) {
    for (int t0 = 0; t0 < M; t0 += kCiTile) {
      __syncthreads();
      for (int i = threadIdx.x; i < 32 * C; i += 1024) s_wc[i] = 0;
      __syncthreads();
      int lab[8], rank[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {           // all 8 loads of the lane in flight together
        const int i = t0 + warp * 256 + k * 32 + lane;
        const long long l = i < M ? labels[i] : -1;
        lab[k] = (l >= 0 && l < C) ? (int)l : -1;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const unsigned grp = __match_any_sync(0xffffffffu, lab[k]);
        rank[k] = 0;
        if (lab[k] >= 0) {
          rank[k] = s_wc[warp * C + lab[k]] + __popc(grp & lt);
          __syncwarp(grp);
          if ((grp & lt) == 0) s_wc[warp * C + lab[k]] += __popc(grp);
        }
        __syncwarp();
      }
      __syncthreads();
      // per class: exclusive scan of the warps' counts on top of the running position
      for (int c = threadIdx.x; c < C; c += 1024) {
        int run = s_run[c];
        for (int w = 0; w < 32; ++w) {
          const int n = s_wc[w * C + c];
          s_wc[w * C + c] = run;
          run += n;
        }
        s_run[c] = run;
      }
      __syncthreads();
      if (pass == 1) {
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (lab[k] >= 0)
            rows[s_wc[warp * C + lab[k]] + rank[k]] = t0 + warp * 256 + k * 32 + lane;
      }
    }
    if (pass == 0) {
      __syncthreads();
      if (threadIdx.x == 0) {
        int off = 0;
        for (int c = 0; c < C; ++c) {
          const int n = s_run[c];
          counts[c] = n; offsets[c] = off; s_run[c] = off;      // pass 1 starts at the offset
          off += n;
        }
        offsets[C] = off;
      }
    }
  }
}

int launch_class_index_fused(const long long* labels, int M, int C, int* counts, int* offsets,
                             int* rows, cudaStream_t stream) {
  if (C > kCiMaxC) return launch_class_index(labels, M, C, counts, offsets, rows, stream);
  ProfScope prof(kProfRepre, stream);
  const size_t smem = (size_t)(33 * C) * sizeof(int);
  class_index_fused_kernel<<<1, 1024, smem, stream>>>(labels, M, C, counts, offsets, rows);
  NSGP_LAUNCHED();
  return 0;
}

// Plan of one build, computed on the device from the class offsets: per-class extents for the
// threshold / greedy kernels, the tile pairs of the ONE Gram over all foreground rows (sorted
// by class: only tiles that contain a same-class pair are contracted), its work items and the
// row bounds of the Gram problem.
//   hdr[0] = n_fg, [1] = n_pairs, [2] = n_items, [3] = error (1: a class has no rows,
//   2: a replayed mask has the wrong length), [4] = K splits
__global__ void __launch_bounds__(256)
repre_plan_kernel(const int* __restrict__ offsets, int class_first, int n_classes, int ld_s,
                  const int* __restrict__ n_saved, const int* __restrict__ saved_len, int nkb,
                  int max_items, ClassExtent* __restrict__ ext, GreedyClass* __restrict__ cls,
                  int2* __restrict__ pairs, tc::TcItem* __restrict__ items,
                  tc::TcProblem* __restrict__ prob, int* __restrict__ hdr, int det) {
  __shared__ int s_npairs, s_splits;
  extern __shared__ int plan_smem[];          // [n_classes + 1] offsets, [n] n_saved, [n] saved_len
  int* s_o = plan_smem;
  int* s_ns = plan_smem + n_classes + 1;
  int* s_sl = s_ns + n_classes;
  // one parallel read of everything the (sequential) plan needs
  for (int k = threadIdx.x; k <= n_classes; k += blockDim.x) s_o[k] = offsets[class_first + k];
  for (int k = threadIdx.x; k < n_classes; k += blockDim.x) {
    s_ns[k] = n_saved ? n_saved[k] : 0;
    s_sl[k] = saved_len ? saved_len[k] : 0;
  }
  __syncthreads();
  const int base = s_o[0];
  if (threadIdx.x == 0) {
    int err = 0;
    long long moff = 0, soff = 0;
    for (int k = 0; k < n_classes; ++k) {
      const int a = s_o[k] - base, b = s_o[k + 1] - base;
      const int n = b - a;
      if (n == 0) err = 1;
      const int ns = s_ns[k];
      if (ns > 0 && s_sl[k] != n) err = 2;
      ext[k] = ClassExtent{(long long)a * ld_s + a, moff, a, n, ld_s, 0};
      cls[k] = GreedyClass{moff, soff, a, n, ns, class_first + k};
      moff += (long long)n * n;
      soff += (long long)ns * n;
    }
    const int n_fg = s_o[n_classes] - base;
    // tile pairs (rb <= cb) that hold a pair of rows of one class; classes are contiguous
    // and ascending, so cb_max(rb) is non-decreasing and comes from the classes touching rb
    int np = 0;
    const int tiles = (n_fg + 127) >> 7;
    int k = 0;
    for (int rb = 0; rb < tiles; ++rb) {
      int cb_max = rb;
      // classes intersecting tile rb: advance k to the first class that ends after the tile start
      while (k < n_classes && s_o[k + 1] - base <= rb * 128) ++k;
      for (int q = k; q < n_classes && s_o[q] - base < (rb + 1) * 128; ++q) {
        const int last = (s_o[q + 1] - base - 1) >> 7;
        if (s_o[q + 1] > s_o[q] && last > cb_max) cb_max = last;
      }
      for (int cb = rb; cb <= cb_max; ++cb) pairs[np++] = make_int2(rb, cb);
    }
    // K splits: the fp32 accumulation chain allows 64 K blocks; more splits when there are
    // few tile pairs, so that every SM gets a couple of items
    int splits = (nkb + 63) / 64;
    const int want = np > 0 ? (2 * 148) / np : 1;      // at most two full waves of items
    // deterministic mode: only the splits the chain bound needs (their partial tiles go to
    // slots and are summed in split order by repre_combine_tiles_kernel)
    if (want > splits && !det) splits = want;
    if (splits > nkb / 4 && !det) splits = nkb / 4 > 0 ? nkb / 4 : 1;
    while (np * splits > max_items && splits > 1) --splits;
    s_npairs = np;
    s_splits = splits;
    hdr[0] = n_fg; hdr[1] = np; hdr[2] = np * splits; hdr[3] = err; hdr[4] = splits;
    prob->p.A.rows = n_fg;
    prob->p.B.rows = n_fg;
    prob->p.n_cols = n_fg;
  }
  __syncthreads();
  const int np = s_npairs, splits = s_splits;
  for (int i = threadIdx.x; i < np * splits; i += blockDim.x) {
    const int sp = i / np, pr = i - sp * np;            // K-range-major: one K range of all
    const int2 t = pairs[pr];                           // tiles is in flight together
    const int kb0 = (int)((long long)nkb * sp / splits);
    const int kb1 = (int)((long long)nkb * (sp + 1) / splits);
    items[i] = tc::TcItem{0, t.x, t.y, kb0, kb1, det && splits > 1 ? i + 1 : 0, 0, 0};
  }
}

// deterministic mode: S tile of pair p += sum over the K splits of slots[sp * np + p], in split
// order (the plan gave item i = sp * np + p slot i)
__global__ void __launch_bounds__(256)
repre_combine_tiles_kernel(const int2* __restrict__ pairs, const int* __restrict__ hdr,
                           const float* __restrict__ slots, float* __restrict__ S, int ld_s) {
  const int np = hdr[1], n_fg = hdr[0], splits = hdr[4];
  if (splits <= 1) return;
  for (int p = blockIdx.x; p < np; p += gridDim.x) {
    const int2 t = pairs[p];
    for (int e = threadIdx.x; e < 128 * 32; e += 256) {
      const int r = t.x * 128 + (e >> 5), c = t.y * 128 + (e & 31) * 4;
      if (r >= n_fg || c >= ld_s) continue;
      const size_t off = (size_t)(e >> 5) * 128 + (e & 31) * 4;
      float4 s = *reinterpret_cast<const float4*>(slots + (size_t)p * kSlotElems + off);
      for (int sp = 1; sp < splits; ++sp) {
        const float4 v =
            *reinterpret_cast<const float4*>(slots + ((size_t)sp * np + p) * kSlotElems + off);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      float4* o = reinterpret_cast<float4*>(S + (long long)r * ld_s + c);
      float4 a = *o;
      a.x += s.x; a.y += s.y; a.z += s.z; a.w += s.w;
      *o = a;
    }
  }
}

// zero the Gram tiles the plan selected (the buffer is sized for the worst case; only the
// needed 128 x 128 tiles are touched)
__global__ void __launch_bounds__(256)
repre_clear_tiles_kernel(const int2* __restrict__ pairs, const int* __restrict__ hdr,
                         float* __restrict__ S, int ld_s) {
  const int np = hdr[1], n_fg = hdr[0];
  for (int p = blockIdx.x; p < np; p += gridDim.x) {
    const int2 t = pairs[p];
    for (int e = threadIdx.x; e < 128 * 32; e += 256) {
      const int r = t.x * 128 + (e >> 5), c = t.y * 128 + (e & 31) * 4;
      if (r < n_fg && c < ld_s)
        *reinterpret_cast<float4*>(S + (long long)r * ld_s + c) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// L2-normalise + tf32 split of the foreground rows, count read on the device
__global__ void __launch_bounds__(256)
normalize_split_dev_kernel(const float* __restrict__ F, int D, const int* __restrict__ rows,
                           const int* __restrict__ offsets, int class_first,
                           const int* __restrict__ hdr, float* __restrict__ hi,
                           float* __restrict__ lo) {
  const int i = blockIdx.x;
  if (i >= hdr[0]) return;
  const float4* src =
      reinterpret_cast<const float4*>(F + (long long)rows[offsets[class_first] + i] * D);
  const int n4 = D >> 2;
  float ss = 0.f;
  for (int j = threadIdx.x; j < n4; j += 256) {
    float4 v = __ldg(src + j);
    ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  __shared__ float red[8];
  __shared__ float norm_s;
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    norm_s = sqrtf(t);
  }
  __syncthreads();
  const float nrm = norm_s;
  float4* dh = reinterpret_cast<float4*>(hi + (long long)i * D);
  float4* dl = reinterpret_cast<float4*>(lo + (long long)i * D);
  for (int j = threadIdx.x; j < n4; j += 256) {
    float4 v = __ldg(src + j), h, l;
    tf32_split(v.x / nrm, h.x, l.x);
    tf32_split(v.y / nrm, h.y, l.y);
    tf32_split(v.z / nrm, h.z, l.z);
    tf32_split(v.w / nrm, h.w, l.w);
    dh[j] = h;
    dl[j] = l;
  }
}

// threshold + neighbour count, one warp per foreground row; the row's class comes from a
// binary search over the extents the plan wrote
__global__ void __launch_bounds__(256)
threshold_count_dev_kernel(const float* __restrict__ S_all, const ClassExtent* __restrict__ ext,
                           int n_classes, const int* __restrict__ hdr, float thresh,
                           unsigned char* __restrict__ mask_all, int* __restrict__ counts_all) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= hdr[0]) return;
  int lo = 0, hi = n_classes;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (ext[mid].row_off <= i) lo = mid; else hi = mid;
  }
  const ClassExtent e = ext[lo];
  const int li = i - e.row_off;
  const float* S = S_all + e.s_off;
  unsigned char* mask = mask_all + e.mask_off;
  int cnt = 0;
  for (int j = lane; j < e.n; j += 32) {
    const float v = (li <= j) ? S[(long long)li * e.ld + j] : S[(long long)j * e.ld + li];
    const bool m = v >= thresh;
    mask[(long long)li * e.n + j] = m ? 1 : 0;
    cnt += m;
  }
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) counts_all[i] = cnt;
}

int launch_repre_plan(const int* offsets, int class_first, int n_classes, int ld_s,
                      const int* n_saved_dev, const int* saved_len_dev, int nkb, int max_items,
                      ClassExtent* ext, GreedyClass* cls, void* pairs, void* items, void* prob,
                      int* hdr, int det, cudaStream_t stream) {
  ProfScope prof(kProfRepre, stream);
  repre_plan_kernel<<<1, 256, (3 * n_classes + 1) * sizeof(int), stream>>>(offsets, class_first, n_classes, ld_s, n_saved_dev,
                                           saved_len_dev, nkb, max_items, ext, cls,
                                           reinterpret_cast<int2*>(pairs),
                                           reinterpret_cast<tc::TcItem*>(items),
                                           reinterpret_cast<tc::TcProblem*>(prob), hdr, det);
  NSGP_LAUNCHED();
  return 0;
}

int launch_repre_prepare(const float* F, int D, int M, const int* rows, const int* offsets,
                         int class_first, const int* hdr, float* hi, float* lo,
                         const void* pairs, float* S, int ld_s, cudaStream_t stream) {
  ProfScope prof(kProfRepre, stream);
  repre_clear_tiles_kernel<<<148 * 2, 256, 0, stream>>>(reinterpret_cast<const int2*>(pairs), hdr,
                                                        S, ld_s);
  NSGP_LAUNCHED();
  normalize_split_dev_kernel<<<M, 256, 0, stream>>>(F, D, rows, offsets, class_first, hdr, hi, lo);
  NSGP_LAUNCHED();
  return 0;
}

int launch_repre_combine(const void* pairs, const int* hdr, const float* slots, float* S, int ld_s,
                         cudaStream_t stream) {
  ProfScope prof(kProfRepre, stream);
  repre_combine_tiles_kernel<<<148 * 2, 256, 0, stream>>>(reinterpret_cast<const int2*>(pairs),
                                                          hdr, slots, S, ld_s);
  NSGP_LAUNCHED();
  return 0;
}

int launch_threshold_count_dev(const float* S, const ClassExtent* ext, int n_classes, int M,
                               const int* hdr, float thresh, unsigned char* mask, int* counts,
                               cudaStream_t stream) {
  ProfScope prof(kProfRepre, stream);
  threshold_count_dev_kernel<<<ceil_div(M, 8), 256, 0, stream>>>(S, ext, n_classes, hdr, thresh,
                                                                 mask, counts);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Replay gather (:458-463 stages ALL prototypes every step; :58-59 a sampled
// subset): out[p][:] = protos[idx[p]][:]  (+ sigma[idx[p]][:] * eps, extension).
// eps is counter-based: Philox4x32-10 keyed by seed, counter (col/4, p, 0, 0),
// Box-Muller on (u0,u1),(u2,u3) - identical to oracle.restated.gaussian_noise.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ float u01(uint32_t x) {
  return (float)(((double)x + 0.5) * (1.0 / 4294967296.0));
}

__global__ void __launch_bounds__(128)
replay_gather_kernel(const float* __restrict__ protos, const float* __restrict__ sigma,
                     const long long* __restrict__ idx, int D, unsigned long long seed,
                     float* __restrict__ out) {
  const int p = blockIdx.y;
  const int q = blockIdx.x * 128 + threadIdx.x;   // float4 column group
  if (q * 4 >= D) return;
  const long long src = idx ? idx[p] : p;
  float4 v = __ldg(reinterpret_cast<const float4*>(protos + src * D) + q);
  if (sigma) {
    float4 s = __ldg(reinterpret_cast<const float4*>(sigma + src * D) + q);
    uint32_t r[4];
    philox4x32_10((uint32_t)q, (uint32_t)p, 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    float u0 = u01(r[0]), u1 = u01(r[1]), u2 = u01(r[2]), u3 = u01(r[3]);
    const float two_pi = 6.283185307179586f;
    float rad0 = sqrtf(-2.0f * logf(u0)), rad1 = sqrtf(-2.0f * logf(u2));
    v.x += s.x * (rad0 * cosf(two_pi * u1));
    v.y += s.y * (rad0 * sinf(two_pi * u1));
    v.z += s.z * (rad1 * cosf(two_pi * u3));
    v.w += s.w * (rad1 * sinf(two_pi * u3));
  }
  reinterpret_cast<float4*>(out + (long long)p * D)[q] = v;
}

int launch_replay_gather(const float* protos, const float* sigma, const long long* idx, int P,
                         int D, unsigned long long seed, float* out, cudaStream_t stream) {
  NSGP_REQUIRE(D % 4 == 0, "replay_gather: D must be a multiple of 4");
  if (P == 0) return 0;
  dim3 grid(ceil_div(D / 4, 128), P);
  replay_gather_kernel<<<grid, 128, 0, stream>>>(protos, sigma, idx, D, seed, out);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// Sampled RoI replay (StandardRoIReplayHead.loss, standard_roi_replay_head.py:53-69):
// idx = randperm(M)[:64]; the six stored tensors are gathered at idx.  One launch: the
// feature rows (D = 12544) as float4 columns, the five small per-RoI records by the
// first threads of the row's first block.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
replay_gather_rois_kernel(const float* __restrict__ feats, const long long* __restrict__ cls_t,
                          const float* __restrict__ cls_w, const float* __restrict__ bbox_t,
                          const float* __restrict__ bbox_w, const float* __restrict__ rois,
                          const long long* __restrict__ idx, int D, float* __restrict__ o_feats,
                          long long* __restrict__ o_cls_t, float* __restrict__ o_cls_w,
                          float* __restrict__ o_bbox_t, float* __restrict__ o_bbox_w,
                          float* __restrict__ o_rois) {
  const int p = blockIdx.y;
  const long long src = idx[p];
  const int q = blockIdx.x * 128 + threadIdx.x;
  if (q * 4 < D)
    reinterpret_cast<float4*>(o_feats + (long long)p * D)[q] =
        __ldg(reinterpret_cast<const float4*>(feats + src * D) + q);
  if (blockIdx.x == 0) {
    const int t = threadIdx.x;
    if (t == 0) { o_cls_t[p] = cls_t[src]; o_cls_w[p] = cls_w[src]; }
    if (t < 4) {
      o_bbox_t[p * 4 + t] = bbox_t[src * 4 + t];
      o_bbox_w[p * 4 + t] = bbox_w[src * 4 + t];
    }
    if (t < 5) o_rois[p * 5 + t] = rois[src * 5 + t];
  }
}

int launch_replay_gather_rois(const float* feats, const long long* cls_t, const float* cls_w,
                              const float* bbox_t, const float* bbox_w, const float* rois,
                              const long long* idx, int P, int D, float* o_feats,
                              long long* o_cls_t, float* o_cls_w, float* o_bbox_t,
                              float* o_bbox_w, float* o_rois, cudaStream_t stream) {
  NSGP_REQUIRE(D % 4 == 0, "replay_gather_rois: D must be a multiple of 4");
  if (P == 0) return 0;
  dim3 grid(ceil_div(D / 4, 128), P);
  ProfScope prof(kProfRepre, stream);
  replay_gather_rois_kernel<<<grid, 128, 0, stream>>>(feats, cls_t, cls_w, bbox_t, bbox_w, rois,
                                                      idx, D, o_feats, o_cls_t, o_cls_w, o_bbox_t,
                                                      o_bbox_w, o_rois);
  NSGP_LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------
// k-means assignment epilogue (extension, parity unpinned): given the dot
// products X C^T from the contraction engine and the centre norms, label =
// argmin_k (|c_k|^2 - 2 x.c_k), ties -> lowest k.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
row_sqnorm_kernel(const float* __restrict__ X, int D, int ld, float* __restrict__ out) {
  const int i = blockIdx.x;
  float ss = 0.f;
  for (int j = threadIdx.x; j < D; j += 256) {
    float v = X[(long long)i * ld + j];
    ss += v * v;
  }
  __shared__ float red[8];
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    out[i] = t;
  }
}

__global__ void __launch_bounds__(256)
kmeans_argmin_kernel(const float* __restrict__ dots, int n, int k, int ld,
                     const float* __restrict__ cnorm, long long* __restrict__ labels) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float best = INFINITY;
  int arg = 0;
  for (int j = 0; j < k; ++j) {
    float s = cnorm[j] - 2.0f * dots[(long long)i * ld + j];
    if (s < best) { best = s; arg = j; }
  }
  labels[i] = arg;
}

int launch_row_sqnorm(const float* X, int n, int D, int ld, float* out, cudaStream_t stream) {
  if (n == 0) return 0;
  row_sqnorm_kernel<<<n, 256, 0, stream>>>(X, D, ld, out);
  NSGP_LAUNCHED();
  return 0;
}

int launch_kmeans_argmin(const float* dots, int n, int k, int ld, const float* cnorm,
                         long long* labels, cudaStream_t stream) {
  if (n == 0) return 0;
  kmeans_argmin_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(dots, n, k, ld, cnorm, labels);
  NSGP_LAUNCHED();
  return 0;
}

}  // namespace nsgp
