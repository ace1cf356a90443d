// SURVEY.md 8(f) rows 3 and 4: the per-step continual-learning side work that the
// reference does in Python loops with one tiny kernel (and often one host sync) per
// tensor or per box.
//
//   EWC (nsrunner_roi_replay.py:946-990, 1038-1073)
//     importance[n] += grad[n]^2 * len(data_batch) / len(dataloader)     per batch, per tensor
//     ewc_loss = 1000 * sum_n sum_t importance[n][t] * (p_n - old[n][t])^2   per training step
//   -> one multi-tensor launch each (plus one for the gradient of the penalty).
//
//   Teacher pseudo-label merge (faster_rcnn_roi_replay.py:67-108)
//     per teacher box, in order: max IoU against the (growing) ground-truth set,
//     skip if > 0.7, append to the RPN targets if score > 0.5 and to the RoI targets
//     (the set the next boxes are compared with) if score > 0.7
//   -> one CTA per image, no host round trip per box.
#include <vector>

#include "../../include/nsgp_repre_b200.h"
#include "common.cuh"

namespace nsgp {

constexpr int kEwcChunk = 1024;     // elements per CTA; BatchNorm tensors are 64..2048 long

struct EwcTensorDev {
  const float* p;        // parameter (penalty) / gradient (accumulate)
  float* imp;            // importance (accumulate: in/out; penalty: [tasks][numel])
  const float* old;      // penalty: previous-task parameters [tasks][numel]
  float* grad;           // penalty backward: gradient buffer of p (accumulated into)
  long long numel;
  int tasks, chunk0;     // first chunk of this tensor
};

__device__ __forceinline__ int ewc_find(const EwcTensorDev* t, int n, int chunk) {
  int lo = 0, hi = n;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (t[mid].chunk0 <= chunk) lo = mid; else hi = mid;
  }
  return lo;
}

// importance += (g * g) * mul / div, the reference's operation order, one rounding each
// (:978-981: "(grad ** 2) * len(data_batch) / len(dataloader)")
__global__ void __launch_bounds__(256)
ewc_accumulate_kernel(const EwcTensorDev* __restrict__ tensors, int n, float mul, float div) {
  const EwcTensorDev t = tensors[ewc_find(tensors, n, blockIdx.x)];
  const long long beg = (long long)(blockIdx.x - t.chunk0) * kEwcChunk;
  const long long end = min(t.numel, beg + kEwcChunk);
  for (long long i = beg + threadIdx.x; i < end; i += 256) {
    const float g = t.p[i];
    const float v = __fdiv_rn(__fmul_rn(__fmul_rn(g, g), mul), div);
    t.imp[i] = __fadd_rn(t.imp[i], v);
  }
}

// MODE 0: loss += coeff * sum imp * (p - old)^2  (double accumulation, one atomic per CTA)
// MODE 1: grad += gout * 2 * coeff * sum_t imp_t * (p - old_t)
template <int MODE>
__global__ void __launch_bounds__(256)
ewc_penalty_kernel(const EwcTensorDev* __restrict__ tensors, int n, float coeff,
                   double* __restrict__ loss, const float* __restrict__ gout) {
  const EwcTensorDev t = tensors[ewc_find(tensors, n, blockIdx.x)];
  const long long beg = (long long)(blockIdx.x - t.chunk0) * kEwcChunk;
  const long long end = min(t.numel, beg + kEwcChunk);
  double acc = 0.0;
  const float go = MODE == 1 ? gout[0] : 0.f;
  for (long long i = beg + threadIdx.x; i < end; i += 256) {
    const float p = t.p[i];
    float s = 0.f;
    for (int k = 0; k < t.tasks; ++k) {
      const float d = p - t.old[(long long)k * t.numel + i];
      const float w = t.imp[(long long)k * t.numel + i];
      if (MODE == 0) acc += (double)w * (double)d * (double)d;
      else s += w * d;
    }
    if (MODE == 1) t.grad[i] += go * (2.f * coeff) * s;
  }
  if (MODE == 0) {
    __shared__ double red[8];
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int w = 0; w < 8; ++w) s += red[w];
      atomicAdd(loss, (double)coeff * s);
    }
  }
}

// Deterministic mode: kEwcDetCtas CTAs stride over the chunks in a fixed order and write one
// fp64 partial each behind the tensor table; one CTA sums them in a fixed order.
constexpr int kEwcDetCtas = 512;

__global__ void __launch_bounds__(256)
ewc_penalty_partial_kernel(const EwcTensorDev* __restrict__ tensors, int n, int total_chunks,
                           double* __restrict__ partial) {
  double acc = 0.0;
  for (int chunk = blockIdx.x; chunk < total_chunks; chunk += gridDim.x) {
    const EwcTensorDev t = tensors[ewc_find(tensors, n, chunk)];
    const long long beg = (long long)(chunk - t.chunk0) * kEwcChunk;
    const long long end = min(t.numel, beg + kEwcChunk);
    for (long long i = beg + threadIdx.x; i < end; i += 256) {
      const float p = t.p[i];
      for (int k = 0; k < t.tasks; ++k) {
        const float d = p - t.old[(long long)k * t.numel + i];
        const float w = t.imp[(long long)k * t.numel + i];
        acc += (double)w * (double)d * (double)d;
      }
    }
  }
  __shared__ double red[8];
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[w];
    partial[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(256)
ewc_penalty_sum_kernel(const double* __restrict__ partial, int n_partial, float coeff,
                       double* __restrict__ loss) {
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_partial; i += 256) acc += partial[i];
  __shared__ double red[8];
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[w];
    *loss = (double)coeff * s;
  }
}

static size_t ewc_tensors_bytes(int n) {
  return (size_t)round_up((long long)(n > 0 ? n : 1) * sizeof(EwcTensorDev), 256);
}

static int ewc_table(const nsgp_ewc_tensor_t* tensors, int n, void* table_dev, size_t table_bytes,
                     cudaStream_t stream, int* total_chunks) {
  NSGP_REQUIRE(tensors && table_dev && n > 0, "ewc: bad arguments");
  NSGP_REQUIRE(table_bytes >= (size_t)n * sizeof(EwcTensorDev), "ewc: table too small");
  std::vector<EwcTensorDev> h(n);
  int chunk = 0;
  for (int i = 0; i < n; ++i) {
    NSGP_REQUIRE(tensors[i].numel > 0 && tensors[i].tasks >= 0, "ewc: tensor %d: bad sizes", i);
    h[i].p = tensors[i].p; h[i].imp = tensors[i].importance; h[i].old = tensors[i].old_params;
    h[i].grad = tensors[i].grad; h[i].numel = tensors[i].numel; h[i].tasks = tensors[i].tasks;
    h[i].chunk0 = chunk;
    chunk += (int)((tensors[i].numel + kEwcChunk - 1) / kEwcChunk);
  }
  *total_chunks = chunk;
  NSGP_CHECK_CUDA(cudaMemcpyAsync(table_dev, h.data(), (size_t)n * sizeof(EwcTensorDev),
                                  cudaMemcpyHostToDevice, stream));
  return 0;
}

// ---------------------------------------------------------------------------
// Pseudo-label merge.  box_iou is torchvision's arithmetic (boxes.py: area from
// (x2-x1)*(y2-y1), clamp(min=0) of the intersection extents, inter / (a1 + a2 - inter)),
// every operation rounded separately so that the fp32 values - and with them the
// "> 0.7" decisions - are the reference's bit for bit.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float box_area(const float4 b) {
  return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}
__device__ __forceinline__ float box_iou(const float4 a, const float4 b) {
  const float ltx = fmaxf(a.x, b.x), lty = fmaxf(a.y, b.y);
  const float rbx = fminf(a.z, b.z), rby = fminf(a.w, b.w);
  // torch.max / torch.min / clamp propagate NaN; fmaxf / fminf do not
  float w = __fsub_rn(rbx, ltx), h = __fsub_rn(rby, lty);
  const bool nan_in = isnan(a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w);
  w = w < 0.f ? 0.f : w;
  h = h < 0.f ? 0.f : h;
  const float inter = __fmul_rn(w, h);
  const float uni = __fsub_rn(__fadd_rn(box_area(a), box_area(b)), inter);
  const float iou = __fdiv_rn(inter, uni);
  return nan_in ? __int_as_float(0x7fc00000) : iou;
}
// torch.Tensor.max(): NaN wins
__device__ __forceinline__ float nan_max(float m, float v) {
  if (isnan(m) || isnan(v)) return __int_as_float(0x7fc00000);
  return fmaxf(m, v);
}

constexpr int kMaxPseudo = 1024;     // teacher boxes per image (test_cfg.rcnn.max_per_img = 100)

__global__ void __launch_bounds__(128)
pseudo_merge_kernel(const float4* __restrict__ gt, const int* __restrict__ gt_off,
                    const float4* __restrict__ ps, const float* __restrict__ score,
                    const int* __restrict__ ps_off, float rpn_thresh, float roi_thresh,
                    double iou_thresh, unsigned char* __restrict__ keep_rpn,
                    unsigned char* __restrict__ keep_roi, int* __restrict__ counts) {
  const int b = blockIdx.x, tid = threadIdx.x;
  const int g0 = gt_off[b], ng = gt_off[b + 1] - g0;
  const int p0 = ps_off[b], np = ps_off[b + 1] - p0;
  __shared__ float s_iou_gt[kMaxPseudo];
  __shared__ short s_acc[kMaxPseudo];
  __shared__ float s_warp[4];
  __shared__ int s_nacc, s_nrpn;
  // max IoU of every teacher box with the original ground truth
  for (int k = tid; k < np; k += 128) {
    const float4 box = ps[p0 + k];
    float m = -INFINITY;
    for (int j = 0; j < ng; ++j) m = nan_max(m, box_iou(box, gt[g0 + j]));
    s_iou_gt[k] = m;
  }
  if (tid == 0) { s_nacc = 0; s_nrpn = 0; }
  __syncthreads();
  // in order: the set grows by the boxes accepted for the RoI head (:104-106)
  for (int k = 0; k < np; ++k) {
    const float4 box = ps[p0 + k];
    const int nacc = s_nacc;
    float m = -INFINITY;
    for (int j = tid; j < nacc; j += 128) m = nan_max(m, box_iou(box, ps[p0 + s_acc[j]]));
    for (int o = 16; o; o >>= 1) m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) s_warp[tid >> 5] = m;
    __syncthreads();
    if (tid == 0) {
      float mm = ng > 0 ? s_iou_gt[k] : -INFINITY;
      for (int w = 0; w < 4; ++w) mm = nan_max(mm, s_warp[w]);
      const float max_iou = (ng + nacc > 0) ? mm : 0.f;            // :86-90
      unsigned char kr = 0, ko = 0;
      if (!((double)max_iou > iou_thresh)) {                       // :93 (python float compare)
        const float sc = score[p0 + k];
        kr = sc > rpn_thresh;                                      // :101 (fp32 compare)
        ko = sc > roi_thresh;                                      // :105
        if (ko) s_acc[s_nacc++] = (short)k;
        if (kr) ++s_nrpn;
      }
      keep_rpn[p0 + k] = kr;
      keep_roi[p0 + k] = ko;
    }
    __syncthreads();
  }
  if (tid == 0) { counts[2 * b] = s_nrpn; counts[2 * b + 1] = s_nacc; }
}

}  // namespace nsgp

using namespace nsgp;

extern "C" {

int nsgp_ewc_accumulate(const nsgp_ewc_tensor_t* tensors, int n, float mul, float div,
                        void* table_dev, size_t table_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n == 0) return 0;
  int chunks = 0;
  int rc = ewc_table(tensors, n, table_dev, table_bytes, stream, &chunks);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    NSGP_REQUIRE(tensors[i].p && tensors[i].importance, "ewc_accumulate: tensor %d: null pointer", i);
  ewc_accumulate_kernel<<<chunks, 256, 0, stream>>>(
      reinterpret_cast<const EwcTensorDev*>(table_dev), n, mul, div);
  NSGP_LAUNCHED();
  return 0;
}

int nsgp_ewc_penalty(const nsgp_ewc_tensor_t* tensors, int n, float coeff, double* loss_dev,
                     void* table_dev, size_t table_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(loss_dev != nullptr, "ewc_penalty: null loss");
  NSGP_CHECK_CUDA(cudaMemsetAsync(loss_dev, 0, sizeof(double), stream));
  if (n == 0) return 0;
  int chunks = 0;
  int rc = ewc_table(tensors, n, table_dev, table_bytes, stream, &chunks);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    NSGP_REQUIRE(tensors[i].p && (tensors[i].tasks == 0 || (tensors[i].importance && tensors[i].old_params)),
                 "ewc_penalty: tensor %d: null pointer", i);
  if (g_deterministic) {
    NSGP_REQUIRE(table_bytes >= ewc_tensors_bytes(n) + kEwcDetCtas * sizeof(double),
                 "ewc_penalty: table too small for the deterministic sum (%zu < %zu)",
                 table_bytes, ewc_tensors_bytes(n) + kEwcDetCtas * sizeof(double));
    double* partial = reinterpret_cast<double*>((char*)table_dev + ewc_tensors_bytes(n));
    const int ctas = chunks < kEwcDetCtas ? chunks : kEwcDetCtas;
    ewc_penalty_partial_kernel<<<ctas, 256, 0, stream>>>(
        reinterpret_cast<const EwcTensorDev*>(table_dev), n, chunks, partial);
    NSGP_LAUNCHED();
    ewc_penalty_sum_kernel<<<1, 256, 0, stream>>>(partial, ctas, coeff, loss_dev);
    NSGP_LAUNCHED();
    return 0;
  }
  ewc_penalty_kernel<0><<<chunks, 256, 0, stream>>>(
      reinterpret_cast<const EwcTensorDev*>(table_dev), n, coeff, loss_dev, nullptr);
  NSGP_LAUNCHED();
  return 0;
}

int nsgp_ewc_penalty_backward(const nsgp_ewc_tensor_t* tensors, int n, float coeff,
                              const float* grad_out_dev, void* table_dev, size_t table_bytes,
                              void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  NSGP_REQUIRE(grad_out_dev != nullptr, "ewc_penalty_backward: null grad_out");
  if (n == 0) return 0;
  int chunks = 0;
  int rc = ewc_table(tensors, n, table_dev, table_bytes, stream, &chunks);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    NSGP_REQUIRE(tensors[i].p && tensors[i].grad, "ewc_penalty_backward: tensor %d: null pointer", i);
  ewc_penalty_kernel<1><<<chunks, 256, 0, stream>>>(
      reinterpret_cast<const EwcTensorDev*>(table_dev), n, coeff, nullptr, grad_out_dev);
  NSGP_LAUNCHED();
  return 0;
}

size_t nsgp_ewc_table_bytes(int n) {
  // deterministic mode: + the fp64 partial sums of the penalty
  if (g_deterministic) return ewc_tensors_bytes(n) + kEwcDetCtas * sizeof(double);
  return (size_t)(n > 0 ? n : 1) * sizeof(EwcTensorDev);
}

int nsgp_pseudo_label_merge(const float* gt_boxes, const int32_t* gt_offsets,
                            const float* pseudo_boxes, const float* pseudo_scores,
                            const int32_t* pseudo_offsets, int n_images, int max_pseudo,
                            float rpn_thresh, float roi_thresh, double iou_thresh,
                            uint8_t* keep_rpn, uint8_t* keep_roi, int32_t* counts,
                            void* stream_) {
  NSGP_REQUIRE(gt_offsets && pseudo_offsets && keep_rpn && keep_roi && counts,
               "pseudo_label_merge: null pointer");
  NSGP_REQUIRE(n_images >= 0 && max_pseudo >= 0 && max_pseudo <= kMaxPseudo,
               "pseudo_label_merge: at most %d teacher boxes per image", kMaxPseudo);
  if (n_images == 0) return 0;
  NSGP_REQUIRE((reinterpret_cast<uintptr_t>(gt_boxes) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(pseudo_boxes) & 15) == 0,
               "pseudo_label_merge: boxes must be 16-byte aligned (N,4) fp32");
  pseudo_merge_kernel<<<n_images, 128, 0, (cudaStream_t)stream_>>>(
      reinterpret_cast<const float4*>(gt_boxes), gt_offsets,
      reinterpret_cast<const float4*>(pseudo_boxes), pseudo_scores, pseudo_offsets, rpn_thresh,
      roi_thresh, iou_thresh, keep_rpn, keep_roi, counts);
  NSGP_LAUNCHED();
  return 0;
}

}  // extern "C"
