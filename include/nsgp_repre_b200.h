/* nsgp_repre_b200.h - C ABI of the B200-native NSGP-RePRE hot path.
 *
 * The reference (yyl404/NSGP-RePRE, a pure-Python MMDetection fork) has no FFI
 * of its own: its plug-in surface is the mmengine registries.  This header is the
 * boundary a maintainer binds UNDER those Python classes (ctypes stubs in
 * INTEGRATION.md).  Each entry point cites the reference code it replaces
 * (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless marked host;
 *   - fp32, row-major, contiguous unless a pitch is given;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered,
 *     nothing synchronises the device;
 *   - return 0 on success, <0 invalid argument, >0 a cudaError_t value;
 *     nsgp_last_error() returns the message of the last failure on this thread;
 *   - no internal device allocation: scratch comes from the caller through the
 *     *_workspace_bytes queries;
 *   - sm_100a only.  There is no CPU fallback.
 */
#ifndef NSGP_REPRE_B200_H_
#define NSGP_REPRE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSGP_ABI_VERSION 1

int nsgp_abi_version(void);
const char* nsgp_last_error(void);
/* number of kernels this library has launched in this process (bench.py reports
 * the delta over the timed region as "gpu_launches") */
unsigned long long nsgp_launch_count(void);

/* Optional device timing per kernel kind (bench.py's roofline leg): when enabled,
 * every launch of that kind is bracketed by a cudaEvent pair on its stream.
 * kinds: 0 Gram contraction (tcgen05), 1 GEMM contraction (tcgen05), 2 staging,
 * 3 SGD prologue, 4 RePRE statistics.  nsgp_profile_read synchronises, returns the
 * summed milliseconds and launch count since the last read, and clears them. */
/* Deterministic mode, process-wide (mirrors torch.use_deterministic_algorithms).  While it is
 * set, size queries and table / plan builds produce work whose partial results meet in a fixed
 * order: two launches with identical inputs give bitwise identical outputs on the same GPU model
 * and library build, whatever the CTA count, SM partition or scheduling.  The size queries
 * nsgp_cov_conv2d_layout (workspace_bytes), nsgp_cov_group_bytes, nsgp_sgd_plan_bytes,
 * repre_build_prototypes_workspace_bytes, repre_cosine_count_batched_workspace_bytes and
 * nsgp_ewc_table_bytes grow (partial-tile slots, fp64 partial sums).  A built table or plan
 * keeps the mode it was built in.  Calls that have no deterministic form fail while it is set
 * (nsgp_sgd_nscl_step and single-problem contractions that need a K split).  Returns the
 * previous value. */
int nsgp_set_deterministic(int on);
int nsgp_get_deterministic(void);

int nsgp_profile_enable(int on);
int nsgp_profile_read(int kind, double* ms_total /* host */,
                      unsigned long long* launches /* host */);

/* ------------------------------------------------------------------------- *
 * a1/a2  per-layer input covariance
 *   replaces BRNullSpaceRunner.compute_cov + update_cov
 *   (mmdet/engine/runner/nsrunner_roi_replay.py:876-916, 923-934)
 * ------------------------------------------------------------------------- */

/* Geometry of the internal accumulator for one hooked Conv2d.
 *   d      = Cin*kh*kw, the covariance dimension of the reference
 *   d_int  = rows/cols of the internal accumulator (>= d)
 *   taps   = 1 or kh*kw: internal row order is (tap, channel) when taps > 1
 *   ld     = leading dimension (elements) of the accumulator, = round_up(d_int,4) */
typedef struct {
  int d, d_int, taps, ld;
  int kind;                /* 0: tap-major upper block-triangle of the d_int x d_int Gram
                              1: autocorrelation layout (3x3 s1 p1): 29 running C x C matrices */
  size_t acc_bytes;        /* zero it once before the first call */
  size_t workspace_bytes;  /* scratch for one accumulate call */
} nsgp_cov_layout_t;

int nsgp_cov_conv2d_layout(int Cin, int H, int W, int kh, int kw, int sh, int sw, int ph,
                           int pw, nsgp_cov_layout_t* out /* host */);
int nsgp_cov_linear_layout(int d, nsgp_cov_layout_t* out /* host */);

/* acc += X^T X with X = unfold(mean_b(x)) - the batch mean is taken first, exactly
 * like nsrunner_roi_replay.py:908.  x: (B,Cin,H,W).  Only the upper block-
 * triangle of acc (internal row order) is maintained; nsgp_cov_finalize expands
 * it.  Fuses torch.mean (:908), F.unfold+permute+reshape (:908-912), torch.mm
 * (:930) and the running add (:931-934). */
int nsgp_cov_conv2d_accumulate(const float* x, int B, int Cin, int H, int W, int kh, int kw,
                               int sh, int sw, int ph, int pw, float* acc, void* workspace,
                               size_t workspace_bytes, void* stream);

/* The two halves of nsgp_cov_conv2d_accumulate as separate stream-ordered calls, so
 * a caller can run the HBM-bound staging of layer i+1 (on the stream that produced
 * x) concurrently with the tensor-bound contraction of layer i (on a side stream):
 *   stage:    workspace <- tf32 hi/lo planes of the batch-averaged, im2col-free operand
 *   contract: acc += X^T X from a staged workspace (same geometry arguments). */
int nsgp_cov_conv2d_stage(const float* x, int B, int Cin, int H, int W, int kh, int kw, int sh,
                          int sw, int ph, int pw, void* workspace, size_t workspace_bytes,
                          void* stream);
int nsgp_cov_conv2d_contract(int Cin, int H, int W, int kh, int kw, int sh, int sw, int ph,
                             int pw, float* acc, const void* workspace, size_t workspace_bytes,
                             void* stream);

/* Linear: acc += m^T m with m = mean over the R rows of x (R,d)
 * (nsrunner_roi_replay.py:900-901, 930-934). */
int nsgp_cov_linear_accumulate(const float* x, int R, int d, float* acc, void* workspace,
                               size_t workspace_bytes, void* stream);

/* cov_out (d x d, dense, symmetric, reference (Cin,kh,kw) order) = expand(acc),
 * or += when accumulate != 0 (the "+ old covariance.pth" merge of :750-753). */
int nsgp_cov_finalize(const float* acc, const nsgp_cov_layout_t* layout /* host */,
                      float* cov_out, int accumulate, void* stream);

/* ------------------------------------------------------------------------- *
 * a7/a8  SGD update + null-space projection
 *   replaces SGDNSCL.get_update + the projection loop of SGDNSCL.step
 *   (mmdet/engine/optimizers/SGD_NSCL.py:387-415, 59-96)
 * ------------------------------------------------------------------------- */

/* pt_hi/pt_lo (d rows, pitch round_up(d,4)) = tf32 hi/lo split of P^T, the K-major
 * operand of update @ P (SGD_NSCL.py:85-90).  Done once per task after
 * get_transforms. */
int nsgp_projector_prepare(const float* P, int d, float* pt_hi, float* pt_lo, void* stream);

typedef struct {
  float* w;          /* parameter, updated in place (:95) */
  float* g;          /* p.grad, modified in place by weight decay (:399-400) */
  float* buf;        /* state['previous_grad'] (:394) */
  long long numel;
  int first_step;    /* 1 when state['step'] becomes 1: buf = grad (:405-406) */
  int layer;         /* index into layers[] when the name is in transforms, else -1 */
} nsgp_sgd_tensor_t;

typedef struct {
  int cout, d;             /* update.view(cout, d) @ P(d,d) */
  const float* pt_hi;      /* from nsgp_projector_prepare */
  const float* pt_lo;
  float* u_hi;             /* scratch, cout rows of pitch round_up(d,4) each: staged update */
  float* u_lo;
  /* Low-rank form (r > 0):  W += scale * (update - (update @ U) @ U^T)  with U (d x r) the
   * kept-out top eigenvectors, i.e. P = scale * (I - U U^T) - the same projector as the
   * dense V0 V0^T (/ ||P||_F for 'backbone' names, SGD_NSCL.py:270-285) without the d x d
   * matrix: 4*cout*d*r instead of 2*cout*d*d FLOPs.  pt_hi / pt_lo are unused then. */
  int r;
  float scale;
  const float* ut_hi;      /* U^T: r rows of pitch round_up(d,4) (nsgp_projector_prepare_lowrank) */
  const float* ut_lo;
  const float* un_hi;      /* U:   d rows of pitch round_up(r,4) */
  const float* un_lo;
  float* t;                /* scratch T = update @ U: cout rows of pitch round_up(r,4), fp32 ... */
  float* t_hi;             /* ... and its tf32 split; all T of a step live in one arena */
  float* t_lo;
} nsgp_proj_layer_t;

/* ut/un (hi, lo) = tf32 splits of U^T and U for the low-rank form.  U: (d x r) row-major. */
int nsgp_projector_prepare_lowrank(const float* U, int d, int r, float* ut_hi, float* ut_lo,
                                   float* un_hi, float* un_lo, void* stream);

size_t nsgp_sgd_step_workspace_bytes(int n_tensors, int n_layers);

/* One optimizer step over all tensors: a fused multi-tensor prologue (weight
 * decay, momentum, -lr) followed by the projection GEMMs W += update @ P for the
 * protected layers.  tensors/layers are HOST arrays. */
int nsgp_sgd_nscl_step(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                       const nsgp_proj_layer_t* layers, int n_layers, double lr,
                       double momentum, double dampening, double weight_decay, int nesterov,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Prepared plan of the same step: the grouped projection GEMM (all protected layers
 * in ONE persistent tcgen05 launch, work items sorted by cost) is encoded once into a
 * caller-provided device buffer; every step then uploads the small tensor table and
 * makes two launches.  Rebuild when a weight / projector / staging pointer or a shape
 * changes (gradient and momentum pointers may change freely between steps). */
typedef struct {
  int kind;
  int n_problems[4], n_items[4];   /* [0] single-CTA kernel, [1] CTA-pair (cta_group::2) kernel,
                                      [2] sliding-window autocorrelation kernel,
                                      [3] ordered combine of a deterministic table: n_problems
                                          partial-tile slots, n_items output tiles (zero when
                                          built with nsgp_set_deterministic(0)) */
  size_t off_probs[4], off_items[4];
  size_t bytes;
} nsgp_group_t;

typedef struct {
  int n_tensors, total_chunks, all_have_buf;
  size_t off_chunks, off_group, off_group2;
  nsgp_group_t group;      /* dense projections and T = update @ U of the low-rank layers */
  nsgp_group_t group2;     /* W -= scale * T @ U^T of the low-rank layers */
  float* t_arena;          /* [T | T_hi | T_lo], t_elems floats each (low-rank layers) */
  size_t t_elems;
  size_t bytes;
} nsgp_sgd_plan_t;

size_t nsgp_sgd_plan_bytes(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                           const nsgp_proj_layer_t* layers, int n_layers);
int nsgp_sgd_plan_build(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                        const nsgp_proj_layer_t* layers, int n_layers,
                        float* t_arena, size_t t_elems,
                        void* plan_dev /* 256-byte aligned */, size_t plan_bytes,
                        nsgp_sgd_plan_t* plan /* host, out */, void* stream);
/* tensors == NULL: reuse the tensor table uploaded by the previous nsgp_sgd_plan_step of this
 * plan (valid while no gradient / momentum pointer and no first_step flag has changed). */
int nsgp_sgd_plan_step(const nsgp_sgd_tensor_t* tensors, int n_tensors,
                       const nsgp_proj_layer_t* layers, int n_layers, void* plan_dev,
                       const nsgp_sgd_plan_t* plan /* host */, double lr, double momentum,
                       double dampening, double weight_decay, int nesterov, void* stream);

/* Grouped covariance contraction: the Gram updates of many staged layers (one job
 * per nsgp_cov_conv2d_stage call, each with its own workspace) as ONE persistent
 * launch - no per-layer launch gaps or tails.  The table is built once per set of
 * (geometry, workspace, accumulator) jobs and re-launched every forward. */
typedef struct {
  int Cin, H, W, kh, kw, sh, sw, ph, pw;
  float* acc;
  const void* workspace;
  size_t workspace_bytes;
} nsgp_cov_job_t;

size_t nsgp_cov_group_bytes(const nsgp_cov_job_t* jobs /* host */, int n_jobs);
int nsgp_cov_group_build(const nsgp_cov_job_t* jobs /* host */, int n_jobs,
                         void* table_dev /* 64-byte aligned */, size_t table_bytes,
                         nsgp_group_t* group /* host, out */, void* stream);
int nsgp_group_launch(const void* table_dev, const nsgp_group_t* group /* host */, void* stream);

/* Deferred staging (a1): the layer inputs of a whole forward (the jobs' `workspace`s are the
 * per-layer staged operands, as for nsgp_cov_conv2d_stage) staged by ONE launch - two when a
 * gather layout first needs the batch mean - instead of 1-3 short launches per layer.  The
 * table is built once per set of layer geometries and batch size B; every launch takes the
 * current input pointers xs[n_jobs] (host array of 16-byte aligned device pointers, each a
 * contiguous (B,Cin,H,W) fp32 tensor that must not change until the launch has run). */
typedef struct {
  int n_jobs, B;
  int n_items[2];
  size_t off_jobs, off_items[2], off_xs, bytes;
  int n_items_tma, pad;            /* items of the TMA-fed staging kernel (heavy routines) */
  size_t off_items_tma, off_maps;  /* ... and one 3-D tensor map per job, re-encoded per launch */
} nsgp_stage_group_t;
size_t nsgp_cov_stage_group_bytes(const nsgp_cov_job_t* jobs /* host */, int n_jobs, int B);
/* same_input (host, n_jobs entries, or NULL): same_input[i] = k >= 0 promises that job i is
 * given the SAME tensor as job k at every launch of this table (else -1).  Used for a 1x1
 * stride-2 conv next to a 1x1 stride-1 conv on one tensor (ResNet: layerN.0.downsample.0 /
 * layerN.0.conv1): its staged operand is written along with the other's, the input is read
 * once. */
int nsgp_cov_stage_group_build(const nsgp_cov_job_t* jobs /* host */, int n_jobs, int B,
                               const int* same_input /* host or NULL */,
                               void* table_dev /* 128-byte aligned */, size_t table_bytes,
                               nsgp_stage_group_t* out /* host */, void* stream);
int nsgp_cov_stage_group_launch(void* table_dev, const nsgp_stage_group_t* sg /* host */,
                                const nsgp_cov_job_t* jobs /* host: as given to the build */,
                                const void* const* xs /* host */, void* stream);

/* Pipelined covariance pass (a1 + a2): the tensor-bound contraction of the PREVIOUS forward
 * (prev_table / prev_group from nsgp_cov_group_build, may be NULL) and the HBM-bound staging of
 * THIS forward (stage_table / sg / xs as for nsgp_cov_stage_group_launch, may be NULL) issued
 * so that they run side by side: the contraction kernels take (SMs - stage_sms) SMs, the
 * first staging phase the other stage_sms, started through programmatic dependent launch as
 * soon as the contraction CTAs are resident.  stage_sms <= 0, or only one of the two halves
 * given: plain back-to-back launches on the whole GPU.  The two halves must use different
 * workspace sets. */
int nsgp_cov_pipeline_launch(const void* prev_table, const nsgp_group_t* prev_group,
                             void* stage_table, const nsgp_stage_group_t* sg,
                             const nsgp_cov_job_t* stage_jobs /* host: as given to the build */,
                             const void* const* xs /* host */, int stage_sms, void* stream);

/* ------------------------------------------------------------------------- *
 * a9/a10/a11  RePRE prototypes
 *   replaces the prototype build of StandardMultiPrototypeReplayHead.__init__
 *   and the per-step staging of .loss
 *   (mmdet/models/roi_heads/standard_roi_replay_head.py:411-449, 458-463)
 * ------------------------------------------------------------------------- */

/* Stable class index of labels (M,) int64 over classes [0,C): counts[C],
 * offsets[C+1], rows[M] (rows of class c = rows[offsets[c]:offsets[c+1]],
 * ascending) - the boolean-mask gather of :412. Labels outside [0,C) (background)
 * are skipped. */
int repre_class_index(const int64_t* labels, int M, int C, int32_t* counts, int32_t* offsets,
                      int32_t* rows, void* stream);

/* out[s][:] = mean over rows[seg_offsets[s]:seg_offsets[s+1]] of F (M,D):
 * coarse class means (:412-414) and masked fine-grained means (:443).
 * max_seg_rows: upper bound of the segment lengths (host hint for the grid). */
int repre_segment_mean(const float* F, int D, const int32_t* seg_offsets,
                       const int32_t* rows, int n_segments, int max_seg_rows, float* out,
                       void* stream);

/* extension (no reference counterpart): out[s][:] = mean((F[row]-mu[s])^2) */
int repre_segment_var(const float* F, int D, const int32_t* seg_offsets, const int32_t* rows,
                      int n_segments, int max_seg_rows, const float* mu, float* out,
                      void* stream);

size_t repre_cosine_count_workspace_bytes(int n, int D);

/* For the n gathered rows F[rows[i]]: L2-normalise, Gram, mask = Gram >= thresh,
 * counts = row sums (:417-421).  mask: (n,n) uint8; counts: (n,) int32;
 * sim_out: optional (n,n) fp32 copy of the Gram (may be NULL). */
int repre_cosine_count(const float* F, int D, const int32_t* rows, int n, float thresh,
                       uint8_t* mask, int32_t* counts, float* sim_out, void* workspace,
                       size_t workspace_bytes, void* stream);

/* The same for n_classes classes in four launches (normalise, clear, ONE grouped
 * tcgen05 Gram over all classes, threshold+count).  rows: device, the classes' row
 * lists concatenated; sizes: HOST, rows per class.  mask: the (n_c x n_c) uint8
 * masks packed back to back; counts: concatenated like rows. */
size_t repre_cosine_count_batched_workspace_bytes(const int32_t* sizes /* host */, int n_classes,
                                                  int D);
int repre_cosine_count_batched(const float* F, int D, const int32_t* rows,
                               const int32_t* sizes /* host */, int n_classes, float thresh,
                               uint8_t* mask, int32_t* counts, void* workspace,
                               size_t workspace_bytes, void* stream);

/* out[p][:] = protos[idx[p]][:] (idx NULL: identity, the reference stages every
 * prototype every step, :458-463; idx = randperm()[:64] is :58-59).  Extension:
 * sigma != NULL adds sigma[idx[p]] * N(0,1) noise from Philox4x32-10 keyed by
 * (seed, p, column/4). */
int repre_replay_gather(const float* protos, const float* sigma, const int64_t* idx, int P,
                        int D, uint64_t seed, float* out, void* stream);

/* a12  sampled RoI replay: StandardRoIReplayHead.loss
 * (mmdet/models/roi_heads/standard_roi_replay_head.py:53-69) draws idx = randperm(M)[:64] and
 * gathers the six tensors of rois_etc.pth at idx.  All six live on the device; one launch
 * gathers feats (M,D), cls_targets (M,) int64, cls_weights (M,), bbox_targets (M,4),
 * bbox_weights (M,4), rois (M,5) into the P-row outputs. */
int repre_replay_gather_rois(const float* feats, const int64_t* cls_targets,
                             const float* cls_weights, const float* bbox_targets,
                             const float* bbox_weights, const float* rois, const int64_t* idx,
                             int P, int D, float* out_feats, int64_t* out_cls_targets,
                             float* out_cls_weights, float* out_bbox_targets,
                             float* out_bbox_weights, float* out_rois, void* stream);

/* extension (no reference counterpart; sklearn KMeans is imported at
 * standard_roi_replay_head.py:18 and never called): Lloyd assignment
 * labels[i] = argmin_k |x_i - c_k|^2, ties -> lowest k. X (n,D), centres (k,D). */
size_t repre_kmeans_assign_workspace_bytes(int n, int k, int D);
int repre_kmeans_assign(const float* X, int n, int D, const float* centres, int k,
                        int64_t* labels, void* workspace, size_t workspace_bytes,
                        void* stream);

/* Density ordering + greedy cover of every class (:421-448) and the table of prototype
 * segments, all on the device.  Inputs as produced by repre_cosine_count_batched (masks and
 * counts concatenated per class, rows_sel = the classes' rows); `saved`/`n_saved` replay the
 * masks of mask.pth (:425-433; device bytes, n_saved[c] masks of sizes[c] bytes per class).
 * Outputs (device): seg_off[n_classes*(max_picks+1)+1], seg_rows[sum sizes*(max_picks+1)],
 * seg_label[n_classes*(max_picks+1)], info = [n_segments | picks per class | picks
 * (row within the class, -2 = replayed mask)], n_classes*(max_picks+1)+1 ints. */
size_t repre_greedy_segments_workspace_bytes(const int32_t* sizes /* host */, int n_classes,
                                             int max_picks);
int repre_greedy_segments(const uint8_t* masks, const int32_t* counts, const int32_t* rows_sel,
                          const int32_t* sizes /* host */, const int32_t* class_ids /* host */,
                          int n_classes, int max_picks, const uint8_t* saved,
                          const int32_t* n_saved /* host */, int32_t* seg_off, int32_t* seg_rows,
                          int32_t* seg_label, int32_t* info, void* workspace,
                          size_t workspace_bytes, void* stream);
/* The whole prototype build of StandardMultiPrototypeReplayHead.__init__ (:404-449) for the
 * consecutive classes [class_first, class_first + n_classes) as a FIXED sequence of launches:
 * no class size is ever read back, every buffer is sized from M.  rows / offsets: the class
 * index (repre_class_index).  Steps: plan (device: per-class extents, the tile pairs of ONE Gram
 * over the class-sorted foreground rows, its work items), L2-normalise + tf32 split, tcgen05
 * Gram, threshold + neighbour counts, density ordering + greedy cover + segment table, segment
 * means.  saved / n_saved / saved_len replay mask.pth (:425-433): n_saved[c] masks of
 * saved_len[c] bytes per class, packed.
 * Outputs (device): masks (class c's n_c x n_c mask at byte offset sum_{c'<c} n_c'^2; size
 * M*M worst case), counts[M], seg_off[n_classes*(max_picks+1)+1], seg_rows[M*(max_picks+1)],
 * seg_label, protos (n_classes*(max_picks+1), D),
 * info = [n_segments | picks per class (n_classes) | picks (n_classes*max_picks) | status |
 *         n_foreground]; status 1: a class has no rows (the reference raises IndexError at
 *         :422), 2: a replayed mask does not match its class's row count.
 * flags & 1: the Gram problem (tensor maps over this workspace) is still in the workspace from
 * an earlier call with the same F-independent arguments (M, D, workspace) - the call is then
 * launches and device-to-device copies only, i.e. capturable into a CUDA graph; needs
 * saved == NULL. */
size_t repre_build_prototypes_workspace_bytes(int M, int D, int n_classes, int max_picks);
int repre_build_prototypes(const float* F, int D, int M, const int32_t* rows,
                           const int32_t* offsets, int class_first, int n_classes, float thresh,
                           int max_picks, const uint8_t* saved, const int32_t* n_saved /* host */,
                           const int32_t* saved_len /* host */, uint8_t* masks, int32_t* counts,
                           int32_t* seg_off, int32_t* seg_rows, int32_t* seg_label, int32_t* info,
                           float* protos, void* workspace, size_t workspace_bytes, int flags,
                           void* stream);

/* repre_segment_mean over at most max_segments segments, the live count read on the device */
int repre_segment_mean_dev(const float* F, int D, const int32_t* seg_offsets, const int32_t* rows,
                           int max_segments, const int32_t* n_segments_dev, int max_seg_rows,
                           float* out, void* stream);

/* ------------------------------------------------------------------------- *
 * SURVEY 8(f)-2  RoIAlign over the FPN levels, optionally fused with the per-class sums
 *   replaces SingleRoIExtractor.forward
 *   (mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:45-118, pooling =
 *   mmcv.ops.RoIAlign: average pooling, adaptive grid when sampling_ratio = 0, `aligned`)
 *   feats[l]: (batch, channels, heights[l], widths[l]) fp32 NCHW device tensors (host array
 *   of pointers), rois (n_rois,5) = [batch index, x1, y1, x2, y2] in image coordinates.
 *   Level of a RoI: levels[r] when `levels` (device int32, n_rois) is given, else
 *   floor(log2(sqrt(w*h)/finest_scale + 1e-6)) clamped to the levels, evaluated in the kernel.
 *   roi_feats (n_rois, channels*pooled*pooled) and/or class_sums (n_classes, same) +
 *   class_counts (n_classes; labels outside [0,n_classes) are skipped); either output
 *   may be NULL.  class_sums / class_counts are cleared by the call.
 * ------------------------------------------------------------------------- */
int repre_roi_align(const float* const* feats /* host */, const int32_t* heights /* host */,
                    const int32_t* widths /* host */, const float* spatial_scales /* host */,
                    int n_levels, int batch, int channels, const float* rois, int n_rois,
                    int pooled, int sampling_ratio, int aligned, float finest_scale,
                    const int32_t* levels, const int64_t* labels, int n_classes, float* roi_feats,
                    float* class_sums, int32_t* class_counts, void* stream);

/* gradient of repre_roi_align w.r.t. the feature maps: grad_feats[l] (batch, channels, H_l, W_l),
 * zero-filled (or holding a gradient to add to) by the caller, accumulated into with atomics */
int repre_roi_align_backward(float* const* grad_feats /* host */, const int32_t* heights,
                             const int32_t* widths, const float* spatial_scales, int n_levels,
                             int batch, int channels, const float* rois, int n_rois, int pooled,
                             int sampling_ratio, int aligned, float finest_scale,
                             const int32_t* levels, const float* grad_out, void* stream);

/* ------------------------------------------------------------------------- *
 * SURVEY 8(f)-4  EWC importance and penalty
 *   replaces the per-tensor loops of BRNullSpaceRunner.calculate_save_importance
 *   (mmdet/engine/runner/nsrunner_roi_replay.py:978-981) and EWCHook.__call__ (:1056-1069)
 *   with one multi-tensor launch each.  `tensors` is a host array; table_dev is a device
 *   scratch of nsgp_ewc_table_bytes(n) bytes.
 * ------------------------------------------------------------------------- */
typedef struct {
  const float* p;          /* accumulate: the gradient; penalty: the parameter */
  float* importance;       /* accumulate: (numel) in/out; penalty: (tasks, numel) */
  const float* old_params; /* penalty: (tasks, numel) */
  float* grad;             /* penalty backward: gradient of p, accumulated into */
  long long numel;
  int tasks;
} nsgp_ewc_tensor_t;
size_t nsgp_ewc_table_bytes(int n);
/* importance += (grad * grad) * mul / div   (one rounding per operation, reference order) */
int nsgp_ewc_accumulate(const nsgp_ewc_tensor_t* tensors /* host */, int n, float mul, float div,
                        void* table_dev, size_t table_bytes, void* stream);
/* *loss_dev = coeff * sum_n sum_t importance * (p - old)^2   (fp64 accumulation) */
int nsgp_ewc_penalty(const nsgp_ewc_tensor_t* tensors /* host */, int n, float coeff,
                     double* loss_dev, void* table_dev, size_t table_bytes, void* stream);
/* grad += *grad_out_dev * 2 * coeff * sum_t importance_t * (p - old_t) */
int nsgp_ewc_penalty_backward(const nsgp_ewc_tensor_t* tensors /* host */, int n, float coeff,
                              const float* grad_out_dev, void* table_dev, size_t table_bytes,
                              void* stream);

/* ------------------------------------------------------------------------- *
 * SURVEY 8(f)-3  teacher pseudo-label merge
 *   replaces the per-box loop of FasterRCNNRoIReplay.loss
 *   (mmdet/models/detectors/faster_rcnn_roi_replay.py:78-108): for every image, every
 *   teacher box in order: max torchvision box_iou against the ground truth plus the teacher
 *   boxes already accepted for the RoI head; > iou_thresh (0.7, compared as a python float)
 *   drops it; score > rpn_thresh (0.5) keeps it for the RPN targets, score > roi_thresh
 *   (0.7) for the RoI targets.  Boxes are (N,4) fp32 xyxy, concatenated over the images
 *   with offsets[n_images+1]; outputs keep_rpn / keep_roi per teacher box and
 *   counts[2*b] / counts[2*b+1] = kept boxes of image b.
 * ------------------------------------------------------------------------- */
int nsgp_pseudo_label_merge(const float* gt_boxes, const int32_t* gt_offsets,
                            const float* pseudo_boxes, const float* pseudo_scores,
                            const int32_t* pseudo_offsets, int n_images, int max_pseudo,
                            float rpn_thresh, float roi_thresh, double iou_thresh,
                            uint8_t* keep_rpn, uint8_t* keep_roi, int32_t* counts, void* stream);

/* generic tf32 hi/lo split of n floats (used by tests and the host layer) */
int nsgp_split_tf32(const float* src, float* hi, float* lo, size_t n, void* stream);

/* C (M x ldc) += A (M x K) * B^T (B is N x K) through the 3xTF32 tcgen05 contraction engine;
 * a_/b_ are tf32 hi/lo pairs (nsgp_split_tf32) with pitch K. */
int nsgp_gemm_nt(const float* a_hi, const float* a_lo, const float* b_hi,
                       const float* b_lo, int M, int N, int K, float* C, int ldc,
                       void* stream);

/* ------------------------------------------------------------------------- *
 * Bring-up build only (make BRINGUP=1 -> libnsgp_repre_b200_bringup.so, -DNSGP_BRINGUP):
 * a second (SIMT fp32) contraction engine for on-device cross-checks, experiment kernels and
 * in-kernel counters.  None of this is in the shipped library.
 * ------------------------------------------------------------------------- */
#ifdef NSGP_BRINGUP
/* contraction engine: 0 = tcgen05/TMA 3xTF32 (product), 1 = SIMT fp32 FFMA.  Returns the
 * previous value. */
int nsgp_set_engine(int engine);
int nsgp_get_engine(void);

/* bring-up: per-CTA wait/issue cycle counters of the last tcgen05 contraction launched
 * with NSGP_DBG_COUNTERS=1 in the environment (8 counters per CTA, host buffer) */
int nsgp_debug_read_counters(unsigned long long* out /* host */, int n);

/* bring-up: cycles one CTA per SM needs for `iters` K blocks of tcgen05 MMAs on
 * shared-memory-resident operands (mode: see csrc/mma_rate.cu); out_dev: n_ctas u64 */
int nsgp_debug_mma_rate(int mode, int iters, unsigned long long* out_dev /* device */,
                        int n_ctas, void* stream);

/* bring-up: cycles per CTA for `iters` 64 KB TMA stages (4 boxes of 128 rows x 128 B) with
 * `depth` stages in flight, from a (rows x K) fp32 matrix of the given row pitch */
int nsgp_debug_tma_probe(const float* base, long long pitch_elems, int K, int rows, int iters,
                         int depth, unsigned long long* out_dev /* device */, int n_ctas,
                         void* stream);

/* bring-up: the same with one 3-D tensor-map box (256 floats x box_rows x B images) per stage */
int nsgp_debug_tma3d_probe(const float* base, long long img_elems, int B, int box_rows,
                           int boxes_per_cta, int depth, unsigned long long* out_dev, int n_ctas,
                           void* stream);

/* bring-up: every CTA streams bytes_per_cta contiguous bytes of src into shared memory with
 * `depth` cp.async.bulk chunks of `chunk` bytes in flight; out_dev: n_ctas u64 cycle counts */
int nsgp_debug_bulk_probe(const void* src, long long bytes_per_cta, int chunk, int depth,
                          unsigned long long* out_dev /* device */, int n_ctas, void* stream);

/* bring-up: with NSGP_TIMELINE=1 in the environment the grouped staging kernel (kind 2) and
 * the two covariance contraction kernels (kind 0 generic, kind 10 sliding-window) record
 * {first block start, last block end} in globaltimer ns per launch; returns the number of
 * launches copied to out[2*i], out[2*i+1], kinds[i] and resets the log */
int nsgp_debug_timeline_read(unsigned long long* out /* host */, int* kinds /* host */,
                             int max_slots);

/* bring-up: n_ctas blocks of `threads` threads holding `smem` bytes of shared memory for
 * `cycles` SM clocks, no memory traffic (co-residency probe, scripts/overlap_probe.py) */
int nsgp_debug_occupy(int threads, size_t smem, long long cycles, int n_ctas, void* stream);

#endif /* NSGP_BRINGUP */

#ifdef __cplusplus
}
#endif
#endif /* NSGP_REPRE_B200_H_ */
