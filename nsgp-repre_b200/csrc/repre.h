// Launchers of the RePRE statistics kernels (repre.cu).
#pragma once
#include "common.cuh"

namespace nsgp {
int launch_class_index(const long long* labels, int M, int C, int* counts, int* offsets,
                       int* rows, cudaStream_t s);
// nseg_dev != null: the grid covers `nseg` segments at most, the live count is read on
// the device (segments built by launch_greedy_segments)
int launch_segment_mean(const float* F, int D, const int* seg_off, const int* rows, int nseg,
                        int max_seg_rows, const float* mu, int mode, float* out, cudaStream_t s,
                        const int* nseg_dev = nullptr);
struct GreedyClass {          // one class of a greedy-cover call
  long long mask_off;         // byte offset of its (n x n) neighbour mask
  long long saved_off;        // byte offset of its replayed masks (n_saved x n)
  int row_off;                // first row in the concatenated row / count arrays
  int n, n_saved, class_id;
};
int launch_greedy_segments(const GreedyClass* cls_dev, int n_classes, int max_n,
                           const unsigned char* masks, const int* counts,
                           const unsigned char* saved, const int* rows_sel, int max_picks,
                           int* order_ws, unsigned char* covered_ws, int* seg_sizes,
                           int* seg_base, int* picks, int* npicks, int* seg_off, int* seg_rows,
                           int* seg_label, int* nseg_out, cudaStream_t s,
                           const int* rows_base = nullptr);
int launch_normalize_split(const float* F, int D, const int* rows, int n, float* hi, float* lo,
                           cudaStream_t s);
int launch_threshold_count(const float* S, int n, int ld, float thresh, unsigned char* mask,
                           int* counts, float* sim_out, cudaStream_t s);
struct ClassExtent {          // one class of a batched cosine-count call
  long long s_off;            // element offset of its Gram in the similarity buffer
  long long mask_off;         // byte offset of its (n x n) mask
  int row_off;                // first row in the concatenated row / count arrays
  int n, ld, pad;
};
int launch_threshold_count_batched(const float* S_all, const ClassExtent* ext_dev, int n_classes,
                                   int max_n, float thresh, unsigned char* mask_all,
                                   int* counts_all, cudaStream_t s);
// device-sized build (repre_build_prototypes)
int launch_class_index_fused(const long long* labels, int M, int C, int* counts, int* offsets,
                             int* rows, cudaStream_t s);
int launch_repre_plan(const int* offsets, int class_first, int n_classes, int ld_s,
                      const int* n_saved_dev, const int* saved_len_dev, int nkb, int max_items,
                      ClassExtent* ext, GreedyClass* cls, void* pairs, void* items, void* prob,
                      int* hdr, int det, cudaStream_t s);
// deterministic mode: the K-split partial Gram tiles (slots) summed into S in split order
int launch_repre_combine(const void* pairs, const int* hdr, const float* slots, float* S, int ld_s,
                         cudaStream_t s);
int launch_repre_prepare(const float* F, int D, int M, const int* rows, const int* offsets,
                         int class_first, const int* hdr, float* hi, float* lo,
                         const void* pairs, float* S, int ld_s, cudaStream_t s);
int launch_threshold_count_dev(const float* S, const ClassExtent* ext, int n_classes, int M,
                               const int* hdr, float thresh, unsigned char* mask, int* counts,
                               cudaStream_t s);
int launch_replay_gather(const float* protos, const float* sigma, const long long* idx, int P,
                         int D, unsigned long long seed, float* out, cudaStream_t s);
int launch_replay_gather_rois(const float* feats, const long long* cls_t, const float* cls_w,
                              const float* bbox_t, const float* bbox_w, const float* rois,
                              const long long* idx, int P, int D, float* o_feats,
                              long long* o_cls_t, float* o_cls_w, float* o_bbox_t,
                              float* o_bbox_w, float* o_rois, cudaStream_t s);
int launch_row_sqnorm(const float* X, int n, int D, int ld, float* out, cudaStream_t s);
int launch_kmeans_argmin(const float* dots, int n, int k, int ld, const float* cnorm,
                         long long* labels, cudaStream_t s);
}  // namespace nsgp
