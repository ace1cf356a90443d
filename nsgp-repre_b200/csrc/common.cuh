// Shared declarations for the NSGP-RePRE B200 library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <vector>

namespace nsgp {

// ---- error handling / launch accounting -----------------------------------
void set_error(const char* fmt, ...);
extern unsigned long long g_launches;   // kernels launched by this library

#define NSGP_CHECK_CUDA(expr)                                                     \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      nsgp::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                      __FILE__, __LINE__);                                        \
      return (int)_e;                                                             \
    }                                                                             \
  } while (0)

#define NSGP_REQUIRE(cond, ...)                                                   \
  do {                                                                            \
    if (!(cond)) {                                                                \
      nsgp::set_error(__VA_ARGS__);                                               \
      return -1;                                                                  \
    }                                                                             \
  } while (0)

#define NSGP_LAUNCHED()                                                           \
  do {                                                                            \
    ++nsgp::g_launches;                                                           \
    NSGP_CHECK_CUDA(cudaGetLastError());                                          \
  } while (0)

// ---- deterministic mode (nsgp_set_deterministic) -------------------------------
// Size queries and table builds read it; a built table carries its mode in its work items,
// so launching it never depends on the flag.
extern int g_deterministic;

// ---- optional per-kernel-kind device timing (bench.py's roofline leg) --------
// When enabled every launch of a profiled kind is bracketed by a cudaEvent pair on
// the launch stream; nsgp_profile_read synchronises and sums them.
enum ProfKind : int { kProfGram = 0, kProfGemm = 1, kProfStage = 2, kProfSgd = 3,
                      kProfRepre = 4, kProfKinds = 5 };
extern int g_profile;
// bring-up timeline (NSGP_TIMELINE=1): every launch of an instrumented kernel gets a slot
// {first block start, last block end} in globaltimer ns, read by nsgp_debug_timeline_read
unsigned long long* timeline_slot(int kind);       // nullptr when disabled
#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long tl_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void tl_begin(unsigned long long* tl) {
  if (tl != nullptr && threadIdx.x == 0) atomicMin(tl, tl_now());
}
__device__ __forceinline__ void tl_end(unsigned long long* tl) {
  if (tl != nullptr && threadIdx.x == 0) atomicMax(tl + 1, tl_now());
}
#endif
void profile_begin(int kind, cudaStream_t s);
void profile_end(int kind, cudaStream_t s);
struct ProfScope {
  int kind; cudaStream_t s;
  ProfScope(int k, cudaStream_t st) : kind(k), s(st) { if (g_profile) profile_begin(kind, s); }
  ~ProfScope() { if (g_profile) profile_end(kind, s); }
};

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline long long round_up(long long a, long long b) { return (a + b - 1) / b * b; }

// ---- 3xTF32 split ------------------------------------------------------------
// hi = rna_tf32(x); lo = rna_tf32(x - hi).  x - hi is exact in fp32, so hi + lo
// carries ~21 mantissa bits and both words have their low 13 bits clear, i.e. the
// tensor core's tf32 truncation of the smem operand is a no-op.
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - hi);
}

// ---- K-major virtual operand ---------------------------------------------------
// Both engines (SIMT bring-up and tcgen05) consume operands described this way.
// A virtual matrix of `rows` = T * Cs rows and K columns: row r = t * Cs + c
// (tap-major) is the K contiguous fp32 words at
//     base + hl * hl_stride + tap_off[t] + c * row_pitch          (hl: 0 = tf32 hi, 1 = lo)
// and reads as zero for k >= K.  Plain row-major matrices are the T = 1 case; the
// staged conv layouts (geometry.h) put every tap at its own offset.
constexpr int kMaxTaps = 9;

struct Operand {
  const float* base;       // hi part
  long long hl_stride;     // elements between the hi and the lo copy
  long long row_pitch;     // elements between consecutive rows c of one tap (% 4 == 0)
  int T, Cs;               // taps, rows per tap
  int K;                   // valid columns
  int rows;                // valid virtual rows (<= T*Cs)
  long long tap_off[kMaxTaps];   // element offset of tap t (% 4 == 0)
};

// Epilogue of the contraction engines.
enum EpiMode : int {
  kEpiGramAtomic = 0,  // upper block-triangle of A*A^T, red.add into out (split-K ok)
  kEpiGemmRmw = 1,     // full A*B^T, out[m][n] += alpha * acc (exclusive tiles, no split-K)
};

struct ContractionArgs {
  Operand A, B;
  float* out;       // (A.rows x ld)
  int ld;           // leading dimension of out (elements)
  int n_cols;       // valid output columns (= B.rows)
  float alpha;
  int epi;          // EpiMode
  int splits;       // split-K factor (SIMT engine, Gram only)
  int chain;        // tcgen05 engine: K blocks per accumulator chain (0 = default for epi)
  int l2_group;     // grouped launches: problems with the same non-zero id read the same
                    // operand planes - their items are ordered K-range-major so that
                    // one K range of all of them is in flight together (L2 reuse)
};

// grouped contraction (tcgen05 engine only): a host-side list of problems that is
// uploaded once as a device table and launched as ONE persistent kernel
struct SubGroup {
  int n_problems, n_items;
  size_t off_probs, off_items;
};
struct GroupInfo {
  SubGroup sub[4];                 // [0] single-CTA kernel, [1] CTA-pair kernel,
                                   // [2] sliding-window autocorrelation kernel,
                                   // [3] ordered combine (deterministic mode): n_problems =
                                   //     partial-tile slots at off_probs, n_items = output
                                   //     tiles (CombTile) at off_items
  int kind;                        // ProfKind of the launches (kProfGram / kProfGemm)
  size_t bytes;
};

// ---- ordered combine of partial tiles (deterministic mode) -------------------------
// A work item whose output tile has other contributors in the same launch stores its fp32
// partial tile (128 x 128, row-major, alpha applied, zeros where the epilogue masks) to a
// slot instead of red.add'ing it; one short launch after the contraction then adds each
// tile's slots into the running sum in slot order.  Slots are numbered by the table build,
// so the result does not depend on which CTA ran which item or when.
constexpr int kSlotElems = 128 * 128;
struct alignas(16) CombTile {
  float* out;              // first element of the output tile
  int ld, rows, cols;      // leading dimension, valid rows / columns of the tile
  int n, first;            // slot ids: list[first .. first + n), in summation order
  int pad[2];
};
// Host side: count every (output tile, contributor) of a launch first, then assign.  A tile
// with one contributor keeps the plain red.add (a single addend is exact and order-free).
struct DetCombine {
  std::unordered_map<const float*, int> counts;     // tile address -> contributors
  std::unordered_map<const float*, int> tile_of;    // tile address -> index into tiles
  std::vector<CombTile> tiles;
  std::vector<std::vector<int>> per_tile;           // slot ids, in build order
  int n_slots = 0;
  void count(const float* tile) { ++counts[tile]; }
  int contributors(const float* tile) const {
    auto it = counts.find(tile);
    return it == counts.end() ? 0 : it->second;
  }
  // slot id of one contribution to `tile`
  int assign(float* tile, int ld, int rows, int cols);
  // table memory from `off` on: CombTile[n] | int list | 256-aligned slots; fills sg and
  // returns the end offset
  size_t layout(size_t off, SubGroup* sg) const;
  static size_t bytes_bound(size_t items) {
    return items * ((size_t)kSlotElems * 4 + sizeof(CombTile) + 4) + 1024;
  }
};
int det_combine_upload(const DetCombine& det, void* table_dev, const SubGroup& sg,
                       cudaStream_t stream);
int det_combine_launch(const void* table_dev, const SubGroup& sg, int kind, cudaStream_t stream);

size_t group_table_bytes(const ContractionArgs* probs, int n);
// det != nullptr: the caller counted every contribution of the launch into det (and lays
// the combine out itself); det == nullptr in deterministic mode: the build does both
void group_table_count(const ContractionArgs* probs, int n, DetCombine* det);
int group_table_build(const ContractionArgs* probs, int n, int kind, void* table_dev,
                      size_t table_bytes, GroupInfo* info, cudaStream_t stream,
                      DetCombine* det = nullptr);
int group_launch(const void* table_dev, const GroupInfo& info, cudaStream_t stream);
// one sub-table of a group (0 generic kernel, 2 sliding-window kernel) on at most max_ctas
// SMs (0: all); pdl: programmatic dependent launch behind the kernel queued before it;
// partitioned: the CTA claims a whole SM's shared memory so that nothing else joins it
int group_launch_sub(const void* table_dev, const GroupInfo& info, int which, int max_ctas,
                     int pdl, cudaStream_t stream);

// slots: partial tiles of the items that carry a slot id (deterministic mode), else NULL
int contraction_launch_dev_items(const void* prob_dev, const void* items_dev, int max_items,
                                 const int* n_items_dev, int kind, float* slots,
                                 cudaStream_t stream);
int contraction_build_problem(const ContractionArgs& a, void* prob_host);
size_t contraction_problem_bytes();
size_t contraction_item_bytes();

int debug_read_counters(unsigned long long* out, int n);
int debug_tma_probe(const float* base, long long pitch_elems, int K, int rows, int iters,
                    int depth, unsigned long long* out_dev, int n_ctas, cudaStream_t stream);
int debug_occupy(int threads, size_t smem, long long cycles, int n_ctas, cudaStream_t stream);
int debug_tma3d_probe(const float* base, long long img_elems, int B, int box_rows,
                      int boxes_per_cta, int depth, unsigned long long* out_dev, int n_ctas,
                      cudaStream_t stream);
int debug_bulk_probe(const void* src, long long bytes_per_cta, int chunk, int depth,
                     unsigned long long* out_dev, int n_ctas, cudaStream_t stream);
int debug_mma_rate(int mode, int iters, unsigned long long* out_dev, int n_ctas,
                   cudaStream_t stream);

// sliding-window autocorrelation kernel (contraction_ac.cu)
struct ConvGeom;
bool autocorr_kernel_enabled();
int debug_read_ac_counters(unsigned long long* out, int n);
size_t autocorr_table_bytes(const ConvGeom* geoms, int n);
// deterministic mode: autocorr_count adds the output tiles of the layers to det before the
// build, which then gives every item whose tiles have other contributors its slots
void autocorr_count(const ConvGeom* geoms, float* const* accs, int n, DetCombine* det);
int autocorr_table_build(const ConvGeom* geoms, const float* const* stages, float* const* accs,
                         int n, void* table_dev, size_t table_bytes, SubGroup* sg,
                         cudaStream_t stream, DetCombine* det = nullptr);
int autocorr_launch(const void* table_dev, const SubGroup& sg, cudaStream_t stream,
                    int max_ctas = 0, int pdl = 0, float* slots = nullptr);

// engines
int contraction_simt(const ContractionArgs& a, cudaStream_t stream);
int contraction_tc(const ContractionArgs& a, cudaStream_t stream);      // tcgen05/TMA
int contraction(const ContractionArgs& a, cudaStream_t stream);         // dispatch on g_engine
// One engine ships: tcgen05.  A -DNSGP_BRINGUP build (make BRINGUP=1) adds the SIMT
// cross-check engine, the CTA-pair kernel and the environment switches of DESIGN.md 6b.
#ifdef NSGP_BRINGUP
extern int g_engine;   // 0 = tcgen05 (product), 1 = SIMT (bring-up / cross-check)
static inline const char* nsgp_env(const char* name) { return getenv(name); }
#else
constexpr int g_engine = 0;
static inline const char* nsgp_env(const char*) { return nullptr; }
#endif

namespace tc { int sm_count(); }
// 3-D fp32 tensor map (x: 256 floats, y: rows of 1 KB, z: images `img_elems` apart), box
// (256, box_rows, B), no swizzle: the batch-mean staging kernel's view of a layer input
int encode_batch_rows_map(CUtensorMap* dst, const float* base, long long img_elems, int B,
                          int box_rows);

// number of 32-wide K blocks of an operand
static inline int k_blocks(const Operand& o) { return ceil_div(o.K, 32); }

}  // namespace nsgp
