// Sliding-window autocorrelation kernel (tcgen05 / TMEM / TMA, 3xTF32) for the 3x3 s1 p1
// covariance (geometry.h, "autocorrelation layout").
//
// The 13 blocks  R_(dy,dx)[c,c'] = sum_{u,x} a[c][u][x] * b[c'][u+dy][x]   (a, b = column-
// shifted copies of the batch-mean map) share operands: for a fixed column strip x0..x0+31
// and a fixed pair of copies, the B tile of row u+1 serves dy = 1 at row u and dy = 0 at
// row u+1.  Walking the rows of a strip with a 3-tile window of B,
//     acc[dy] += A(u) * B(u+dy)^T ,  dy = 0,1,2 ,
// costs ONE new A tile and ONE new B tile per row for THREE MMA sets - three times the
// tensor work per byte brought into shared memory of the generic GEMM kernel, whose
// operand ring is latency-bound (profiles/counters_r01.txt).
//
//   warps 0, 6  TMA producers: B ring (4 x 32 KB: hi|lo of 128 channels x 32 columns) and
//               A ring (3 x 32 KB); operands staged tile-major, one contiguous 16 KB box
//               per plane (SWIZZLE_128B)
//   warp 1      MMA issuer: per row 3 x 12 tcgen05.mma.kind::tf32 (M=128, N<=128, K=8) into
//               three TMEM accumulators (one per dy), commits free the A slot and the
//               oldest B slot
//   warps 2..5  epilogue: three 128 x 128 tiles -> red.global.add.v4.f32 into R_(dy,dx)
//
// Work item = (copy pair / dx, tile (rb, cb), column strip, row range <= 32 rows): the row
// range bounds the accumulation chain (12 accumulate steps per row, see DESIGN.md).
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "geometry.h"
#include "tc_common.cuh"

namespace nsgp {

using namespace tc;

namespace {

constexpr int SA = 3;                       // A ring stages
constexpr int SB = 4;                       // B ring stages (3 in the window + 1 in flight)
constexpr uint32_t kPlane = BM * BK * 4;    // 16 KB: one hi or lo plane of a tile
constexpr uint32_t kTile = 2 * kPlane;      // hi | lo
// rows per work item = accumulation chain of 12 steps per row (bias of the truncating tensor-core
// accumulate ~1.9e-8 per step)
constexpr int kRowsPerItem = 48;
constexpr int kThreadsAc = 224;             // 7 warps: B producer, MMA, 4 epilogue, A producer
constexpr size_t kSmemAc = (size_t)(SA + SB) * kTile + 1024 + 256;

struct alignas(64) AcProblem {
  CUtensorMap maps[2];                      // [hi/lo]: (32, n_tiles * 128), rows 128 B apart
  float* acc;                               // 29 matrices C x ldc (geometry.h)
  int C, H, W, ldc;
  int Hs, NS;                               // staged rows per copy, column strips
  int tiles;                                // channel blocks = ceil(C / 128)
  int pad0;
};
struct alignas(16) AcItem {
  int prob, pass, rb, cb;
  int x0, u0, u1, slot;       // slot > 0: the tiles dy0..2 go to slots slot-1, slot, ...
};

// pass -> (A copy, B copy, dx, first dy)
__host__ __device__ __forceinline__ void pass_info(int pass, int rb, int cb, int* sa, int* sb, int* dx,
                                          int* dy0) {
  *sa = pass == 3 ? 1 : (pass == 4 ? 2 : 0);
  *sb = pass == 1 ? 1 : (pass == 2 ? 2 : 0);
  *dx = pass == 0 ? 0 : (pass == 1 ? 1 : (pass == 2 ? 2 : (pass == 3 ? -1 : -2)));
  // dx = 0: R_(0,0) is symmetric - tiles below the diagonal only need dy = 1, 2;
  // dx < 0 occurs only with dy >= 1 in the upper triangle of the covariance
  *dy0 = (pass >= 3 || (pass == 0 && rb > cb)) ? 1 : 0;
}

__device__ __forceinline__ void tma_load_3d_elect(uint32_t dst, const CUtensorMap* map,
                                                  uint64_t* bar, int x, int u, int c) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];\n\t}" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(x), "r"(u), "r"(c)
      : "memory");
}

__device__ unsigned long long g_ac_counters[160 * 8];

__global__ void __launch_bounds__(kThreadsAc, 1)
autocorr_tc_kernel(const AcProblem* __restrict__ probs, const AcItem* __restrict__ items,
                   int n_items, int dbg, unsigned long long* tl, int* __restrict__ sched,
                   float* __restrict__ slots) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_ring = smem;                          // SA tiles
  uint8_t* b_ring = smem + SA * kTile;             // SB tiles
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + (SA + SB) * kTile);
  uint64_t* a_empty = a_full + SA;
  uint64_t* b_full = a_empty + SA;
  uint64_t* b_empty = b_full + SB;
  uint64_t* tmem_full = b_empty + SB;
  uint64_t* tmem_empty = tmem_full + 1;
  // dynamic work distribution: warp 0 draws item indices from a global ticket counter (the
  // list is sorted by descending cost, so this is longest-processing-time-first) and hands
  // them to the other six warps through a 4-deep ring
  constexpr int kSched = 4;
  uint64_t* sched_full = tmem_empty + 1;
  uint64_t* sched_empty = sched_full + kSched;
  int* sched_item = reinterpret_cast<int*>(sched_empty + kSched);
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(sched_item + kSched);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long t_start = clock64();
  long long c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0;
  // programmatic dependent launch: the staging kernel of the NEXT forward, queued behind this
  // launch, may start on the SMs this grid leaves free as soon as all CTAs are running
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  tl_begin(tl);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < SA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < SB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 4);
    for (int s = 0; s < kSched; ++s) { mbar_init(&sched_full[s], 1); mbar_init(&sched_empty[s], 6); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_base_slot)),
                 "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  uint32_t sched_cnt = 0;
  // warp 0: draw the next item (-1: list exhausted) and publish it
  auto sched_draw = [&]() -> int {
    const uint32_t s = sched_cnt % kSched, par = (sched_cnt / kSched) & 1;
    mbar_wait_warp(&sched_empty[s], par ^ 1, lane);
    int idx = 0;
    if (lane == 0) {
      idx = atomicAdd(sched, 1);
      if (idx >= n_items) idx = -1;
      sched_item[s] = idx;
      mbar_arrive(&sched_full[s]);
    }
    idx = __shfl_sync(0xffffffffu, idx, 0);
    ++sched_cnt;
    return idx;
  };
  // the other warps: take the next published item
  auto sched_take = [&]() -> int {
    const uint32_t s = sched_cnt % kSched, par = (sched_cnt / kSched) & 1;
    mbar_wait_warp(&sched_full[s], par, lane);
    const int idx = *reinterpret_cast<volatile int*>(&sched_item[s]);
    __syncwarp();
    if (lane == 0) mbar_arrive(&sched_empty[s]);
    ++sched_cnt;
    return idx;
  };

  if (warp == 0 || warp == 6) {
    // ============================ TMA producers ============================
    // warp 0 feeds the B ring, warp 6 the A ring: each runs as far ahead as its own ring
    // allows (one warp for both made every A load wait behind the next B slot)
    const bool is_b = warp == 0;
    uint32_t cnt = 0;
    for (;;) {
      const int idx = is_b ? sched_draw() : sched_take();
      if (idx < 0) break;
      const AcItem it = items[idx];
      const AcProblem& p = probs[it.prob];
      int sa, sb, dx, dy0;
      pass_info(it.pass, it.rb, it.cb, &sa, &sb, &dx, &dy0);
      // tile (copy s, channel block cb, row u, strip st) starts at row
      // (((s * tiles + cb) * Hs + u) * NS + st) * 128 of the tile matrix
      const int st = it.x0 / BK;
      const int n = it.u1 - it.u0;
      if (is_b) {
        const long long tile0 = ((long long)(sb * p.tiles + it.cb) * p.Hs + it.u0) * p.NS + st;
        for (int i = 0; i < n + 2; ++i) {
          const uint32_t s = cnt % SB, par = (cnt / SB) & 1;
          long long q0 = dbg ? clock64() : 0;
          mbar_wait_warp(&b_empty[s], par ^ 1, lane);
          if (dbg) c0 += clock64() - q0;
          mbar_expect_tx_elect(&b_full[s], kTile);
          // B ring = [hi planes of the SB slots | lo planes]: neighbouring window tiles are
          // contiguous per plane, so one N = 256 MMA can cover two of them
          const uint32_t dst = smem_u32(b_ring + s * kPlane);
          const int row = (int)((tile0 + (long long)i * p.NS) * BM);
          tma_load_2d_elect(dst, &p.maps[0], &b_full[s], 0, row);
          tma_load_2d_elect(dst + SB * kPlane, &p.maps[1], &b_full[s], 0, row);
          ++cnt;
        }
      } else {
        const long long tile0 = ((long long)(sa * p.tiles + it.rb) * p.Hs + it.u0) * p.NS + st;
        for (int j = 0; j < n; ++j) {
          const uint32_t s = cnt % SA, par = (cnt / SA) & 1;
          long long q0 = dbg ? clock64() : 0;
          mbar_wait_warp(&a_empty[s], par ^ 1, lane);
          if (dbg) c1 += clock64() - q0;
          mbar_expect_tx_elect(&a_full[s], kTile);
          const uint32_t dst = smem_u32(a_ring + s * kTile);
          const int row = (int)((tile0 + (long long)j * p.NS) * BM);
          tma_load_2d_elect(dst, &p.maps[0], &a_full[s], 0, row);
          tma_load_2d_elect(dst + kPlane, &p.maps[1], &a_full[s], 0, row);
          ++cnt;
        }
      }
    }
    if (dbg && lane == 0) {
      if (is_b) g_ac_counters[blockIdx.x * 8 + 5] = c0;
      else g_ac_counters[blockIdx.x * 8 + 6] = c1;
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ============================
    uint32_t a_cnt = 0, b_cnt = 0, n_done = 0;
    for (;; ++n_done) {
      const int idx = sched_take();
      if (idx < 0) break;
      const AcItem it = items[idx];
      const AcProblem& p = probs[it.prob];
      int sa, sb, dx, dy0;
      pass_info(it.pass, it.rb, it.cb, &sa, &sb, &dx, &dy0);
      int n_valid = p.C - it.cb * BM;
      if (n_valid > BM) n_valid = BM;
      const uint32_t idesc = make_idesc_tf32(BM, (n_valid + 15) & ~15);
      // two accumulators at once need full 128-column tiles (the second starts at column 128)
      const uint32_t idesc2 = make_idesc_tf32(BM, 2 * BM);
      const bool wide = n_valid == BM;
      const int n = it.u1 - it.u0;
      long long q0 = dbg ? clock64() : 0;
      mbar_wait_warp(tmem_empty, (n_done & 1) ^ 1, lane);     // epilogue drained the accumulators
      if (dbg) c2 += clock64() - q0;
      tc_fence_after();
      // B tiles 0 and 1 of this item
      for (int i = 0; i < 2; ++i) {
        const uint32_t c = b_cnt + i;
        mbar_wait_warp(&b_full[c % SB], (c / SB) & 1, lane);
      }
      for (int j = 0; j < n; ++j) {
        const uint32_t as = a_cnt % SA, ap = (a_cnt / SA) & 1;
        const uint32_t b2 = b_cnt + 2;
        long long q1 = dbg ? clock64() : 0;
        mbar_wait_warp(&a_full[as], ap, lane);
        long long q2 = dbg ? clock64() : 0;
        mbar_wait_warp(&b_full[b2 % SB], (b2 / SB) & 1, lane);
        long long q3 = dbg ? clock64() : 0;
        c0 += q2 - q1; c1 += q3 - q2; ++c4;
        tc_fence_after();
        const uint32_t abase = smem_u32(a_ring + as * kTile);
        const uint64_t a_hi = make_kmajor_sw128_desc(abase);
        const uint64_t a_lo = make_kmajor_sw128_desc(abase + kPlane);
        // An M128 x N128 x K8 tf32 MMA reads 8 KB of operands per 64 cycles = the SM's whole
        // shared-memory bandwidth (DESIGN.md 4).  Two neighbouring window tiles that are also
        // neighbours in the ring (no wrap) go through ONE N = 256 MMA into their two
        // neighbouring accumulators: A is read once for both.
        for (int dy = dy0; dy < 3;) {
          const uint32_t bs = (b_cnt + dy) % SB;
          const bool two = wide && dy + 1 < 3 && bs + 1 < SB;
          const uint32_t bbase = smem_u32(b_ring + bs * kPlane);
          const uint64_t b_hi = make_kmajor_sw128_desc(bbase);
          const uint64_t b_lo = make_kmajor_sw128_desc(bbase + SB * kPlane);
          const uint32_t d = tmem_base + dy * BM;
          tc_mma_kblock_3xtf32(d, d, a_hi, a_lo, b_hi, b_lo, two ? idesc2 : idesc,
                               j > 0 ? 1u : 0u, 1u);
          dy += two ? 2 : 1;
        }
        tc_commit_elect(&a_empty[as]);                // A(j) free when these MMAs retire
        tc_commit_elect(&b_empty[b_cnt % SB]);        // B(j) is not needed after row j
        if (dbg) c3 += clock64() - q3;
        ++a_cnt;
        ++b_cnt;
      }
      // the last two window tiles, then hand the accumulators to the epilogue
      tc_commit_elect(&b_empty[b_cnt % SB]);
      tc_commit_elect(&b_empty[(b_cnt + 1) % SB]);
      b_cnt += 2;
      tc_commit_elect(tmem_full);
    }
    if (dbg && lane == 0) {
      g_ac_counters[blockIdx.x * 8 + 0] = c0;     // wait A
      g_ac_counters[blockIdx.x * 8 + 1] = c1;     // wait B
      g_ac_counters[blockIdx.x * 8 + 2] = c2;     // wait accumulators (epilogue)
      g_ac_counters[blockIdx.x * 8 + 3] = c3;     // issue
      g_ac_counters[blockIdx.x * 8 + 4] = c4;     // row steps
      g_ac_counters[blockIdx.x * 8 + 7] = clock64() - t_start;
    }
  } else {
    // ============================ epilogue ============================
    const int quad = warp & 3;
    uint32_t n_done = 0;
    for (;; ++n_done) {
      const int idx = sched_take();
      if (idx < 0) break;
      const AcItem it = items[idx];
      const AcProblem& p = probs[it.prob];
      int sa, sb, dx, dy0;
      pass_info(it.pass, it.rb, it.cb, &sa, &sb, &dx, &dy0);
      mbar_wait_warp(tmem_full, n_done & 1, lane, 200);
      tc_fence_after();
      const int row = it.rb * BM + quad * 32 + lane;
      const bool row_ok = row < p.C;
      const int C = p.C;
      const bool vec = (p.ldc % 4 == 0);
      for (int dy = dy0; dy < 3; ++dy) {
        float* mat = p.acc + (long long)ac_ridx(dy, dx) * C * p.ldc;
        float* orow = mat + (long long)row * p.ldc;
        // deterministic mode: the partial tile goes to its slot (zeros where masked)
        float* srow = it.slot > 0 ? slots + (size_t)(it.slot - 1 + dy - dy0) * kSlotElems +
                                        (quad * 32 + lane) * 128
                                  : nullptr;
#pragma unroll 1
        for (int chunk = 0; chunk < BM / 32; ++chunk) {
          uint32_t v[32];
          const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + dy * BM + chunk * 32;
          tc_ld32(taddr, v);
          tc_wait_ld();
          const int col0 = it.cb * BM + chunk * 32;
          if (srow != nullptr) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const int col = col0 + j;
              float4 x;
              x.x = row_ok && col < C ? __uint_as_float(v[j]) : 0.f;
              x.y = row_ok && col + 1 < C ? __uint_as_float(v[j + 1]) : 0.f;
              x.z = row_ok && col + 2 < C ? __uint_as_float(v[j + 2]) : 0.f;
              x.w = row_ok && col + 3 < C ? __uint_as_float(v[j + 3]) : 0.f;
              *reinterpret_cast<float4*>(srow + chunk * 32 + j) = x;
            }
          } else if (row_ok && col0 < C) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const int col = col0 + j;
              const float x0 = __uint_as_float(v[j]), x1 = __uint_as_float(v[j + 1]),
                          x2 = __uint_as_float(v[j + 2]), x3 = __uint_as_float(v[j + 3]);
              if (vec && col + 3 < C) {
                red_add_v4(orow + col, x0, x1, x2, x3);
              } else {
                if (col < C) atomicAdd(orow + col, x0);
                if (col + 1 < C) atomicAdd(orow + col + 1, x1);
                if (col + 2 < C) atomicAdd(orow + col + 2, x2);
                if (col + 3 < C) atomicAdd(orow + col + 3, x3);
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty);
    }
  }

  tc_fence_before();
  __syncthreads();
  tl_end(tl);
  // the last CTA to leave rewinds the ticket counter for the next launch of this table
  if (threadIdx.x == 0 && atomicAdd(sched + 1, 1) == (int)gridDim.x - 1) {
    atomicExch(sched, 0);
    atomicExch(sched + 1, 0);
  }
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(512)
                 : "memory");
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) ==
            cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<EncodeTiledFn>(p);
    return (EncodeTiledFn) nullptr;
  }();
  return fn;
}

}  // namespace

int debug_read_ac_counters(unsigned long long* out, int n) {
  NSGP_CHECK_CUDA(cudaMemcpyFromSymbol(out, g_ac_counters, (size_t)n * sizeof(unsigned long long)));
  return 0;
}

bool autocorr_kernel_enabled() {
  static const bool on = [] {
    const char* e = nsgp_env("NSGP_AC_KERNEL");          // 0 disables (generic GEMM problems)
    return !(e && e[0] == '0');
  }();
  return on;
}

size_t autocorr_table_bytes(const ConvGeom* geoms, int n) {
  size_t items = 0;
  for (int i = 0; i < n; ++i) {
    const ConvGeom& g = geoms[i];
    const size_t t = (size_t)ceil_div(g.C, BM);
    items += 5 * t * t * (size_t)ceil_div(g.W, BK) * (size_t)ceil_div(g.H, kRowsPerItem);
  }
  // deterministic mode: up to three partial tiles per item
  return (size_t)n * sizeof(AcProblem) + items * sizeof(AcItem) + 1024 +
         (g_deterministic ? DetCombine::bytes_bound(3 * items) : 0);
}

// output tile of (layer accumulator, pass, dy, tile) - the address the epilogue adds into
static float* ac_tile(float* acc, const ConvGeom& g, int pass, int dy, int rb, int cb) {
  int sa, sb, dx, dy0;
  pass_info(pass, rb, cb, &sa, &sb, &dx, &dy0);
  const int ldc = (int)round_up(g.C, 4);
  return acc + (long long)ac_ridx(dy, dx) * g.C * ldc + (long long)rb * BM * ldc + cb * BM;
}

void autocorr_count(const ConvGeom* geoms, float* const* accs, int n, DetCombine* det) {
  for (int i = 0; i < n; ++i) {
    const ConvGeom& g = geoms[i];
    const int tiles = ac_cblocks(g), strips = ceil_div(g.W, BK);
    for (int u0 = 0; u0 < g.H; u0 += kRowsPerItem)
      for (int st = 0; st < strips; ++st)
        for (int pass = 0; pass < 5; ++pass)
          for (int rb = 0; rb < tiles; ++rb)
            for (int cb = 0; cb < tiles; ++cb) {
              int sa, sb, dx, dy0;
              pass_info(pass, rb, cb, &sa, &sb, &dx, &dy0);
              for (int dy = dy0; dy < 3; ++dy) det->count(ac_tile(accs[i], g, pass, dy, rb, cb));
            }
  }
}

// geoms[i] / stages[i] / accs[i]: staged autocorrelation layers.  Uploads the table.
int autocorr_table_build(const ConvGeom* geoms, const float* const* stages, float* const* accs,
                         int n, void* table_dev, size_t table_bytes, SubGroup* sg,
                         cudaStream_t stream, DetCombine* det) {
  EncodeTiledFn enc = encode_fn();
  NSGP_REQUIRE(enc != nullptr, "autocorr kernel: cuTensorMapEncodeTiled is unavailable");
  std::vector<AcProblem> hp(n);
  struct Key { int rows, layer, u0, x0, pass, tile; AcItem it; };
  std::vector<Key> keys;
  for (int i = 0; i < n; ++i) {
    const ConvGeom& g = geoms[i];
    AcProblem& p = hp[i];
    memset(&p, 0, sizeof(p));
    p.acc = accs[i];
    p.C = g.C; p.H = g.H; p.W = g.W;
    p.ldc = (int)round_up(g.C, 4);
    p.tiles = ac_cblocks(g);
    p.Hs = g.Hs;
    p.NS = ac_strips(g);
    NSGP_REQUIRE(g.tiled, "autocorr kernel needs the tiled staging layout");
    const long long hl = stage_hl_stride(g);
    const long long n_rows = 3LL * p.tiles * g.Hs * p.NS * BM;
    NSGP_REQUIRE(n_rows < (1LL << 31), "autocorr kernel: staged operand too large");
    for (int h = 0; h < 2; ++h) {
      const float* base = stages[i] + h * hl;
      cuuint64_t gdim[2] = {(cuuint64_t)BK, (cuuint64_t)n_rows};
      cuuint64_t gstr[1] = {(cuuint64_t)BK * 4};
      cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&p.maps[h], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr,
                       box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      NSGP_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (autocorr) failed (%d)", (int)r);
    }
    const int strips = ceil_div(g.W, BK);
    for (int u0 = 0; u0 < g.H; u0 += kRowsPerItem) {
      const int u1 = u0 + kRowsPerItem < g.H ? u0 + kRowsPerItem : g.H;
      for (int st = 0; st < strips; ++st)
        for (int pass = 0; pass < 5; ++pass)
          for (int rb = 0; rb < p.tiles; ++rb)
            for (int cb = 0; cb < p.tiles; ++cb) {
              Key k;
              k.rows = u1 - u0; k.layer = i; k.u0 = u0; k.x0 = st * BK; k.pass = pass;
              k.tile = rb * p.tiles + cb;
              int slot = 0;
              if (det != nullptr) {
                int sa, sb, dx, dy0;
                pass_info(pass, rb, cb, &sa, &sb, &dx, &dy0);
                bool shared = false;
                for (int dy = dy0; dy < 3; ++dy)
                  shared |= det->contributors(ac_tile(accs[i], g, pass, dy, rb, cb)) > 1;
                if (shared) {
                  // consecutive slots, one per tile dy0..2
                  const int rows = g.C - rb * BM, cols = g.C - cb * BM;
                  for (int dy = dy0; dy < 3; ++dy) {
                    const int s = det->assign(ac_tile(accs[i], g, pass, dy, rb, cb), p.ldc,
                                              rows < BM ? rows : BM, cols < BM ? cols : BM);
                    if (dy == dy0) slot = s + 1;
                  }
                }
              }
              k.it = AcItem{i, pass, rb, cb, st * BK, u0, u1, slot};
              keys.push_back(k);
            }
    }
  }
  // long items first; within a layer all (pass, tile) items of one (row range, strip) are
  // adjacent so that they run together and share the operand rows in L2
  std::stable_sort(keys.begin(), keys.end(), [](const Key& a, const Key& b) {
    if (a.rows != b.rows) return a.rows > b.rows;
    if (a.layer != b.layer) return a.layer < b.layer;
    if (a.u0 != b.u0) return a.u0 < b.u0;
    if (a.x0 != b.x0) return a.x0 < b.x0;
    if (a.pass != b.pass) return a.pass < b.pass;
    return a.tile < b.tile;
  });
  sg->n_problems = n;
  sg->n_items = (int)keys.size();
  sg->off_probs = 0;
  sg->off_items = (size_t)n * sizeof(AcProblem);
  const size_t need = sg->off_items + keys.size() * sizeof(AcItem) + 64;   // + ticket, done
  NSGP_REQUIRE(need <= table_bytes, "autocorr table too small (%zu < %zu)", table_bytes, need);
  NSGP_REQUIRE((reinterpret_cast<uintptr_t>(table_dev) & 63) == 0,
               "autocorr table must be 64-byte aligned");
  std::vector<AcItem> hi(keys.size());
  for (size_t i = 0; i < keys.size(); ++i) hi[i] = keys[i].it;
  if (n > 0) {
    NSGP_CHECK_CUDA(cudaMemcpyAsync(table_dev, hp.data(), (size_t)n * sizeof(AcProblem),
                                    cudaMemcpyHostToDevice, stream));
    NSGP_CHECK_CUDA(cudaMemcpyAsync((char*)table_dev + sg->off_items, hi.data(),
                                    hi.size() * sizeof(AcItem), cudaMemcpyHostToDevice, stream));
    NSGP_CHECK_CUDA(cudaMemsetAsync((char*)table_dev + sg->off_items + hi.size() * sizeof(AcItem),
                                    0, 64, stream));
  }
  return 0;
}

int autocorr_launch(const void* table_dev, const SubGroup& sg, cudaStream_t stream, int max_ctas,
                    int pdl, float* slots) {
  if (sg.n_items == 0) return 0;
  static bool configured = false;
  if (!configured) {
    NSGP_CHECK_CUDA(cudaFuncSetAttribute(autocorr_tc_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSmemAc));
    configured = true;
  }
  const AcProblem* probs = reinterpret_cast<const AcProblem*>((const char*)table_dev + sg.off_probs);
  const AcItem* items = reinterpret_cast<const AcItem*>((const char*)table_dev + sg.off_items);
  int grid = sg.n_items < sm_count() ? sg.n_items : sm_count();
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  ProfScope prof(kProfGram, stream);
  static const int dbg = nsgp_env("NSGP_DBG_COUNTERS") ? 1 : 0;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreadsAc);
  cfg.dynamicSmemBytes = kSmemAc;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  int* sched = reinterpret_cast<int*>(const_cast<char*>((const char*)table_dev) + sg.off_items +
                                      (size_t)sg.n_items * sizeof(AcItem));
  NSGP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, autocorr_tc_kernel, probs, items, sg.n_items, dbg,
                                     timeline_slot(10), sched, slots));
  NSGP_LAUNCHED();
  return 0;
}

}  // namespace nsgp
