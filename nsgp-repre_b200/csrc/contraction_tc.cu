// tcgen05 / TMEM / TMA contraction engine (sm_100a), 3xTF32 with fp32 accumulation.
//
//   out (+)= A * B^T      A: rows_a x K, B: rows_b x K, both K-major "virtual"
//                         operands over staged hi/lo planes (common.cuh).
//
// Every operand element was pre-split into hi = rna_tf32(x), lo = rna_tf32(x - hi)
// so the tensor core's tf32 truncation of the shared-memory words is a no-op and
//   A*B^T ~= A_hi*B_hi + A_hi*B_lo + A_lo*B_hi        (error ~2^-21 relative)
// is accumulated in fp32 in TMEM.
//
// One persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer   (cp.async.bulk.tensor.3d, SWIZZLE_128B, mbarrier tx)
//   warp 1      MMA issuer     (tcgen05.mma kind::tf32, M=128, N=BN, K=8), TMEM owner
//   warps 2..5  epilogue       (tcgen05.ld 32x32b -> registers -> global)
// Three pipelines: smem full/empty ring (TMA <-> MMA), TMEM full/empty double
// buffer (MMA <-> epilogue), static round-robin work list (tile, K-split).
//
// Work item = (output tile 128 x BN, K range).  For the Gram epilogue only tiles
// touching the upper block-triangle are visited, K is split across items and the
// tile is red.add'ed into the running sum; the K chain per item is bounded so the
// fp32 accumulation chain inside the tensor core stays short.  For the GEMM
// epilogue tiles are exclusive and the tile is read-modify-written
// (out += alpha * acc).
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <vector>
#include <unordered_map>

#include "common.cuh"
#include "tc_common.cuh"

namespace nsgp {

using namespace tc;

namespace {

// ---------------------------------------------------------------- work items
constexpr int BN = 128;            // tile columns (UMMA N)
constexpr int STAGES = 3;
constexpr uint32_t kABytes = BM * BK * 4;       // 16 KB, one operand plane of a stage
constexpr uint32_t kStageBytes = 4 * kABytes;   // A_hi | A_lo | B_hi | B_lo
// TMEM: 2 buffers x (main accumulator | correction accumulator) x 128 columns.
// hi*hi goes to `main`, the two 2^-11-sized cross terms to `corr`: the long chain
// of large addends is a third as long, and the small terms do not get truncated at
// the scale of the large sum.  The epilogue adds them in fp32 (round-to-nearest).
constexpr uint32_t kTmemCols = 512;
// K blocks the L2 prefetch cursor of the producer runs ahead of its loads
constexpr int kPrefetchDist = 8;

// number of br-row TMA boxes covering [r0, r0+128) below `rows`
__device__ __forceinline__ int seg_count(int r0, int rows, int br) {
  int n = 0;
  for (int r = r0; r < r0 + BM && r < rows; r += br) ++n;
  return n;
}

struct Item {
  const TcMaps* maps;
  const TcParams* p;
  int rb, cb, kb0, kb1;
  int slot;                  // > 0: partial tile goes to slot (slot - 1), see DetCombine
};

// Single problem: items are (K split, tile) pairs enumerated arithmetically; Gram
// problems visit the upper block-triangle only.  Group: the list is in global memory.
__device__ __forceinline__ Item fetch_item(const TcMaps* pmaps, const TcParams* pp,
                                           const TcProblem* gprobs, const TcItem* gitems,
                                           int idx) {
  Item it;
  if (gitems != nullptr) {
    const int4 a = *reinterpret_cast<const int4*>(&gitems[idx]);
    const int4 b = *reinterpret_cast<const int4*>(&gitems[idx].kb1);
    it.maps = &gprobs[a.x].maps;
    it.p = &gprobs[a.x].p;
    it.rb = a.y; it.cb = a.z; it.kb0 = a.w; it.kb1 = b.x;
    it.slot = b.y;
    return it;
  }
  it.maps = pmaps;
  it.p = pp;
  it.slot = 0;
  const int split = idx / pp->n_tiles;
  int tile = idx - split * pp->n_tiles;
  if (pp->gram) {
    int rb = 0;
    for (;; ++rb) {                       // tiles_m <= 36: short walk
      const int cnt = pp->tiles_n - rb;
      if (tile < cnt) break;
      tile -= cnt;
    }
    it.rb = rb; it.cb = rb + tile;
  } else {
    it.rb = tile / pp->tiles_n;
    it.cb = tile - it.rb * pp->tiles_n;
  }
  it.kb0 = (int)((long long)pp->nkb * split / pp->splits);
  it.kb1 = (int)((long long)pp->nkb * (split + 1) / pp->splits);
  return it;
}

// Bring-up instrumentation (NSGP_DBG_COUNTERS=1): per-CTA cycle counters of where the
// producer and the MMA issuer spend their time.  [0] MMA warp waiting for operands
// (full barrier), [1] MMA warp issuing (blocks on the tensor pipe), [2] MMA warp waiting
// for a free accumulator, [3] producer waiting for a free stage, [4] producer issuing
// (blocks on the TMA unit), [5] total, [6] K blocks.
__device__ unsigned long long g_dbg_counters[160 * 8];

// ---------------------------------------------------------------- the kernel
// PAIR = false: one CTA per 128 x 128 tile.
// PAIR = true : a CTA pair (cluster of 2, cta_group::2) per 256 x 256 tile.  Each CTA
//   owns 128 of the tile rows (its A tile) and stages half of the B rows; the MMA unit
//   of each SM reads the other half from the peer.  Per output element that is half
//   the TMA traffic of the single-CTA kernel - and TMA issue throughput (~58 B/cycle/SM
//   measured with NSGP_DBG_COUNTERS) is what bounds the single-CTA kernel.
template <bool PAIR>
__global__ void __launch_bounds__(kThreads, 1)
contraction_tc_kernel(const __grid_constant__ TcMaps pmaps, const __grid_constant__ TcParams pp,
                      const TcProblem* __restrict__ gprobs, const TcItem* __restrict__ gitems,
                      int n_items_max, int dbg,
                      unsigned long long* tl, const int* __restrict__ n_items_dev,
                      float* __restrict__ slots) {
  // the item count may live in device memory (work lists generated on the device)
  const int n_items = n_items_dev != nullptr ? min(n_items_max, __ldg(n_items_dev)) : n_items_max;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * kStageBytes);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* peer_full = tmem_empty + 2;          // pair: "the peer's half of stage s landed"
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(peer_full + STAGES);

  constexpr int TILE = PAIR ? 256 : 128;         // tile edge in rows / columns
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = PAIR ? (int)cluster_ctarank() : 0;
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const long long t_start = clock64();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // see autocorr_tc_kernel
  tl_begin(tl);
  long long c_wait = 0, c_issue = 0, c_acc = 0, c_kb = 0;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
      mbar_init(&peer_full[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], PAIR ? 8 : 4);   // epilogue warps (of both CTAs)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(tmem_base_slot)),
                   "r"(kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(tmem_base_slot)),
                   "r"(kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;

  if (warp == 0) {
    // ============================ TMA producer ============================
    // The whole warp runs the loop with warp-uniform values; the single issuing thread
    // is elected inside each asm block (see tc_common.cuh).  A second cursor runs
    // kPrefetchDist K blocks ahead and pulls the operand rows into L2 - by exactly one
    // worker per row block (diagonal tile for Gram, first tile of the row / column for
    // GEMM) - so that the ring's load latency is an L2 hit, not a DRAM fill that every
    // CTA of the wave waits for together.
    uint32_t stage = 0, phase = 0;
    int pf_idx = worker, pf_kb = 0;
    Item pf_it{};
    bool pf_live = pf_idx < n_items;
    if (pf_live) { pf_it = fetch_item(&pmaps, &pp, gprobs, gitems, pf_idx); pf_kb = pf_it.kb0; }
    auto prefetch_step = [&]() {
      if (!pf_live) return;
      const TcParams& q = *pf_it.p;
      const bool pa = q.gram ? (pf_it.rb == pf_it.cb) : (pf_it.cb == 0);
      const bool pb = q.gram ? false : (pf_it.rb == 0);
      const int kx = pf_kb * BK;
      if (pa) {
        const int r0 = pf_it.rb * TILE + rank * BM;
        for (int r = r0; r < r0 + BM && r < q.A.rows; r += q.A.br) {
          const int t = r / q.A.Cs, c = r - t * q.A.Cs;
          tma_prefetch_2d_elect(&pf_it.maps->a[0][t], kx, c);
          tma_prefetch_2d_elect(&pf_it.maps->a[1][t], kx, c);
        }
      }
      if (pb) {
        const int c0 = pf_it.cb * TILE + rank * BM;
        for (int r = c0; r < c0 + BM && r < q.B.rows; r += q.B.br) {
          const int t = r / q.B.Cs, c = r - t * q.B.Cs;
          tma_prefetch_2d_elect(&pf_it.maps->b[0][t], kx, c);
          tma_prefetch_2d_elect(&pf_it.maps->b[1][t], kx, c);
        }
      }
      if (++pf_kb >= pf_it.kb1) {
        pf_idx += n_workers;
        pf_live = pf_idx < n_items;
        if (pf_live) { pf_it = fetch_item(&pmaps, &pp, gprobs, gitems, pf_idx); pf_kb = pf_it.kb0; }
      }
    };
    for (int i = 0; i < kPrefetchDist; ++i) prefetch_step();
    for (int idx = worker; idx < n_items; idx += n_workers) {
      const Item it = fetch_item(&pmaps, &pp, gprobs, gitems, idx);
      const TcParams& p = *it.p;
      const int r0 = it.rb * TILE + rank * BM;    // this CTA's A rows
      const int c0 = it.cb * TILE + rank * BM;    // the B rows this CTA stages
      const bool share = p.gram && p.same_operand && it.rb == it.cb;
      const int a_rows = p.A.rows, a_br = p.A.br, a_cs = p.A.Cs;
      const int b_rows = p.B.rows, b_br = p.B.br, b_cs = p.B.Cs;
      const int segs_a = seg_count(r0, a_rows, a_br);
      const int segs_b = share ? 0 : seg_count(c0, b_rows, b_br);
      // bytes landing on this CTA's full barrier per stage; full boxes always count
      const uint32_t tx = 2u * (uint32_t)(segs_a * a_br + segs_b * b_br) * BK * 4u;
      for (int kb = it.kb0; kb < it.kb1; ++kb) {
        prefetch_step();
        long long t0 = dbg ? clock64() : 0;
        mbar_wait_warp(&empty_bar[stage], phase ^ 1, lane);
        long long t1 = dbg ? clock64() : 0;
        c_wait += t1 - t0;
        mbar_expect_tx_elect(&full_bar[stage], tx);
        const uint32_t sbase = smem_u32(smem + stage * kStageBytes);
        const int kx0 = kb * BK;
        for (int s = 0; s < segs_a; ++s) {
          const int r = r0 + s * a_br;
          const int t = r / a_cs, c = r - t * a_cs;
          const uint32_t off = (uint32_t)(s * a_br) * (BK * 4);
          tma_load_2d_elect(sbase + off, &it.maps->a[0][t], &full_bar[stage], kx0, c);
          tma_load_2d_elect(sbase + kABytes + off, &it.maps->a[1][t], &full_bar[stage], kx0, c);
        }
        for (int s = 0; s < segs_b; ++s) {
          const int r = c0 + s * b_br;
          const int t = r / b_cs, c = r - t * b_cs;
          const uint32_t off = (uint32_t)(s * b_br) * (BK * 4);
          tma_load_2d_elect(sbase + 2 * kABytes + off, &it.maps->b[0][t], &full_bar[stage], kx0, c);
          tma_load_2d_elect(sbase + 3 * kABytes + off, &it.maps->b[1][t], &full_bar[stage], kx0, c);
        }
        if (dbg) c_issue += clock64() - t1;
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    if (dbg && lane == 0) {
      g_dbg_counters[blockIdx.x * 8 + 3] = c_wait;
      g_dbg_counters[blockIdx.x * 8 + 4] = c_issue;
    }
  } else if (warp == 1) {
    // ============================ MMA issuer (pair: leader CTA only) ============================
    if (!PAIR || rank == 0) {
      uint32_t stage = 0, phase = 0;
      uint32_t local_item = 0;
      for (int idx = worker; idx < n_items; idx += n_workers, ++local_item) {
        const Item it = fetch_item(&pmaps, &pp, gprobs, gitems, idx);
        const TcParams& p = *it.p;
        const bool share = p.gram && p.same_operand && it.rb == it.cb;
        // single-CTA: ragged right edge issues only the valid columns (N in steps of 16)
        int n_valid = p.n_cols - it.cb * TILE;
        if (n_valid > TILE) n_valid = TILE;
        const uint32_t idesc = PAIR ? make_idesc_tf32(256, 256)
                                    : make_idesc_tf32(BM, (n_valid + 15) & ~15);
        const uint32_t buf = local_item & 1;
        const uint32_t use = local_item >> 1;
        long long ta = dbg ? clock64() : 0;
        mbar_wait_warp(&tmem_empty[buf], (use & 1) ^ 1, lane);   // epilogue drained this buffer
        if (dbg) c_acc += clock64() - ta;
        tc_fence_after();
        // single-CTA: [main | corr] x 128 columns per buffer; pair: one 256-column accumulator
        const uint32_t d_main = tmem_base + buf * 256;
        const uint32_t d_corr = d_main + 128;
        for (int kb = it.kb0; kb < it.kb1; ++kb) {
          long long t0 = dbg ? clock64() : 0;
          mbar_wait_warp(&full_bar[stage], phase, lane);
          if (PAIR) mbar_wait_warp(&peer_full[stage], phase, lane);
          long long t1 = dbg ? clock64() : 0;
          c_wait += t1 - t0;
          ++c_kb;
          tc_fence_after();
          const uint32_t sbase = smem_u32(smem + stage * kStageBytes);
          const uint64_t a_hi = make_kmajor_sw128_desc(sbase);
          const uint64_t a_lo = make_kmajor_sw128_desc(sbase + kABytes);
          const uint64_t b_hi = share ? a_hi : make_kmajor_sw128_desc(sbase + 2 * kABytes);
          const uint64_t b_lo = share ? a_lo : make_kmajor_sw128_desc(sbase + 3 * kABytes);
          const uint32_t first = kb > it.kb0 ? 1u : 0u;
          if (PAIR) {
            tc_mma_kblock_3xtf32_2sm(d_main, a_hi, a_lo, b_hi, b_lo, idesc, first);
            tc_commit_2sm_mc_elect(&empty_bar[stage]);        // frees the slot in both CTAs
            if (kb == it.kb1 - 1) tc_commit_2sm_mc_elect(&tmem_full[buf]);
          } else {
            tc_mma_kblock_3xtf32(d_main, d_corr, a_hi, a_lo, b_hi, b_lo, idesc, first, 0u);
            tc_commit_elect(&empty_bar[stage]);               // slot free when these retire
            if (kb == it.kb1 - 1) tc_commit_elect(&tmem_full[buf]);
          }
          if (dbg) c_issue += clock64() - t1;
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (it.kb1 <= it.kb0) {                               // defensive: empty K range
          if (PAIR) tc_commit_2sm_mc_elect(&tmem_full[buf]);
          else tc_commit_elect(&tmem_full[buf]);
        }
      }
      if (dbg && lane == 0) {
        g_dbg_counters[blockIdx.x * 8 + 0] = c_wait;
        g_dbg_counters[blockIdx.x * 8 + 1] = c_issue;
        g_dbg_counters[blockIdx.x * 8 + 2] = c_acc;
        g_dbg_counters[blockIdx.x * 8 + 5] = clock64() - t_start;
        g_dbg_counters[blockIdx.x * 8 + 6] = c_kb;
      }
    } else {
      // pair, peer CTA: forward "my half of the stage has landed" to the leader's barrier
      // (plain per-CTA TMA + this hop measured faster than cta_group::2 TMA whose issue
      // rate per SM is half)
      uint32_t stage = 0, phase = 0;
      for (int idx = worker; idx < n_items; idx += n_workers) {
        const Item it = fetch_item(&pmaps, &pp, gprobs, gitems, idx);
        for (int kb = it.kb0; kb < it.kb1; ++kb) {
          mbar_wait_warp(&full_bar[stage], phase, lane);
          mbar_arrive_remote_elect(&peer_full[stage], 0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ============================ epilogue (own 128 accumulator rows) ============================
    const int quad = warp & 3;                         // TMEM lane quadrant of this warp
    uint32_t local_item = 0;
    for (int idx = worker; idx < n_items; idx += n_workers, ++local_item) {
      const Item it = fetch_item(&pmaps, &pp, gprobs, gitems, idx);
      const TcParams& p = *it.p;
      const uint32_t buf = local_item & 1;
      const uint32_t use = local_item >> 1;
      mbar_wait_warp(&tmem_full[buf], use & 1, lane, 200);
      tc_fence_after();
      const int rblk = it.rb * TILE + rank * BM;
      const int row = rblk + quad * 32 + lane;
      const bool row_ok = row < p.A.rows && it.kb1 > it.kb0;
      float* orow = p.out + (long long)row * p.ld;
      const float alpha = p.alpha;
      const int n_cols = p.n_cols;
      const bool vec = p.vec_red != 0;
      const bool gram = p.gram != 0;
      // deterministic mode: the whole partial tile goes to its slot (zeros where masked)
      float* srow = (!PAIR && it.slot > 0)
                        ? slots + (size_t)(it.slot - 1) * kSlotElems + (quad * 32 + lane) * 128
                        : nullptr;
#pragma unroll 1
      for (int chunk = 0; chunk < TILE / 32; ++chunk) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * 256 + chunk * 32;
        tc_ld32(taddr, v);
        if (!PAIR) {
          uint32_t w[32];
          tc_ld32(taddr + 128, w);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j)
            v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(w[j]));
        } else {
          tc_wait_ld();
        }
        const int col0 = it.cb * TILE + chunk * 32;
        // Gram: chunks strictly left of this CTA's diagonal block carry nothing needed
        const bool wanted = !gram || (col0 + 31 >= rblk);
        if (srow != nullptr) {
          const bool ok = row_ok && wanted;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const int col = col0 + j;
            float4 x;
            x.x = ok && col < n_cols ? alpha * __uint_as_float(v[j]) : 0.f;
            x.y = ok && col + 1 < n_cols ? alpha * __uint_as_float(v[j + 1]) : 0.f;
            x.z = ok && col + 2 < n_cols ? alpha * __uint_as_float(v[j + 2]) : 0.f;
            x.w = ok && col + 3 < n_cols ? alpha * __uint_as_float(v[j + 3]) : 0.f;
            *reinterpret_cast<float4*>(srow + chunk * 32 + j) = x;
          }
        } else if (row_ok && col0 < n_cols && wanted) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const int col = col0 + j;
            const float x0 = alpha * __uint_as_float(v[j]), x1 = alpha * __uint_as_float(v[j + 1]),
                        x2 = alpha * __uint_as_float(v[j + 2]), x3 = alpha * __uint_as_float(v[j + 3]);
            if (vec && col + 3 < n_cols) {
              red_add_v4(orow + col, x0, x1, x2, x3);
            } else {
              if (col < n_cols) atomicAdd(orow + col, x0);
              if (col + 1 < n_cols) atomicAdd(orow + col + 1, x1);
              if (col + 2 < n_cols) atomicAdd(orow + col + 2, x2);
              if (col + 3 < n_cols) atomicAdd(orow + col + 3, x3);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (!PAIR || rank == 0) {
        if (lane == 0) mbar_arrive(&tmem_empty[buf]);
      } else {
        mbar_arrive_remote_elect(&tmem_empty[buf], 0);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  tl_end(tl);
  if (PAIR) cluster_sync();          // the peer may still be reading this CTA's smem / barriers
  if (warp == 1) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"(kTmemCols)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"(kTmemCols)
                   : "memory");
  }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) ==
            cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// Rows per TMA box.  A single-tap operand takes the largest power of two <= Cs (at most 128)
// but never less than 8 rows, the 128-byte swizzle atom: box rows at or past Cs are out of
// bounds, land in shared memory as zeros and are masked by the epilogue, so an operand of
// 1..7 rows (a layer with 3 output channels, 3 kept-out directions, 5 centres) is one 8-row
// box.  The rows of tap t > 0 start at t * Cs, so a multi-tap operand needs boxes that
// divide Cs.
int pick_box_rows(const Operand& o) {
  if (o.T == 1) {
    int br = 128;
    while (br > 8 && br > o.Cs) br >>= 1;
    return br;
  }
  for (int br = 128; br >= 8; br >>= 1)
    if (o.Cs % br == 0) return br;
  return 0;
}

// One 2-D tensor map per (hi/lo, tap): dims (k: K valid columns, c: rows of the
// tap), box (32, br).  Columns >= K are out of bounds and read as zero - that is
// what masks the K tail.
int encode_operand(const Operand& o, int br, CUtensorMap (*dst)[kMaxTaps]) {
  EncodeTiledFn enc = get_encode_fn();
  NSGP_REQUIRE(enc != nullptr, "tcgen05 engine: cuTensorMapEncodeTiled is unavailable");
  for (int hl = 0; hl < 2; ++hl)
    for (int t = 0; t < o.T; ++t) {
      const float* base = o.base + (long long)hl * o.hl_stride + o.tap_off[t];
      NSGP_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0,
                   "tcgen05 engine: operand base must be 16-byte aligned");
      cuuint64_t gdim[2] = {(cuuint64_t)o.K, (cuuint64_t)o.Cs};
      cuuint64_t gstr[1] = {(cuuint64_t)o.row_pitch * 4};
      cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)br};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&dst[hl][t], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr,
                       box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      NSGP_REQUIRE(r == CUDA_SUCCESS,
                   "cuTensorMapEncodeTiled failed (%d): K=%d Cs=%d pitch=%lld br=%d", (int)r, o.K,
                   o.Cs, o.row_pitch, br);
    }
  return 0;
}

void fill_operand(const Operand& o, int br, TcOperand* d) {
  d->T = o.T; d->Cs = o.Cs; d->rows = o.rows; d->br = br;
}

constexpr size_t kSmemBytes = (size_t)STAGES * kStageBytes + 1024 + 256;
// partitioned launches (pipelined covariance pass): the CTA claims the whole SM's shared
// memory, like the sliding-window kernel, so that no staging block can join its SM
constexpr size_t kSmemBytesFullSm = (size_t)7 * 32768 + 1024 + 256;

int dbg_counters() {
  static const int d = nsgp_env("NSGP_DBG_COUNTERS") ? 1 : 0;
  return d;
}

template <bool PAIR>
int configure_kernel() {
  static bool configured = false;
  if (!configured) {
    NSGP_CHECK_CUDA(cudaFuncSetAttribute(contraction_tc_kernel<PAIR>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSmemBytesFullSm));
    configured = true;
  }
  return 0;
}

// Launch over `n_items` work items with `workers` CTAs (single) or CTA pairs (pair).
int launch_kernel(bool pair, const TcMaps& maps, const TcParams& p, const TcProblem* gprobs,
                  const TcItem* gitems, int n_items, int kind, cudaStream_t stream,
                  int max_ctas = 0, int pdl = 0, const int* n_items_dev = nullptr,
                  float* slots = nullptr) {
  if (n_items <= 0) return 0;
  ProfScope prof(kind, stream);
#ifndef NSGP_BRINGUP
  NSGP_REQUIRE(!pair, "the CTA-pair kernel is a bring-up build feature");
#else
  if (pair) {
    int rc = configure_kernel<true>();
    if (rc) return rc;
    int clusters = sm_count() / 2;
    if (n_items < clusters) clusters = n_items;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * clusters);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    NSGP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, contraction_tc_kernel<true>, maps, p, gprobs, gitems,
                                       n_items, dbg_counters(),
                                       (unsigned long long*)nullptr, (const int*)nullptr,
                                       (float*)nullptr));
    NSGP_LAUNCHED();
    return 0;
  }
#endif
  {
    int rc = configure_kernel<false>();
    if (rc) return rc;
    int grid = n_items < sm_count() ? n_items : sm_count();
    if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = max_ctas > 0 ? kSmemBytesFullSm : kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    NSGP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, contraction_tc_kernel<false>, maps, p, gprobs, gitems,
                                       n_items, dbg_counters(),
                                       kind == kProfGram ? timeline_slot(0) : nullptr,
                                       n_items_dev, slots));
  }
  NSGP_LAUNCHED();
  return 0;
}

// CTA-pair kernel or single-CTA kernel?  The pair kernel moves half the operand bytes
// per output element (256 x 256 tile over two SMs) but pads to 256-row blocks and has
// one accumulator chain.  Measured (scripts/bench_gram.py, NSGP_DBG_COUNTERS): both
// kernels are bound by operand delivery into the 3-stage ring, and the pair kernel is
// ~15 % faster per issued FLOP once its TMA is the plain per-CTA form with the peer
// forwarding readiness (cta_group::2 TMA issues at half the rate per SM).  Default:
// pair for covariance problems whose rows are a multiple of 256 (no padding waste);
// NSGP_PAIR_KERNEL=0 never, 1 every same-operand Gram, 3 everything with > 128 rows.
bool want_pair(const ContractionArgs& a) {
#ifndef NSGP_BRINGUP
  (void)a;
  return false;      // measured slower end to end (DESIGN.md 4): bring-up builds only
#else
  static const int force = [] {
    const char* e = nsgp_env("NSGP_PAIR_KERNEL");
    return e ? atoi(e) : -1;
  }();
  const bool gram = a.epi == kEpiGramAtomic;
  const bool same = gram && a.A.base == a.B.base && a.A.hl_stride == a.B.hl_stride &&
                    a.A.rows == a.B.rows;
  if (force == 0 || g_deterministic) return false;   // the pair kernel has no slot epilogue
  if (force == 3) return a.A.rows > 128;
  if (force == 1) return gram && same;
  // default: autocorrelation-layout problems (they carry an l2_group) on 256-multiples
  return a.l2_group > 0 && a.A.rows % 256 == 0 && a.n_cols % 256 == 0 && a.A.K >= 1024;
#endif
}

// Validates one problem, encodes its tensor maps and fills every field of the
// parameter block except `splits`.  Returns 1 for an empty problem (nothing to do).
int build_problem(const ContractionArgs& a, bool pair, TcProblem* out) {
  NSGP_REQUIRE(a.A.T >= 1 && a.A.T <= kMaxTaps && a.B.T >= 1 && a.B.T <= kMaxTaps,
               "tcgen05 engine: bad tap count");
  NSGP_REQUIRE(a.A.row_pitch % 4 == 0 && a.B.row_pitch % 4 == 0,
               "tcgen05 engine: row pitch must be 16-byte");
  NSGP_REQUIRE(ceil_div(a.A.K, BK) == ceil_div(a.B.K, BK),
               "contraction: operands disagree on K blocks");
  const int br_a = pick_box_rows(a.A), br_b = pick_box_rows(a.B);
  NSGP_REQUIRE(br_a > 0 && br_b > 0,
               "tcgen05 engine: operand rows per tap must be a multiple of 8 when taps > 1");
  TcParams& p = out->p;
  p = TcParams{};
  p.nkb = k_blocks(a.A);
  if (a.A.rows == 0 || a.n_cols == 0 || p.nkb == 0) return 1;
  int rc = encode_operand(a.A, br_a, out->maps.a);
  if (rc) return rc;
  rc = encode_operand(a.B, br_b, out->maps.b);
  if (rc) return rc;
  fill_operand(a.A, br_a, &p.A);
  fill_operand(a.B, br_b, &p.B);
  p.out = a.out; p.ld = a.ld; p.n_cols = a.n_cols; p.alpha = a.alpha;
  p.gram = (a.epi == kEpiGramAtomic) ? 1 : 0;
  p.same_operand = (p.gram && a.A.base == a.B.base && a.A.hl_stride == a.B.hl_stride &&
                    a.A.rows == a.B.rows) ? 1 : 0;
  p.pair = pair ? 1 : 0;
  p.chain = a.chain;
  const int tile = pair ? 256 : 128;
  p.tiles_m = ceil_div(a.A.rows, tile);
  p.tiles_n = ceil_div(a.n_cols, tile);
  NSGP_REQUIRE(!p.gram || p.tiles_m == p.tiles_n, "Gram: operands must have the same rows");
  p.n_tiles = p.gram ? p.tiles_m * (p.tiles_m + 1) / 2 : p.tiles_m * p.tiles_n;
  p.vec_red = (a.ld % 4 == 0 && (reinterpret_cast<uintptr_t>(a.out) & 15) == 0) ? 1 : 0;
  p.splits = 1;
  return 0;
}

// K blocks one TMEM accumulator chain may cover.  The tensor core accumulates with
// truncation (~2^-25.6 relative per accumulate step, measured); the single-CTA kernel
// keeps hi*hi in its own accumulator (4 steps per K block), the pair kernel has one
// accumulator for all three products (12 steps per K block).
int chain_limit(const TcParams& p) {
  if (p.chain > 0) return p.pair && p.chain > 32 ? 32 : p.chain;
  if (!p.gram) return kChainGemm;
  return p.pair ? 32 : kChainGram;
}

}  // namespace

int encode_batch_rows_map(CUtensorMap* dst, const float* base, long long img_elems, int B,
                          int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  NSGP_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is unavailable");
  NSGP_REQUIRE(img_elems % 256 == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0,
               "batch rows map: input must be 16-byte aligned with a multiple of 256 elements");
  cuuint64_t gdim[3] = {256, (cuuint64_t)(img_elems / 256), (cuuint64_t)B};
  cuuint64_t gstr[2] = {1024, (cuuint64_t)img_elems * 4};
  cuuint32_t box[3] = {256, (cuuint32_t)box_rows, (cuuint32_t)B};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(dst, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)base, gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  NSGP_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (batch rows) failed (%d)", (int)r);
  return 0;
}

namespace tc {
int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}
}  // namespace tc

int contraction_tc(const ContractionArgs& a, cudaStream_t stream) {
  TcProblem prob;
  const bool pair = want_pair(a);
  int rc = build_problem(a, pair, &prob);
  if (rc == 1) return 0;
  if (rc) return rc;
  TcParams& p = prob.p;
  // K splits: bound the accumulation chain, then choose the split count that
  // minimises  waves x (K blocks per item + per-item overhead) - the last wave of the
  // static round-robin deal is the tail.  Partial tiles are red.add'ed, so splits need
  // no workspace.  GEMM (W += update @ P): one chain per tile up to kChainGemm blocks
  // (d <= 5120), so every W element takes ONE fp32 rounding like the reference's add_
  // and the result is deterministic.
  const int workers = pair ? sm_count() / 2 : sm_count();
  {
    const int s_min = ceil_div(p.nkb, chain_limit(p));
    int s_max = p.nkb / 4 > s_min ? p.nkb / 4 : s_min;
    if (s_max > s_min + 64) s_max = s_min + 64;
    if (!p.gram) s_max = s_min;
    const int overhead = 4;            // K-block equivalents of pipeline fill + epilogue
    long long best = -1;
    int best_s = s_min;
    for (int sp = s_min; sp <= s_max; ++sp) {
      long long waves = ceil_div((long long)p.n_tiles * sp, workers);
      long long cost = waves * (ceil_div(p.nkb, sp) + overhead);
      if (best < 0 || cost < best) { best = cost; best_s = sp; }
    }
    p.splits = best_s;
    // deterministic mode: one item per output tile, whose red.add is then the only addend
    if (g_deterministic) {
      NSGP_REQUIRE(s_min == 1, "deterministic mode: a single-problem contraction over %d K "
                   "blocks needs a K split; it has no deterministic form (use a group table)",
                   p.nkb);
      p.splits = 1;
    }
  }
  return launch_kernel(pair, prob.maps, p, nullptr, nullptr, p.n_tiles * p.splits,
                       p.gram ? kProfGram : kProfGemm, stream);
}

int debug_read_counters(unsigned long long* out, int n) {
  NSGP_CHECK_CUDA(cudaMemcpyFromSymbol(out, g_dbg_counters, (size_t)n * sizeof(unsigned long long)));
  return 0;
}

// ---------------------------------------------------------------- grouped launches
// A group table holds up to two sub-tables: problems run by the single-CTA kernel and
// problems run by the CTA-pair kernel (one launch each).
size_t group_table_bytes(const ContractionArgs* probs, int n) {
  size_t items = 0, det_items = 0;
  for (int i = 0; i < n; ++i) {
    const int tm = ceil_div(probs[i].A.rows, BM), tn = ceil_div(probs[i].n_cols, BN);
    const int nkb = k_blocks(probs[i].A);
    const bool gram = probs[i].epi == kEpiGramAtomic;
    const size_t tiles = gram ? (size_t)tm * (tm + 1) / 2 : (size_t)tm * tn;
    // upper bound for either kernel: 128-tiles with the shortest chain
    const int chain = probs[i].chain > 0 ? (probs[i].chain < 32 ? probs[i].chain : 32)
                                         : (gram ? 32 : kChainGemm);
    items += tiles * (size_t)ceil_div(nkb > 0 ? nkb : 1, chain);
    // deterministic mode (single-CTA kernel only): exact item count, each may need a slot
    const int chain_d = probs[i].chain > 0 ? probs[i].chain : (gram ? kChainGram : kChainGemm);
    det_items += tiles * (size_t)ceil_div(nkb > 0 ? nkb : 1, chain_d);
  }
  return (size_t)n * sizeof(TcProblem) + items * sizeof(TcItem) + 1024 +
         (g_deterministic ? DetCombine::bytes_bound(det_items) : 0);
}

// Output tiles of every work item of the problems, as group_table_build enumerates them in
// deterministic mode (single-CTA kernel)
void group_table_count(const ContractionArgs* probs, int n, DetCombine* det) {
  for (int i = 0; i < n; ++i) {
    const ContractionArgs& a = probs[i];
    const int nkb = k_blocks(a.A);
    if (a.A.rows == 0 || a.n_cols == 0 || nkb == 0) continue;
    const bool gram = a.epi == kEpiGramAtomic;
    const int tm = ceil_div(a.A.rows, BM), tn = ceil_div(a.n_cols, BN);
    const int chain = a.chain > 0 ? a.chain : (gram ? kChainGram : kChainGemm);
    const int splits = ceil_div(nkb, chain);
    for (int sp = 0; sp < splits; ++sp)
      for (int rb = 0; rb < tm; ++rb)
        for (int cb = gram ? rb : 0; cb < tn; ++cb)
          det->count(a.out + (long long)rb * BM * a.ld + cb * BN);
  }
}

int group_table_build(const ContractionArgs* probs, int n, int kind, void* table_dev,
                      size_t table_bytes, GroupInfo* info, cudaStream_t stream, DetCombine* det) {
  NSGP_REQUIRE((probs || n == 0) && table_dev && info && n >= 0, "group_build: bad arguments");
  NSGP_REQUIRE((reinterpret_cast<uintptr_t>(table_dev) & 63) == 0,
               "group_build: table must be 64-byte aligned");
  // deterministic mode: the slots of this launch, counted here unless the caller shares the
  // combine with another sub-table
  DetCombine local;
  const bool own_det = det == nullptr && g_deterministic;
  if (own_det) {
    det = &local;
    group_table_count(probs, n, det);
  }
  struct Cost { long long c; int grp, split; TcItem it; };
  std::vector<TcProblem> hp[2];
  std::vector<Cost> items[2];
  for (int i = 0; i < n; ++i) {
    const ContractionArgs& a = probs[i];
    const int k = want_pair(a) ? 1 : 0;
    TcProblem pr;
    int rc = build_problem(a, k == 1, &pr);
    if (rc == 1) continue;
    if (rc) return rc;
    const TcParams& p = pr.p;
    const int prob = (int)hp[k].size();
    const int splits = ceil_div(p.nkb, chain_limit(p));
    for (int sp = 0; sp < splits; ++sp) {
      const int kb0 = (int)((long long)p.nkb * sp / splits);
      const int kb1 = (int)((long long)p.nkb * (sp + 1) / splits);
      for (int rb = 0; rb < p.tiles_m; ++rb)
        for (int cb = p.gram ? rb : 0; cb < p.tiles_n; ++cb) {
          Cost c;
          int slot = 0;
          if (det != nullptr) {
            NSGP_REQUIRE(k == 0, "group_build: deterministic tables use the single-CTA kernel");
            float* tile = a.out + (long long)rb * BM * a.ld + cb * BN;
            if (det->contributors(tile) > 1) {
              const int rows = a.A.rows - rb * BM, cols = a.n_cols - cb * BN;
              slot = 1 + det->assign(tile, a.ld, rows < BM ? rows : BM, cols < BN ? cols : BN);
            }
          }
          c.it = TcItem{prob, rb, cb, kb0, kb1, slot, 0, 0};
          c.c = (long long)(kb1 - kb0) * 8 + 16;       // ~ K blocks + a fixed part
          c.grp = a.l2_group > 0 ? a.l2_group : -(i + 1);
          c.split = sp;
          items[k].push_back(c);
        }
    }
    hp[k].push_back(pr);
  }
  size_t off = 0;
  info->kind = kind;
  for (int k = 0; k < 2; ++k) {
    // big items first; ties keep (problem, K range, tile) order so that tiles sharing
    // operand rows of one K range run at the same time (L2 reuse)
    // ... and problems that share operand planes (l2_group) walk their K ranges together
    std::stable_sort(items[k].begin(), items[k].end(), [](const Cost& x, const Cost& y) {
      if (x.c != y.c) return x.c > y.c;
      if (x.grp != y.grp) return x.grp < y.grp;
      return x.split < y.split;
    });
    SubGroup& sg = info->sub[k];
    sg.n_problems = (int)hp[k].size();
    sg.n_items = (int)items[k].size();
    sg.off_probs = off;
    sg.off_items = off + hp[k].size() * sizeof(TcProblem);
    off = (size_t)round_up((long long)(sg.off_items + items[k].size() * sizeof(TcItem)), 64);
  }
  info->sub[2] = SubGroup{0, 0, 0, 0};
  info->sub[3] = SubGroup{0, 0, 0, 0};
  if (own_det) off = local.layout(off, &info->sub[3]);
  info->bytes = off;
  NSGP_REQUIRE(info->bytes <= table_bytes, "group_build: table too small (%zu < %zu)",
               table_bytes, info->bytes);
  if (own_det) {
    int rc = det_combine_upload(local, table_dev, info->sub[3], stream);
    if (rc) return rc;
  }
  for (int k = 0; k < 2; ++k) {
    const SubGroup& sg = info->sub[k];
    if (sg.n_items == 0) continue;
    std::vector<TcItem> hi(items[k].size());
    for (size_t i = 0; i < items[k].size(); ++i) hi[i] = items[k][i].it;
    NSGP_CHECK_CUDA(cudaMemcpyAsync((char*)table_dev + sg.off_probs, hp[k].data(),
                                    hp[k].size() * sizeof(TcProblem), cudaMemcpyHostToDevice,
                                    stream));
    NSGP_CHECK_CUDA(cudaMemcpyAsync((char*)table_dev + sg.off_items, hi.data(),
                                    hi.size() * sizeof(TcItem), cudaMemcpyHostToDevice, stream));
  }
  return 0;
}

static float* group_slots(const void* table_dev, const GroupInfo& info) {
  if (info.sub[3].n_items == 0) return nullptr;
  return reinterpret_cast<float*>(const_cast<char*>((const char*)table_dev) + info.sub[3].off_probs);
}

int group_launch_sub(const void* table_dev, const GroupInfo& info, int which, int max_ctas,
                     int pdl, cudaStream_t stream) {
  static const TcMaps dummy_maps{};
  TcParams dummy{};
  float* slots = group_slots(table_dev, info);
  if (which == 2) return autocorr_launch(table_dev, info.sub[2], stream, max_ctas, pdl, slots);
  const SubGroup& sg = info.sub[0];
  if (sg.n_items == 0) return 0;
  const TcProblem* probs = reinterpret_cast<const TcProblem*>((const char*)table_dev + sg.off_probs);
  const TcItem* items = reinterpret_cast<const TcItem*>((const char*)table_dev + sg.off_items);
  return launch_kernel(false, dummy_maps, dummy, probs, items, sg.n_items, info.kind, stream,
                       max_ctas, pdl, nullptr, slots);
}

// one problem, work items written by a device kernel (at most max_items of them, the live
// count in *n_items_dev): RePRE's Gram over the class-sorted foreground rows
int contraction_launch_dev_items(const void* prob_dev, const void* items_dev, int max_items,
                                 const int* n_items_dev, int kind, float* slots,
                                 cudaStream_t stream) {
  static const TcMaps dummy_maps{};
  TcParams dummy{};
  return launch_kernel(false, dummy_maps, dummy, reinterpret_cast<const TcProblem*>(prob_dev),
                       reinterpret_cast<const TcItem*>(items_dev), max_items, kind, stream, 0, 0,
                       n_items_dev, slots);
}
// host part of the same: validates the problem and encodes its tensor maps
int contraction_build_problem(const ContractionArgs& a, void* prob_host /* TcProblem */) {
  int rc = build_problem(a, false, reinterpret_cast<TcProblem*>(prob_host));
  NSGP_REQUIRE(rc != 1, "contraction_build_problem: empty problem");
  return rc;
}
size_t contraction_problem_bytes() { return sizeof(TcProblem); }
size_t contraction_item_bytes() { return sizeof(TcItem); }

int group_launch(const void* table_dev, const GroupInfo& info, cudaStream_t stream) {
  static const TcMaps dummy_maps{};
  TcParams dummy{};
  float* slots = group_slots(table_dev, info);
  for (int k = 1; k >= 0; --k) {          // pair sub-table first: it holds the big layers
    const SubGroup& sg = info.sub[k];
    if (sg.n_items == 0) continue;
    const TcProblem* probs = reinterpret_cast<const TcProblem*>((const char*)table_dev + sg.off_probs);
    const TcItem* items = reinterpret_cast<const TcItem*>((const char*)table_dev + sg.off_items);
    int rc = launch_kernel(k == 1, dummy_maps, dummy, probs, items, sg.n_items, info.kind, stream,
                           0, 0, nullptr, slots);
    if (rc) return rc;
  }
  // autocorrelation sub-table last: its long items fill the machine best once the small
  // problems are out of the way
  int rc = autocorr_launch(table_dev, info.sub[2], stream, 0, 0, slots);
  if (rc) return rc;
  return det_combine_launch(table_dev, info.sub[3], info.kind, stream);
}

// ---------------------------------------------------------------- ordered combine
int DetCombine::assign(float* tile, int ld, int rows, int cols) {
  auto it = tile_of.find(tile);
  int t;
  if (it == tile_of.end()) {
    t = (int)tiles.size();
    tile_of.emplace(tile, t);
    CombTile c{};
    c.out = tile; c.ld = ld; c.rows = rows; c.cols = cols;
    tiles.push_back(c);
    per_tile.emplace_back();
  } else {
    t = it->second;
  }
  per_tile[t].push_back(n_slots);
  return n_slots++;
}

size_t DetCombine::layout(size_t off, SubGroup* sg) const {
  off = (size_t)round_up((long long)off, 256);
  sg->n_items = (int)tiles.size();
  sg->off_items = off;
  sg->n_problems = n_slots;
  off += tiles.size() * sizeof(CombTile) + (size_t)n_slots * sizeof(int);
  sg->off_probs = (size_t)round_up((long long)off, 256);
  return sg->off_probs + (size_t)n_slots * kSlotElems * sizeof(float);
}

int det_combine_upload(const DetCombine& det, void* table_dev, const SubGroup& sg,
                       cudaStream_t stream) {
  if (sg.n_items == 0) return 0;
  std::vector<CombTile> t(det.tiles);
  std::vector<int> list;
  list.reserve(det.n_slots);
  for (size_t i = 0; i < t.size(); ++i) {
    t[i].first = (int)list.size();
    t[i].n = (int)det.per_tile[i].size();
    list.insert(list.end(), det.per_tile[i].begin(), det.per_tile[i].end());
  }
  char* base = (char*)table_dev + sg.off_items;
  NSGP_CHECK_CUDA(cudaMemcpyAsync(base, t.data(), t.size() * sizeof(CombTile),
                                  cudaMemcpyHostToDevice, stream));
  NSGP_CHECK_CUDA(cudaMemcpyAsync(base + t.size() * sizeof(CombTile), list.data(),
                                  list.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
  return 0;
}

namespace {
// One CTA per output tile: sum the tile's slots in list order, then one read-modify-write of
// the running sum.  The contraction launch before it on the stream wrote the slots.
__global__ void __launch_bounds__(256)
det_combine_kernel(const CombTile* __restrict__ tiles, const float* __restrict__ slots) {
  const CombTile t = tiles[blockIdx.x];
  const int* ids = reinterpret_cast<const int*>(tiles + gridDim.x) + t.first;
  for (int e = threadIdx.x; e < kSlotElems / 4; e += 256) {
    const int r = e >> 5, c = (e & 31) * 4;
    if (r >= t.rows || c >= t.cols) continue;
    const size_t off = (size_t)r * 128 + c;
    float4 s = *reinterpret_cast<const float4*>(slots + (size_t)ids[0] * kSlotElems + off);
    for (int k = 1; k < t.n; ++k) {
      const float4 v = *reinterpret_cast<const float4*>(slots + (size_t)ids[k] * kSlotElems + off);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    float* o = t.out + (long long)r * t.ld + c;
    o[0] += s.x;
    if (c + 1 < t.cols) o[1] += s.y;
    if (c + 2 < t.cols) o[2] += s.z;
    if (c + 3 < t.cols) o[3] += s.w;
  }
}
}  // namespace

int det_combine_launch(const void* table_dev, const SubGroup& sg, int kind, cudaStream_t stream) {
  if (sg.n_items == 0) return 0;
  ProfScope prof(kind, stream);
  det_combine_kernel<<<sg.n_items, 256, 0, stream>>>(
      reinterpret_cast<const CombTile*>((const char*)table_dev + sg.off_items),
      reinterpret_cast<const float*>((const char*)table_dev + sg.off_probs));
  NSGP_LAUNCHED();
  return 0;
}

}  // namespace nsgp
