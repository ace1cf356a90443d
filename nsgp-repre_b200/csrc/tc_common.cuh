// Shared pieces of the tcgen05 contraction kernels: parameter blocks and PTX wrappers.
#pragma once
#include "common.cuh"

namespace nsgp {
namespace tc {

constexpr int BM = 128;            // tile rows  (UMMA M)
constexpr int BK = 32;             // fp32 elements per K block = one 128-byte swizzle row
constexpr int UMMA_K = 8;          // tf32: 32 bytes per instruction
constexpr int kThreads = 192;      // 6 warps
constexpr int kEpiWarp0 = 2;

struct alignas(64) TcMaps {
  CUtensorMap a[2][kMaxTaps];   // [hi/lo][tap]
  CUtensorMap b[2][kMaxTaps];
};

struct TcOperand {
  int T, Cs, rows, br;            // taps, rows per tap, valid rows, rows per TMA box
  int pad[4];
};

struct TcParams {
  TcOperand A, B;
  float* out;
  int ld, n_cols;
  float alpha;
  int nkb;                        // K blocks in total
  int splits;                     // K splits
  int tiles_m, tiles_n, n_tiles;  // tile grid (Gram: n_tiles counts visited pairs)
  int same_operand;               // Gram: B is A
  int vec_red;                    // use red.global.add.v4.f32 in the epilogue
  int gram;                       // 1: upper block-triangle of A*A^T, 0: full A*B^T
  int pair;                       // tiles are 256 x 256 over a CTA pair (cta_group::2)
  int chain;                      // K blocks per accumulator chain (0: default)
};

// Grouped launches: many problems in one persistent launch.  The table lives in
// device memory: TcProblem[n_problems] followed by TcItem[n_items] (sorted by
// descending cost so that the static round-robin deal is balanced).
struct alignas(64) TcProblem {
  TcMaps maps;
  TcParams p;
};
struct alignas(16) TcItem {
  int prob, rb, cb, kb0;
  int kb1, pad0, pad1, pad2;
};

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  const uint32_t addr = smem_u32(bar);
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// One lane polls, the warp reconverges on it: 31 fewer spinning lanes per waiting warp
// (the part is power-capped, idle polling costs clock).  `backoff_ns` > 0 sleeps
// between polls - for waits that are expected to be long (epilogue).
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity, int lane,
                                               unsigned backoff_ns = 0) {
  if (lane == 0) {
    uint32_t done;
    const uint32_t addr = smem_u32(bar);
    for (;;) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(addr), "r"(parity)
          : "memory");
      if (done) break;
      if (backoff_ns) __nanosleep(backoff_ns);
    }
  }
  __syncwarp();
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint64_t* bar,
                                            int x, int c) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(x), "r"(c)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b),
               "f"(c), "f"(d)
               : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor: 128-byte rows, 8-row
// swizzle atoms 1024 bytes apart (SBO), LBO unused (1), descriptor version 1.
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// kind::tf32, fp32 accumulate, both operands K-major.
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}


// ---- warp-convergent single-thread issue ------------------------------------------
// tcgen05.mma / TMA / commit are issued by ONE thread, but putting them inside an
// `if (lane == 0)` region makes the compiler wrap every one of them in an
// ELECT + R2UR.BROADCAST + branch loop (uniform-datapath instructions under
// divergence): ~20 extra instructions per MMA, enough to starve the tensor pipe of
// 64-cycle MMAs.  These wrappers are executed by the whole (converged) warp with
// warp-uniform operands and elect the issuing thread inside the asm block.
__device__ __forceinline__ void mbar_expect_tx_elect(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
      "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_elect(uint32_t dst, const CUtensorMap* map,
                                                  uint64_t* bar, int x, int c) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(x), "r"(c)
      : "memory");
}
__device__ __forceinline__ void tc_commit_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::
      "r"(smem_u32(bar))
      : "memory");
}
// One K block (32 fp32 = 4 K steps of 8) of the 3xTF32 product, 12 MMAs in one asm
// block: hi*hi -> d_main, lo*hi and hi*lo -> d_corr (d_corr == d_main: one accumulator).
// Descriptors advance by 2 (32 bytes >> 4) per K step.  `first` = 0 overwrites the
// accumulators at the first K step.
__device__ __forceinline__ void tc_mma_kblock_3xtf32(uint32_t d_main, uint32_t d_corr,
                                                     uint64_t a_hi, uint64_t a_lo, uint64_t b_hi,
                                                     uint64_t b_lo, uint32_t idesc,
                                                     uint32_t first, uint32_t same_acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred pe, pf, pc, pt;\n\t"
      "setp.eq.b32 pt, 0, 0;\n\t"
      ".reg .b64 ah, al, bh, bl;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "setp.ne.b32 pf, %7, 0;\n\t"            // accumulate into d_main at K step 0?
      "setp.eq.b32 pc, %8, 1;\n\t"            // same accumulator: corr never overwrites
      "or.pred pc, pc, pf;\n\t"
      ".reg .pred ps, pq;\n\t"                // bring-up: same_acc == 2 skips the hi*lo product,
      "setp.lt.u32 ps, %8, 2;\n\t"            //           same_acc == 3 both cross products
      "and.pred ps, ps, pe;\n\t"
      "setp.ne.b32 pq, %8, 3;\n\t"
      "and.pred pq, pq, pe;\n\t"
      // K step 0
      "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], %2, %4, %6, pf;\n\t"
      "@pq tcgen05.mma.cta_group::1.kind::tf32 [%1], %3, %4, %6, pc;\n\t"
      "@ps tcgen05.mma.cta_group::1.kind::tf32 [%1], %2, %5, %6, pt;\n\t"
      // K step 1
      "add.u64 ah, %2, 2; add.u64 al, %3, 2; add.u64 bh, %4, 2; add.u64 bl, %5, 2;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bh, %6, pt;\n\t"
      "@pq tcgen05.mma.cta_group::1.kind::tf32 [%1], al, bh, %6, pt;\n\t"
      "@ps tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bl, %6, pt;\n\t"
      // K step 2
      "add.u64 ah, %2, 4; add.u64 al, %3, 4; add.u64 bh, %4, 4; add.u64 bl, %5, 4;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bh, %6, pt;\n\t"
      "@pq tcgen05.mma.cta_group::1.kind::tf32 [%1], al, bh, %6, pt;\n\t"
      "@ps tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bl, %6, pt;\n\t"
      // K step 3
      "add.u64 ah, %2, 6; add.u64 al, %3, 6; add.u64 bh, %4, 6; add.u64 bl, %5, 6;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bh, %6, pt;\n\t"
      "@pq tcgen05.mma.cta_group::1.kind::tf32 [%1], al, bh, %6, pt;\n\t"
      "@ps tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bl, %6, pt;\n\t"
      "}" ::"r"(d_main),
      "r"(d_corr), "l"(a_hi), "l"(a_lo), "l"(b_hi), "l"(b_lo), "r"(idesc), "r"(first),
      "r"(same_acc)
      : "memory");
}

// ---- CTA-pair (cta_group::2) versions of the same ---------------------------------
__device__ __forceinline__ void tma_load_2d_2sm_elect(uint32_t dst, const CUtensorMap* map,
                                                      uint64_t* bar, int x, int c) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(x), "r"(c)
      : "memory");
}
__device__ __forceinline__ void tc_commit_2sm_mc_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t.reg .b16 m;\n\t"
      "mov.b16 m, 3;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], m;\n\t}" ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote_elect(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t.reg .b32 ra;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "@pe mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(
          smem_u32(bar)),
      "r"(rank)
      : "memory");
}
// one K block, 12 MMAs over the CTA pair (M = 256), single accumulator
__device__ __forceinline__ void tc_mma_kblock_3xtf32_2sm(uint32_t d, uint64_t a_hi, uint64_t a_lo,
                                                         uint64_t b_hi, uint64_t b_lo,
                                                         uint32_t idesc, uint32_t first) {
  asm volatile(
      "{\n\t"
      ".reg .pred pe, pf, pt;\n\t"
      ".reg .b64 ah, al, bh, bl;\n\t"
      "setp.eq.b32 pt, 0, 0;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "setp.ne.b32 pf, %6, 0;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], %2, %3, %5, pf;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %4, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %3, %5, pt;\n\t"
      "add.u64 ah, %1, 2; add.u64 al, %2, 2; add.u64 bh, %3, 2; add.u64 bl, %4, 2;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], al, bh, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], ah, bl, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], ah, bh, %5, pt;\n\t"
      "add.u64 ah, %1, 4; add.u64 al, %2, 4; add.u64 bh, %3, 4; add.u64 bl, %4, 4;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], al, bh, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], ah, bl, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], ah, bh, %5, pt;\n\t"
      "add.u64 ah, %1, 6; add.u64 al, %2, 6; add.u64 bh, %3, 6; add.u64 bl, %4, 6;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], al, bh, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], ah, bl, %5, pt;\n\t"
      "@pe tcgen05.mma.cta_group::2.kind::tf32 [%0], ah, bh, %5, pt;\n\t"
      "}" ::"r"(d),
      "l"(a_hi), "l"(a_lo), "l"(b_hi), "l"(b_lo), "r"(idesc), "r"(first)
      : "memory");
}

// TMA prefetch of one box into L2 (no shared memory, no barrier)
__device__ __forceinline__ void tma_prefetch_2d_elect(const CUtensorMap* map, int x, int c) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];\n\t}" ::"l"(
          reinterpret_cast<uint64_t>(map)),
      "r"(x), "r"(c)
      : "memory");
}

// ---- cluster / 2-CTA variants ------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // shared::cluster address of the same
                                                 // offset in the even CTA of a pair
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)),
      "r"(rank)
      : "memory");
}
// TMA load into THIS CTA's smem, completion bytes credited to the even CTA's barrier
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map,
                                                uint64_t* bar, int x, int c) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(x), "r"(c)
      : "memory");
}
__device__ __forceinline__ void tc_commit_2sm_mc(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                                uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---- host helpers shared by the launchers --------------------------------------
int sm_count();
// chain limits (K blocks accumulated in one TMEM accumulator pair)
constexpr int kChainGram = 64;
constexpr int kChainGemm = 160;

}  // namespace tc
}  // namespace nsgp
