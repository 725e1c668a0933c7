// K2 v2 — unified tcgen05 kind::tf32 GEMM with the 3-term error-compensated split ("3xTF32")
//
//   C[M,N] = act( sum_s opA(A_s)[M,K_s] opB(B_s)[K_s,N] + bias ) (+C)        fp32 in / out, fp32-class accuracy
//
// for every operand layout (A stored [M,K] or [K,M]; B stored [N,K] or [K,N]), any M, N, K.  What changed against
// gemm_tc.cu (round-1 K2 / K3), and why (profiles/r01_*, DESIGN.md section 6):
//   * The tensor core truncates its fp32 TMEM accumulator on every MMA, so an accumulation chain is cut every
//     `drain_kb` k-blocks.  v1 drained a chain by read-modify-writing the C tile in global memory while the MMA
//     pipe waited (45 % of the kernel at K = 1024, 60 % at K = 3048).  Here a tile is 128 x 128, TMEM holds two
//     accumulator pairs [main | cross terms] (256 columns each, alternating per chain), and the eight epilogue
//     warps add finished chains into REGISTERS (64 fp32 per thread, round-to-nearest) while the next chain runs:
//     no global traffic, no MMA stall; C is written once.
//   * The B_lo tile sits right behind the B_hi tile in shared memory, so A_hi [B_hi ; B_lo]^T is ONE N = 256 MMA that
//     fills main and cross halves at once; a second N = 128 MMA adds A_lo B_hi^T to the cross half: two MMAs and 20 KB
//     of operand reads per K = 8 step instead of three and 24 KB.
//   * Both operands arrive as raw fp32 tiles by TMA and are split into hi / lo in shared memory (v1 loaded
//     pre-split B_hi and B_lo: 80 KB per k-block, L2-bound at ~207 TFLOP/s; now 32 KB per k-block), so there is
//     no packing pre-kernel and no workspace for it.
//   * MN-major operands (transposed A, untransposed B) use the SWIZZLE_128B_BASE32B canonical layout
//     (TMA: SWIZZLE_128B_ATOM_32B boxes of 32 x 32) found on hardware in round 1 — no explicit transposes.
//   * Work item = (row tile, column chunk, k part): when M x N alone gives fewer tiles than SMs the contraction
//     is cut into parts whose partial tiles go to slabs that a second kernel sums in fixed order (deterministic).
//   * Template PAIR (round 2): clusters of two CTAs drive one cta_group::2 MMA (M = 256), each CTA loading / splitting half of B.
//   * Template TEPI (round 2, CTA pairs; which products take it: t2_tepi_mode): TMA epilogue — three stages and a 64 KB epilogue area of per-warp SWIZZLE_128B
//     blocks; the fused epilogue operand arrives by TMA while the tile's MMAs run, the output tile leaves by TMA stores
//     (profiles/r02c_tepi_ab.txt: fused softmax-backward product 12.9 -> 10.0 ms).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace dcb {
namespace {

constexpr int T2_BM = 128, T2_BN = 128, T2_BK = 32;
constexpr int T2_STAGES = 3;
constexpr int T2_THREADS = 512;
constexpr int T2_TILE_BYTES = T2_BM * T2_BK * 4;              // 16 KB (A and B tiles have the same shape)
constexpr int T2_STAGE_BYTES = 4 * T2_TILE_BYTES;             // A hi(raw), A lo, B hi(raw), B lo
constexpr int T2_EPI_ROW = 20;                                // staging row: 16 floats + 4 pad
constexpr int T2_EPI_WARP_FLOATS = 32 * T2_EPI_ROW;
constexpr int T2_SMEM_BYTES = T2_STAGES * T2_STAGE_BYTES + 8 * T2_EPI_WARP_FLOATS * 4 + 256 + 1024;
constexpr int T2_DRAIN_KB = 4;                                // chain length in k-blocks (16 main MMA steps), long contractions
constexpr int T2_DRAIN_KB_SHORT = 4;                          // ... short contractions (kb_total <= T2_SHORT_KB); lab knob
constexpr int T2_SHORT_KB = 16;                               // K <= 512
constexpr int T2_PART_KB = 8;                                 // k parts are whole multiples of 8 k-blocks (independent of the chain length)
constexpr int T2_MAX_KPARTS = 64;   // weight gradients: 256 x 256 outputs over 512k nodes need ~37 parts to fill 148 SMs

// one problem of a batched launch (device table; the tensor maps are read by TMA straight from global memory)
struct alignas(64) T2Problem {
  CUtensorMap mapA, mapB;
  CUtensorMap mapC, mapE;   // TMA epilogue (T2Params::tepi): 32 x 32 fp32 boxes of the output and of the fused epilogue operand
  float* C;
  long long ldc;
  int M, N, kb_total, n_chunks;
  const float* E;      // optional epilogue operand [M, N] (lde) and row vector [M]:  C = E o (acc - rowv[row])
  const float* rowv;
  long long lde;
  int pad[2];
};

struct T2Params {
  const T2Problem* batch;   // != nullptr: batched launch (single segment, no k parts); item_off[i] = first item of problem i
  const int* item_off;
  int n_problems;
  int nseg;
  int kb_seg[4];          // k-blocks per segment
  int kb_total;
  int M, N;
  int m_tiles, n_chunks, k_parts, kb_per_part, items;
  int a_mn, b_mn;         // 1 = operand is MN-major in memory (A stored [K,M] / B stored [K,N])
  int drain_kb;
  float* C;
  long long ldc;
  const float* bias;
  int relu, accumulate;
  float* partial;         // [k_parts, M, N] when k_parts > 1
  int pair;               // 1: launched as clusters of two CTAs driving one cta_group::2 MMA (template PAIR)
  int raw_hi;             // 1: the MMA reads the raw fp32 tile as the hi operand (the tensor core ignores the low 13 bits); 0: masked copy
  int lo_rn;              // 1: lo = x - hi is pre-biased by half a tf32 ulp, so the tensor core's truncation rounds it to nearest
  float comp;             // per-MMA compensation of the accumulator's round-towards-zero bias (0 = off); see t2_numerics()
  int tepi;               // 1: TMA epilogue (template TEPI): E tiles arrive by TMA while the tile's MMAs run, C tiles leave by TMA stores
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
// the same two transfers with an L2 evict-first policy: tiles of matrices that stream through once (P / dS: 97 MB per group and head)
// should not push the operand tiles every CTA re-reads out of L2
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* map, uint32_t src, int c0, int c1, uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(map), "r"(src),
               "r"(c0), "r"(c1), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tensormap_acquire(const CUtensorMap* map) {
  asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" ::"l"(map) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// ---- CTA pair (cta_group::2): one MMA spans two SMs; the peer's threads signal barriers that live in the leader's shared memory
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  __syncthreads();   // redundant for the hardware; compute-sanitizer's racecheck does not take the cluster barrier as a CTA barrier
}
__device__ __forceinline__ void mbar_arrive_rank(uint32_t bar, uint32_t rank) {   // arrive on the barrier at the same offset in CTA `rank`
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar), "r"(rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ void umma2_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit2(uint32_t bar) {   // arrives on the barrier at this offset in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((unsigned short)3)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major operand tile [128 rows x 32 k]: SWIZZLE_128B, 8-row groups 1024 B apart; one K = 8 step = +32 B
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major operand tile: 4 TMA boxes [32 k-rows x 32 elements] (SWIZZLE_128B_ATOM_32B) 4096 B apart;
// SWIZZLE_128B_BASE32B canonical layout: LBO = 4096 (next 32 elements along M/N), SBO = 512 (next 4 k-rows);
// one K = 8 step = +1024 B
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((4096 >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((512 >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}

#define T2_TMEM_LD32(R, ADDR)                                                                                            \
  asm volatile(                                                                                                         \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                         \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, " \
      "%24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                                                                 \
      : "=r"(R[0]), "=r"(R[1]), "=r"(R[2]), "=r"(R[3]), "=r"(R[4]), "=r"(R[5]), "=r"(R[6]), "=r"(R[7]), "=r"(R[8]),    \
        "=r"(R[9]), "=r"(R[10]), "=r"(R[11]), "=r"(R[12]), "=r"(R[13]), "=r"(R[14]), "=r"(R[15]), "=r"(R[16]),         \
        "=r"(R[17]), "=r"(R[18]), "=r"(R[19]), "=r"(R[20]), "=r"(R[21]), "=r"(R[22]), "=r"(R[23]), "=r"(R[24]),        \
        "=r"(R[25]), "=r"(R[26]), "=r"(R[27]), "=r"(R[28]), "=r"(R[29]), "=r"(R[30]), "=r"(R[31])                       \
      : "r"(ADDR))

struct T2Item {
  int m0, n0, part, kb0, kb1;
  int M, N;
  float* C;
  long long ldc;
  const CUtensorMap *mapA, *mapB;   // batched launches only
  const CUtensorMap *mapC, *mapE;   // batched launches only (TMA epilogue)
  const float *E, *rowv;            // batched launches only: C = E o (acc - rowv[row])
  long long lde;
};
// work item w of this CTA's sequence (w increases monotonically, so the problem index only moves forward)
__device__ __forceinline__ T2Item t2_item(const T2Params& p, int w, int& pidx, int rank = 0) {
  // p.pair: w counts PAIRS of row tiles (tile 2 q + rank for CTA `rank` of the cluster); a missing odd tile lies beyond M and
  // is all zeros for TMA and all skipped rows for the epilogue
  T2Item it;
  if (p.batch) {
    while (w >= p.item_off[pidx + 1]) ++pidx;
    const T2Problem* q = p.batch + pidx;
    const int local = w - p.item_off[pidx];
    const int nch = q->n_chunks;
    it.part = 0;
    it.n0 = (local % nch) * T2_BN;
    it.m0 = (p.pair ? (local / nch) * 2 + rank : (local / nch)) * T2_BM;
    it.kb0 = 0;
    it.kb1 = q->kb_total;
    it.M = q->M; it.N = q->N; it.C = q->C; it.ldc = q->ldc;
    it.mapA = &q->mapA; it.mapB = &q->mapB;
    it.mapC = &q->mapC; it.mapE = &q->mapE;
    it.E = q->E; it.rowv = q->rowv; it.lde = q->lde;
    return it;
  }
  it.part = w % p.k_parts;
  const int mn = w / p.k_parts;
  it.n0 = (mn % p.n_chunks) * T2_BN;
  it.m0 = (p.pair ? (mn / p.n_chunks) * 2 + rank : (mn / p.n_chunks)) * T2_BM;
  it.kb0 = it.part * p.kb_per_part;
  it.kb1 = min(p.kb_total, it.kb0 + p.kb_per_part);
  it.M = p.M; it.N = p.N; it.C = p.C; it.ldc = p.ldc;
  it.mapA = nullptr; it.mapB = nullptr;
  it.mapC = nullptr; it.mapE = nullptr;
  it.E = nullptr; it.rowv = nullptr; it.lde = 0;
  return it;
}

template <bool PAIR, bool TEPI>
__global__ void __launch_bounds__(T2_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapA3,
                const __grid_constant__ CUtensorMap mapB0, const __grid_constant__ CUtensorMap mapB1,
                const __grid_constant__ CUtensorMap mapB2, const __grid_constant__ CUtensorMap mapB3,
                const __grid_constant__ CUtensorMap mapC0, const T2Params p) {
  static_assert(PAIR || !TEPI, "the TMA epilogue exists for CTA pairs only");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  // A CTA of a pair holds half a B tile: 48 KB per stage instead of 64, so the same 192 KB make FOUR stages — the hand-offs that
  // cross the pair (split warps -> leader's MMA thread, MMA commit -> both producers) take a few hundred cycles longer.
  // TEPI: three stages (144 KB) and a 64 KB epilogue area instead of the 20 KB staging tiles: per epilogue warp one 32 x 64 block as
  // two SWIZZLE_128B boxes of 32 x 32 floats — the landing zone of the fused epilogue operand AND the source of the TMA stores.
  constexpr int NST = PAIR ? (TEPI ? 3 : 4) : T2_STAGES;
  constexpr int STB = PAIR ? 3 * T2_TILE_BYTES : T2_STAGE_BYTES;
  constexpr int RING = NST * STB;
  constexpr int EPI_WARP_BYTES = TEPI ? 8192 : T2_EPI_WARP_FLOATS * 4;
  constexpr int B_OFF = 2 * T2_TILE_BYTES;                              // B hi (raw) behind A hi (raw), A lo
  constexpr int BLO_OFF = PAIR ? B_OFF + T2_TILE_BYTES / 2 : B_OFF + T2_TILE_BYTES;   // B lo right behind B hi
  static_assert(RING + 8 * EPI_WARP_BYTES + 256 + 1024 <= T2_SMEM_BYTES, "shared memory carve");
  static_assert(TEPI || RING == T2_STAGES * T2_STAGE_BYTES, "stage ring size");
  float* epi_stage = reinterpret_cast<float*>(base_ptr + RING);
  const uint32_t bar_base = base + RING + 8 * EPI_WARP_BYTES;
  // barriers (8 B each): full[4], xform[4], empty[4], tfull[2], tempty[2]; the TMEM pointer at +144; TEPI: ebar[8] at +160
  auto ebar = [&](int slot) { return bar_base + 160u + 8u * slot; };
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto xform_bar = [&](int s) { return bar_base + 32u + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 64u + 8u * s; };
  auto tfull_bar = [&](int j) { return bar_base + 96u + 8u * j; };
  auto tempty_bar = [&](int j) { return bar_base + 112u + 8u * j; };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(base_ptr + RING + 8 * EPI_WARP_BYTES + 144);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // PAIR: the two CTAs of a cluster own row tiles 2 q and 2 q + 1 and HALF of the B tile each (64 of its 128 rows); CTA 0 (the
  // leader) issues every MMA with cta_group::2 — M = 256 across the two SMs, each tensor core reading its own A tile and both B
  // halves — so a CTA reads 2 KB of B per MMA instead of 4 and loads / splits 8 KB of B per k-block instead of 16.  The barriers
  // the MMA thread waits on (xform, tempty) live in the leader and count the threads of both CTAs; what the MMA completes
  // (empty, tfull) is committed to both CTAs at once.
  const int rank = PAIR ? (int)cluster_ctarank() : 0;
  const int w0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int wstep = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(xform_bar(s), PAIR ? 8 : 128);      // PAIR: one (remote) arrival per split warp of both CTAs
      mbar_init(empty_bar(s), 1);
    }
    for (int j = 0; j < 2; ++j) {
      mbar_init(tfull_bar(j), 1);
      mbar_init(tempty_bar(j), PAIR ? 16 : 256);   // PAIR: one arrival per epilogue warp of both CTAs
    }
    if (TEPI)
      for (int sl = 0; sl < 8; ++sl) mbar_init(ebar(sl), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_ptr_smem)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_ptr_smem)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // the peer's barriers exist before anything is signalled across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      const CUtensorMap* mA[4] = {&mapA0, &mapA1, &mapA2, &mapA3};
      const CUtensorMap* mB[4] = {&mapB0, &mapB1, &mapB2, &mapB3};
      int it = 0, pidx = 0, fenced = -1;
      for (int w = w0; w < p.items; w += wstep) {
        const T2Item item = t2_item(p, w, pidx, rank);
        if (p.batch) {
          mA[0] = item.mapA; mB[0] = item.mapB;
          if (fenced != pidx) {
            // Tensor maps that live in GLOBAL memory (the uploaded problem table; its workspace address is recycled from
            // launch to launch) must be acquired through the tensormap proxy before the TMA unit may use them, or it can
            // serve a stale descriptor cached under the same address (CUDA programming guide, tensor maps in global memory).
            tensormap_acquire(item.mapA);
            tensormap_acquire(item.mapB);
            fenced = pidx;
          }
        }
        int seg = 0, seg_kb0 = 0;   // segment containing k-block kb, and its first k-block
        for (int kb = item.kb0; kb < item.kb1; ++kb, ++it) {
          if (!p.batch)
            while (kb >= seg_kb0 + p.kb_seg[seg]) { seg_kb0 += p.kb_seg[seg]; ++seg; }
          const int k0 = (kb - seg_kb0) * T2_BK;
          const int st = it % NST;
          const uint32_t ph = (it / NST) & 1;
          mbar_wait(empty_bar(st), ph ^ 1);
          const uint32_t sbase = base + st * STB;
          mbar_expect_tx(full_bar(st), PAIR ? T2_TILE_BYTES + T2_TILE_BYTES / 2 : 2 * T2_TILE_BYTES);
          if (p.a_mn) {
#pragma unroll
            for (int c = 0; c < 4; ++c) tma_load_2d(sbase + c * 4096, mA[seg], full_bar(st), item.m0 + c * 32, k0);
          } else {
            tma_load_2d(sbase, mA[seg], full_bar(st), k0, item.m0);
          }
          if (PAIR) {   // this CTA's half of the B tile: rows [64 rank, 64 rank + 64) of the chunk (box of 64 rows / two 32-wide boxes)
            const int nb0 = item.n0 + rank * (T2_BN / 2);
            if (p.b_mn) {
#pragma unroll
              for (int c = 0; c < 2; ++c) tma_load_2d(sbase + 2 * T2_TILE_BYTES + c * 4096, mB[seg], full_bar(st), nb0 + c * 32, k0);
            } else {
              tma_load_2d(sbase + 2 * T2_TILE_BYTES, mB[seg], full_bar(st), k0, nb0);
            }
          } else if (p.b_mn) {
#pragma unroll
            for (int c = 0; c < 4; ++c) tma_load_2d(sbase + 2 * T2_TILE_BYTES + c * 4096, mB[seg], full_bar(st), item.n0 + c * 32, k0);
          } else {
            tma_load_2d(sbase + 2 * T2_TILE_BYTES, mB[seg], full_bar(st), k0, item.n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (PAIR: the leader CTA only)
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)p.a_mn << 15) | ((uint32_t)p.b_mn << 16) |
                             ((uint32_t)(T2_BN >> 3) << 17) | ((uint32_t)(T2_BM >> 4) << 24);
      const uint32_t a_adv = p.a_mn ? (1024u >> 4) : (32u >> 4), b_adv = p.b_mn ? (1024u >> 4) : (32u >> 4);
      // N = 256 form of the same descriptor: the B_lo tile follows the B_hi tile in shared memory (same canonical layout), so
      // ONE MMA gives [ A_hi B_hi | A_hi B_lo ] in 256 adjacent TMEM columns; a second N = 128 MMA adds A_lo B_hi onto the
      // cross half.  2 MMAs and 20 KB of operand reads per K = 8 step instead of 3 and 24 KB.
      const uint32_t idesc256 = (idesc & ~(0x3Fu << 17)) | ((uint32_t)(2 * T2_BN >> 3) << 17);
      // PAIR: M = 256 over the two CTAs, N = 128; three N = 128 MMAs per K = 8 step (the stacked [B_hi ; B_lo] form would interleave
      // main and cross columns per CTA half, which a single N = 128 cross-term MMA cannot follow)
      const uint32_t idesc_pair = (idesc & ~(0x1Fu << 24)) | ((uint32_t)(2 * T2_BM >> 4) << 24);
      int it = 0, chain = 0, pidx = 0;
      for (int w = w0; w < p.items; w += wstep) {
        const T2Item item = t2_item(p, w, pidx, rank);
        for (int kc0 = item.kb0; kc0 < item.kb1; kc0 += p.drain_kb, ++chain) {
          const int kc1 = min(item.kb1, kc0 + p.drain_kb);
          const int j = chain & 1;   // TMEM columns [256 j, 256 j + 128) main, [256 j + 128, 256 j + 256) cross terms
          const uint32_t d_main = tmem_base + (uint32_t)(2 * T2_BN * j), d_cross = d_main + (uint32_t)T2_BN;
          mbar_wait(tempty_bar(j), ((chain >> 1) & 1) ^ 1);
          tc_fence_after();
          for (int kb = kc0; kb < kc1; ++kb, ++it) {
            const int st = it % NST;
            const uint32_t ph = (it / NST) & 1;
            mbar_wait(full_bar(st), ph);
            mbar_wait(xform_bar(st), ph);   // PAIR: both CTAs' tiles have landed and are split
            tc_fence_after();
            const uint32_t sbase = base + st * STB;
            const uint64_t a_hi = p.a_mn ? desc_mnmajor(sbase) : desc_kmajor(sbase);
            const uint64_t a_lo = p.a_mn ? desc_mnmajor(sbase + T2_TILE_BYTES) : desc_kmajor(sbase + T2_TILE_BYTES);
            const uint64_t b_hi = p.b_mn ? desc_mnmajor(sbase + 2 * T2_TILE_BYTES) : desc_kmajor(sbase + 2 * T2_TILE_BYTES);
            if (PAIR) {
              const uint64_t b_lo = p.b_mn ? desc_mnmajor(sbase + BLO_OFF) : desc_kmajor(sbase + BLO_OFF);
#pragma unroll
              for (int kk = 0; kk < T2_BK / 8; ++kk) {
                const uint64_t aa = (uint64_t)(kk * a_adv), bb = (uint64_t)(kk * b_adv);
                const uint32_t acc = (kb > kc0 || kk > 0) ? 1u : 0u;
                umma2_tf32(d_main, a_hi + aa, b_hi + bb, idesc_pair, acc);    // main  = A_hi B_hi
                umma2_tf32(d_cross, a_hi + aa, b_lo + bb, idesc_pair, acc);   // cross = A_hi B_lo
                umma2_tf32(d_cross, a_lo + aa, b_hi + bb, idesc_pair, 1u);    //       + A_lo B_hi
              }
              umma_commit2(empty_bar(st));
            } else {
#pragma unroll
            for (int kk = 0; kk < T2_BK / 8; ++kk) {
              const uint64_t aa = (uint64_t)(kk * a_adv), bb = (uint64_t)(kk * b_adv);
              const uint32_t acc = (kb > kc0 || kk > 0) ? 1u : 0u;   // both halves restart with every chain
              umma_tf32(d_main, a_hi + aa, b_hi + bb, idesc256, acc);   // [main | A_hi B_lo]
              umma_tf32(d_cross, a_lo + aa, b_hi + bb, idesc, 1u);      // cross += A_lo B_hi
            }
            umma_commit(empty_bar(st));
            }
          }
          if (PAIR) umma_commit2(tfull_bar(j)); else umma_commit(tfull_bar(j));
        }
      }
    }
  } else if (warp >= 8 && warp < 12) {
    // ------------------------------------------------------------------ split warps: X -> X_hi (in place), X_lo
    const int t = threadIdx.x - 256;
    const uint32_t rb = p.lo_rn ? 0x1000u : 0u;
    int it = 0, pidx = 0;
    for (int w = w0; w < p.items; w += wstep) {
      const T2Item item = t2_item(p, w, pidx, rank);
      for (int kb = item.kb0; kb < item.kb1; ++kb, ++it) {
        const int st = it % NST;
        const uint32_t ph = (it / NST) & 1;
        mbar_wait(full_bar(st), ph);
        uint4* a = reinterpret_cast<uint4*>(base_ptr + st * STB);
        uint4* b = reinterpret_cast<uint4*>(base_ptr + st * STB + B_OFF);
        constexpr int LO = T2_TILE_BYTES / 16;   // the lo tile follows its hi tile (PAIR: half a B tile -> half the distance)
        constexpr int LO_B = (BLO_OFF - B_OFF) / 16;
#pragma unroll
        for (int i = 0; i < 2 * T2_TILE_BYTES / 16 / 128; ++i) {
          if (PAIR && (i & 1) && (i >> 1) >= T2_TILE_BYTES / 32 / 128) continue;   // PAIR: half a B tile (8 KB)
          uint4* src = (i & 1) ? b : a;
          const int idx = t + (i >> 1) * 128;
          const uint4 v = src[idx];
          // Branch-free on purpose: this loop is the critical path of the kernel, fully unrolled so that all 16 shared-memory
          // loads are in flight before the first use; an if / else around the arithmetic serialised them and cost 17 % of the
          // kernel (A/B against the round-1 build on the same box, profiles/r02_gemm_ab.txt).
          //   hi = trunc_tf32(x): the raw tile itself serves as hi (the tensor core ignores the low 13 bits of a tf32 operand);
          //   lo = (x - hi) + rb on the bit pattern: rb = 0x1000 pre-biases the remainder by half a tf32 ulp, so that the same
          //        truncation rounds lo to nearest (ties away) instead of towards zero: the cross terms lose their systematic
          //        shrink for one integer add per element (a cvt.rna.tf32 here is quarter-rate and cost 17 % as well).
          const uint4 h = make_uint4(v.x & 0xFFFFE000u, v.y & 0xFFFFE000u, v.z & 0xFFFFE000u, v.w & 0xFFFFE000u);
          uint4 l;
          l.x = __float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)) + rb;
          l.y = __float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)) + rb;
          l.z = __float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)) + rb;
          l.w = __float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)) + rb;
          if (!p.raw_hi) src[idx] = h;
          src[idx + ((i & 1) ? LO_B : LO)] = l;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (PAIR) {
          __syncwarp();   // every lane's tile writes (and its proxy fence) precede the one arrival of the warp
          if (lane == 0) mbar_arrive_rank(xform_bar(st), 0);
        } else {
          mbar_arrive(xform_bar(st));
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue: warps 4-7 columns 0-63, warps 12-15 columns 64-127
    const int q = warp & 3;               // TMEM lane quarter == warp % 4
    const int half = warp >= 12 ? 1 : 0;
    float* stg = epi_stage + ((half * 4) + q) * T2_EPI_WARP_FLOATS;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 64);
    int chain = 0, pidx = 0;
    // TEPI: this warp's 32 x 64 block lives in two SWIZZLE_128B boxes (32 rows x 32 floats, 4 KB each): row r at r * 128 B, its
    // 16-byte chunk c at physical chunk c ^ (r & 7) — the 8 lanes of a quarter-warp touch 8 different chunks: conflict-free
    const int slot = half * 4 + q;
    const uint32_t ebuf = base + RING + slot * 8192;
    uint8_t* ebuf_ptr = base_ptr + RING + slot * 8192;
    uint32_t eph = 0;
    int efenced = -1;
    const bool ehint = TEPI && (p.tepi & 2);
    const uint64_t epol = ehint ? l2_evict_first_policy() : 0ull;
    for (int w = w0; w < p.items; w += wstep) {
      const T2Item item = t2_item(p, w, pidx, rank);
      const bool vec_ok = ((item.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(item.C) & 15) == 0) &&
                          (!p.bias || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0) && ((item.N & 3) == 0 || p.k_parts == 1);
      float acc[64];
#pragma unroll
      for (int i = 0; i < 64; ++i) acc[i] = 0.f;
      const CUtensorMap* mC = TEPI ? (p.batch ? item.mapC : &mapC0) : nullptr;
      const int ecol0 = item.n0 + half * 64, erow0 = item.m0 + q * 32;
      if (TEPI) {
        // The previous item's stores have read the block; then the fused epilogue operand of THIS item starts its way into it
        // while the tile's MMAs are still running: no load latency is left on the epilogue's critical path.
        if (lane == 0) {
          bulk_wait_read0();
          if (p.batch && efenced != pidx) {
            tensormap_acquire(item.mapC);
            if (item.E != nullptr) tensormap_acquire(item.mapE);
            efenced = pidx;
          }
          if (item.E != nullptr) {
            mbar_expect_tx(ebar(slot), 8192);
            if (ehint) {
              tma_load_2d_hint(ebuf, item.mapE, ebar(slot), ecol0, erow0, epol);
              tma_load_2d_hint(ebuf + 4096, item.mapE, ebar(slot), ecol0 + 32, erow0, epol);
            } else {
              tma_load_2d(ebuf, item.mapE, ebar(slot), ecol0, erow0);
              tma_load_2d(ebuf + 4096, item.mapE, ebar(slot), ecol0 + 32, erow0);
            }
          }
        }
        __syncwarp();
      }
      if (!TEPI && item.E != nullptr) {
        // The fused epilogue operand of a 32 x 64 block (2-3 lines per row) is pulled into L2 ONE ITEM AHEAD: with the fused
        // epilogue this warp is the bottleneck of the tile pipeline (the MMAs of its current item are long done when it gets
        // here), so a prefetch for the current item would be issued just before its first use.
        auto prefetch_block = [&](const T2Item& it2) {
          const int prow = it2.m0 + q * 32 + lane;
          const int pcol = it2.n0 + half * 64;
          if (it2.E != nullptr && prow < it2.M && pcol < it2.N) {
            const float* pe = it2.E + (long long)prow * it2.lde + pcol;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pe));
            if (pcol + 32 < it2.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(pe + 32));
            if (pcol + 63 < it2.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(pe + 63));
          }
        };
        if (w == w0) prefetch_block(item);
        if (w + wstep < p.items) {
          int pidx2 = pidx;
          prefetch_block(t2_item(p, w + wstep, pidx2, rank));
        }
      }
      for (int kc0 = item.kb0; kc0 < item.kb1; kc0 += p.drain_kb, ++chain) {
        const int j = chain & 1;
        mbar_wait(tfull_bar(j), (chain >> 1) & 1);
        tc_fence_after();
        const uint32_t cbase = lane_addr + (uint32_t)(2 * T2_BN * j);
        // the main chain just drained went through 4 MMAs per k-block, each rounding the accumulator towards zero
        const float comp = 1.0f + p.comp * (float)(4 * (min(item.kb1, kc0 + p.drain_kb) - kc0));
        uint32_t r[32];
#pragma unroll
        for (int part = 0; part < 4; ++part) {   // main columns 0-31, 32-63 of this warp's half, then the cross-term columns
          T2_TMEM_LD32(r, cbase + (uint32_t)((part >> 1) * T2_BN + (part & 1) * 32));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (part == 3) {
            tc_fence_before();
            if (PAIR) {   // the accumulator pair is free again as soon as it sits in registers
              __syncwarp();
              if (lane == 0) mbar_arrive_rank(tempty_bar(j), 0);
            } else {
              mbar_arrive(tempty_bar(j));
            }
          }
          if (part < 2) {   // main (hi x hi) columns: add the chain with its expected truncation loss given back
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[(part & 1) * 32 + i] = fmaf(__uint_as_float(r[i]), comp, acc[(part & 1) * 32 + i]);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[(part & 1) * 32 + i] += __uint_as_float(r[i]);
          }
        }
      }
      if (TEPI) {
        // ---- registers -> (o E) -> swizzled block -> TMA stores (rows / columns beyond M / N are clipped by the TMA unit; the
        // operand's out-of-range elements arrive as zeros)
        const int row = erow0 + lane;
        float d = 0.f;
        if (item.E != nullptr) {
          if (row < item.M) d = __ldg(item.rowv + row);
          mbar_wait(ebar(slot), eph);
          eph ^= 1;
        }
        const float* bias = p.bias;
        const bool bias_vec = bias && ((reinterpret_cast<uintptr_t>(bias) & 15) == 0);
#pragma unroll
        for (int b = 0; b < 2; ++b) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            float4* cell = reinterpret_cast<float4*>(ebuf_ptr + b * 4096 + lane * 128 + ((c ^ (lane & 7)) << 4));
            float4 v = make_float4(acc[b * 32 + c * 4], acc[b * 32 + c * 4 + 1], acc[b * 32 + c * 4 + 2], acc[b * 32 + c * 4 + 3]);
            if (bias) {
              const int col = ecol0 + b * 32 + c * 4;
              if (bias_vec && col + 3 < item.N) {
                const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + col));
                v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
              } else {
                if (col < item.N) v.x += __ldg(bias + col);
                if (col + 1 < item.N) v.y += __ldg(bias + col + 1);
                if (col + 2 < item.N) v.z += __ldg(bias + col + 2);
                if (col + 3 < item.N) v.w += __ldg(bias + col + 3);
              }
            }
            if (item.E != nullptr) {   // fused softmax backward  dS = P o (dP - rowsum(dP o P))  (E = P, rowv = rowdot(dO, O))
              const float4 e = *cell;
              v.x = e.x * (v.x - d); v.y = e.y * (v.y - d); v.z = e.z * (v.z - d); v.w = e.w * (v.w - d);
            }
            if (p.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            *cell = v;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          if (ehint) {
            tma_store_2d_hint(mC, ebuf, ecol0, erow0, epol);
            tma_store_2d_hint(mC, ebuf + 4096, ecol0 + 32, erow0, epol);
          } else {
            tma_store_2d(mC, ebuf, ecol0, erow0);
            tma_store_2d(mC, ebuf + 4096, ecol0 + 32, erow0);
          }
          bulk_commit();
        }
        continue;
      }
      // ---- write the 32 x 64 block of this warp, 16 columns at a time through a padded staging tile
      const bool to_slab = p.k_parts > 1;
      float* outp = to_slab ? p.partial + (size_t)item.part * (size_t)item.M * item.N : item.C;
      const long long ldo = to_slab ? (long long)item.N : item.ldc;
      const bool add_c = !to_slab && p.accumulate;
      const bool do_relu = !to_slab && p.relu;
      const float* bias = to_slab ? nullptr : p.bias;
      const int row0 = item.m0 + q * 32;
      if (item.E != nullptr && vec_ok && !add_c && !do_relu && !bias && (item.N & 3) == 0 && (item.lde & 3) == 0 &&
          (reinterpret_cast<uintptr_t>(item.E) & 15) == 0) {
        // ---- fused softmax backward  dS = P o (dP - rowsum(dP o P))  (E = P, rowv = rowdot(dO, O)): the operand loads of a
        // 16-column group are issued one group AHEAD of the stores.  Inside the store loop the compiler has to keep them in
        // program order behind the stores (C may alias E), which serialised 16 DRAM round trips per tile and ran this product
        // at 89 TFLOP/s against 196 for its plain siblings (profiles/r02_launches_train_c3.csv, launch 294).
        // lane -> (row, 16-byte column chunk) of the staged 32 x 16 block: the 8 lanes of a quarter-warp read 8 DIFFERENT rows at the
        // same chunk (row pitch 80 B = 5 chunks: 5 r mod 8 is a permutation -> conflict-free); 4 chunks x 8 rows per store instruction
        const int c4 = (lane >> 3) * 4;
        const int rsub = lane & 7;
        const int colbase = item.n0 + half * 64 + c4;
        const float* erow = item.E + (long long)(row0 + rsub) * item.lde + colbase;
        float* orow = outp + (long long)(row0 + rsub) * ldo + colbase;
        float4 xa[4], xb[4];
        float dv[4];
#pragma unroll
        for (int it4 = 0; it4 < 4; ++it4) dv[it4] = (row0 + it4 * 8 + rsub < item.M) ? __ldg(item.rowv + row0 + it4 * 8 + rsub) : 0.f;
        auto load_group = [&](float4 (&x)[4], int g) {
#pragma unroll
          for (int it4 = 0; it4 < 4; ++it4) {
            x[it4] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row0 + it4 * 8 + rsub < item.M && colbase + g * 16 < item.N)
              x[it4] = __ldcs(reinterpret_cast<const float4*>(erow + (long long)(it4 * 8) * item.lde + g * 16));
          }
        };
        load_group(xa, 0);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
#pragma unroll
          for (int jv = 0; jv < 16; jv += 4)
            *reinterpret_cast<float4*>(stg + lane * T2_EPI_ROW + jv) = make_float4(acc[g * 16 + jv], acc[g * 16 + jv + 1], acc[g * 16 + jv + 2], acc[g * 16 + jv + 3]);
          __syncwarp();
          if (g + 1 < 4) { if (g & 1) load_group(xa, g + 1); else load_group(xb, g + 1); }
#pragma unroll
          for (int it4 = 0; it4 < 4; ++it4) {
            const int rr = it4 * 8 + rsub;
            if (row0 + rr < item.M && colbase + g * 16 < item.N) {
              float4 v = *reinterpret_cast<const float4*>(stg + rr * T2_EPI_ROW + c4);
              const float4 e = (g & 1) ? xb[it4] : xa[it4];
              const float d = dv[it4];
              v.x = e.x * (v.x - d); v.y = e.y * (v.y - d); v.z = e.z * (v.z - d); v.w = e.w * (v.w - d);
              // streaming store: 2 x 12.5 GB of P / dS pass through L2 per train step next to operand tiles that every CTA re-reads
              __stcs(reinterpret_cast<float4*>(orow + (long long)(it4 * 8) * ldo + g * 16), v);
            }
          }
          __syncwarp();
        }
        continue;
      }
#pragma unroll
      for (int g = 0; g < 4; ++g) {
#pragma unroll
        for (int jv = 0; jv < 16; jv += 4)
          *reinterpret_cast<float4*>(stg + lane * T2_EPI_ROW + jv) = make_float4(acc[g * 16 + jv], acc[g * 16 + jv + 1], acc[g * 16 + jv + 2], acc[g * 16 + jv + 3]);
        __syncwarp();
        const int c4 = (lane >> 3) * 4;   // see the fused path: conflict-free reads of the staging tile
        const int col = item.n0 + half * 64 + g * 16 + c4;
        if (vec_ok && col + 3 < item.N) {
          const float4 bv = bias ? *reinterpret_cast<const float4*>(bias + col) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int it4 = 0; it4 < 4; ++it4) {
            const int rr = it4 * 8 + (lane & 7);
            const int row = row0 + rr;
            if (row < item.M) {
              float4 v = *reinterpret_cast<const float4*>(stg + rr * T2_EPI_ROW + c4);
              v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
              if (item.E) {   // fused softmax backward: dS = P o (dP - rowsum(dP o P)), the row sums precomputed as rowdot(dO, O)
                const float d = item.rowv[row];
                const float* ep = item.E + (long long)row * item.lde + col;
                float4 e4;
                if (((item.lde & 3) == 0) && ((reinterpret_cast<uintptr_t>(item.E) & 15) == 0)) e4 = *reinterpret_cast<const float4*>(ep);
                else e4 = make_float4(ep[0], ep[1], ep[2], ep[3]);
                v.x = e4.x * (v.x - d); v.y = e4.y * (v.y - d); v.z = e4.z * (v.z - d); v.w = e4.w * (v.w - d);
              }
              float4* dst = reinterpret_cast<float4*>(outp + (long long)row * ldo + col);
              if (add_c) { const float4 o = *dst; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
              if (do_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
              *dst = v;
            }
          }
        } else {
          for (int it4 = 0; it4 < 4; ++it4) {
            const int rr = it4 * 8 + (lane & 7);
            const int row = row0 + rr;
            for (int e = 0; e < 4; ++e) {
              if (row < item.M && col + e < item.N) {
                float v = stg[rr * T2_EPI_ROW + c4 + e] + (bias ? bias[col + e] : 0.f);
                if (item.E) v = item.E[(long long)row * item.lde + col + e] * (v - item.rowv[row]);
                float* dst = outp + (long long)row * ldo + col + e;
                if (add_c) v += *dst;
                if (do_relu) v = fmaxf(v, 0.f);
                *dst = v;
              }
            }
          }
        }
        __syncwarp();
      }
    }
  }

  if (TEPI && warp >= 4 && !(warp >= 8 && warp < 12) && lane == 0) bulk_wait0();   // this warp's last TMA stores have left the block
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // PAIR: neither CTA may leave while the other can still signal its barriers
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// C = act( sum over k parts (fixed order) + bias ) (+C)
__global__ void t2_reduce_kernel(const float* __restrict__ partial, int parts, long long MN, int N, float* __restrict__ C,
                                 long long ldc, const float* __restrict__ bias, int relu, int accumulate) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= MN) return;
  const long long m = idx / N;
  const int n = (int)(idx % N);
  float s = 0.f;
  for (int z = 0; z < parts; ++z) s += partial[(size_t)z * MN + idx];
  if (bias) s += bias[n];
  float* dst = C + m * ldc + n;
  if (accumulate) s += *dst;
  if (relu) s = fmaxf(s, 0.f);
  *dst = s;
}

typedef CUresult (*EncodeFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn2 get_encode2() {
  static EncodeFn2 fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn2>(sym);
  }
  return fn;
}

// operand stored as `rows` x `inner` fp32 with leading dimension ld; box = [32 inner, box_rows]
int make_map2(CUtensorMap* map, const float* ptr, uint64_t inner, uint64_t rows, uint64_t ld_elems, uint32_t box_rows,
              CUtensorMapSwizzle swz) {
  EncodeFn2 enc = get_encode2();
  DC_REQUIRE(enc, DC_ECUDA, "gemm_tc2: cuTensorMapEncodeTiled not available");
  cuuint64_t gdim[2] = {inner, rows};
  cuuint64_t gstr[1] = {ld_elems * 4};
  cuuint32_t box[2] = {T2_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DC_REQUIRE(r == CUDA_SUCCESS, DC_ECUDA, "gemm_tc2: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return DC_OK;
}

// Chain length in k-blocks.  The tensor core rounds its fp32 accumulator towards zero on every MMA, a bias of ~0.5 ulp per
// MMA on the main (hi x hi) chain: 32 MMAs per chain gave 0.8-1.0e-6 against fp64 (round 1), 16 give 4.6e-7, 4 give ~3e-7
// (profiles/r02_gemm_drain_lab.txt).  A separate length for short contractions (K <= 512: the attention scores Q K^T and
// dP = dO Xr^T, whose absolute error the unscaled softmax amplifies) was measured too: no gain, so both classes use 4
// (DCB200_DRAIN_KB / DCB200_DRAIN_KB_SHORT remain as lab knobs).
int t2_drain_kb(int64_t kb_total) {
  static int d_long = -1, d_short = -1;
  if (d_long < 0) {
    const char* e = getenv("DCB200_DRAIN_KB");
    d_long = (e && atoi(e) > 0) ? atoi(e) : T2_DRAIN_KB;
    const char* es = getenv("DCB200_DRAIN_KB_SHORT");
    d_short = (es && atoi(es) > 0) ? atoi(es) : T2_DRAIN_KB_SHORT;
  }
  return kb_total <= T2_SHORT_KB ? (d_short < d_long ? d_short : d_long) : d_long;
}

// Numerics of the split and of the TMEM accumulation (both measured in profiles/r02_gemm_numerics_lab.txt):
//  * lo_rn: the tensor core truncates tf32 operands; pre-biasing the lo remainder by half a tf32 ulp turns that into
//    round-to-nearest (the hi part is the raw tile itself and stays truncated).
//  * comp: the tensor core rounds its fp32 accumulator TOWARDS ZERO on every MMA.  One such rounding loses u * ulp(acc) with
//    u ~ U[0, 1): 0.5 * 2^-23 * E[1/mantissa] = 4.3e-8 of |acc| on average.  Over a chain of n MMAs whose partial sums grow
//    from 0 to x (|acc_t| / |x| ~ t/n for sign-coherent products such as P Xr, ~ sqrt(t/n) for random signs) that is
//    ~ 0.6 n * 4.3e-8 |x|, always towards zero: a BIAS, which is what sum-with-cancellation reductions downstream (bias
//    gradients, softmax backward) amplify.  The epilogue gives that expectation back when it adds a drained chain:
//    acc += x * (1 + comp * n), comp = 2.6e-8.  Deterministic; exact when no rounding happened it over-corrects by at most
//    comp * n = 4e-7 relative (n = 16), the size of the error it removes on dense data.
void t2_numerics(T2Params& p) {
  static int lo_rn = -1;
  static float comp = -1.f;
  if (lo_rn < 0) {
    const char* e = getenv("DCB200_T2_LO_RN");
    lo_rn = e ? (e[0] == '1') : 1;
    const char* c = getenv("DCB200_T2_COMP");
    comp = c ? (float)atof(c) : 2.6e-8f;
  }
  p.lo_rn = lo_rn;
  p.comp = comp;
}

// CTA pairs (cta_group::2) unless DCB200_T2_PAIR=0
int t2_pair() {
  static int pair = -1;
  if (pair < 0) {
    const char* e = getenv("DCB200_T2_PAIR");
    pair = e ? (e[0] == '1') : 1;
  }
  return pair;
}

// TMA epilogue (CTA pairs only): DCB200_T2_TEPI = 0 off, 1 for short contractions (K <= 512: the products whose tile time is set by
// the epilogue — attention scores, the fused softmax-backward product, the K = 256 layer products), 2 for every K, 3 (default) = as 2,
// but a batched launch takes it only when a problem carries a fused epilogue operand: the plain batched scores product prefers the
// fourth pipeline stage (same-box A/B, profiles/r02c_tepi_ab.txt: 92.10 -> 91.79 ms per step)
int t2_tepi_mode() {
  static int mode = -1;
  if (mode < 0) {
    const char* e = getenv("DCB200_T2_TEPI");
    mode = e ? atoi(e) : 3;
  }
  return mode;
}
bool t2_tepi_ok(int pair, int64_t kb_max, int k_parts, int accumulate) {
  const int mode = t2_tepi_mode();
  return pair && mode > 0 && k_parts == 1 && !accumulate && (mode > 1 || kb_max <= T2_SHORT_KB);
}
// An [M, N] operand the TMA epilogue can address.  N % 4 == 0 as well: the TMA stores of the swizzled output boxes write the whole
// 16-byte chunk that holds column N - 1, so a row of N % 4 != 0 floats would get up to three floats past its end overwritten
// (measured on the B200 with C a view into a wider buffer).
bool t2_tepi_operand_ok(const float* ptr, int64_t ld, int64_t N) {
  return ptr && (ld & 3) == 0 && (N & 3) == 0 && (reinterpret_cast<uintptr_t>(ptr) & 15) == 0;
}

// one persistent CTA per SM; PAIR: clusters of two CTAs (an even grid)
int t2_launch(const CUtensorMap* mA, const CUtensorMap* mB, const CUtensorMap& mC, const T2Params& p, cudaStream_t st) {
  static DeviceOnce attr_set;
  if (attr_set.first()) {
    DC_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
    DC_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
    DC_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
  }
  if (!p.pair) {
    const int grid = p.items < sm_count() ? p.items : sm_count();
    gemm_tc2_kernel<false, false><<<grid, T2_THREADS, T2_SMEM_BYTES, st>>>(mA[0], mA[1], mA[2], mA[3], mB[0], mB[1], mB[2], mB[3], mC, p);
  } else {
    const int pairs = p.items < sm_count() / 2 ? p.items : sm_count() / 2;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(2 * pairs));
    cfg.blockDim = dim3(T2_THREADS);
    cfg.dynamicSmemBytes = T2_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (p.tepi) DC_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc2_kernel<true, true>, mA[0], mA[1], mA[2], mA[3], mB[0], mB[1], mB[2], mB[3], mC, p));
    else DC_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc2_kernel<true, false>, mA[0], mA[1], mA[2], mA[3], mB[0], mB[1], mB[2], mB[3], mC, p));
  }
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int t2_k_parts(int64_t M, int64_t N, int64_t kb_total) {
  const int64_t mn = cdiv(M, T2_BM) * cdiv(N, T2_BN);
  if (mn >= sm_count()) return 1;
  int64_t parts = sm_count() / mn;                          // fill the machine once
  const int64_t max_parts = kb_total / T2_PART_KB;    // at least 8 k-blocks per part
  if (parts > max_parts) parts = max_parts;
  if (parts > T2_MAX_KPARTS) parts = T2_MAX_KPARTS;
  return parts < 1 ? 1 : (int)parts;
}
}  // namespace

bool gemm_tc2_supported(const dc_gemm_seg* segs, int nseg, int transA, int transB, int64_t M, int64_t N) {
  if (nseg < 1 || nseg > 4 || M < 1 || N < 1 || M >= (1ll << 31) || N >= (1ll << 31)) return false;
  if (nseg > 1 && (transA || !transB)) return false;   // multi-segment: K-major A and B only (the TAGConv layer GEMM)
  for (int s = 0; s < nseg; ++s) {
    if (segs[s].K <= 0 || segs[s].K >= (1ll << 31)) return false;
    if (segs[s].lda % 4 != 0 || segs[s].ldb % 4 != 0) return false;   // TMA: 16-byte row pitch
    if ((reinterpret_cast<uintptr_t>(segs[s].A) & 15) || (reinterpret_cast<uintptr_t>(segs[s].B) & 15)) return false;
  }
  return true;
}

size_t gemm_tc2_workspace_bytes(int64_t M, int64_t N, int64_t Ktot) {
  const int parts = t2_k_parts(M, N, cdiv(Ktot, T2_BK));
  return parts > 1 ? align_up((size_t)parts * M * N * sizeof(float), 256) + 256 : 0;
}

int gemm_tc2(const dc_gemm_seg* segs, int nseg, int transA, int transB, int64_t M, int64_t N, float* C, int64_t ldc,
             const float* bias, int relu, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  DC_REQUIRE(gemm_tc2_supported(segs, nseg, transA, transB, M, N), DC_ENOSUP, "gemm_tc2: layout not supported by the tcgen05 path");
  T2Params p{};
  p.nseg = nseg;
  p.a_mn = transA ? 1 : 0;
  p.b_mn = transB ? 0 : 1;
  p.pair = t2_pair();
  const uint32_t b_box_rows = p.pair ? T2_BN / 2 : T2_BN;   // a CTA of a pair loads half of the B tile
  CUtensorMap mA[4], mB[4];
  int64_t ktot = 0, kelems = 0;
  for (int s = 0; s < 4; ++s) {
    const int ss = s < nseg ? s : 0;
    const uint64_t K = (uint64_t)segs[ss].K;
    if (transA) {   // stored [K, M]: inner = M
      if (int rc = make_map2(&mA[s], segs[ss].A, (uint64_t)M, K, (uint64_t)segs[ss].lda, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    } else {        // stored [M, K]: inner = K
      if (int rc = make_map2(&mA[s], segs[ss].A, K, (uint64_t)M, (uint64_t)segs[ss].lda, T2_BM, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    if (transB) {   // stored [N, K]: inner = K
      if (int rc = make_map2(&mB[s], segs[ss].B, K, (uint64_t)N, (uint64_t)segs[ss].ldb, b_box_rows, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    } else {        // stored [K, N]: inner = N
      if (int rc = make_map2(&mB[s], segs[ss].B, (uint64_t)N, K, (uint64_t)segs[ss].ldb, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    }
    p.kb_seg[s] = s < nseg ? (int)cdiv(segs[s].K, T2_BK) : (1 << 30);
    if (s < nseg) ktot += cdiv(segs[s].K, T2_BK), kelems += segs[s].K;
  }
  p.kb_total = (int)ktot;
  p.M = (int)M; p.N = (int)N;
  p.m_tiles = (int)cdiv(M, T2_BM);
  p.n_chunks = (int)cdiv(N, T2_BN);
  // the number of parts follows the contraction length, as in gemm_tc2_workspace_bytes: segments whose K is not a multiple of
  // 32 each add a partial k-block, which must not raise the part count above what the workspace query promised
  p.k_parts = t2_k_parts(M, N, cdiv(kelems, T2_BK));
  p.kb_per_part = (int)(cdiv(cdiv(p.kb_total, p.k_parts), T2_PART_KB) * T2_PART_KB);   // whole chains per part
  p.k_parts = (int)cdiv(p.kb_total, p.kb_per_part);
  p.items = (p.pair ? (p.m_tiles + 1) / 2 : p.m_tiles) * p.n_chunks * p.k_parts;   // pair: items are pairs of row tiles
  p.drain_kb = t2_drain_kb(p.kb_total);
  p.C = C; p.ldc = ldc; p.bias = bias; p.relu = relu; p.accumulate = accumulate;
  // measured r01: identical error against fp64 with and without the masked copy (the tensor core reads only the
  // upper 19 bits of a tf32 operand), 7-10 % faster without the extra shared-memory write
  p.raw_hi = 1;
  if (const char* e = getenv("DCB200_T2_RAWHI")) p.raw_hi = e[0] == '1';
  t2_numerics(p);
  if (p.k_parts > 1) {
    const size_t need = align_up((size_t)p.k_parts * M * N * sizeof(float), 256) + 256;
    DC_REQUIRE(workspace && workspace_bytes >= need, DC_EWORKSPACE, "gemm_tc2: workspace %zu < %zu", workspace_bytes, need);
    p.partial = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  }
  CUtensorMap mC{};
  p.tepi = t2_tepi_ok(p.pair, p.kb_total, p.k_parts, accumulate) && t2_tepi_operand_ok(C, ldc, N);
  if (p.tepi)
    if (int rc = make_map2(&mC, C, (uint64_t)N, (uint64_t)M, (uint64_t)ldc, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = t2_launch(mA, mB, mC, p, st)) return rc;
  if (p.k_parts > 1) {
    const long long MN = (long long)M * N;
    t2_reduce_kernel<<<(unsigned)cdiv(MN, 256), 256, 0, st>>>(p.partial, p.k_parts, MN, (int)N, C, ldc, bias, relu, accumulate);
    DC_LAUNCH_CHECK();
  }
  return DC_OK;
}

size_t gemm_tc2_batched_workspace_bytes(int count) {
  if (count < 0) count = 0;
  return align_up((size_t)count * sizeof(T2Problem), 256) + align_up((size_t)(count + 1) * sizeof(int), 256) + 512;
}

// `count` independent single-segment problems with common transposes in ONE persistent launch: work items of all
// problems are dealt to the CTAs round-robin, so problems that are too small to fill the machine alone (the
// per-group attention products) run at the rate of a large one.  The problem table (tensor maps + sizes) is built
// on the host — in `host_staging` (caller-owned PINNED memory, at least the workspace size) when given, so that the
// upload is a truly asynchronous, CUDA-graph-capturable copy — and copied into `workspace` on the stream.
int gemm_tc2_batched(const dc_gemm_problem* probs, int count, int transA, int transB, int relu, int accumulate, void* workspace,
                     size_t workspace_bytes, void* host_staging, size_t host_staging_bytes, cudaStream_t st) {
  DC_REQUIRE(probs && count > 0, DC_EINVAL, "gemm_batched: no problems");
  const size_t need = gemm_tc2_batched_workspace_bytes(count);
  DC_REQUIRE(workspace && workspace_bytes >= need, DC_EWORKSPACE, "gemm_batched: workspace %zu < %zu", workspace_bytes, need);
  const size_t tab_bytes = align_up((size_t)count * sizeof(T2Problem), 256);
  const size_t off_bytes = (size_t)(count + 1) * sizeof(int);
  // host image of the table (tensor maps must be 64-byte aligned in device memory: the workspace is aligned to 256)
  std::vector<unsigned char> host;
  unsigned char* hraw = static_cast<unsigned char*>(host_staging);
  if (hraw) {
    DC_REQUIRE(host_staging_bytes >= tab_bytes + off_bytes + 64, DC_EWORKSPACE, "gemm_batched: host staging %zu < %zu",
               host_staging_bytes, tab_bytes + off_bytes + 64);
  } else {   // legacy form: pageable image, staged by the runtime before cudaMemcpyAsync returns (NOT capturable)
    host.resize(tab_bytes + off_bytes + 64);
    hraw = host.data();
  }
  unsigned char* hbase = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(hraw) + 63) & ~(uintptr_t)63);
  T2Problem* tab = reinterpret_cast<T2Problem*>(hbase);
  int* item_off = reinterpret_cast<int*>(hbase + tab_bytes);
  const int pair = t2_pair();
  const uint32_t b_box_rows = pair ? T2_BN / 2 : T2_BN;
  int64_t items = 0;
  int64_t max_kb = 0;
  // TMA epilogue: every problem's output (and epilogue operand) must be addressable by a tensor map
  int64_t kb_all = 0;
  bool tepi_operands = true;
  for (int i = 0; i < count; ++i) {
    const dc_gemm_problem& q = probs[i];
    if (q.M <= 0 || q.N <= 0) continue;
    if (cdiv(q.K, T2_BK) > kb_all) kb_all = cdiv(q.K, T2_BK);
    if (!t2_tepi_operand_ok(q.C, q.ldc, q.N) || (q.E && !t2_tepi_operand_ok(q.E, q.lde, q.N))) tepi_operands = false;
  }
  // mode 3 (lab): batched launches take the TMA epilogue only when a problem carries a fused epilogue operand
  bool any_e = false;
  for (int i = 0; i < count; ++i) any_e = any_e || probs[i].E != nullptr;
  const int tepi = t2_tepi_ok(pair, kb_all, 1, accumulate) && tepi_operands && (t2_tepi_mode() != 3 || any_e);
  for (int i = 0; i < count; ++i) {
    const dc_gemm_problem& q = probs[i];
    DC_REQUIRE(q.M >= 0 && q.N >= 0 && q.K >= 0, DC_EINVAL, "gemm_batched: negative size in problem %d", i);
    item_off[i] = (int)items;
    T2Problem& t = tab[i];
    memset(&t, 0, sizeof(t));
    if (q.M == 0 || q.N == 0) continue;   // empty problem: no items
    DC_REQUIRE(q.K > 0, DC_ENOSUP, "gemm_batched: K = 0 in problem %d (zero the output instead)", i);
    dc_gemm_seg seg{q.A, q.lda, q.B, q.ldb, q.K};
    DC_REQUIRE(gemm_tc2_supported(&seg, 1, transA, transB, q.M, q.N) && q.C && q.ldc >= q.N, DC_ENOSUP,
               "gemm_batched: problem %d is not supported by the tcgen05 path (needs lda/ldb %% 4 == 0, 16-byte aligned operands)", i);
    if (transA) {
      if (int rc = make_map2(&t.mapA, q.A, (uint64_t)q.M, (uint64_t)q.K, (uint64_t)q.lda, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    } else {
      if (int rc = make_map2(&t.mapA, q.A, (uint64_t)q.K, (uint64_t)q.M, (uint64_t)q.lda, T2_BM, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    if (transB) {
      if (int rc = make_map2(&t.mapB, q.B, (uint64_t)q.K, (uint64_t)q.N, (uint64_t)q.ldb, b_box_rows, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    } else {
      if (int rc = make_map2(&t.mapB, q.B, (uint64_t)q.N, (uint64_t)q.K, (uint64_t)q.ldb, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    }
    t.C = q.C; t.ldc = q.ldc; t.M = (int)q.M; t.N = (int)q.N;
    t.E = q.E; t.rowv = q.rowv; t.lde = q.lde;
    DC_REQUIRE(!q.E || (q.rowv && q.lde >= q.N), DC_EINVAL, "gemm_batched: problem %d: epilogue operand needs rowv and lde >= N", i);
    if (tepi) {
      if (int rc = make_map2(&t.mapC, q.C, (uint64_t)q.N, (uint64_t)q.M, (uint64_t)q.ldc, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
      if (q.E)
        if (int rc = make_map2(&t.mapE, q.E, (uint64_t)q.N, (uint64_t)q.M, (uint64_t)q.lde, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    t.kb_total = (int)cdiv(q.K, T2_BK);
    if (t.kb_total > max_kb) max_kb = t.kb_total;
    t.n_chunks = (int)cdiv(q.N, T2_BN);
    items += (pair ? cdiv(cdiv(q.M, T2_BM), 2) : cdiv(q.M, T2_BM)) * t.n_chunks;
    DC_REQUIRE(items < (1ll << 30), DC_ENOSUP, "gemm_batched: too many work items");
  }
  item_off[count] = (int)items;
  if (items == 0) return DC_OK;
  unsigned char* dbase = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  DC_CUDA(cudaMemcpyAsync(dbase, hbase, tab_bytes + off_bytes, cudaMemcpyHostToDevice, st));   // pinned source: async / a graph copy node
  T2Params p{};
  p.batch = reinterpret_cast<const T2Problem*>(dbase);
  p.item_off = reinterpret_cast<const int*>(dbase + tab_bytes);
  p.n_problems = count;
  p.nseg = 1;
  p.kb_seg[0] = 1 << 30;
  p.a_mn = transA ? 1 : 0;
  p.b_mn = transB ? 0 : 1;
  p.k_parts = 1;
  p.pair = pair;
  p.items = (int)items;
  p.drain_kb = t2_drain_kb(max_kb);
  p.relu = relu; p.accumulate = accumulate;
  p.raw_hi = 1;
  if (const char* e = getenv("DCB200_T2_RAWHI")) p.raw_hi = e[0] == '1';
  t2_numerics(p);
  // batched products write matrices far larger than L2 that the next kernel reads from the start again: evict-first (DCB200_T2_TEPI_HINT=0: off)
  static int hint = -1;
  if (hint < 0) { const char* e = getenv("DCB200_T2_TEPI_HINT"); hint = e ? atoi(e) : 1; }
  p.tepi = tepi ? (hint ? 3 : 1) : 0;
  CUtensorMap dummy[4]{};
  return t2_launch(dummy, dummy, dummy[0], p, st);
}

}  // namespace dcb
