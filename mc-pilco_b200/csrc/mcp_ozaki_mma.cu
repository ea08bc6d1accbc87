// The digit-plane contraction of the error-compensated INT8 variant (mcp_ozaki.cu) as ONE persistent tcgen05 kernel.
//
//   V[M,N] (fp64) = 2^(eA[m] + eB[n]) * sum_seg sum_{w<S} 256^-(w+2) * C_w,     C_w = sum_{t+u=w} A_t * B_u^T   (exact, int32)
//
// replaces the contraction `K_X_star @ K_X_inv` of the reference (gpr_lib/GP_prior/GP_prior.py:152) when the caller opted in.
//
// Structure (Blackwell, sm_100a; no library templates):
//   * CTA pairs (cluster 2x1x1) own a 256 x 128 output tile: tcgen05.mma.cta_group::2.kind::i8 with M = 256, N = 128, K = 32.  Each CTA
//     stages ITS 128 rows of an A plane and ITS 64 rows of a B plane (the pair shares B through the tensor core's 2-SM data path).
//   * FOUR plane sums C_w live in tensor memory at once (4 x 128 columns = all 512): the kernel sweeps the contraction index once for
//     the four least significant sums (w = S-4 .. S-1) and once for the rest, and inside a 128-byte k-block it multiplies every
//     resident A plane with every B plane it pairs with.  A plane k-block is therefore fetched from L2 once per sweep instead of once
//     per product: 26 (then 10) products per 8 + 8 (then 4 + 4) plane blocks for S = 8 — half the L2 -> shared-memory bytes per MAC of a
//     plain 256 x 256-tile int8 GEMM (which would need 64 B/clk/SM, more than the chip's L2 delivers at full clocks).
//   * operands arrive by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle, boxes of 128 (A) / 64 (B) rows x 128 bytes, out-of-range rows
//     zero-filled) into per-plane slots (8 x 16 KB + 8 x 8 KB), each with its own full / empty mbarrier pair: a slot is released by a
//     multicast tcgen05.commit right after the last product of its plane in the k-block and refilled with the next k-block while the
//     other planes are still being multiplied.  Both CTAs' boxes complete on the LEADER CTA's `full` barrier (cta_group::2 TMA form).
//   * after a sweep the accumulators are committed to the epilogue warps, which read them with tcgen05.ld (32 lanes x 16 columns per
//     warp and instruction), fold the up to four sums in fp64 — least significant first — and write V: once after the first sweep,
//     one read-modify-write after the second, which also applies the row / column power-of-two scales.  Nothing int32 is ever written
//     to memory, and all S(S+1)/2 plane products of a contraction are one launch.
//   * persistent: cluster c processes tiles c, c + #clusters, ... in a grouped raster order (8 tile rows per group) so that the
//     clusters running at the same time read a compact set of operand panels through L2.
//
// Warp roles per CTA (384 threads): warp 0 = TMA producer (one lane), warp 1 = TMEM allocator + (leader CTA) MMA issuer (one lane),
// warps 4..11 = epilogue (TMEM lane quarter = warp % 4, column half = (warp - 4) / 4); warps 2, 3 idle.
#include <cuda.h>

#include "mcp_common.cuh"

namespace mcp {

namespace {

constexpr int OZ_BM = 128;                       // A rows per CTA (pair: 256)
constexpr int OZ_BN = 128;                       // output columns per pair tile; each CTA stages 64 B rows
constexpr int OZ_BK = 128;                       // contraction bytes per k-block (= the 128-byte swizzle span), 4 MMAs of K = 32
constexpr int OZ_SLOTS = 8;                      // plane slots per operand
constexpr int OZ_A_BYTES = OZ_BM * OZ_BK;        // 16 KB
constexpr int OZ_B_BYTES = (OZ_BN / 2) * OZ_BK;  // 8 KB
constexpr int OZ_EPI_WARPS = 8;                  // two per TMEM lane quarter, 64 output columns each
constexpr int OZ_THREADS = 32 * (4 + OZ_EPI_WARPS);
constexpr int OZ_GROUP = 8;                      // tile rows per raster group
constexpr int OZ_NACC = 4;                       // plane sums resident in tensor memory
constexpr int OZ_NBAR = 4 * OZ_SLOTS + 2;
constexpr size_t OZ_SMEM_BYTES = (size_t)OZ_SLOTS * (OZ_A_BYTES + OZ_B_BYTES) + 8 * OZ_NBAR + 16 + 1024;
constexpr uint32_t OZ_TMEM_COLS = 512;
static_assert(OZ_NACC * OZ_BN == (int)OZ_TMEM_COLS, "the resident plane sums fill the tensor memory");

// tcgen05 instruction descriptor, kind::i8: D = s32 (bits 4-5 = 2), A = B = signed 8 bit (bits 7-9, 10-12 = 1), both K-major (bits 15, 16
// = 0), N >> 3 at bits 17-22, M >> 4 at bits 24-28 (M = 256 across the CTA pair)
constexpr uint32_t OZ_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BN >> 3) << 17) | ((uint32_t)((2 * OZ_BM) >> 4) << 24);

__device__ __forceinline__ uint32_t oz_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t oz_cta_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of the same shared-memory location in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t oz_mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void oz_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void oz_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void oz_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void oz_mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void oz_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "OZ_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra OZ_DONE_%=;\n"
      "bra OZ_WAIT_%=;\n"
      "OZ_DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// TMA load of one [128 rows x 128 bytes] box into this CTA's shared memory; completion bytes are credited to `bar0`, an mbarrier of the
// LEADER CTA (shared::cluster address) — the cta_group::2 form allows the barrier to live in the peer CTA
__device__ __forceinline__ void oz_tma_load_2sm(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar0) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(map), "r"(c0), "r"(c1), "r"(bar0)
               : "memory");
}
// shared-memory matrix descriptor of a K-major [rows x 128 B] tile in the TMA 128-byte-swizzle layout: start address >> 4 (bits 0-13),
// leading byte offset (unused for swizzled K-major; 1), stride byte offset = 8 rows x 128 B = 1024 B (>> 4 = 64, bits 32-45), descriptor
// version 1 (bit 46), layout type SWIZZLE_128B = 2 (bits 61-63).  Tiles are 1024-byte aligned (base offset 0); advancing K by 32 bytes
// inside the swizzle span adds 2 to the start-address field.
__device__ __forceinline__ uint64_t oz_smem_desc(uint32_t addr) {
  return (uint64_t)((addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void oz_mma_i8_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(OZ_IDESC), "r"(accumulate)
      : "memory");
}
// all tcgen05 operations issued so far by this thread arrive (once) on the mbarrier at the same shared-memory offset in both CTAs of the pair
__device__ __forceinline__ void oz_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}
// 32 lanes x 16 columns of one accumulator into registers (asynchronous: oz_tmem_wait() before the registers are read)
__device__ __forceinline__ void oz_tmem_ld16(uint32_t taddr, int32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void oz_tmem_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// one lane of the (converged) warp; the surrounding code stays warp-uniform so that descriptors and addresses live in uniform registers
__device__ __forceinline__ bool oz_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void oz_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void oz_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

struct OzTile {
  int m0, n0;
};
__device__ __forceinline__ OzTile oz_tile(int tile, int tiles_m, int tiles_n) {
  const int per_group = OZ_GROUP * tiles_n, group = tile / per_group, first_m = group * OZ_GROUP;
  const int rows_here = min(tiles_m - first_m, OZ_GROUP), in_group = tile - group * per_group;
  OzTile t;
  t.m0 = (first_m + in_group % rows_here) * (2 * OZ_BM);
  t.n0 = (in_group / rows_here) * OZ_BN;
  return t;
}

// The plane sums of one tile are produced in (at most) two sweeps over the contraction index: sweep 0 holds the (up to) four least
// significant sums w = max(0, S-4) .. S-1, sweep 1 the remaining w = 0 .. S-5.  Planes 0 .. whi take part in a sweep.
struct OzSweep {
  int wlo, whi;
};
__device__ __forceinline__ int oz_num_sweeps(int S) { return S > OZ_NACC ? 2 : 1; }
__device__ __forceinline__ OzSweep oz_sweep(int S, int i) {
  OzSweep g;
  if (i == 0) {
    g.wlo = S > OZ_NACC ? S - OZ_NACC : 0;
    g.whi = S - 1;
  } else {
    g.wlo = 0;
    g.whi = S - OZ_NACC - 1;
  }
  return g;
}
// slot of plane p in k-block kb: sweeps with at most 4 planes keep two k-blocks in flight
__device__ __forceinline__ int oz_slot(int p, int kb, int whi) { return whi < OZ_SLOTS / 2 ? p + (OZ_SLOTS / 2) * (kb & 1) : p; }

// One sweep of the MMA issuer over the contraction index with the plane-sum range [WLO, WHI] known at compile time: the product schedule
// of a k-block (which planes meet, which accumulator they feed, where a slot is first needed and where it is released) unrolls into
// straight-line code — per product one (rare) barrier wait, four UTCIMMA from uniform registers and the commits.  The whole warp runs
// it; one elected lane issues.  bars: fullA at +0, fullB at +8 SLOTS, emptyA at +16 SLOTS, emptyB at +24 SLOTS (bytes: x8).
template <int WLO, int WHI>
__device__ __forceinline__ void oz_mma_sweep(uint32_t smemA, uint32_t smemB, uint32_t bars, uint32_t tmem_base, int kblocks, uint32_t& pfA,
                                             uint32_t& pfB) {
  constexpr bool DBL = WHI < OZ_SLOTS / 2;  // at most four planes: two k-blocks in flight (slot = plane + 4 (kb & 1))
  constexpr uint32_t USED = (1u << (WHI + 1)) - 1u;
  const uint64_t descA0 = oz_smem_desc(smemA), descB0 = oz_smem_desc(smemB);
  for (int kb = 0; kb < kblocks; kb++) {
    const int so = DBL ? (kb & 1) * (OZ_SLOTS / 2) : 0;
#pragma unroll
    for (int t = 0; t <= WHI; t++) {
      const int ia = t + so;
      oz_mbar_wait(bars + 8u * (uint32_t)ia, (pfA >> ia) & 1u);
      const uint64_t adesc = descA0 + (uint64_t)(ia * (OZ_A_BYTES >> 4));
#pragma unroll
      for (int u = 0; u <= WHI; u++) {
        if (u < (WLO - t > 0 ? WLO - t : 0) || u > WHI - t) continue;  // the products of this sweep: WLO <= t + u <= WHI
        const int ib = u + so;
        if (t == (WLO - u > 0 ? WLO - u : 0)) oz_mbar_wait(bars + 8u * (uint32_t)(OZ_SLOTS + ib), (pfB >> ib) & 1u);  // first use of B_u
        oz_fence_after();
        const uint64_t bdesc = descB0 + (uint64_t)(ib * (OZ_B_BYTES >> 4));
        const uint32_t d_tmem = tmem_base + (uint32_t)((t + u - WLO) * OZ_BN);
        if (oz_elect_one()) {
          oz_mma_i8_2sm(d_tmem, adesc, bdesc, (t > 0 || kb > 0) ? 1u : 0u);
          oz_mma_i8_2sm(d_tmem, adesc + 2u, bdesc + 2u, 1u);
          oz_mma_i8_2sm(d_tmem, adesc + 4u, bdesc + 4u, 1u);
          oz_mma_i8_2sm(d_tmem, adesc + 6u, bdesc + 6u, 1u);
          if (t == WHI - u) oz_commit_pair(bars + 8u * (uint32_t)(3 * OZ_SLOTS + ib));  // last use of B_u in this k-block
          if (u == WHI - t) oz_commit_pair(bars + 8u * (uint32_t)(2 * OZ_SLOTS + ia));  // ... and of A_t
        }
        __syncwarp();
      }
    }
    pfA ^= USED << so;
    pfB ^= USED << so;
  }
}

}  // namespace

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(OZ_THREADS, 1)
ozaki_mma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int M, int N, int S, int nseg, int Ksp,
                 const int32_t* __restrict__ eA, const int32_t* __restrict__ eB, double* __restrict__ V, int ldv) {
  extern __shared__ unsigned char oz_smem_raw[];
  const uint32_t base = (oz_smem_u32(oz_smem_raw) + 1023u) & ~1023u;  // SWIZZLE_128B tiles want 1024-byte alignment
  const uint32_t smemA = base, smemB = base + OZ_SLOTS * OZ_A_BYTES;
  const uint32_t bars = smemB + OZ_SLOTS * OZ_B_BYTES;
  auto fullA = [&](int i) { return bars + 8u * (uint32_t)i; };                       // `full` barriers are used in the leader CTA only
  auto fullB = [&](int i) { return bars + 8u * (uint32_t)(OZ_SLOTS + i); };
  auto emptyA = [&](int i) { return bars + 8u * (uint32_t)(2 * OZ_SLOTS + i); };      // one per CTA
  auto emptyB = [&](int i) { return bars + 8u * (uint32_t)(3 * OZ_SLOTS + i); };
  const uint32_t tfull = bars + 8u * (4 * OZ_SLOTS), tempty = tfull + 8u;             // accumulators ready (per CTA) / drained (leader)
  const uint32_t tmem_slot = bars + 8u * OZ_NBAR;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = oz_cta_rank();
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int tiles_m = (M + 2 * OZ_BM - 1) / (2 * OZ_BM), tiles_n = (N + OZ_BN - 1) / OZ_BN, tiles = tiles_m * tiles_n;
  const int kblocks = Ksp / OZ_BK, nsweeps = oz_num_sweeps(S);

  if (threadIdx.x == 0) {
    for (int i = 0; i < OZ_SLOTS; i++) {
      oz_mbar_init(fullA(i), 1);
      oz_mbar_init(fullB(i), 1);
      oz_mbar_init(emptyA(i), 1);
      oz_mbar_init(emptyB(i), 1);
    }
    oz_mbar_init(tfull, 1);
    oz_mbar_init(tempty, 2 * OZ_EPI_WARPS);  // every epilogue warp of both CTAs
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 1) {  // the same warp of both CTAs allocates (and later frees) the pair's tensor memory: all 512 columns
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(OZ_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  oz_fence_before();
  oz_cluster_sync();
  oz_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (warp == 0) {
    // ------------------------------- TMA producer (both CTAs; the whole warp runs the loops, one elected lane issues) -------------
    uint32_t peA = 0xFFFFu, peB = 0xFFFFu;  // parity to wait for on each slot's `empty` barrier (a fresh barrier passes parity 1)
    for (int tile = cluster_id; tile < tiles; tile += num_clusters) {
      const OzTile tl = oz_tile(tile, tiles_m, tiles_n);
      const int a_row = tl.m0 + (int)rank * OZ_BM, b_row = tl.n0 + (int)rank * (OZ_BN / 2);
      for (int seg = 0; seg < nseg; seg++) {
        for (int sw = 0; sw < nsweeps; sw++) {
          const OzSweep g = oz_sweep(S, sw);
          for (int kb = 0; kb < kblocks; kb++) {
            const int kcol = kb * OZ_BK;
            for (int t = 0; t <= g.whi; t++) {
              // B planes first needed by A_t (in the order the MMA thread touches them), then A_t itself
              const int ufirst = t == 0 ? g.wlo : g.wlo - t, ulast = t == 0 ? g.whi : g.wlo - t;
              for (int u = ufirst; u <= ulast; u++) {
                if (u < 0) continue;
                const int i = oz_slot(u, kb, g.whi);
                oz_mbar_wait(emptyB(i), (peB >> i) & 1u);
                peB ^= 1u << i;
                if (oz_elect_one()) {
                  if (rank == 0) oz_mbar_expect_tx(fullB(i), 2 * OZ_B_BYTES);  // both CTAs' boxes land on the leader's barrier
                  oz_tma_load_2sm(smemB + (uint32_t)i * OZ_B_BYTES, &tmB, (seg * S + (S - 1 - u)) * Ksp + kcol, b_row, oz_mapa(fullB(i), 0));
                }
                __syncwarp();
              }
              const int i = oz_slot(t, kb, g.whi);
              oz_mbar_wait(emptyA(i), (peA >> i) & 1u);
              peA ^= 1u << i;
              if (oz_elect_one()) {
                if (rank == 0) oz_mbar_expect_tx(fullA(i), 2 * OZ_A_BYTES);
                oz_tma_load_2sm(smemA + (uint32_t)i * OZ_A_BYTES, &tmA, (seg * S + t) * Ksp + kcol, a_row, oz_mapa(fullA(i), 0));
              }
              __syncwarp();
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer (leader CTA; the whole warp runs the loops, one elected lane issues) -------------
    if (rank == 0) {
      uint32_t pfA = 0, pfB = 0, pte = 1;  // parities to wait for: slots' `full` barriers, accumulators drained
      for (int tile = cluster_id; tile < tiles; tile += num_clusters) {
        for (int seg = 0; seg < nseg; seg++) {
          for (int sw = 0; sw < nsweeps; sw++) {
            const OzSweep g = oz_sweep(S, sw);
            oz_mbar_wait(tempty, pte);  // the epilogue has read the previous sweep's sums out of tensor memory
            pte ^= 1u;
            oz_fence_after();
            if (g.wlo == 4 && g.whi == 7) oz_mma_sweep<4, 7>(smemA, smemB, bars, tmem_base, kblocks, pfA, pfB);        // S = 8, low sums
            else if (g.wlo == 0 && g.whi == 3) oz_mma_sweep<0, 3>(smemA, smemB, bars, tmem_base, kblocks, pfA, pfB);   // S = 8, high sums
            else if (g.wlo == 3 && g.whi == 6) oz_mma_sweep<3, 6>(smemA, smemB, bars, tmem_base, kblocks, pfA, pfB);   // S = 7, low sums
            else if (g.wlo == 0 && g.whi == 2) oz_mma_sweep<0, 2>(smemA, smemB, bars, tmem_base, kblocks, pfA, pfB);   // S = 7, high sums
            else
            for (int kb = 0; kb < kblocks; kb++) {  // any other plane count: the same schedule with run-time bounds
              for (int t = 0; t <= g.whi; t++) {
                const int ia = oz_slot(t, kb, g.whi);
                oz_mbar_wait(fullA(ia), (pfA >> ia) & 1u);
                pfA ^= 1u << ia;
                const uint64_t adesc = oz_smem_desc(smemA + (uint32_t)ia * OZ_A_BYTES);
                const int ulo = g.wlo - t > 0 ? g.wlo - t : 0, uhi = g.whi - t;
                for (int u = ulo; u <= uhi; u++) {
                  const int ib = oz_slot(u, kb, g.whi);
                  if (t == (g.wlo - u > 0 ? g.wlo - u : 0)) {  // first product of this k-block that reads B_u
                    oz_mbar_wait(fullB(ib), (pfB >> ib) & 1u);
                    pfB ^= 1u << ib;
                  }
                  oz_fence_after();
                  const uint64_t bdesc = oz_smem_desc(smemB + (uint32_t)ib * OZ_B_BYTES);
                  const uint32_t d_tmem = tmem_base + (uint32_t)(t + u - g.wlo) * OZ_BN;
                  const uint32_t acc0 = (kb > 0 || t > 0) ? 1u : 0u;
                  if (oz_elect_one()) {
                    oz_mma_i8_2sm(d_tmem, adesc, bdesc, acc0);
                    oz_mma_i8_2sm(d_tmem, adesc + 2u, bdesc + 2u, 1u);
                    oz_mma_i8_2sm(d_tmem, adesc + 4u, bdesc + 4u, 1u);
                    oz_mma_i8_2sm(d_tmem, adesc + 6u, bdesc + 6u, 1u);
                    if (t == g.whi - u) oz_commit_pair(emptyB(ib));  // last product of this k-block that reads B_u: slot free in both CTAs
                    if (u == uhi) oz_commit_pair(emptyA(ia));        // ... and A_t
                  }
                  __syncwarp();
                }
              }
            }
            if (oz_elect_one()) oz_commit_pair(tfull);  // the sweep's plane sums are complete in both CTAs' tensor memory
            __syncwarp();
          }
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------- epilogue (both CTAs): TMEM -> fp64 recombination into V -------------------------------
    const int q = warp & 3;                                    // TMEM lane quarter this warp may read
    constexpr int CHUNKS = OZ_BN / 16 / (OZ_EPI_WARPS / 4);    // 16-column chunks per warp
    const int c_first = ((warp - 4) >> 2) * CHUNKS;
    uint32_t ptf = 0;
    const uint32_t tempty0 = oz_mapa(tempty, 0);
    for (int tile = cluster_id; tile < tiles; tile += num_clusters) {
      const OzTile tl = oz_tile(tile, tiles_m, tiles_n);
      const int row = tl.m0 + (int)rank * OZ_BM + q * 32 + lane;
      const bool row_ok = row < M;
      double* vrow = V + (size_t)(row_ok ? row : 0) * ldv;
      const int ea = row_ok ? eA[row] : 0;
      for (int seg = 0; seg < nseg; seg++) {
        for (int sw = 0; sw < nsweeps; sw++) {
          const OzSweep g = oz_sweep(S, sw);
          const int nacc = g.whi - g.wlo + 1;
          const bool first = (seg == 0 && sw == 0), last = (seg == nseg - 1 && sw == nsweeps - 1);
          oz_mbar_wait(tfull, ptf);
          ptf ^= 1u;
          oz_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
          for (int c = c_first; c < c_first + CHUNKS; c++) {
            int32_t r[OZ_NACC][16];
#pragma unroll
            for (int a = 0; a < OZ_NACC; a++)
              if (a < nacc) oz_tmem_ld16(taddr + (uint32_t)(a * OZ_BN + c * 16), r[a]);
            oz_tmem_wait();
            if (c == c_first + CHUNKS - 1) {  // everything this warp reads of the sweep is in registers: hand the tensor memory back to the MMA thread
              oz_fence_before();
              __syncwarp();
              if (lane == 0) oz_mbar_arrive_cluster(tempty0);
            }
            const int col0 = tl.n0 + c * 16;
            if (row_ok && col0 < N) {
              double* p = vrow + col0;
              const bool vec = col0 + 16 <= N && (((uintptr_t)p) & 15) == 0;
              double v[16];
#pragma unroll
              for (int j = 0; j < 16; j += 2) {
                if (first) {
                  v[j] = v[j + 1] = 0.0;
                } else if (vec) {
                  const double2 t2 = *reinterpret_cast<const double2*>(p + j);
                  v[j] = t2.x;
                  v[j + 1] = t2.y;
                } else {
                  v[j] = col0 + j < N ? p[j] : 0.0;
                  v[j + 1] = col0 + j + 1 < N ? p[j + 1] : 0.0;
                }
              }
#pragma unroll
              for (int a = OZ_NACC - 1; a >= 0; a--) {  // least significant plane sum first
                if (a < nacc) {
                  const double sc = scalbn(1.0, -8 * (g.wlo + a + 2));
#pragma unroll
                  for (int j = 0; j < 16; j++) v[j] = fma((double)r[a][j], sc, v[j]);
                }
              }
              if (last) {  // row / column scales; a row of A or of B marked non-finite by the slicer makes the element NaN (finite
                           // rows have exponents within +-1100, so a sum above half the marker holds one)
#pragma unroll
                for (int j = 0; j < 16; j++) {
                  const int ex = ea + (col0 + j < N ? eB[col0 + j] : 0);
                  v[j] = ex > MCP_OZAKI_EXP_NONFINITE / 2 ? __longlong_as_double(0x7FF8000000000000ll) : scalbn(v[j], ex);
                }
              }
              if (vec) {
#pragma unroll
                for (int j = 0; j < 16; j += 2) *reinterpret_cast<double2*>(p + j) = make_double2(v[j], v[j + 1]);
              } else {
#pragma unroll
                for (int j = 0; j < 16; j++)
                  if (col0 + j < N) p[j] = v[j];
              }
            }
          }
        }
      }
    }
  }

  // ------------------------------- teardown -------------------------------
  oz_fence_before();
  oz_cluster_sync();  // no CTA of the pair leaves (or frees tensor memory) while the other may still signal its barriers / read its smem
  if (warp == 1) {
    oz_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(OZ_TMEM_COLS) : "memory");
  }
}

// ---- host side ------------------------------------------------------------------------------------------------------------
typedef CUresult (*OzEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static OzEncodeTiledFn oz_encode_fn() {
  static OzEncodeTiledFn fn = nullptr;
  static bool tried = false;
  std::lock_guard<std::mutex> lock(init_mutex());
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = (OzEncodeTiledFn)p;
  }
  return fn;
}

// digit planes [rows x row_bytes] int8, row-major -> boxes of [box_rows x 128 bytes], 128-byte swizzle, rows past the end read as zero
static int oz_make_map(CUtensorMap* map, const int8_t* ptr, int rows, size_t row_bytes, int box_rows) {
  OzEncodeTiledFn fn = oz_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return MCP_E_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
  cuuint32_t box[2] = {(cuuint32_t)OZ_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for digit planes [%d x %zu]", (int)r, rows, row_bytes);
    return MCP_E_CUDA;
  }
  return MCP_OK;
}

// V[M, N] = 2^(eA + eB) sum_w 256^-(w+2) sum_{t+u=w} A_t B_u^T from the digit planes (layouts: ozaki_slice_kernel); one launch
int ozaki_mma(const int8_t* Ap, const int32_t* Ae, const int8_t* Bp, const int32_t* Be, int M, int N, int S, int nseg, int Ksp, double* V, int ldv,
              cudaStream_t st) {
  MCP_CHECK_ARG(M >= 1 && N >= 1 && S >= 2 && S <= 8 && nseg >= 1 && Ksp >= OZ_BK && Ksp % OZ_BK == 0, "ozaki_mma: bad geometry (M=%d N=%d S=%d nseg=%d Ksp=%d)",
                M, N, S, nseg, Ksp);
  MCP_CHECK_ARG(((uintptr_t)Ap % 16) == 0 && ((uintptr_t)Bp % 16) == 0, "ozaki_mma: digit planes must be 16-byte aligned");
  static bool configured[MCP_MAX_DEVICES] = {};
  MCP_CUDA(ensure_dynamic_smem(configured, ozaki_mma_kernel, (int)OZ_SMEM_BYTES));
  const size_t row_bytes = (size_t)nseg * S * Ksp;
  CUtensorMap tmA, tmB;
  if (int e = oz_make_map(&tmA, Ap, M, row_bytes, OZ_BM)) return e;
  if (int e = oz_make_map(&tmB, Bp, N, row_bytes, OZ_BN / 2)) return e;
  int dev = 0, sms = 148;
  MCP_CUDA(cudaGetDevice(&dev));
  MCP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int tiles = cdiv(M, 2 * OZ_BM) * cdiv(N, OZ_BN);
  int clusters = sms / 2;
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)sms / 2 * 2);
    cfg.blockDim = dim3(OZ_THREADS);
    cfg.dynamicSmemBytes = OZ_SMEM_BYTES;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = 2;
    at.val.clusterDim.y = 1;
    at.val.clusterDim.z = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, ozaki_mma_kernel, &cfg) == cudaSuccess && n >= 1) clusters = n < clusters ? n : clusters;
    else (void)cudaGetLastError();
  }
  if (clusters > tiles) clusters = tiles;
  ozaki_mma_kernel<<<2 * clusters, OZ_THREADS, OZ_SMEM_BYTES, st>>>(tmA, tmB, M, N, S, nseg, Ksp, Ae, Be, V, ldv);
  MCP_LAUNCH_CHECK();
  return MCP_OK;
}

}  // namespace mcp
