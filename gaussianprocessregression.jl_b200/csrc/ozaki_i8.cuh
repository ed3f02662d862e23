// FP64 GEMM through the INT8 tensor cores (tcgen05.mma kind::i8, TMEM accumulators): an Ozaki-type splitting.
//
//   C (M x N) = alpha * op(A)^T-form product + beta * C,   op(A)[m, k] = A[k + m lda], op(B)[k, n] = B[k + n ldb]   (T,N form)
//
// sm_100a has no FP64 kind of tcgen05.mma; its FP64 tensor path is the warp-level DMMA (35.9 TFLOP/s measured with the
// TMA-fed kernel of dgemm_tma.cuh = the roof of that pipe).  The INT8 path of the 5th-generation tensor cores is
// ~120x wider, so an FP64 product can be bought with several exact integer products:
//
//   1. every row of op(A) (a vector over k) is scaled by a power of two 2^-ea so that |a| < 1/2 and cut into S signed
//      7-bit digits:  a 2^-ea = sum_{s=1..S} A_s 2^(-7 s),  A_s in [-64, 64]  (round-to-nearest digits, exact);
//      likewise every column of op(B).  (oz_slice_kernel)
//   2. the integer products A_s B_t^T are EXACT in int32 for K <= 2^17 (|sum| <= K 2^12), and all pairs of one
//      diagonal d = s + t share the weight 2^(-7 d), so a diagonal accumulates in ONE int32 TMEM accumulator over all
//      its pairs and the whole contraction (K <= 32768: |sum| <= 8 K 2^12 = 2^30);
//   3. pairs with s + t > S + 1 are dropped (their weight is below 2^(-7 (S + 2)), i.e. 2^-70 for S = 8 relative to the
//      row / column maxima): S (S + 1) / 2 = 36 integer products for S = 8;
//   4. the epilogue converts the S diagonals to FP64, weights and sums them (smallest first), rescales by
//      2^(ea_m + eb_n) and applies alpha / beta.
// Error: every retained term is exact, so the result differs from the exact product by the dropped digits only:
// <= ~2^-56 max_k|a_mk| max_k|b_kn| K for S = 8 -- a NORM-wise FP64 product (measured against DGEMM in
// tests/test_gpu_parity.py::test_ozaki_*).  It is not component-wise accurate for rows with a huge dynamic range.
//
// Kernel (oz_gemm_kernel): one CTA per 128 x 64 tile of C, 6 warps:
//   warp 0  TMA producer: per k-tile of 64 (bytes) ONE cp.async.bulk.tensor.3d per operand brings all S digit planes
//           (A: S x 128 x 64 B, B: S x 64 x 64 B, SWIZZLE_64B) into one of two 96 KB stages;
//   warp 1  one thread issues tcgen05.mma.cta_group::1.kind::i8 (M 128, N 64, K 32) for the 36 (s, t) pairs x 2 k-steps
//           of the stage into accumulator (s + t - 2) of the 8 x 64-column TMEM accumulators (all 512 columns), then
//           tcgen05.commit releases the stage; after the last k-tile a commit signals the epilogue;
//   warps 2-5  epilogue: tcgen05.ld (32 lanes x 16 columns) per diagonal, int32 -> FP64, weighted sum, scaling, C update.
// ncu (profiles/ozaki_ncu_full_r2t.md): tensor-core pipe 94 % busy -- every 128 x 64 x 32 product re-reads its 4 KB A operand from
// shared memory, and eight accumulators cannot be wider than 64 of the 512 TMEM columns: the roof of this instruction shape.
//
// Kernel (oz_gemm_win_kernel): the same roles for ONE window of diagonals d = DLO..DHI with BN = 96 / 128 columns per
// accumulator.  Used for NINE digits (45 products: the W^T W of the inverse, whose operand columns span many orders of magnitude
// under one scale): d = 6..10 in five 96-column accumulators, then d = 2..5, each launch accumulating into C.
//
// Launch flag of launch_ozaki_dgemm only: 512 two-window form of the 8-digit product.
// Forms (flags, same meaning as dgemm_sm100.cuh): upper only (1), K-from-N (2: triangular operand, masked in the digit extraction),
// skip tile (0,0) (64), and, in the single-pass kernel only, the tile-mapped forms of the block-cyclic multi-GPU drivers: MAP_UPPER (8),
// MAP_KUPTO (16: per-column contraction limit, masked in the digit extraction; long K comes in k-chunks <= 32768 with their own scales).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dgemm_tma.cuh"
#include "kbuild_tma.cuh"

namespace gpr {

constexpr int OZ_BM = 128, OZ_BN = 64, OZ_BK = 64;        // tile of C; k-tile in int8 elements (= bytes)
constexpr int OZ_SMAX = 8;
constexpr int OZ_THREADS = 192;
constexpr int OZ_STAGES = 2;

// pair: a CTA of a cta_group::2 pair holds half of the op(B) tile
__host__ __device__ inline size_t oz_stage_bytes(int S, bool pair = false) { return (size_t)S * (OZ_BM + (pair ? OZ_BN / 2 : OZ_BN)) * OZ_BK; }
__host__ __device__ inline size_t oz_smem_bytes(int S, bool pair = false) { return OZ_STAGES * oz_stage_bytes(S, pair) + 1024 + 128; }

// ---------------------------------------------------------------------------------------------------------------
// digit planes: X is K x R column major (column r = the vector over k of row / column r of the product operand).
// planes[s][r][k] (int8, k contiguous, row pitch Kp), scale[r] = 2^e_r (so that x = scale * sum_s planes_s 2^(-7 s)).
// One warp per column r.
// ---------------------------------------------------------------------------------------------------------------
// kfrom != 0: column r only holds data for k >= 128 * (r / 128) (lower-triangular operand of a K-from-N product, whose
// upper part may be uninitialised): everything above is treated as zero.
// kfrom == 2 (GEMM_MAP_KUPTO, the row-panel recurrence of the block-cyclic trtri): column r belongs to global 128-tile column
// gt = col_gtile[r / 128] and only holds data for k + k_off < (gt - k_gtile0 + 1) * 128; everything below is treated as zero.
__global__ void __launch_bounds__(256) oz_slice_kernel(const double* __restrict__ X, long long ldx, int K, int R, int S, int8_t* __restrict__ planes,
                                                       long long Kp, long long Rp, double* __restrict__ scale, int kfrom, int k_off,
                                                       const int* __restrict__ col_gtile = nullptr, int k_gtile0 = 0) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = blockIdx.x * 8 + warp;
  if (r >= Rp) return;
  if (r >= R) {   // padding rows: zero digits
    for (int s = 0; s < S; ++s)
      for (long long k = lane * 16; k < Kp; k += 32 * 16) *reinterpret_cast<int4*>(planes + ((long long)s * Rp + r) * Kp + k) = make_int4(0, 0, 0, 0);
    if (lane == 0) scale[r] = 1.0;
    return;
  }
  const double* col = X + (long long)r * ldx;
  const int kbeg = (kfrom == 1) ? max(0, 128 * (r / 128) - k_off) : 0;   // k_off: global row of this operand's first k (k-panel of a larger product)
  if (kfrom == 2) K = max(0, min(K, (col_gtile[r / 128] - k_gtile0 + 1) * 128 - k_off));
  double amax = 0.0;
  for (int k = kbeg + lane; k < K; k += 32) amax = fmax(amax, fabs(col[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  int e = 0;
  if (amax > 0.0) { (void)frexp(amax, &e); e += 1; }          // amax = m 2^(e-1), m in [0.5, 1)  ->  |x| 2^-e < 1/2
  const double down = ldexp(1.0, -e);
  if (lane == 0) scale[r] = ldexp(1.0, e);
  // 16 consecutive k per lane and step: one 16-byte store per plane
  for (long long k0 = lane * 16; k0 < Kp; k0 += 32 * 16) {
    double rem[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) rem[i] = (k0 + i < K && k0 + i >= kbeg) ? col[k0 + i] * down : 0.0;
    for (int s = 0; s < S; ++s) {
      unsigned w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const double sc = rem[i] * 128.0;                     // exact
        const double q = rint(sc);                            // |q| <= 64
        rem[i] = sc - q;                                      // exact, |rem| <= 1/2
        w[i >> 2] |= ((unsigned)(int)q & 0xffu) << (8 * (i & 3));
      }
      *reinterpret_cast<uint4*>(planes + ((long long)s * Rp + r) * Kp + k0) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

// (A variant with the column spread over up to 1024 threads so that the second pass hits L2 -- the launch list shows 42.9 GB read
// for 21.5 GB written per evaluation -- measured SLOWER: 16.5 vs 16.1 ms per 8192^3 product, evaluation +7 ms; removed.)

// ---------------------------------------------------------------------------------------------------------------
// tcgen05 primitives
// ---------------------------------------------------------------------------------------------------------------
// mbarrier wait that gives up (trap -> launch failure) instead of hanging the device if a barrier is never completed
__device__ __forceinline__ void oz_wait(uint64_t* bar, unsigned parity) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  const long long t0 = clock64();
  for (;;) {
    unsigned ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
    if (ok) return;
    if (clock64() - t0 > 4000000000ll) __trap();   // ~2 s
  }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"((unsigned)__cvta_generic_to_shared(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] B[smem]^T, int8 x int8 -> int32, M = 128, N = 64, K = 32
__device__ __forceinline__ void tc_mma_i8(unsigned tmem_d, uint64_t desc_a, uint64_t desc_b, unsigned idesc, unsigned accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
// ---- CTA pairs (tcgen05 cta_group::2): one MMA of M = 256 reads 128 rows of op(A) and half of op(B) from each CTA's shared memory
// at the same offset and accumulates into both CTAs' TMEM (128 lanes each) ----
__device__ __forceinline__ unsigned oz_cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
// every thread of both CTAs (release / acquire at cluster scope)
__device__ __forceinline__ void oz_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// shared::cluster address of the object at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ unsigned oz_mapa(const void* p, unsigned rank) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"((unsigned)__cvta_generic_to_shared(p)), "r"(rank));
  return r;
}
// TMA load into this CTA's shared memory whose bytes complete on the mbarrier at cluster address `bar` (the leader's)
__device__ __forceinline__ void tma_load_3d_pair(void* smem_dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(
                   (unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// completion of the pair's MMAs issued so far arrives on the mbarrier at this offset in both CTAs
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
                   (unsigned)__cvta_generic_to_shared(bar)),
               "h"((unsigned short)0x3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_i8_pair(unsigned tmem_d, uint64_t desc_a, uint64_t desc_b, unsigned idesc, unsigned accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TMEM: all 512 columns; with cta_group::2 one warp of EACH CTA of the pair takes part
template <bool PAIR> __device__ __forceinline__ void oz_tmem_alloc(unsigned* slot) {
  if constexpr (PAIR) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"((unsigned)__cvta_generic_to_shared(slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"((unsigned)__cvta_generic_to_shared(slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
}
template <bool PAIR> __device__ __forceinline__ void oz_tmem_dealloc(unsigned base) {
  if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;\n" ::"r"(base) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(base) : "memory");
}
// A pair works on row tiles 2j (leader, cluster rank 0) and 2j + 1 of one column tile.  It leaves only when both tiles are skipped;
// otherwise a CTA whose own tile is skipped (below the diagonal of an upper-only product, tile (0,0) of a skip-tile product, the row
// tile past M of an odd row-tile count: TMA zero fill) runs as a ghost: same loads, its half of the MMAs, no stores.

// K-major operand tile with 64-byte rows, SWIZZLE_64B: 8-row groups are 512 bytes apart
__device__ __forceinline__ uint64_t oz_smem_desc(const void* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  uint64_t d = 0;
  d |= (uint64_t)((a & 0x3FFFFu) >> 4);          // start address, bits [0, 14)
  d |= (uint64_t)1 << 16;                        // leading byte offset: 1 (16 B) for swizzled K-major layouts (CUTLASS make_umma_desc)
  d |= (uint64_t)(512u >> 4) << 32;              // stride byte offset: 8 rows x 64 B
  d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
  d |= (uint64_t)4 << 61;                        // layout type: SWIZZLE_64B
  return d;
}
// instruction descriptor: D = S32, A = B = signed int8, both K-major, N = 64, M = 128
constexpr unsigned OZ_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(OZ_BN >> 3) << 17) | ((unsigned)(OZ_BM >> 4) << 24);
constexpr unsigned OZ_IDESC_PAIR = (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(OZ_BN >> 3) << 17) | ((unsigned)((2 * OZ_BM) >> 4) << 24);   // M = 256

struct OzParams {
  int M, N, K, S;
  double alpha, beta;
  double* C; long long ldc;
  const double* scaleA; const double* scaleB;    // 2^ea (M), 2^eb (N)
  int flags;                                     // GEMM_UPPER_ONLY, GEMM_K_FROM_N (same meaning as dgemm_sm100.cuh)
  int k_off;                                     // K-from-N: global index of the first contraction row (k-panels of one product)
  const int* col_gtile; int row_gtile0;          // GEMM_MAP_UPPER (flag 8): global 128-tile column of each local 128-tile column (csrc/dist_blocked.hpp)
  int k_gtile0;                                  // GEMM_MAP_KUPTO (flag 16): the tile column contracts over k + k_off < (gt - k_gtile0 + 1) * 128 only
  const double* E; long long lde;                // Hadamard epilogue: C = alpha (A^T B) .* E + beta C  (split-predict mean)
};

// PAIR: clusters of two CTAs issuing tcgen05.mma.cta_group::2 of M = 256 (256 x 64 tile per pair; mapB's box holds 32 rows)
template <int S, bool PAIR = false>
__global__ void __launch_bounds__(OZ_THREADS, 1)
oz_gemm_kernel(const OzParams p, const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB) {
  constexpr int BNC = PAIR ? OZ_BN / 2 : OZ_BN;      // op(B) rows in this CTA's shared memory
  extern __shared__ unsigned char oz_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)oz_smem_raw + 1023) & ~(uintptr_t)1023);
  const size_t stage_bytes = oz_stage_bytes(S, PAIR);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + OZ_STAGES * stage_bytes);
  uint64_t* empty = full + OZ_STAGES;
  uint64_t* tfull = empty + OZ_STAGES;
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(tfull + 1);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // CTA rasterisation as in dgemm128_kernel: consecutive CTAs walk 16 row tiles x all column tiles, so one wave of 148 CTAs
  // touches ~16 x 9 tiles of C and re-reads few digit planes (issued x-fastest, a wave would stream every plane of op(A)
  // from DRAM once per column tile: 467 GB for a 16384^3 product against 4.3 GB of planes).
  // (a pair is one unit of the rasterisation: x counts pairs of row tiles, 8 pairs = 16 row tiles per group)
  constexpr int NC = PAIR ? 2 : 1;
  int tile_m, tile_n;
  {
    constexpr int GM = 16 / NC;
    const int Mx = gridDim.x / NC, Ny = gridDim.y;
    const int pid = blockIdx.x / NC + blockIdx.y * Mx;
    const int group = pid / (GM * Ny), first_m = group * GM;
    const int gsize = min(Mx - first_m, GM);
    const int rem = pid - group * GM * Ny;
    tile_m = first_m + rem % gsize;
    tile_n = rem / gsize;
  }
  const int blk_n = (tile_n * OZ_BN) >> 7;
  [[maybe_unused]] unsigned crank = 0;
  [[maybe_unused]] bool ghost = false;
  if constexpr (!PAIR) {
    if ((p.flags & 1) && tile_m > blk_n) return;                       // GEMM_UPPER_ONLY: whole CTA leaves before any allocation
    if ((p.flags & 64) && tile_m == 0 && blk_n == 0) return;           // GEMM_SKIP_TILE00
  } else {
    crank = oz_cluster_ctarank();
    const int m_lead = 2 * tile_m;
    tile_m = m_lead + (int)crank;
    const bool skip_lead = ((p.flags & 1) && m_lead > blk_n) || ((p.flags & 64) && m_lead == 0 && blk_n == 0);
    const bool skip_peer = ((p.flags & 1) && m_lead + 1 > blk_n) || (m_lead + 1) * OZ_BM >= p.M;
    if (skip_lead && skip_peer) return;
    ghost = crank ? skip_peer : skip_lead;
  }
  int gt = 0;
  if (p.flags & 8) {                                                  // GEMM_MAP_UPPER: tile-mapped trailing update of the block-cyclic potrf
    gt = p.col_gtile[blk_n];
    if (p.row_gtile0 + tile_m > gt) return;
  }
  const int kt0 = (p.flags & 2) ? max(0, blk_n * 128 - p.k_off) / OZ_BK : 0;   // GEMM_K_FROM_N
  int KT = p.K / OZ_BK - kt0;
  if (p.flags & 16) {                                                 // GEMM_MAP_KUPTO: per-column contraction limit (k-chunk of a longer product)
    KT = min(KT, ((p.col_gtile[blk_n] - p.k_gtile0 + 1) * 128 - p.k_off) / OZ_BK);
    if (KT <= 0) return;                                              // nothing of this column in this chunk (the caller accumulates: beta = 1)
  }
  const int m0 = tile_m * OZ_BM, n0 = tile_n * OZ_BN;

  if (tid == 0) {
    for (int s = 0; s < OZ_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tfull, 1);
    mbar_fence_init();
  }
  if (warp == 1) oz_tmem_alloc<PAIR>(tmem_slot);   // TMEM: all 512 columns (8 diagonals x 64)
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) oz_cluster_sync();         // the peer's barriers exist before anything signals them
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kt = 0; kt < KT; ++kt) {
        const int s = kt & 1;
        if (kt >= OZ_STAGES) oz_wait(&empty[s], (unsigned)(((kt >> 1) - 1) & 1));
        unsigned char* st = smem + (size_t)s * stage_bytes;
        if constexpr (!PAIR) {
          if ((p.flags & 256) && kt >= OZ_STAGES) { mbar_arrive(&full[s]); continue; }   // timing probe: no reload (results are garbage)
          mbar_expect_tx(&full[s], (unsigned)stage_bytes);
          tma_load_3d(st, &mapA, &full[s], (kt0 + kt) * OZ_BK, m0, 0);                               // S x 128 x 64 B
          tma_load_3d(st + (size_t)S * OZ_BM * OZ_BK, &mapB, &full[s], (kt0 + kt) * OZ_BK, n0, 0);   // S x  64 x 64 B
        } else {
          // both CTAs' bytes complete on the leader's full[s]; the leader's MMA thread is the only one waiting on it
          if ((p.flags & 256) && kt >= OZ_STAGES) { if (crank == 0) mbar_arrive(&full[s]); continue; }
          if (crank == 0) mbar_expect_tx(&full[s], (unsigned)(2 * stage_bytes));
          const unsigned bar = oz_mapa(&full[s], 0);
          tma_load_3d_pair(st, &mapA, bar, (kt0 + kt) * OZ_BK, m0, 0);                                            // S x 128 x 64 B
          tma_load_3d_pair(st + (size_t)S * OZ_BM * OZ_BK, &mapB, bar, (kt0 + kt) * OZ_BK, n0 + (int)crank * BNC, 0);   // S x 32 x 64 B
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    // One thread issues every MMA of the CTA, so its instruction stream is the critical path: S is a template parameter,
    // the pair loops are fully unrolled and a descriptor is the stage's base descriptor plus a compile-time constant.
    // The whole warp runs the (warp-uniform) control flow and one elected lane issues: inside a divergent `if (lane == 0)` the
    // compiler wraps every uniform-datapath instruction (UTCIMMA, its descriptor arithmetic) into an ELECT / BRA.U.ANY loop,
    // ~8 SASS instructions per MMA, and the issue stream -- not the tensor pipe -- sets the pace (58 cycles per MMA measured).
    {
      unsigned elected = 0;
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "elect.sync _|p, 0xffffffff;\n"
          "selp.u32 %0, 1, 0, p;\n"
          "}\n"
          : "=r"(elected));
      uint64_t baseA[OZ_STAGES], baseB[OZ_STAGES];
#pragma unroll
      for (int s = 0; s < OZ_STAGES; ++s) {
        baseA[s] = oz_smem_desc(smem + (size_t)s * stage_bytes);
        baseB[s] = oz_smem_desc(smem + (size_t)s * stage_bytes + (size_t)S * OZ_BM * OZ_BK);
      }
      if (PAIR && crank != 0) KT = 0;        // the leader issues the pair's MMAs
      for (int kt = 0; kt < KT; ++kt) {
        const int s = kt & 1;
        oz_wait(&full[s], (unsigned)((kt >> 1) & 1));
        tc_fence_after();
        const uint64_t dA = s ? baseA[1] : baseA[0], dB = s ? baseB[1] : baseB[0];
        const unsigned acc_first = (kt > 0) ? 1u : 0u;
        if (elected) {
#pragma unroll
          for (int t = 1; t <= S; ++t) {
#pragma unroll
            for (int sa = 1; sa + t <= S + 1; ++sa) {
#pragma unroll
              for (int kk = 0; kk < OZ_BK / 32; ++kk) {   // 32-byte k-steps inside the 64-byte swizzle atom: +2 in the 16-byte address field
                const uint64_t da = dA + (uint64_t)(((sa - 1) * OZ_BM * OZ_BK + 32 * kk) >> 4);
                const uint64_t db = dB + (uint64_t)(((t - 1) * BNC * OZ_BK + 32 * kk) >> 4);
                if constexpr (PAIR) tc_mma_i8_pair(tmem_base + (unsigned)((sa + t - 2) * OZ_BN), da, db, OZ_IDESC_PAIR, (kk > 0 || t > 1) ? 1u : acc_first);
                else tc_mma_i8(tmem_base + (unsigned)((sa + t - 2) * OZ_BN), da, db, OZ_IDESC, (kk > 0 || t > 1) ? 1u : acc_first);
              }
            }
          }
          if constexpr (PAIR) tc_commit_pair(&empty[s]); else tc_commit(&empty[s]);   // the stage may be refilled once these MMAs have read it
        }
        __syncwarp();
      }
      if constexpr (PAIR) { if (elected && crank == 0) tc_commit_pair(tfull); }
      else if (elected) tc_commit(tfull);       // all accumulators complete
    }
  } else {
    // ===== epilogue: warps 2..5 own TMEM lanes 32 (warp % 4) .. +31 = rows of the tile =====
    oz_wait(tfull, 0);
    tc_fence_after();
    const int q = warp & 3;
    const int row = 32 * q + lane;
    const unsigned lane_addr = tmem_base + ((unsigned)(32 * q) << 16);
    const bool diag_tile = ((p.flags & 1) && (tile_m == blk_n)) || ((p.flags & 8) && (p.row_gtile0 + tile_m == gt));
    const int coff = n0 & 127;
    const double sa = p.scaleA[m0 + row] * p.alpha;
    double* Crow = p.C + (long long)(m0 + row) + (long long)n0 * p.ldc;
    for (int c0 = 0; c0 < OZ_BN; c0 += 16) {
      if constexpr (PAIR) { if (ghost) break; }
      double acc[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = 0.0;
      for (int d = S + 1; d >= 2; --d) {   // smallest weights first
        unsigned v[16];
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
              "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
            : "r"(lane_addr + (unsigned)((d - 2) * OZ_BN + c0)));
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        const double w = __hiloint2double((1023 - 7 * d) << 20, 0);   // 2^(-7 d)
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = fma((double)(int)v[j], w, acc[j]);
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int col = c0 + j;
        if (diag_tile && row > col + coff) continue;
        double* cp = Crow + (long long)col * p.ldc;
        double r = acc[j] * sa * p.scaleB[n0 + col];
        if (p.E) r *= p.E[(long long)(m0 + row) + (long long)(n0 + col) * p.lde];
        *cp = (p.beta != 0.0) ? fma(p.beta, *cp, r) : r;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if constexpr (PAIR) oz_cluster_sync();      // no CTA leaves (or frees TMEM) while its peer may still signal or use it
  if (warp == 1) {
    tc_fence_after();
    oz_tmem_dealloc<PAIR>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Second-generation kernel: a WINDOW of diagonals per launch, 128 x 128 tile.
// One UTCIMMA of shape M128 N64 K32 occupies the tensor pipe for ~58 cycles however cleanly it is issued (measured with and
// without operand reloads, tools/ozaki_probe.py) -- 0.58 of the INT8 rate the pipe reaches with wide N -- and the eight diagonal
// accumulators of one pass cannot be wider than 64 TMEM columns each.  Splitting the 36 pairs into two launches by diagonal,
//   low order  d = 6 .. 9  (26 pairs, all 8 digit planes, k-tile 32 bytes / SWIZZLE_32B),  C  = alpha * (...) + beta * C
//   high order d = 2 .. 5  (10 pairs, digit planes 1-4,   k-tile 64 bytes / SWIZZLE_64B),  C += alpha * (...)
// needs four accumulators per launch, i.e. N = 128 per MMA: half as many tensor-pipe instructions for the same work.
// The digit planes are streamed twice (once per window).  MEASURED (profiles/ozaki_probe_r2p.log): an N = 128 instruction takes
// twice as long as an N = 64 one -- 73.5 against 69.1 TFLOP/s FP64-equivalent at 8192^3, nothing inside the factorization --
// so the tensor pipe itself (~2.65 INT8 POPS in this access pattern), not the instruction shape, is the limit.  Launch flag 512:
// the largest products take it (context option "ozaki_win_mink").
// ---------------------------------------------------------------------------------------------------------------
// PAIR: clusters of two CTAs issuing tcgen05.mma.cta_group::2 of M = 256; a CTA holds BN / 2 rows of op(B) per plane, so a stage is
// smaller and more of them fit (three -> four for every window below).
template <int S, int BN, int BK, int DLO, int DHI, bool PAIR = false> struct OzWin {
  static constexpr int NACC = DHI - DLO + 1;
  static constexpr int PL = (DHI - 1 < S) ? DHI - 1 : S;                  // digit planes needed
  static constexpr int BNC = PAIR ? BN / 2 : BN;                          // op(B) rows in this CTA's shared memory
  static constexpr size_t STAGE = (size_t)PL * (OZ_BM + BNC) * BK;
  static constexpr int NST = (int)(231000 / STAGE) > 4 ? 4 : (int)(231000 / STAGE);      // 227 KB of shared memory per CTA
  static constexpr size_t SMEM = NST * STAGE + 1024 + 256;
  static constexpr unsigned IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(BN >> 3) << 17) | ((unsigned)(((PAIR ? 2 : 1) * OZ_BM) >> 4) << 24);
  static_assert(NACC * BN <= 512, "accumulators exceed TMEM");
  static_assert(NST >= 2, "need two stages");
};

template <int BK> __device__ __forceinline__ uint64_t oz_smem_desc_k(const void* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  uint64_t d = 0;
  d |= (uint64_t)((a & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8u * BK) >> 4) << 32;          // 8-row groups are 8 * BK bytes apart
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(BK == 64 ? 4 : 6) << 61;         // SWIZZLE_64B / SWIZZLE_32B
  return d;
}

template <int S, int BN, int BK, int DLO, int DHI, bool PAIR = false>
__global__ void __launch_bounds__(OZ_THREADS, 1)
oz_gemm_win_kernel(const OzParams p, const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB) {
  using W = OzWin<S, BN, BK, DLO, DHI, PAIR>;
  constexpr int NST = W::NST, PL = W::PL, BNC = W::BNC;
  extern __shared__ unsigned char oz_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)oz_smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NST * W::STAGE);
  uint64_t* empty = full + NST;
  uint64_t* tfull = empty + NST;
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(tfull + 1);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NC = PAIR ? 2 : 1;
  int tile_m, tile_n;
  {
    constexpr int GM = 8 / NC;      // 8 row tiles x all column tiles per pass (tiles are 128 x 128 here); x counts pairs of row tiles
    const int Mx = gridDim.x / NC, Ny = gridDim.y;
    const int pid = blockIdx.x / NC + blockIdx.y * Mx;
    const int group = pid / (GM * Ny), first_m = group * GM;
    const int gsize = min(Mx - first_m, GM);
    const int rem = pid - group * GM * Ny;
    tile_m = first_m + rem % gsize;
    tile_n = rem / gsize;
  }
  const int blk_n = (tile_n * BN) >> 7;                       // first 128-block of the tile's columns
  if (tile_n * BN >= p.N) return;
  [[maybe_unused]] unsigned crank = 0;
  [[maybe_unused]] bool ghost = false;
  if constexpr (!PAIR) {
    if ((p.flags & 1) && tile_m > ((tile_n * BN + BN - 1) >> 7)) return;
    if ((p.flags & 64) && tile_m == 0 && blk_n == 0) return;
  } else {
    crank = oz_cluster_ctarank();
    const int m_lead = 2 * tile_m, last_blk = (tile_n * BN + BN - 1) >> 7;
    tile_m = m_lead + (int)crank;
    const bool skip_lead = ((p.flags & 1) && m_lead > last_blk) || ((p.flags & 64) && m_lead == 0 && blk_n == 0);
    const bool skip_peer = ((p.flags & 1) && m_lead + 1 > last_blk) || (m_lead + 1) * OZ_BM >= p.M;
    if (skip_lead && skip_peer) return;
    ghost = crank ? skip_peer : skip_lead;
  }
  const int kt0 = (p.flags & 2) ? max(0, blk_n * 128 - p.k_off) / BK : 0;
  int KT = p.K / BK - kt0;
  const int m0 = tile_m * OZ_BM, n0 = tile_n * BN;

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tfull, 1);
    mbar_fence_init();
  }
  if (warp == 1) oz_tmem_alloc<PAIR>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) oz_cluster_sync();      // the peer's barriers exist before anything signals them
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kt = 0; kt < KT; ++kt) {
        const int s = kt % NST;
        if (kt >= NST) oz_wait(&empty[s], (unsigned)((kt / NST - 1) & 1));
        unsigned char* st = smem + (size_t)s * W::STAGE;
        if constexpr (!PAIR) {
          mbar_expect_tx(&full[s], (unsigned)W::STAGE);
          tma_load_3d(st, &mapA, &full[s], (kt0 + kt) * BK, m0, 0);                               // PL x 128 x BK
          tma_load_3d(st + (size_t)PL * OZ_BM * BK, &mapB, &full[s], (kt0 + kt) * BK, n0, 0);     // PL x BN  x BK
        } else {
          // both CTAs' bytes complete on the leader's full[s]
          if (crank == 0) mbar_expect_tx(&full[s], (unsigned)(2 * W::STAGE));
          const unsigned bar = oz_mapa(&full[s], 0);
          tma_load_3d_pair(st, &mapA, bar, (kt0 + kt) * BK, m0, 0);                                            // PL x 128 x BK
          tma_load_3d_pair(st + (size_t)PL * OZ_BM * BK, &mapB, bar, (kt0 + kt) * BK, n0 + (int)crank * BNC, 0);   // PL x BN / 2 x BK
        }
      }
    }
  } else if (warp == 1) {
    unsigned elected = 0;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(elected));
    const uint64_t baseA0 = oz_smem_desc_k<BK>(smem), baseB0 = oz_smem_desc_k<BK>(smem + (size_t)PL * OZ_BM * BK);
    if (PAIR && crank != 0) KT = 0;          // the leader issues the pair's MMAs
    for (int kt = 0; kt < KT; ++kt) {
      const int s = kt % NST;
      oz_wait(&full[s], (unsigned)((kt / NST) & 1));
      tc_fence_after();
      const uint64_t dA = baseA0 + (uint64_t)((s * W::STAGE) >> 4), dB = baseB0 + (uint64_t)((s * W::STAGE) >> 4);
      const unsigned acc_first = (kt > 0) ? 1u : 0u;
      if (elected) {
#pragma unroll
        for (int t = 1; t <= PL; ++t) {
#pragma unroll
          for (int sa = 1; sa <= PL; ++sa) {
            if (sa + t < DLO || sa + t > DHI) continue;
            // first pair of diagonal d = sa + t in this loop order: t = max(1, d - PL)
            const bool first_pair = (t == ((sa + t - PL) > 1 ? (sa + t - PL) : 1));
#pragma unroll
            for (int kk = 0; kk < BK / 32; ++kk) {
              const uint64_t da = dA + (uint64_t)(((sa - 1) * OZ_BM * BK + 32 * kk) >> 4);
              const uint64_t db = dB + (uint64_t)(((t - 1) * BNC * BK + 32 * kk) >> 4);
              if constexpr (PAIR) tc_mma_i8_pair(tmem_base + (unsigned)((sa + t - DLO) * BN), da, db, W::IDESC, (kk > 0 || !first_pair) ? 1u : acc_first);
              else tc_mma_i8(tmem_base + (unsigned)((sa + t - DLO) * BN), da, db, W::IDESC, (kk > 0 || !first_pair) ? 1u : acc_first);
            }
          }
        }
        if constexpr (PAIR) tc_commit_pair(&empty[s]); else tc_commit(&empty[s]);
      }
      __syncwarp();
    }
    if constexpr (PAIR) { if (elected && crank == 0) tc_commit_pair(tfull); }
    else if (elected) tc_commit(tfull);
  } else {
    oz_wait(tfull, 0);
    tc_fence_after();
    const int q = warp & 3;
    const int row = 32 * q + lane;
    const unsigned lane_addr = tmem_base + ((unsigned)(32 * q) << 16);
    const bool diag_local = (p.flags & 1) && (tile_m >= blk_n);     // upper only: rows below the diagonal stay untouched
    const double sa = p.scaleA[m0 + row] * p.alpha;
    double* Crow = p.C + (long long)(m0 + row) + (long long)n0 * p.ldc;
    for (int c0 = 0; c0 < BN; c0 += 16) {
      if (n0 + c0 >= p.N) break;
      if constexpr (PAIR) { if (ghost) break; }
      double acc[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = 0.0;
#pragma unroll
      for (int d = DHI; d >= DLO; --d) {
        unsigned v[16];
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
              "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
            : "r"(lane_addr + (unsigned)((d - DLO) * BN + c0)));
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        const double w = __hiloint2double((1023 - 7 * d) << 20, 0);
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = fma((double)(int)v[j], w, acc[j]);
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int col = c0 + j;
        if (diag_local && m0 + row > n0 + col) continue;
        double* cp = Crow + (long long)col * p.ldc;
        double r = acc[j] * sa * p.scaleB[n0 + col];
        if (p.E) r *= p.E[(long long)(m0 + row) + (long long)(n0 + col) * p.lde];       // Hadamard epilogue: linear, so every window applies it
        *cp = (p.beta != 0.0) ? fma(p.beta, *cp, r) : r;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if constexpr (PAIR) oz_cluster_sync();      // no CTA leaves (or frees TMEM) while its peer may still signal or use it
  if (warp == 1) {
    tc_fence_after();
    oz_tmem_dealloc<PAIR>(tmem_base);
  }
}

// ---- host side ----
// int8 digit planes as a 3-D tensor {k (bytes), rows, plane}: box = {64, box_rows, S}, SWIZZLE_64B
inline bool oz_make_map(CUtensorMap* map, const int8_t* base, uint64_t Kp, uint64_t Rp, int S, uint32_t box_rows) {
  PFN_encodeTiled fn = tma_encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {Kp, Rp, (cuuint64_t)S};
  cuuint64_t strides[2] = {Kp, Kp * Rp};
  cuuint32_t box[3] = {OZ_BK, box_rows, (cuuint32_t)S};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int S, bool PAIR = false> inline cudaError_t oz_set_attr_s() {
  return cudaFuncSetAttribute(oz_gemm_kernel<S, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz_smem_bytes(S, PAIR));
}
inline bool oz_make_map_k(CUtensorMap* map, const int8_t* base, uint64_t Kp, uint64_t Rp, int planes_total, int box_planes, uint32_t box_rows, int BK) {
  PFN_encodeTiled fn = tma_encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {Kp, Rp, (cuuint64_t)planes_total};
  cuuint64_t strides[2] = {Kp, Kp * Rp};
  cuuint32_t box[3] = {(cuuint32_t)BK, box_rows, (cuuint32_t)box_planes};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            BK == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
using OzWinLo = OzWin<8, 128, 32, 6, 9>;
using OzWinHi = OzWin<8, 128, 64, 2, 5>;      // (k-tiles of 32 with seven stages instead of 64 with three: measured slower, 20.1 vs 18.7 ms per 8192^3 nine-digit product)
using OzWin9Z = OzWin<9, 96, 32, 6, 10>;      // nine digits in TWO windows: d = 6..10 in five 96-column accumulators (480 TMEM columns, 35 pairs)
using OzWinLoP = OzWin<8, 128, 32, 6, 9, true>;
using OzWinHiP = OzWin<8, 128, 64, 2, 5, true>;
using OzWin9ZP = OzWin<9, 96, 32, 6, 10, true>;

inline cudaError_t oz_set_attr() {
  cudaError_t e = cudaFuncSetAttribute(oz_gemm_win_kernel<8, 128, 32, 6, 9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OzWinLo::SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_win_kernel<8, 128, 64, 2, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OzWinHi::SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_win_kernel<9, 96, 32, 6, 10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OzWin9Z::SMEM);
  if (e == cudaSuccess) e = oz_set_attr_s<8>();
  if (e == cudaSuccess) e = oz_set_attr_s<7>();
  if (e == cudaSuccess) e = oz_set_attr_s<6>();
  if (e == cudaSuccess) e = oz_set_attr_s<2>();
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_win_kernel<8, 128, 32, 6, 9, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OzWinLoP::SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_win_kernel<8, 128, 64, 2, 5, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OzWinHiP::SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_win_kernel<9, 96, 32, 6, 10, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OzWin9ZP::SMEM);
  if (e == cudaSuccess) e = oz_set_attr_s<8, true>();
  if (e == cudaSuccess) e = oz_set_attr_s<7, true>();
  if (e == cudaSuccess) e = oz_set_attr_s<6, true>();
  return e;
}

// launch as clusters of two CTAs along x (the cta_group::2 pairs): grid.x = row tiles rounded up to even
template <typename Kern>
inline cudaError_t oz_launch_pairs(Kern kern, int row_tiles, int col_tiles, size_t smem, cudaStream_t st, const OzParams& p, const CUtensorMap& a,
                                   const CUtensorMap& b) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(row_tiles + (row_tiles & 1)), (unsigned)col_tiles, 1);
  cfg.blockDim = dim3(OZ_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, p, a, b);
}

// workspace (bytes) for the digit planes and scales of one product
inline size_t oz_workspace_bytes(int M, int N, int K, int S) {
  const size_t Kp = ((size_t)K + 127) / 128 * 128;
  return (size_t)S * Kp * ((size_t)M + (size_t)N) + sizeof(double) * ((size_t)M + (size_t)N) + 512;
}

// C = alpha A^T B + beta C through the int8 tensor cores.  M % 128 == 0, N % 128 == 0, K % 128 == 0, K <= 32768.
// flags: GEMM_UPPER_ONLY (1), GEMM_K_FROM_N (2), GEMM_SKIP_TILE00 (64), 512 (above); the tile-mapped MAP_UPPER (8) and MAP_KUPTO (16)
// and the timing probe (256) are forms of the single-pass kernel (S <= 8 without 512).  2048: CTA pairs (tcgen05 cta_group::2) for
// S = 6..9 in every form but the tile-mapped and Hadamard ones, bit-identical to the single-CTA kernels (exact integer accumulation,
// same epilogue).  When A and B are the same matrix (the symmetric
// updates of potrf and the W^T W product of the inverse) its digit planes are formed once and shared.
inline cudaError_t launch_ozaki_dgemm(cudaStream_t st, int M, int N, int K, int S, double alpha, const double* A, long long lda, const double* B,
                                      long long ldb, double beta, double* C, long long ldc, int flags, void* workspace, int k_off = 0,
                                      const int* col_gtile = nullptr, int row_gtile0 = 0, int k_gtile0 = 0, const double* E = nullptr,
                                      long long lde = 0) {
  if (flags & ~(1 | 2 | 8 | 16 | 64 | 256 | 512 | 2048)) return cudaErrorInvalidValue;
  if (E && (flags & (8 | 16))) return cudaErrorInvalidValue;                         // Hadamard epilogue: plain forms only
  if ((flags & (8 | 16)) && (!col_gtile || S == 9 || (flags & 512))) return cudaErrorInvalidValue;   // tile-mapped: single-pass kernel only
  if ((flags & 16) && ((flags & (1 | 2 | 8 | 64)) || (A == B && lda == ldb))) return cudaErrorInvalidValue;   // KUPTO: plain form only
  if (S == 9 && (flags & 64)) return cudaErrorInvalidValue;                           // a 96-wide tile straddles tile (0,0)'s columns
  if ((S != 9 && S != 8 && S != 7 && S != 6 && S != 2) || (M % OZ_BM) || (N % 128) || (K % 128) || K > 32768) return cudaErrorInvalidValue;
  const size_t Kp = (size_t)K;
  const bool shared = (A == B && lda == ldb);
  const int kfrom = (flags & 2) ? 1 : 0;
  const int Ra = shared ? (M > N ? M : N) : M;
  int8_t* pa = reinterpret_cast<int8_t*>(workspace);
  int8_t* pb = shared ? pa : pa + (size_t)S * Kp * Ra;
  const int Rb = shared ? Ra : N;
  double* sa = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(pa + (size_t)S * Kp * ((size_t)Ra + (shared ? 0 : (size_t)N))) + 255) & ~(uintptr_t)255);
  double* sb = shared ? sa : sa + Ra;
  // K-from-N: only op(B)'s columns are triangular (column block J holds data for k >= 128 J).  With shared planes (W^T W, upper
  // only) the rows I <= J of op(A)^T are the same columns, read for k >= 128 J >= 128 I only, so the same masking is exact.
  oz_slice_kernel<<<(Ra + 7) / 8, 256, 0, st>>>(A, lda, K, Ra, S, pa, (long long)Kp, Ra, sa, shared ? kfrom : 0, k_off);
  if (!shared) {
    if (flags & 16) oz_slice_kernel<<<(N + 7) / 8, 256, 0, st>>>(B, ldb, K, N, S, pb, (long long)Kp, N, sb, 2, k_off, col_gtile, k_gtile0);
    else oz_slice_kernel<<<(N + 7) / 8, 256, 0, st>>>(B, ldb, K, N, S, pb, (long long)Kp, N, sb, kfrom, k_off);
  }
  const OzParams p{M, N, K, S, alpha, beta, C, ldc, sa, sb, flags & ~(512 | 2048), k_off, col_gtile, row_gtile0, k_gtile0, E, lde};
  // CTA pairs: each SM reads its own 128 rows of op(A) and half of the op(B) tile from shared memory per MMA
  const bool pair = (flags & 2048) && !(flags & (8 | 16)) && !E && S != 2;
  const int mt = M / OZ_BM;
  if (S == 9 || (S == 8 && (flags & 512))) {
    // Two windows of diagonals, lowest order first, the second accumulating into C.
    // NINE digits (products whose operands span several orders of magnitude under one scale per column: the W^T W of the inverse):
    // nine 64-column accumulators do not fit the 512 TMEM columns, so d = 6..10 runs in five 96-column accumulators (35 pairs,
    // 128 x 96 tiles; the last column tile is partial: TMA zero fill, masked epilogue), then d = 2..5 (10 pairs, 128 x 128 tiles):
    // 19.4 ms at 8192^3.
    // EIGHT digits (flag 512): d = 6..9 then d = 2..5, 128 x 128 tiles; measured 73.5 against 69.1 TFLOP/s at 8192^3 and no gain inside
    // the factorization below 8192, so the single-pass 128 x 64 kernel stays the default there.  ncu (profiles/ozaki_ncu_full_r2t.md):
    // the single-pass kernel keeps the tensor-core pipe 94 % busy (sm__pipe_tc_cycles_active; every N = 64 product re-reads its 4 KB
    // A operand from shared memory), the windows load the planes twice and sit at 81 % of the L2 -> SM fill rate instead.
    const bool nine = (S == 9);
    const int plLo = nine ? OzWin9Z::PL : OzWinLo::PL, bnLo = nine ? 96 : 128;
    const int bdiv = pair ? 2 : 1;       // a CTA of a pair loads half of the op(B) tile
    CUtensorMap aLo, bLo, aHi, bHi;
    if (!oz_make_map_k(&aLo, pa, Kp, (uint64_t)Ra, S, plLo, OZ_BM, 32) || !oz_make_map_k(&bLo, pb, Kp, (uint64_t)Rb, S, plLo, bnLo / bdiv, 32) ||
        !oz_make_map_k(&aHi, pa, Kp, (uint64_t)Ra, S, OzWinHi::PL, OZ_BM, 64) || !oz_make_map_k(&bHi, pb, Kp, (uint64_t)Rb, S, OzWinHi::PL, 128 / bdiv, 64))
      return cudaErrorInvalidValue;
    if (pair) {
      OzParams p2 = p;
      p2.beta = 1.0;
      cudaError_t e = nine ? oz_launch_pairs(oz_gemm_win_kernel<9, 96, 32, 6, 10, true>, mt, (N + 95) / 96, OzWin9ZP::SMEM, st, p, aLo, bLo)
                           : oz_launch_pairs(oz_gemm_win_kernel<8, 128, 32, 6, 9, true>, mt, N / 128, OzWinLoP::SMEM, st, p, aLo, bLo);
      if (e == cudaSuccess) e = oz_launch_pairs(oz_gemm_win_kernel<8, 128, 64, 2, 5, true>, mt, N / 128, OzWinHiP::SMEM, st, p2, aHi, bHi);
      return e != cudaSuccess ? e : cudaGetLastError();
    }
    if (nine) oz_gemm_win_kernel<9, 96, 32, 6, 10><<<dim3(M / OZ_BM, (N + 95) / 96), OZ_THREADS, OzWin9Z::SMEM, st>>>(p, aLo, bLo);
    else oz_gemm_win_kernel<8, 128, 32, 6, 9><<<dim3(M / OZ_BM, N / 128), OZ_THREADS, OzWinLo::SMEM, st>>>(p, aLo, bLo);
    OzParams p2 = p;
    p2.beta = 1.0;
    oz_gemm_win_kernel<8, 128, 64, 2, 5><<<dim3(M / OZ_BM, N / 128), OZ_THREADS, OzWinHi::SMEM, st>>>(p2, aHi, bHi);
    return cudaGetLastError();
  }
  CUtensorMap mA, mB;
  if (!oz_make_map(&mA, pa, Kp, (uint64_t)Ra, S, OZ_BM) || !oz_make_map(&mB, pb, Kp, (uint64_t)Rb, S, pair ? OZ_BN / 2 : OZ_BN)) return cudaErrorInvalidValue;
  if (pair) {
    cudaError_t e = (S == 8)   ? oz_launch_pairs(oz_gemm_kernel<8, true>, mt, N / OZ_BN, oz_smem_bytes(8, true), st, p, mA, mB)
                    : (S == 7) ? oz_launch_pairs(oz_gemm_kernel<7, true>, mt, N / OZ_BN, oz_smem_bytes(7, true), st, p, mA, mB)
                               : oz_launch_pairs(oz_gemm_kernel<6, true>, mt, N / OZ_BN, oz_smem_bytes(6, true), st, p, mA, mB);
    return e != cudaSuccess ? e : cudaGetLastError();
  }
  dim3 grid(M / OZ_BM, N / OZ_BN);
  if (S == 8) oz_gemm_kernel<8><<<grid, OZ_THREADS, oz_smem_bytes(8), st>>>(p, mA, mB);
  else if (S == 7) oz_gemm_kernel<7><<<grid, OZ_THREADS, oz_smem_bytes(7), st>>>(p, mA, mB);
  else if (S == 6) oz_gemm_kernel<6><<<grid, OZ_THREADS, oz_smem_bytes(6), st>>>(p, mA, mB);
  else oz_gemm_kernel<2><<<grid, OZ_THREADS, oz_smem_bytes(2), st>>>(p, mA, mB);
  return cudaGetLastError();
}

}  // namespace gpr
