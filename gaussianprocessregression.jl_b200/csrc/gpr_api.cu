// libgpr_sm100a.so: C ABI (include/gpr_sm100a.h) over the sm_100a kernels.
// Host orchestration only; all arithmetic is in the kernels of this directory.
// There is deliberately no CPU path: without a usable CUDA device every entry
// point fails with GPR_ERR_CUDA.
#include "../../include/gpr_sm100a.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "blocked.hpp"
#include "dist_blocked.hpp"
#include "cov_kernels.cuh"
#include "dgemm_sm100.cuh"
#include "kbuild_tma.cuh"
#include "grad_wide.cuh"
#include "dgemm_tma.cuh"
#include "ozaki_i8.cuh"
#include "leaf_kernels.cuh"

using namespace gpr;

namespace {

thread_local std::string g_create_error;

// Live-handle registry.  A host with finalizers (the Julia glue, julia/GPRsm100a.jl) may release a context before the
// models created on it, or a handle twice at exit: a *_destroy call on a handle that is not (or no longer) registered
// is a no-op, and destroying a context first releases the models it still owns.
std::mutex g_live_mu;
std::set<const void*> g_live;
bool live_take(const void* h) { std::lock_guard<std::mutex> l(g_live_mu); return g_live.erase(h) > 0; }
void live_add(const void* h) { std::lock_guard<std::mutex> l(g_live_mu); g_live.insert(h); }

inline int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

struct Timer {
  cudaEvent_t beg[GPR_T_COUNT], end[GPR_T_COUNT];
  bool used[GPR_T_COUNT];
  double acc_ms[GPR_T_COUNT];
};

// phase of the factorization / inverse being run (gpr_ctx::oz_cur); the values are the bits of the public option "ozaki_phases"
constexpr int OZ_PH_POTRF = 1, OZ_PH_TRTRI = 2, OZ_PH_LAUUM = 4, OZ_PH_OTHER = 8;

}  // namespace

struct gpr_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int sm_count = 0;
  int64_t predict_tile = 16384;
  int inplace_lauum = 0;   // option "inplace_lauum": force the recursive in-place W W^T (saves one N x N buffer)
  int leaf_lookahead = 1;  // option "leaf_lookahead": factor the next diagonal leaf on the side queue (csrc/blocked.hpp)
  int alpha_from_inverse = 1;   // option "alpha_from_inverse": alpha = K^-1 y by a symmetric product on the gradient path
  int gemm_cfg = 0;             // option "gemm_cfg": forced tile configuration of dgemm128 (0 = automatic), per context
  int ozaki = -1;               // option "ozaki": number of 7-bit digits S of the INT8-tensor-core FP64 product (csrc/ozaki_i8.cuh)
                                // used for large T,N products: 0 = off, 6 / 7 / 8 = forced, -1 = automatic (default): 8 digits for
                                // models whose condition-number bound allows a norm-wise accurate product (ozaki_digits_for below),
                                // DMMA otherwise; "ozaki_min": smallest M, N, K routed there
  int oz_active = 0;            // digits in force for the model being worked on (set by the entry points)
  int64_t ozaki_min = 1024;
  int ozaki_lauum = 9;          // option "ozaki_lauum": digits of the INT8 route for the W^T W product of the inverse (0 = DMMA, 8, 9 = default)
  int64_t ozaki_win_mink = 8192;   // option "ozaki_win_mink": two-diagonal-window form (128 x 128 tiles) of the 8-digit product for products with M, N,
                                   // K >= this (0 = never): the windows pay for their second pass over the digit planes only on the largest products --
                                   // N = 32768 evaluation 680 -> 667 ms at 8192, 670 at 4096, 680 at 2048 (profiles/ozaki_win_mink_r2an.log)
  int ozaki_pair = 1;           // option "ozaki_pair": the plain INT8 products run as CTA pairs (tcgen05 cta_group::2, launch flag 2048): each SM
                                // reads half of the op(B) tile from shared memory per MMA; bit-identical to the single-CTA kernels
  int ozaki_split = 9;          // option "ozaki_split": digits of the INT8 route for the split-predict mean products (0 = DMMA, 8, 9)
  int64_t ozaki_kchunk = 32768; // option "ozaki_kchunk": k-chunk of the long-K tile-mapped products (tests lower it to exercise the chunk loop)
  int64_t ozaki_panel = 32768;  // option "ozaki_panel": k-panel of the W^T W product (own digit scales per panel)
  int oz_mask = OZ_PH_POTRF | OZ_PH_TRTRI | OZ_PH_OTHER, oz_cur = OZ_PH_OTHER;
                                  // option "ozaki_phases": bit 0 potrf, 1 trtri, 3 everything else (prediction solves); the W^T W product of the
                                  // inverse (lauum) is governed by "ozaki_lauum": its operand columns span many orders of magnitude under ONE
                                  // power-of-two scale per column, and with 8 digits the gradient keeps only 7 digits (1.1e-7 vs the oracle);
                                  // NINE digits restore it (4.0e-11, DMMA: 6.1e-11 at N = 32768; profiles/ozaki_lauum9_r2s.log)
  void* oz_ws = nullptr; size_t oz_ws_bytes = 0;
  int gemm_tma = 1;             // option "gemm_tma": T,N products through the TMA-fed kernel (csrc/dgemm_tma.cuh)
  int kbuild_gram = 1;          // option "kbuild_gram": TMA-fed Gram-form covariance build (csrc/kbuild_tma.cuh); 0 = direct-difference kernel
  std::vector<gpr_model*> models;   // live models of this context (released by gpr_ctx_destroy if the caller has not)
  long long launches = 0;
  long long* d_info = nullptr;
  cudaError_t pending = cudaSuccess;   // first launch error seen by the backend
  // second queue of the multi-GPU drivers (look-ahead / prefetch, csrc/dist_blocked.hpp); `stream` is the queue
  // launches currently go to and equals main_stream outside those drivers
  cudaStream_t main_stream = nullptr, side_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr};   // split predict: chunk-ready events for the overlapped download
  cudaEvent_t ev_d2h[4] = {nullptr, nullptr, nullptr, nullptr};     // ... and chunk-downloaded events (pinned staging buffer)
  double* h_stage = nullptr; size_t h_stage_elems = 0;              // pinned staging buffer of the split-predict mean
  // h_stage grown to `elems` doubles if that is at most 1 GB; nullptr when the buffer is smaller and cannot be grown
  double* host_stage(size_t elems) {
    if (elems > h_stage_elems && elems * sizeof(double) <= ((size_t)1 << 30)) {
      if (h_stage) { cudaFreeHost(h_stage); h_stage = nullptr; h_stage_elems = 0; }
      if (cudaMallocHost(&h_stage, elems * sizeof(double)) == cudaSuccess) h_stage_elems = elems;
      else { cudaGetLastError(); h_stage = nullptr; }
    }
    return h_stage_elems >= elems ? h_stage : nullptr;
  }
};

namespace {

int fail(gpr_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg; else g_create_error = msg;
  return code;
}
int fail_cuda(gpr_ctx* ctx, cudaError_t e, const char* what, int line) {
  char buf[512];
  snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s [gpr_api.cu:%d]", (int)e, cudaGetErrorString(e), what, line);
  return fail(ctx, e == cudaErrorMemoryAllocation ? GPR_ERR_MEMORY : GPR_ERR_CUDA, buf);
}
#define CK(call)                                                              \
  do {                                                                        \
    cudaError_t e_ = (call);                                                  \
    if (e_ != cudaSuccess) return fail_cuda(ctx, e_, #call, __LINE__);        \
  } while (0)

// CUDA backend of csrc/blocked.hpp
struct CudaBE {
  gpr_ctx* ctx;
  void note(cudaError_t e) { if (e != cudaSuccess && ctx->pending == cudaSuccess) ctx->pending = e; }
  // digit-plane workspace of the INT8 route: grown on demand; false if it cannot hold `need` bytes (the product then stays on the DMMA pipe)
  bool oz_reserve(size_t need) {
    if (need > ctx->oz_ws_bytes) {
      cudaStreamSynchronize(ctx->main_stream);
      cudaFree(ctx->oz_ws); ctx->oz_ws = nullptr; ctx->oz_ws_bytes = 0;
      if (cudaMalloc(&ctx->oz_ws, need) == cudaSuccess) ctx->oz_ws_bytes = need; else cudaGetLastError();
    }
    return ctx->oz_ws_bytes >= need;
  }
  // Route of one product: digits of the INT8 tensor cores (csrc/ozaki_i8.cuh), 0 = DMMA pipe; launch flags it adds; k-split
  // (0 = none): ozaki_panel for the W^T W product of the inverse, ozaki_kchunk for the k-upto product.
  enum OzKind { OZ_PLAIN, OZ_HADAMARD, OZ_MAP_UPPER, OZ_MAP_KUPTO };
  struct OzRoute { int digits = 0, flags = 0; int64_t ksplit = 0; };
  OzRoute ozaki_route(OzKind kind, char tA, char tB, int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B,
                      int64_t ldb, const double* C, int flags, int64_t batch = 1) const {
    OzRoute r;
    if (ctx->oz_active <= 0 || ctx->stream != ctx->main_stream || tA != 'T' || tB != 'N') return r;   // (the side queue stays on DMMA)
    if ((const double*)C == A || (const double*)C == B) return r;
    const int64_t mn = ctx->ozaki_min;
    if (M < mn || N < mn || K < mn || (M % 128) || (N % 128) || (K % 128)) return r;
    int digits = ctx->oz_active;
    if (ctx->oz_cur == OZ_PH_LAUUM && kind == OZ_PLAIN) digits = ctx->ozaki_lauum;     // W^T W of the inverse: "ozaki_lauum", not the phase mask
    else if (ctx->oz_cur == OZ_PH_LAUUM && kind == OZ_HADAMARD) return r;
    else if (!(ctx->oz_mask & ctx->oz_cur)) return r;
    switch (kind) {
      case OZ_PLAIN:
      case OZ_HADAMARD:
        if ((flags & ~(BLK_UPPER_ONLY | BLK_K_FROM_N | BLK_SKIP_TILE00)) || batch < 1 || batch > 16 || K > 32768) return r;
        if (kind == OZ_HADAMARD) { r.digits = ctx->ozaki_split; return r; }
        r.digits = digits;
        if (ctx->ozaki_pair) r.flags |= 2048;
        if (batch == 1 && flags == (BLK_UPPER_ONLY | BLK_K_FROM_N) && A == B && lda == ldb && M == N && N == K && K > ctx->ozaki_panel)
          r.ksplit = ctx->ozaki_panel;
        else if (ctx->ozaki_win_mink > 0 && std::min(K, std::min(M, N)) >= ctx->ozaki_win_mink)
          r.flags |= 512;
        return r;
      case OZ_MAP_UPPER:
        if (flags == BLK_MAP_UPPER && K <= 32768) r.digits = digits;
        return r;
      case OZ_MAP_KUPTO:
        if (flags == BLK_MAP_KUPTO && A != B) { r.digits = digits; r.ksplit = std::min<int64_t>(ctx->ozaki_kchunk, 32768); }
        return r;
    }
    return r;
  }
  void gemm(char tA, char tB, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
            const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int64_t batch = 1,
            int64_t sA = 0, int64_t sB = 0, int64_t sC = 0) {
    const OzRoute oz = ozaki_route(OZ_PLAIN, tA, tB, M, N, K, A, lda, B, ldb, C, flags, batch);
    if (oz.digits && oz_reserve(oz_workspace_bytes((int)std::max(M, N), (int)N, (int)K, oz.digits))) {
      if (oz.ksplit) {
        // W^T W of the inverse (lauum_oop_t): the columns of the triangular factor span many orders of magnitude (O(1/sigma_n)
        // next to the diagonal, tiny far from it), and the digit planes of a column share ONE power-of-two scale.  Summing the
        // product over k-panels, each with its own column scales, keeps the error relative to the panel-local magnitudes
        // (measured on the benchmark model: gradient error vs the oracle 1.1e-7 with one scale per column -> see profiles/).
        // The last panel touches every column and initialises C (beta), the earlier ones accumulate into their leading block.
        for (int64_t p1 = K; p1 > 0; p1 -= oz.ksplit) {
          const int64_t p0 = std::max<int64_t>(0, p1 - oz.ksplit);
          const int64_t cols = std::min<int64_t>(N, p1);
          note(launch_ozaki_dgemm(ctx->stream, (int)cols, (int)cols, (int)(p1 - p0), oz.digits, alpha, A + p0, lda, B + p0, ldb,
                                  p1 == K ? beta : 1.0, C, ldc, flags | oz.flags, ctx->oz_ws, (int)p0));
          ctx->launches += 2;
        }
        return;
      }
      // large T,N product: one launch per batch member
      for (int64_t z = 0; z < batch; ++z) {
        note(launch_ozaki_dgemm(ctx->stream, (int)M, (int)N, (int)K, oz.digits, alpha, A + z * sA, lda, B + z * sB, ldb, beta, C + z * sC, ldc,
                                flags | oz.flags, ctx->oz_ws));
        ctx->launches += 3;
      }
      return;
    }
    // grid.z is limited to 65535: split very large batches
    for (int64_t z0 = 0; z0 < batch; z0 += 32768) {
      const int64_t nb = std::min<int64_t>(32768, batch - z0);
      if (ctx->gemm_tma && gemm_tma_supported(tA, tB, (int)M, (int)N, (int)K, A, B, C, flags, (int)nb, sA, sB)) {
        // TMA-fed operand ring (csrc/dgemm_tma.cuh), T,N form
        note(launch_dgemm128_tma(ctx->stream, (int)M, (int)N, (int)K, alpha, A + z0 * sA, lda, B + z0 * sB, ldb, beta, C + z0 * sC, ldc,
                                 flags, (int)nb, sA, sB, sC));
        ctx->launches++;
        continue;
      }
      note(launch_dgemm128(ctx->stream, tA, tB, (int)M, (int)N, (int)K, alpha, A + z0 * sA, lda, B + z0 * sB, ldb, beta,
                           C + z0 * sC, ldc, flags, (int)nb, sA, sB, sC, nullptr, 0, 0, ctx->gemm_cfg));
      ctx->launches++;
    }
  }
  // C = (A^T B) .* E + beta C, T,N form with the Hadamard epilogue (split-predict mean)
  void gemm_hadamard(int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B, int64_t ldb,
                     const double* E, int64_t lde, double beta, double* C, int64_t ldc) {
    // split-predict mean on the INT8 tensor cores; the Hadamard factor and beta ride in the epilogue.  NINE digits by default ("ozaki_split"):
    // the columns of Diagonal(wt) C carry the weights' dynamic range and the sum over the training points cancels heavily -- with eight
    // digits the mean agrees with the dense path to 4e-10 instead of 8e-12 (N = 32768, profiles/README.md)
    const OzRoute oz = ozaki_route(OZ_HADAMARD, 'T', 'N', M, N, K, A, lda, B, ldb, C, 0);
    if (oz.digits && oz_reserve(oz_workspace_bytes((int)M, (int)N, (int)K, oz.digits))) {
      note(launch_ozaki_dgemm(ctx->stream, (int)M, (int)N, (int)K, oz.digits, 1.0, A, lda, B, ldb, beta, C, ldc, oz.flags, ctx->oz_ws, 0,
                              nullptr, 0, 0, E, lde));
      ctx->launches += 3;
      return;
    }
    if (ctx->gemm_tma && gemm_tma_supported('T', 'N', (int)M, (int)N, (int)K, A, B, C, 0, 1, 0, 0))
      note(launch_dgemm128_tma(ctx->stream, (int)M, (int)N, (int)K, 1.0, A, lda, B, ldb, beta, C, ldc, 0, 1, 0, 0, 0, nullptr, 0, 0, E, lde));
    else
      note(launch_dgemm128(ctx->stream, 'T', 'N', (int)M, (int)N, (int)K, 1.0, A, lda, B, ldb, beta, C, ldc, 0, 1, 0, 0, 0, nullptr, 0, 0,
                           0, E, lde));
    ctx->launches++;
  }
  void activate() { note(cudaSetDevice(ctx->device)); }
  void fork() { note(cudaEventRecord(ctx->ev_fork, ctx->main_stream)); note(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_fork, 0)); }
  void join() { note(cudaEventRecord(ctx->ev_join, ctx->side_stream)); note(cudaStreamWaitEvent(ctx->main_stream, ctx->ev_join, 0)); }
  void side(bool on) { ctx->stream = on ? ctx->side_stream : ctx->main_stream; }
  // tile-mapped GEMM of the block-cyclic multi-GPU drivers (csrc/dist_blocked.hpp)
  void gemm_map(char tA, char tB, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
                const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, const TileMap& map) {
    // INT8 tensor cores: the rank-nb trailing update of the block-cyclic potrf (map-upper) and the row-panel recurrence of the
    // block-cyclic trtri (k-upto: M = nb rows, per-column contraction limit, K up to N, in k-chunks of at most 32768 -- the int32
    // accumulators are exact up to there -- each with its own digit scales, accumulated in C)
    const OzRoute oz = ozaki_route(flags == BLK_MAP_KUPTO ? OZ_MAP_KUPTO : OZ_MAP_UPPER, tA, tB, M, N, K, A, lda, B, ldb, C, flags);
    const int64_t KC = oz.ksplit ? oz.ksplit : K;
    if (oz.digits && oz_reserve(oz_workspace_bytes((int)M, (int)N, (int)std::min(K, KC), oz.digits))) {
      for (int64_t k0 = 0; k0 < K; k0 += KC) {
        const int64_t kc = std::min(KC, K - k0);
        note(launch_ozaki_dgemm(ctx->stream, (int)M, (int)N, (int)kc, oz.digits, alpha, A + k0, lda, B + k0, ldb, k0 == 0 ? beta : 1.0, C, ldc,
                                flags | oz.flags, ctx->oz_ws, (int)k0, map.col_gtile, map.row_gtile0, map.k_gtile0));
        ctx->launches += 3;
      }
      return;
    }
    if (ctx->gemm_tma && gemm_tma_supported(tA, tB, (int)M, (int)N, (int)K, A, B, C, flags, 1, 0, 0))
      note(launch_dgemm128_tma(ctx->stream, (int)M, (int)N, (int)K, alpha, A, lda, B, ldb, beta, C, ldc, flags, 1, 0, 0, 0, map.col_gtile,
                               map.row_gtile0, map.k_gtile0));
    else
      note(launch_dgemm128(ctx->stream, tA, tB, (int)M, (int)N, (int)K, alpha, A, lda, B, ldb, beta, C, ldc, flags, 1, 0, 0, 0,
                           map.col_gtile, map.row_gtile0, map.k_gtile0, ctx->gemm_cfg));
    ctx->launches++;
  }
  void potrf_leaf(double* A, int64_t lda, double* dinv, int64_t goff) {
    potrf_leaf_kernel<<<1, LEAF_THREADS, LEAF_SMEM_BYTES, ctx->stream>>>(A, lda, dinv, ctx->d_info, goff);
    note(cudaGetLastError());
    ctx->launches++;
  }
  void gemv(char tA, int64_t M, int64_t K, double alpha, const double* A, int64_t lda, const double* x, double* y) {
    if (tA == 'T') gemv_t_kernel<<<(unsigned)((M + 7) / 8), 256, 0, ctx->stream>>>((int)M, (int)K, alpha, A, lda, x, y);
    else gemv_n_kernel<<<(unsigned)((M + 63) / 64), 256, 0, ctx->stream>>>((int)M, (int)K, alpha, A, lda, x, y);
    note(cudaGetLastError());
    ctx->launches++;
  }
  void leaf_mv(char tA, const double* dinv, double* v, double s) {
    leaf_mv_kernel<<<1, 256, LEAF_MV_SMEM_BYTES, ctx->stream>>>(dinv, v, s, tA == 'T' ? 1 : 0);
    note(cudaGetLastError());
    ctx->launches++;
  }
  void transpose_inplace(double* A, int64_t ld, int64_t n) {
    const int64_t nt = n / 32;
    transpose_inplace_kernel<<<(unsigned)(nt * (nt + 1) / 2), dim3(32, 8), 0, ctx->stream>>>(A, ld, nt);
    note(cudaGetLastError());
    ctx->launches++;
  }
  void copy_dinv_128_t(double* dst, int64_t ldd, const double* src, int64_t batch, int64_t stride, int64_t dstride) {
    copy_dinv_128_t_kernel<<<(unsigned)batch, 256, 0, ctx->stream>>>(dst, ldd, src, stride, dstride);
    note(cudaGetLastError());
    ctx->launches++;
  }
  void copy_dinv_128(double* dst, int64_t ldd, const double* src, int64_t batch, int64_t stride, int64_t dstride,
                     bool full) {
    copy_dinv_128_kernel<<<(unsigned)batch, 256, 0, ctx->stream>>>(dst, ldd, src, stride, dstride, full ? 1 : 0);
    note(cudaGetLastError());
    ctx->launches++;
  }
};

int setup_kernel_attributes(gpr_ctx* ctx) {
  CK(gemm_setup_attributes());
  CK(gemm_tma_set_attr());
  CK(oz_set_attr());
  CK(cudaFuncSetAttribute(potrf_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LEAF_SMEM_BYTES));
  CK(cudaFuncSetAttribute(leaf_mv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LEAF_MV_SMEM_BYTES));
  CK(cudaFuncSetAttribute(kbuild_kernel<DM_EUCLID>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(kbuild_kernel<DM_SPLIT_A>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(kbuild_kernel<DM_SPLIT_C>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(kbuild_gram_kernel<DM_EUCLID>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(kbuild_gram_kernel<DM_SPLIT_A>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(kbuild_gram_kernel<DM_SPLIT_C>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(grad_reduce_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(grad_reduce_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(kbuild_kernel<DM_EUCLID, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KBW_SMEM_BYTES));
  CK(cudaFuncSetAttribute(kbuild_kernel<DM_SPLIT_A, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KBW_SMEM_BYTES));
  CK(cudaFuncSetAttribute(kbuild_kernel<DM_SPLIT_C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KBW_SMEM_BYTES));
  CK(cudaFuncSetAttribute(grad_reduce_wide_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GW_SMEM_BYTES));
  CK(cudaFuncSetAttribute(grad_reduce_wide_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GW_SMEM_BYTES));
  return GPR_OK;
}

int make_spec(gpr_ctx* ctx, const int* types, int ncomp, int D, KSpec* spec, int* P_out, int* nk_out) {
  if (!types || ncomp < 1 || ncomp > KSPEC_MAXC) return fail(ctx, GPR_ERR_ARG, "ncomp must be in 1..8");
  if (D < 1) return fail(ctx, GPR_ERR_ARG, "D must be >= 1");
  int off = 0, nk = 0;
  spec->ncomp = ncomp;
  for (int c = 0; c < KSPEC_MAXC; ++c) { spec->type[c] = 0; spec->hp_off[c] = 0; }
  for (int c = 0; c < ncomp; ++c) {
    spec->type[c] = types[c];
    spec->hp_off[c] = off;
    if (types[c] == GPR_KERN_SE || types[c] == GPR_KERN_MATERN52) { off += D + 1; nk++; }
    else if (types[c] == GPR_KERN_NOISE) off += 1;
    else return fail(ctx, GPR_ERR_ARG, "unknown kernel component type");
  }
  if (nk == 0) return fail(ctx, GPR_ERR_ARG, "covariance needs at least one non-noise component");
  if (P_out) *P_out = off;
  if (nk_out) *nk_out = nk;
  return GPR_OK;
}

// covariance build launcher.  centre: D doubles on the device (Euclidean Gram form), skip_lower: single-GPU training build.
int launch_kbuild(gpr_ctx* ctx, int mode, const KBuildArgs& a, const double* centre = nullptr, int skip_lower = 0) {
  int nk = 0;
  for (int c = 0; c < a.spec.ncomp; ++c) if (a.spec.type[c] != KT_NOISE) nk++;
  if (ctx->kbuild_gram && kgram_supported(a, nk)) {
    // TMA-fed Gram form on the DMMA pipe (csrc/kbuild_tma.cuh)
    KGramArgs ka{a, centre, skip_lower};
    cudaError_t e = mode == DM_EUCLID ? kgram_launch<DM_EUCLID>(ctx->stream, ka, nk)
                  : mode == DM_SPLIT_A ? kgram_launch<DM_SPLIT_A>(ctx->stream, ka, nk) : kgram_launch<DM_SPLIT_C>(ctx->stream, ka, nk);
    ctx->launches++;
    if (e != cudaSuccess) return fail_cuda(ctx, e, "kbuild_gram launch", __LINE__);
    return GPR_OK;
  }
  size_t smem = (size_t)2 * nk * a.D * KB_TILE * sizeof(double);
  if (a.mean_w || a.mean_w_rows) smem = std::max(smem, (size_t)16 * (KB_TILE + 1) * sizeof(double));
  dim3 grid((unsigned)((a.Rp + KB_TILE - 1) / KB_TILE), (unsigned)((a.Cp + KB_TILE - 1) / KB_TILE));
  if (grid.y > 65535) return fail(ctx, GPR_ERR_UNSUPPORTED, "covariance build: too many column tiles");
  if (smem > 200 * 1024) {
    // the scaled point tiles of all components do not fit: stage them one component and KBW_DC coordinates at a time
    if (mode == DM_EUCLID) kbuild_kernel<DM_EUCLID, true><<<grid, KB_THREADS, KBW_SMEM_BYTES, ctx->stream>>>(a);
    else if (mode == DM_SPLIT_A) kbuild_kernel<DM_SPLIT_A, true><<<grid, KB_THREADS, KBW_SMEM_BYTES, ctx->stream>>>(a);
    else kbuild_kernel<DM_SPLIT_C, true><<<grid, KB_THREADS, KBW_SMEM_BYTES, ctx->stream>>>(a);
  } else if (mode == DM_EUCLID) kbuild_kernel<DM_EUCLID><<<grid, KB_THREADS, smem, ctx->stream>>>(a);
  else if (mode == DM_SPLIT_A) kbuild_kernel<DM_SPLIT_A><<<grid, KB_THREADS, smem, ctx->stream>>>(a);
  else kbuild_kernel<DM_SPLIT_C><<<grid, KB_THREADS, smem, ctx->stream>>>(a);
  ctx->launches++;
  CK(cudaGetLastError());
  return GPR_OK;
}

// fused gradient reduction (partial[block][P+1], a.P and a.D set): grad_reduce_kernel where its per-thread accumulators and
// point tiles fit in shared memory, the wide form (csrc/grad_wide.cuh: O(P) state per CTA, DMMA contractions over D in
// chunks) otherwise.  Shared by the single-GPU and the block-cyclic multi-GPU gradient.
template <bool DIST>
cudaError_t launch_grad_reduce(cudaStream_t st, const GradArgs& a, int blocks) {
  const size_t smem = ((size_t)(a.P + 1) * GR_THREADS + 2 * (size_t)a.D * GR_TILE + 2 * GR_TILE + 32) * sizeof(double);
  if (smem <= 200 * 1024) grad_reduce_kernel<DIST><<<blocks, GR_THREADS, smem, st>>>(a);
  else grad_reduce_wide_kernel<DIST><<<blocks, GR_THREADS, GW_SMEM_BYTES, st>>>(a);
  return cudaGetLastError();
}

// rows of the output one CTA of the covariance build covers (the fused-mean partials are per CTA row tile)
int kbuild_rows_per_cta(gpr_ctx* ctx, const KBuildArgs& a) {
  int nk = 0;
  for (int c = 0; c < a.spec.ncomp; ++c) if (a.spec.type[c] != KT_NOISE) nk++;
  return (ctx->kbuild_gram && kgram_supported(a, nk)) ? KG_BM : KB_TILE;
}

struct DevBuf {
  double* p = nullptr;
  size_t n = 0;   // elements
  // grow to hold `need` doubles (no-op when it already does); false on an allocation failure, whose CUDA error is cleared
  bool grow(size_t need) {
    if (need <= n) return true;
    cudaFree(p); p = nullptr; n = 0;
    if (cudaMalloc(&p, need * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return false; }
    n = need;
    return true;
  }
};

}  // namespace

struct gpr_model {
  gpr_ctx* ctx = nullptr;
  KSpec spec;
  std::vector<int> types;
  int ncomp = 0, D = 0, P = 0, nk = 0, ny = 1, train_axis = 1;
  int64_t N = 0, Np = 0, nyp = 128;
  double* d_x = nullptr;      // D x N
  double* d_y = nullptr;      // N x ny
  double* d_hp = nullptr;     // P
  double* d_U = nullptr;      // Np x Np: upper = U, strict lower = K
  double* d_Kinv = nullptr;   // Np x Np upper = K^-1 (may alias d_U when memory is short)
  double* d_W = nullptr;      // Np x Np upper = U^-1 (out-of-place inverse path; optional)
  double* d_dinv = nullptr;   // Np/128 blocks of 128x128
  double* d_wt = nullptr;     // Np x nyp : K^-1 y (all columns), zero padded
  double* d_scal = nullptr;   // [logdet, y.alpha]
  double* d_G = nullptr;      // P
  double* d_gpart = nullptr;  // grad partials
  int gr_blocks = 0;
  bool kinv_alias = false;
  // state
  bool have_factor = false, have_inverse = false, factor_destroyed = false, kinv_symmetric = false;
  bool lower_is_k = false;   // strict lower triangle of d_U holds K (filled on demand by gpr_fetch(U))
  int oz = 0;                // digits of the INT8-tensor-core route in force for the current hyper-parameters (0 = DMMA)
  std::vector<double> hp_host;
  double eps_host = 0.0;
  int64_t info_host = 0;
  // predict workspaces (lazy)
  DevBuf w_kxp, w_xp, w_part, w_mean, w_var;
  DevBuf w_sA, w_sBt, w_sC, w_sCu, w_sx, w_smu;   // split predict (GPRSplitPredictCache)
  Timer tm;
};

namespace {

void timer_init(Timer& t) {
  for (int i = 0; i < GPR_T_COUNT; ++i) {
    cudaEventCreate(&t.beg[i]); cudaEventCreate(&t.end[i]);
    t.used[i] = false; t.acc_ms[i] = 0.0;
  }
}
void timer_free(Timer& t) {
  for (int i = 0; i < GPR_T_COUNT; ++i) { cudaEventDestroy(t.beg[i]); cudaEventDestroy(t.end[i]); }
}
void timer_reset(Timer& t) { for (int i = 0; i < GPR_T_COUNT; ++i) { t.used[i] = false; t.acc_ms[i] = 0.0; } }
void timer_reset_predict(Timer& t) {
  for (int i = GPR_T_PRED_KSTAR; i <= GPR_T_PRED_ROWNORM; ++i) { t.used[i] = false; t.acc_ms[i] = 0.0; }
  for (int i = GPR_T_SPLIT_BUILD; i <= GPR_T_SPLIT_D2H; ++i) { t.used[i] = false; t.acc_ms[i] = 0.0; }
}
// accumulate a previously recorded slot (needs the events to have completed)
void timer_collect(Timer& t, int slot) {
  if (!t.used[slot]) return;
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, t.beg[slot], t.end[slot]) == cudaSuccess) t.acc_ms[slot] += ms;
  t.used[slot] = false;
}
struct Scope {
  Timer& t; int slot; cudaStream_t st;
  Scope(Timer& t_, int s, cudaStream_t st_) : t(t_), slot(s), st(st_) {
    if (t.used[slot]) { cudaEventSynchronize(t.end[slot]); timer_collect(t, slot); }
    cudaEventRecord(t.beg[slot], st);
  }
  ~Scope() { cudaEventRecord(t.end[slot], st); t.used[slot] = true; }
};

int ensure(gpr_ctx* ctx, DevBuf& b, size_t elems) {
  if (b.n >= elems && b.p) return GPR_OK;
  if (b.p) { cudaFree(b.p); b.p = nullptr; b.n = 0; }
  CK(cudaMalloc(&b.p, elems * sizeof(double)));
  b.n = elems;
  return GPR_OK;
}

int check_pending(gpr_ctx* ctx, const char* where) {
  if (ctx->pending != cudaSuccess) {
    cudaError_t e = ctx->pending; ctx->pending = cudaSuccess;
    return fail_cuda(ctx, e, where, __LINE__);
  }
  return GPR_OK;
}

// INT8-tensor-core route (csrc/ozaki_i8.cuh) for this model and these hyper-parameters?  Its products are exact up to
// ~2^-56 of the operand ROW maxima (norm-wise, not component-wise), which a factorization amplifies by cond(K): harmless
// while cond * 2^-53 is far below the 1e-8 tolerances, visible on near-singular models (jitter-only kernels, cond 1e10:
// predictive mean 4e-3 against 6e-6 on the DMMA pipe, tests/test_extended_precision.py with GPR_OZAKI_MIN=128).
// Automatic mode therefore bounds the condition number from the hyper-parameters,
//   cond(K) <= (N * sum_c sigma_c^2 + sigma_n^2 + nk * eps) / (sigma_n^2 + nk * eps),
// and takes the INT8 route only below 1e8 (the benchmark model: 4e6).  Shared with the multi-GPU model (mgpu_factor).
int ozaki_auto_digits(const KSpec& spec, int nk, int64_t N, const double* hp, double eps) {
  double sig2 = 0.0, noise2 = 0.0;
  bool have_noise = false;
  for (int c = 0; c < spec.ncomp; ++c) {
    const double v = hp[spec.hp_off[c]];
    if (spec.type[c] == KT_NOISE) { if (!have_noise) { noise2 = v * v; have_noise = true; } }
    else sig2 += v * v;
  }
  const double floor_ = noise2 + nk * eps;
  if (!(floor_ > 0.0)) return 0;
  const double bound = ((double)N * sig2 + floor_) / floor_;
  return bound <= 1e8 ? 8 : 0;
}
int ozaki_digits_for(const gpr_model* m, const double* hp, double eps) {
  return m->ctx->ozaki >= 0 ? m->ctx->ozaki : ozaki_auto_digits(m->spec, m->nk, m->N, hp, eps);
}

// prior variance of a test point: sum over ALL components (noise included) of hp_c[1]^2, no jitter (src/predict.jl:55-58,67)
double prior_var(const KSpec& spec, const double* hp) {
  double s = 0.0;
  for (int c = 0; c < spec.ncomp; ++c) { const double v = hp[spec.hp_off[c]]; s += v * v; }
  return s;
}

// antideriv2(SquaredExp(), hp, a, b) (src/integrate.jl:33-41): sigma^2 prod_i erf_integ(l_i, a_i, b_i), hp = [sigma, l_1..l_D]
// of the first component whatever the others are, as the reference reads it
double antideriv2_se(const double* hp, const double* a, const double* b, int D) {
  double k2 = hp[0] * hp[0];
  for (int i = 0; i < D; ++i) {
    const double w = hp[1 + i], d = b[i] - a[i];
    k2 *= 1.0 / (w * w) * (std::exp(-(w * d) * (w * d)) - 1.0) + 2.0 * (0.88622692545275801365 / w) * d * std::erf(w * d);
  }
  return k2;
}

// largest dynamic shared memory a CTA can opt in to on sm_100 (227 KB)
constexpr size_t ANTIDERIV_SMEM_MAX = 227 * 1024;

// k1 tile of nbox boxes on ctx's queue (antideriv_se_kernel: np x mtp, ld ldk; a, b D x nbox on the device)
int launch_antideriv(gpr_ctx* ctx, const double* x, int D, int64_t n, int64_t np, const double* hp, const double* a,
                     const double* b, int64_t nbox, int64_t mtp, double* k1, int64_t ldk) {
  const size_t smem = sizeof(double) * 2 * D * ANTIDERIV_BOXES;
  const dim3 grid((unsigned)((np + 255) / 256), (unsigned)std::min<int64_t>((mtp + ANTIDERIV_BOXES - 1) / ANTIDERIV_BOXES, 65535));
  if (smem > ANTIDERIV_SMEM_MAX) {
    // the bounds of D coordinates exceed the 227 KB a CTA can have: stage them ANTIDERIV_DCH coordinates at a time
    const size_t smem_c = sizeof(double) * 2 * ANTIDERIV_DCH * ANTIDERIV_BOXES;
    CK(cudaFuncSetAttribute(antideriv_se_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c));
    antideriv_se_kernel<true><<<grid, 256, smem_c, ctx->stream>>>(x, D, n, np, hp, a, b, nbox, mtp, k1, ldk);
  } else {
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(antideriv_se_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    antideriv_se_kernel<false><<<grid, 256, smem, ctx->stream>>>(x, D, n, np, hp, a, b, nbox, mtp, k1, ldk);
  }
  ctx->launches++;
  CK(cudaGetLastError());
  return GPR_OK;
}

// K (+ noise, + jitter, identity padding) into m->d_U, then blocked potrf; solves for all y columns.
// Reads the factorization status back (the only host <-> device round trip of the factor / inverse sequence) and fixes the cache
// state accordingly.  LAPACK-style info: first failing pivot, 0 = ok (src/cost.jl:104 throws PosDefException the same way).
int finish_factor_status(gpr_model* m, int64_t* info, const char* where) {
  gpr_ctx* ctx = m->ctx;
  long long h_info = 0;
  CK(cudaMemcpyAsync(&h_info, ctx->d_info, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  int rc = check_pending(ctx, where);
  if (rc) { m->have_factor = false; m->have_inverse = false; return rc; }
  m->info_host = h_info;
  if (info) *info = h_info;
  m->have_factor = (h_info == 0);
  if (h_info != 0) {
    m->have_inverse = false;
    char buf[128];
    snprintf(buf, sizeof buf, "matrix is not positive definite; Cholesky failed at pivot %lld", h_info);
    return fail(ctx, GPR_ERR_NOT_POSDEF, buf);
  }
  return GPR_OK;
}

// defer_status: the caller goes straight on to the inverse and reads the status once at the end (finish_factor_status): a failed
// pivot makes potrf_leaf stop writing, the kernels behind it then work on stale data (dense index ranges only -- nothing can fault)
// and the result is discarded.
int factor_and_solve(gpr_model* m, const double* hp, double eps, int64_t* info, bool defer_alpha, bool defer_status = false) {
  gpr_ctx* ctx = m->ctx;
  const int64_t N = m->N, Np = m->Np;
  m->oz = ozaki_digits_for(m, hp, eps);
  ctx->oz_active = m->oz;
  CK(cudaMemcpyAsync(m->d_hp, hp, sizeof(double) * m->P, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->d_info, 0, sizeof(long long), ctx->stream));
  {
    Scope s(m->tm, GPR_T_KBUILD, ctx->stream);
    KBuildArgs a{};
    a.out = m->d_U; a.ldo = Np; a.R = N; a.C = N; a.Rp = Np; a.Cp = Np;
    a.x1 = m->d_x; a.x2 = m->d_x; a.D = m->D; a.hp = m->d_hp; a.spec = m->spec;
    a.eps = eps; a.same = 1; a.add_noise = 1; a.pad_identity = 1; a.sigma_one = 0; a.row_scale = nullptr; a.diag_shift = 0;
    // nothing on the path reads the strict lower triangle; it is only part of the reference's cache contents
    // (kchol_base keeps K there, test/test_loss.jl:46), so it is filled in lazily by gpr_fetch(U)
    a.zero_lower = 1;
    m->lower_is_k = false;
    int rc = launch_kbuild(ctx, DM_EUCLID, a, m->d_x, 1);
    if (rc) return rc;
  }
  CudaBE be{ctx};
  Blocked<CudaBE> blk(be, m->d_dinv);
  blk.leaf_lookahead = ctx->leaf_lookahead != 0;
  {
    Scope s(m->tm, GPR_T_POTRF, ctx->stream);
    ctx->oz_cur = OZ_PH_POTRF;
    blk.potrf(m->d_U, Np, Np, 0);
    ctx->oz_cur = OZ_PH_OTHER;
  }
  {
    Scope s(m->tm, GPR_T_POTRS, ctx->stream);
    const int threads = 256;
    const int64_t total = Np * m->nyp;
    int blocks = (int)std::min<int64_t>((total + threads - 1) / threads, 65535);
    pad_copy_kernel<<<blocks, threads, 0, ctx->stream>>>(m->d_wt, Np, Np, m->nyp, m->d_y, N, N, m->ny);
    ctx->launches++;
    if (!defer_alpha) {
      if (m->ny == 1) blk.potrsv(m->d_U, Np, Np, m->d_wt);        // vector y: memory-bound trsv sweeps
      else blk.potrs(m->d_U, Np, Np, m->d_wt, Np, m->nyp);       // matrix y: GEMM-based trsm on the padded block
      const double* alpha = m->d_wt + (int64_t)(m->train_axis - 1) * Np;
      const double* ycol = m->d_y + (int64_t)(m->train_axis - 1) * N;
      logdet_dot_kernel<<<1, 1024, 0, ctx->stream>>>(m->d_U, Np, N, ycol, alpha, m->d_scal);
      ctx->launches++;
    }
  }
  m->have_inverse = false;
  m->factor_destroyed = false;
  m->kinv_symmetric = false;
  if (defer_status) { m->have_factor = true; return GPR_OK; }     // provisional until finish_factor_status
  return finish_factor_status(m, info, "factor_and_solve");
}

int form_inverse(gpr_model* m) {
  gpr_ctx* ctx = m->ctx;
  const int64_t Np = m->Np;
  ctx->oz_active = m->oz;
  // Buffers: preferred = two extra N x N (W = U^-1 and K^-1 = W W^T out of place, one fully parallel launch);
  // one extra = in-place trtri + recursive lauum on it; none = invert in place over U (destroys the factor).
  if (!m->d_Kinv) {
    cudaError_t e = cudaMalloc(&m->d_Kinv, sizeof(double) * Np * Np);
    if (e != cudaSuccess) {
      cudaGetLastError();
      m->d_Kinv = m->d_U;
      m->kinv_alias = true;
    } else if (!ctx->inplace_lauum) {
      e = cudaMalloc(&m->d_W, sizeof(double) * Np * Np);
      if (e != cudaSuccess) { cudaGetLastError(); m->d_W = nullptr; }
    }
  }
  CudaBE be{ctx};
  Blocked<CudaBE> blk(be, m->d_dinv);
  if (m->d_W) {
    {
      Scope s(m->tm, GPR_T_TRTRI, ctx->stream);
      ctx->oz_cur = OZ_PH_TRTRI;
      blk.trtri_t(m->d_U, Np, m->d_W, Np, Np, 0);      // lower(W) = U^-T, all products in the T,N form
    }
    {
      Scope s(m->tm, GPR_T_LAUUM, ctx->stream);
      ctx->oz_cur = OZ_PH_LAUUM;
      blk.lauum_oop_t(m->d_W, Np, Np, m->d_Kinv, Np);  // K^-1 = (U^-T)^T U^-T
      ctx->oz_cur = OZ_PH_OTHER;
    }
  } else {
    {
      Scope s(m->tm, GPR_T_TRTRI, ctx->stream);
      if (!m->kinv_alias) CK(cudaMemcpyAsync(m->d_Kinv, m->d_U, sizeof(double) * Np * Np, cudaMemcpyDeviceToDevice, ctx->stream));
      else m->factor_destroyed = true;
      blk.trtri(m->d_Kinv, Np, Np, 0, false);
    }
    {
      Scope s(m->tm, GPR_T_LAUUM, ctx->stream);
      blk.lauum(m->d_Kinv, Np, Np, 0);
    }
  }
  m->have_inverse = true;
  m->kinv_symmetric = false;
  return check_pending(ctx, "form_inverse");
}

// true when K^-1 lives (or will live) in its own buffer, i.e. the factor U survives form_inverse
bool inverse_is_out_of_place(gpr_model* m) {
  if (m->d_Kinv) return !m->kinv_alias;
  cudaError_t e = cudaMalloc(&m->d_Kinv, sizeof(double) * m->Np * m->Np);   // what form_inverse would do first
  if (e != cudaSuccess) { cudaGetLastError(); m->d_Kinv = nullptr; return false; }
  if (!m->ctx->inplace_lauum) {
    e = cudaMalloc(&m->d_W, sizeof(double) * m->Np * m->Np);
    if (e != cudaSuccess) { cudaGetLastError(); m->d_W = nullptr; }
  }
  return true;
}

// alpha = K^-1 y (upper-stored symmetric product), then log det U and y . alpha
int alpha_from_inverse(gpr_model* m) {
  gpr_ctx* ctx = m->ctx;
  const int64_t N = m->N, Np = m->Np;
  Scope s(m->tm, GPR_T_POTRS, ctx->stream);
  double* alpha = m->d_wt;                       // ny == 1: column 0 (pad_copy left y there; overwritten below)
  const double* ycol = m->d_y;
  CK(cudaMemsetAsync(alpha, 0, sizeof(double) * Np * m->nyp, ctx->stream));
  symv_upper_cols_kernel<<<(unsigned)((N + 7) / 8), 256, 0, ctx->stream>>>(N, m->d_Kinv, Np, ycol, alpha);
  ctx->launches++;
  CK(cudaGetLastError());
  symv_upper_rows_kernel<<<(unsigned)((N + 63) / 64), 256, 0, ctx->stream>>>(N, m->d_Kinv, Np, ycol, alpha);
  ctx->launches++;
  CK(cudaGetLastError());
  logdet_dot_kernel<<<1, 1024, 0, ctx->stream>>>(m->d_U, Np, N, ycol, alpha, m->d_scal);
  ctx->launches++;
  CK(cudaGetLastError());
  return GPR_OK;
}

int compute_grad(gpr_model* m, int log_scale, double* G_host) {
  gpr_ctx* ctx = m->ctx;
  if (!m->have_inverse) return fail(ctx, GPR_ERR_STATE, "grad: cache holds no K^-1 (call gpr_update_cache with want_inverse = 1)");
  {
    Scope s(m->tm, GPR_T_GRAD, ctx->stream);
    GradArgs a{};
    a.Kinv = m->d_Kinv; a.ld = m->Np; a.alpha = m->d_wt + (int64_t)(m->train_axis - 1) * m->Np;
    a.x = m->d_x; a.D = m->D; a.N = m->N; a.hp = m->d_hp; a.spec = m->spec; a.P = m->P; a.eps = m->eps_host;
    a.partial = m->d_gpart;
    CK(launch_grad_reduce<false>(ctx->stream, a, m->gr_blocks));
    ctx->launches++;
    grad_finalize_kernel<<<1, 256, 0, ctx->stream>>>(m->d_gpart, m->gr_blocks, m->P, m->d_hp, m->spec, m->D, log_scale, m->d_G);
    ctx->launches++;
    CK(cudaGetLastError());
  }
  CK(cudaMemcpyAsync(G_host, m->d_G, sizeof(double) * m->P, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GPR_OK;
}

int compute_loss(gpr_model* m, double* F) {
  gpr_ctx* ctx = m->ctx;
  if (!m->have_factor) return fail(ctx, GPR_ERR_STATE, "loss: no valid factorization in the cache");
  double sc[2];
  CK(cudaMemcpyAsync(sc, m->d_scal, sizeof sc, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  // 0.5 * (dot(y, K^-1 y) + logdet(K) + N log(2 pi))   (src/loss_grad.jl:40)
  *F = 0.5 * (sc[1] + sc[0] + (double)m->N * std::log(2.0 * M_PI));
  return GPR_OK;
}

}  // namespace

extern "C" {

int gpr_version(void) { return 101; }

int gpr_device_count(void) {
  int ndev = 0, ok = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess) { cudaGetLastError(); return 0; }
  for (int d = 0; d < ndev; ++d) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
  }
  return ok;
}

int gpr_ctx_create(int device, gpr_ctx** out) {
  gpr_ctx* ctx = nullptr;
  if (!out) return fail(nullptr, GPR_ERR_ARG, "ctx out pointer is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, GPR_ERR_CUDA, std::string("no CUDA device available (libgpr_sm100a has no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(nullptr, GPR_ERR_ARG, "device index out of range");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(nullptr, GPR_ERR_CUDA, "libgpr_sm100a.so is built for sm_100a only; device compute capability is " +
                                           std::to_string(prop.major) + "." + std::to_string(prop.minor));
  ctx = new gpr_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete ctx; return fail_cuda(nullptr, e, "cudaStreamCreate", __LINE__); }
  e = cudaMalloc(&ctx->d_info, sizeof(long long));
  if (e != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return fail_cuda(nullptr, e, "cudaMalloc", __LINE__); }
  int rc = setup_kernel_attributes(ctx);
  if (rc) { g_create_error = ctx->err; cudaFree(ctx->d_info); cudaStreamDestroy(ctx->stream); delete ctx; return rc; }
  ctx->main_stream = ctx->stream;
  if (const char* ev = getenv("GPR_OZAKI")) {   // run an unmodified caller (the parity suite) with the INT8-tensor-core product
    const int v = atoi(ev);
    if (v == -1 || v == 0 || v == 6 || v == 7 || v == 8) ctx->ozaki = v;
  }
  if (const char* ev = getenv("GPR_OZAKI_MIN")) ctx->ozaki_min = std::max<int64_t>(128, atoll(ev));
  if (const char* ev = getenv("GPR_OZAKI_PHASES")) ctx->oz_mask = atoi(ev) & 15;
  if (const char* ev = getenv("GPR_OZAKI_LAUUM")) { const int v = atoi(ev); if (v == 0 || v == 8 || v == 9) ctx->ozaki_lauum = v; }
  e = cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
  live_add(ctx);
  if (e != cudaSuccess) { gpr_ctx_destroy(ctx); return fail_cuda(nullptr, e, "side queue", __LINE__); }
  *out = ctx;
  return GPR_OK;
}

int gpr_ctx_destroy(gpr_ctx* ctx) {
  if (!ctx || !live_take(ctx)) return GPR_OK;
  cudaSetDevice(ctx->device);
  while (!ctx->models.empty()) gpr_model_destroy(ctx->models.back());   // models the caller has not released yet
  if (ctx->main_stream) ctx->stream = ctx->main_stream;
  cudaStreamSynchronize(ctx->stream);
  if (ctx->side_stream) { cudaStreamSynchronize(ctx->side_stream); cudaStreamDestroy(ctx->side_stream); }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  for (auto& ev : ctx->ev_chunk) if (ev) cudaEventDestroy(ev);
  for (auto& ev : ctx->ev_d2h) if (ev) cudaEventDestroy(ev);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  cudaFree(ctx->oz_ws);
  cudaFree(ctx->d_info);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
  return GPR_OK;
}

const char* gpr_last_error(gpr_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int gpr_ctx_set_option(gpr_ctx* ctx, const char* name, int64_t value) {
  if (!ctx || !name) return GPR_ERR_ARG;
  if (!strcmp(name, "predict_tile")) {
    if (value < 128) return fail(ctx, GPR_ERR_ARG, "predict_tile must be >= 128");
    ctx->predict_tile = round_up(value, 128);
    return GPR_OK;
  }
  if (!strcmp(name, "inplace_lauum")) { ctx->inplace_lauum = value ? 1 : 0; return GPR_OK; }
  if (!strcmp(name, "leaf_lookahead")) { ctx->leaf_lookahead = value ? 1 : 0; return GPR_OK; }
  if (!strcmp(name, "alpha_from_inverse")) { ctx->alpha_from_inverse = value ? 1 : 0; return GPR_OK; }
  if (!strcmp(name, "gemm_tma")) { ctx->gemm_tma = value ? 1 : 0; return GPR_OK; }
  if (!strcmp(name, "ozaki")) {
    if (value != -1 && value != 0 && value != 6 && value != 7 && value != 8)
      return fail(ctx, GPR_ERR_ARG, "ozaki: number of digits must be -1 (automatic), 0 (off), 6, 7 or 8");
    ctx->ozaki = (int)value; ctx->oz_active = value > 0 ? (int)value : 0; return GPR_OK;
  }
  if (!strcmp(name, "ozaki_lauum")) {
    if (value != 0 && value != 8 && value != 9) return fail(ctx, GPR_ERR_ARG, "ozaki_lauum: 0 (DMMA), 8 or 9 digits");
    ctx->ozaki_lauum = (int)value; return GPR_OK;
  }
  if (!strcmp(name, "ozaki_pair")) { ctx->ozaki_pair = value ? 1 : 0; return GPR_OK; }
  if (!strcmp(name, "ozaki_win_mink")) { ctx->ozaki_win_mink = std::max<int64_t>(0, value); return GPR_OK; }
  if (!strcmp(name, "ozaki_split")) {
    if (value != 0 && value != 8 && value != 9) return fail(ctx, GPR_ERR_ARG, "ozaki_split: 0 (DMMA), 8 or 9 digits");
    ctx->ozaki_split = (int)value; return GPR_OK;
  }
  if (!strcmp(name, "ozaki_kchunk")) { ctx->ozaki_kchunk = std::min<int64_t>(32768, std::max<int64_t>(128, (value / 128) * 128)); return GPR_OK; }
  if (!strcmp(name, "ozaki_panel")) { ctx->ozaki_panel = std::max<int64_t>(128, (value / 128) * 128); return GPR_OK; }
  if (!strcmp(name, "ozaki_phases")) { ctx->oz_mask = (int)value & 15; return GPR_OK; }
  if (!strcmp(name, "ozaki_min")) { ctx->ozaki_min = std::max<int64_t>(128, value); return GPR_OK; }
  if (!strcmp(name, "kbuild_gram")) { ctx->kbuild_gram = value ? 1 : 0; return GPR_OK; }
  if (!strcmp(name, "gemm_cfg")) { ctx->gemm_cfg = (int)value; return GPR_OK; }   // 0 auto, 1..3: see dgemm_sm100.cuh
  return fail(ctx, GPR_ERR_ARG, std::string("unknown option ") + name);
}

int64_t gpr_ctx_launch_count(gpr_ctx* ctx) { return ctx ? ctx->launches : 0; }

int gpr_dim_hp(const int* comp_types, int ncomp, int D) {
  int P = 0;
  for (int c = 0; c < ncomp; ++c) {
    if (comp_types[c] == GPR_KERN_SE || comp_types[c] == GPR_KERN_MATERN52) P += D + 1;
    else if (comp_types[c] == GPR_KERN_NOISE) P += 1;
    else return GPR_ERR_ARG;
  }
  return P;
}

int gpr_model_create(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, int64_t N, const double* x, const double* y,
                     int ny, int train_axis, gpr_model** out) {
  if (!ctx) return GPR_ERR_ARG;
  if (!out || !x || !y) return fail(ctx, GPR_ERR_ARG, "NULL argument");
  *out = nullptr;
  if (N < 1) return fail(ctx, GPR_ERR_ARG, "x and y size mismatch.");
  if (ny < 1 || train_axis < 1 || train_axis > ny) return fail(ctx, GPR_ERR_ARG, "train_axis out of range");
  CK(cudaSetDevice(ctx->device));
  gpr_model* m = new gpr_model();
  m->ctx = ctx;
  int rc = make_spec(ctx, comp_types, ncomp, D, &m->spec, &m->P, &m->nk);
  if (rc) { delete m; return rc; }
  timer_init(m->tm);
  m->types.assign(comp_types, comp_types + ncomp);
  m->ncomp = ncomp; m->D = D; m->N = N; m->Np = round_up(N, 128); m->ny = ny; m->train_axis = train_axis;
  m->nyp = round_up(ny, 128);
  const int64_t Np = m->Np;
  cudaError_t e = cudaSuccess;
  auto A = [&](double** p, size_t elems) { if (e == cudaSuccess) e = cudaMalloc(p, elems * sizeof(double)); };
  A(&m->d_x, (size_t)D * N);
  A(&m->d_y, (size_t)N * ny);
  A(&m->d_hp, (size_t)m->P);
  A(&m->d_U, (size_t)Np * Np);
  A(&m->d_dinv, (size_t)Np * 128);
  A(&m->d_wt, (size_t)Np * m->nyp);
  A(&m->d_scal, 2);
  A(&m->d_G, (size_t)m->P);
  const int64_t T = (N + GR_TILE - 1) / GR_TILE;
  m->gr_blocks = (int)std::min<int64_t>(T * (T + 1) / 2, (int64_t)ctx->sm_count * 4);
  A(&m->d_gpart, (size_t)m->gr_blocks * (m->P + 1));
  live_add(m);
  ctx->models.push_back(m);
  if (e != cudaSuccess) { gpr_model_destroy(m); return fail_cuda(ctx, e, "cudaMalloc(model)", __LINE__); }
  e = cudaMemcpyAsync(m->d_x, x, sizeof(double) * D * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(m->d_y, y, sizeof(double) * N * ny, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { gpr_model_destroy(m); return fail_cuda(ctx, e, "upload x,y", __LINE__); }
  *out = m;
  return GPR_OK;
}

int gpr_model_destroy(gpr_model* m) {
  if (!m || !live_take(m)) return GPR_OK;    // unknown / already released (e.g. by gpr_ctx_destroy): nothing to do
  {
    auto& v = m->ctx->models;
    v.erase(std::remove(v.begin(), v.end(), m), v.end());
  }
  cudaSetDevice(m->ctx->device);
  cudaStreamSynchronize(m->ctx->stream);
  cudaFree(m->d_x); cudaFree(m->d_y); cudaFree(m->d_hp); cudaFree(m->d_U);
  if (m->d_Kinv && !m->kinv_alias) cudaFree(m->d_Kinv);
  cudaFree(m->d_W);
  cudaFree(m->d_dinv); cudaFree(m->d_wt); cudaFree(m->d_scal); cudaFree(m->d_G); cudaFree(m->d_gpart);
  cudaFree(m->w_kxp.p); cudaFree(m->w_xp.p); cudaFree(m->w_part.p); cudaFree(m->w_mean.p); cudaFree(m->w_var.p);
  cudaFree(m->w_sA.p); cudaFree(m->w_sBt.p); cudaFree(m->w_sC.p); cudaFree(m->w_sCu.p); cudaFree(m->w_sx.p); cudaFree(m->w_smu.p);
  timer_free(m->tm);
  delete m;
  return GPR_OK;
}

int gpr_model_set_y(gpr_model* m, const double* y) {
  if (!m || !y) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(m->d_y, y, sizeof(double) * m->N * m->ny, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  m->have_factor = m->have_inverse = false;
  m->hp_host.clear();
  return GPR_OK;
}

int gpr_model_set_x(gpr_model* m, const double* x) {
  if (!m || !x) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(m->d_x, x, sizeof(double) * m->N * m->D, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  m->have_factor = m->have_inverse = false;
  m->hp_host.clear();
  return GPR_OK;
}

int gpr_kernel(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, const double* hp, const double* x, int64_t N,
               const double* xp, int64_t M, int same_x, double eps, int add_noise, double* out) {
  if (!ctx) return GPR_ERR_ARG;
  if (!hp || !x || !xp || !out || N < 1 || M < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  if (same_x && N != M) return fail(ctx, GPR_ERR_ARG, "same_x requires N == M");
  CK(cudaSetDevice(ctx->device));
  KSpec spec; int P = 0, nk = 0;
  int rc = make_spec(ctx, comp_types, ncomp, D, &spec, &P, &nk);
  if (rc) return rc;
  double *d_x = nullptr, *d_xp = nullptr, *d_hp = nullptr, *d_out = nullptr;
  cudaError_t e = cudaMalloc(&d_x, sizeof(double) * D * N);
  if (e == cudaSuccess && !same_x) e = cudaMalloc(&d_xp, sizeof(double) * D * M);
  if (e == cudaSuccess) e = cudaMalloc(&d_hp, sizeof(double) * P);
  if (e == cudaSuccess) e = cudaMalloc(&d_out, sizeof(double) * N * M);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_x, x, sizeof(double) * D * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && !same_x) e = cudaMemcpyAsync(d_xp, xp, sizeof(double) * D * M, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_hp, hp, sizeof(double) * P, cudaMemcpyHostToDevice, ctx->stream);
  rc = GPR_OK;
  if (e == cudaSuccess) {
    KBuildArgs a{};
    a.out = d_out; a.ldo = N; a.R = N; a.C = M; a.Rp = N; a.Cp = M;
    a.x1 = d_x; a.x2 = same_x ? d_x : d_xp; a.D = D; a.hp = d_hp; a.spec = spec;
    a.eps = eps; a.same = same_x; a.add_noise = add_noise; a.pad_identity = 0; a.sigma_one = 0; a.row_scale = nullptr; a.diag_shift = 0;
    rc = launch_kbuild(ctx, DM_EUCLID, a, d_x);
    if (!rc) e = cudaMemcpyAsync(out, d_out, sizeof(double) * N * M, cudaMemcpyDeviceToHost, ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  cudaFree(d_x); cudaFree(d_xp); cudaFree(d_hp); cudaFree(d_out);
  if (rc) return rc;
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_kernel", __LINE__);
  return GPR_OK;
}

int gpr_kernel_grad(gpr_ctx* ctx, int comp_type, int D, const double* hp_comp, const double* x, int64_t N, int li,
                    double eps, double* out) {
  if (!ctx) return GPR_ERR_ARG;
  if (!hp_comp || !x || !out || N < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  if (comp_type != GPR_KERN_SE && comp_type != GPR_KERN_MATERN52) return fail(ctx, GPR_ERR_ARG, "gpr_kernel_grad: dense derivative exists for SE / Matern52 only");
  if (li < 0 || li > D) return fail(ctx, GPR_ERR_ARG, "hyper-parameter index out of range");
  CK(cudaSetDevice(ctx->device));
  double *d_x = nullptr, *d_hp = nullptr, *d_out = nullptr;
  cudaError_t e = cudaMalloc(&d_x, sizeof(double) * D * N);
  if (e == cudaSuccess) e = cudaMalloc(&d_hp, sizeof(double) * (D + 1));
  if (e == cudaSuccess) e = cudaMalloc(&d_out, sizeof(double) * N * N);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_x, x, sizeof(double) * D * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_hp, hp_comp, sizeof(double) * (D + 1), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) {
    KGradArgs a{d_out, N, N, d_x, D, d_hp, comp_type, li, eps};
    const int64_t total = N * N;
    int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 16);
    kgrad_dense_kernel<<<blocks, 256, 0, ctx->stream>>>(a);
    ctx->launches++;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, sizeof(double) * N * N, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  cudaFree(d_x); cudaFree(d_hp); cudaFree(d_out);
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_kernel_grad", __LINE__);
  return GPR_OK;
}

int gpr_update_cache(gpr_model* m, const double* hp, int P, double eps, int want_inverse, int64_t* info) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!hp) return fail(ctx, GPR_ERR_ARG, "hp is NULL");
  if (P != m->P) return fail(ctx, GPR_ERR_ARG, "Parameter size mismatch.");
  CK(cudaSetDevice(ctx->device));
  if (info) *info = 0;
  // same hp as the cached evaluation: reuse (SecondOrder optimisers call loss and grad! separately, src/train.jl:58-87)
  const bool same_hp = m->have_factor && !m->factor_destroyed && m->hp_host.size() == (size_t)P && m->eps_host == eps &&
                       std::equal(hp, hp + P, m->hp_host.begin());
  if (!same_hp) {
    timer_reset(m->tm);
    Scope total(m->tm, GPR_T_TOTAL, ctx->stream);
    m->hp_host.assign(hp, hp + P);
    m->eps_host = eps;
    // gradient path with a vector y: K^-1 is formed anyway, so alpha = K^-1 y is one symmetric matrix-vector product
    // with it (8 N^2 bytes, ~1.5 ms at N = 32768) instead of two chains of ~500 dependent triangular-solve launches
    // (12.5 ms).  Needs the separate K^-1 buffer: with the in-place inverse the factor (whose diagonal the log det
    // reads) is gone by then, so that path keeps the solves.
    const bool defer_alpha = want_inverse && m->ny == 1 && ctx->alpha_from_inverse && inverse_is_out_of_place(m);
    // gradient path: potrf, the inverse and alpha are enqueued back to back; the factorization status is read once at the end
    const bool defer_status = want_inverse != 0;
    int rc = factor_and_solve(m, hp, eps, info, defer_alpha, defer_status);
    if (rc) { m->hp_host.clear(); return rc; }
    if (want_inverse) { rc = form_inverse(m); if (rc) { m->hp_host.clear(); m->have_factor = false; return rc; } }
    if (defer_alpha) { rc = alpha_from_inverse(m); if (rc) { m->hp_host.clear(); m->have_factor = false; return rc; } }
    if (defer_status) { rc = finish_factor_status(m, info, "gpr_update_cache"); if (rc) { m->hp_host.clear(); return rc; } }
  } else if (want_inverse && !m->have_inverse) {
    int rc = form_inverse(m);
    if (rc) return rc;
  }
  return GPR_OK;
}

int gpr_loss(gpr_model* m, double* F) {
  if (!m || !F) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  CK(cudaSetDevice(ctx->device));
  return compute_loss(m, F);
}

int gpr_grad(gpr_model* m, int log_scale, double* G) {
  if (!m || !G) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  CK(cudaSetDevice(ctx->device));
  return compute_grad(m, log_scale, G);
}

int gpr_nlml_grad(gpr_model* m, const double* hp_in, int P, int log_scale, double eps, double* F, double* G,
                  int64_t* info) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!hp_in) return fail(ctx, GPR_ERR_ARG, "hp is NULL");
  if (P != m->P) return fail(ctx, GPR_ERR_ARG, "Parameter size mismatch.");
  std::vector<double> hp(hp_in, hp_in + P);
  if (log_scale) for (auto& v : hp) v = std::exp(v);   // hp = exp.(log_hp)  (src/cost.jl:61)
  CK(cudaSetDevice(ctx->device));
  cudaEventRecord(m->tm.beg[GPR_T_EVAL], ctx->stream);   // (timer_reset inside gpr_update_cache leaves the recorded event alone)
  int rc = gpr_update_cache(m, hp.data(), P, eps, G != nullptr, info);
  if (rc) return rc;
  if (G) { rc = compute_grad(m, log_scale, G); if (rc) return rc; }
  if (F) { rc = compute_loss(m, F); if (rc) return rc; }
  cudaEventRecord(m->tm.end[GPR_T_EVAL], ctx->stream);
  m->tm.acc_ms[GPR_T_EVAL] = 0.0;
  m->tm.used[GPR_T_EVAL] = true;
  CK(cudaStreamSynchronize(ctx->stream));
  return GPR_OK;
}

int gpr_fetch(gpr_model* m, int which, double* out) {
  if (!m || !out) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  CK(cudaSetDevice(ctx->device));
  const int64_t N = m->N, Np = m->Np;
  if (which == GPR_FETCH_U) {
    if (!m->have_factor || m->factor_destroyed) return fail(ctx, GPR_ERR_STATE, "fetch U: no factorization in the cache");
    if (!m->lower_is_k) {   // strict lower = K, exactly what dpotrf('U') leaves in tc.kchol_base
      KBuildArgs a{};
      a.out = m->d_U; a.ldo = Np; a.R = N; a.C = N; a.Rp = Np; a.Cp = Np;
      a.x1 = m->d_x; a.x2 = m->d_x; a.D = m->D; a.hp = m->d_hp; a.spec = m->spec;
      a.eps = m->eps_host; a.same = 1; a.add_noise = 1; a.pad_identity = 1; a.lower_only = 1;
      int rc = launch_kbuild(ctx, DM_EUCLID, a);
      if (rc) return rc;
      m->lower_is_k = true;
    }
    CK(cudaMemcpy2DAsync(out, sizeof(double) * N, m->d_U, sizeof(double) * Np, sizeof(double) * N, N, cudaMemcpyDeviceToHost, ctx->stream));
  } else if (which == GPR_FETCH_ALPHA) {
    if (!m->have_factor) return fail(ctx, GPR_ERR_STATE, "fetch alpha: no factorization in the cache");
    CK(cudaMemcpyAsync(out, m->d_wt + (int64_t)(m->train_axis - 1) * Np, sizeof(double) * N, cudaMemcpyDeviceToHost, ctx->stream));
  } else if (which == GPR_FETCH_WT) {
    if (!m->have_factor) return fail(ctx, GPR_ERR_STATE, "fetch wt: no factorization in the cache");
    CK(cudaMemcpy2DAsync(out, sizeof(double) * N, m->d_wt, sizeof(double) * Np, sizeof(double) * N, m->ny, cudaMemcpyDeviceToHost, ctx->stream));
  } else if (which == GPR_FETCH_KINV) {
    if (!m->have_inverse) return fail(ctx, GPR_ERR_STATE, "fetch K^-1: cache holds no inverse");
    if (!m->kinv_symmetric) {
      dim3 grid((unsigned)((Np + 31) / 32), (unsigned)((Np + 31) / 32)), block(32, 8);
      symmetrize_from_upper_kernel<<<grid, block, 0, ctx->stream>>>(m->d_Kinv, Np, Np);
      ctx->launches++;
      CK(cudaGetLastError());
      m->kinv_symmetric = true;
    }
    CK(cudaMemcpy2DAsync(out, sizeof(double) * N, m->d_Kinv, sizeof(double) * Np, sizeof(double) * N, N, cudaMemcpyDeviceToHost, ctx->stream));
  } else {
    return fail(ctx, GPR_ERR_ARG, "unknown fetch selector");
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return GPR_OK;
}

int gpr_model_route(gpr_model* m, int* digits, int* digits_inverse) {
  if (!m) return GPR_ERR_ARG;
  if (digits) *digits = m->oz > 0 ? m->oz : 0;
  if (digits_inverse) {
    // the route form_inverse's lauum_oop_t takes: W^T W (Np^3, upper only, K-from-N) in the lauum phase with the model's digits
    gpr_ctx* ctx = m->ctx;
    const int active = ctx->oz_active, cur = ctx->oz_cur;
    ctx->oz_active = m->oz > 0 ? m->oz : 0;
    ctx->oz_cur = OZ_PH_LAUUM;
    *digits_inverse = m->d_W ? CudaBE{ctx}.ozaki_route(CudaBE::OZ_PLAIN, 'T', 'N', m->Np, m->Np, m->Np, m->d_W, m->Np, m->d_W, m->Np,
                                                       m->d_Kinv, BLK_UPPER_ONLY | BLK_K_FROM_N).digits
                             : 0;
    ctx->oz_active = active;
    ctx->oz_cur = cur;
  }
  return GPR_OK;
}

int gpr_timings(gpr_model* m, double* ms, int n) {
  if (!m || !ms) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < GPR_T_COUNT; ++i) timer_collect(m->tm, i);
  for (int i = 0; i < n && i < GPR_T_COUNT; ++i) ms[i] = m->tm.acc_ms[i];
  return GPR_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// prediction
// ---------------------------------------------------------------------------
namespace {

// One tile of test points resident on the device: d_xp is D x mt (mt valid points, global index m0..m0+mt).
// Writes mean (mt x ny, column stride ldmean) and var (mt) to device memory.
int predict_tile(gpr_model* m, const double* d_xp, int64_t mt, int64_t m0, int same_x, double* d_mean, int64_t ldmean,
                 double* d_var) {
  // The tile is held TRANSPOSED: Kt = K(x, xp) is Np x mtp with the training index fastest (the reference keeps
  // Kxp = K(xp, x), src/predict.jl:37).  V^T = U^-T Kt is then a LEFT solve with U^T whose products are all of the T,N
  // form -- the same instantiation of the DMMA kernel as potrf / trtri / lauum (DMMA pipe 92.9 % active against 90.1 %
  // for the N,N products of the right solve Kxp U^-1) -- and the row norms of V become contiguous column sums.
  gpr_ctx* ctx = m->ctx;
  const int64_t Np = m->Np, N = m->N;
  const int64_t mtp = round_up(mt, 128);
  ctx->oz_active = m->oz;
  int rc = GPR_OK;
  if (d_var || m->ny > 1) {   // the K* tile is only materialised for the variance (or a matrix y)
    rc = ensure(ctx, m->w_kxp, (size_t)mtp * Np);
    if (rc) return rc;
  }
  double* Kt = m->w_kxp.p;
  CudaBE be{ctx};
  {
    Scope s(m->tm, GPR_T_PRED_KSTAR, ctx->stream);
    KBuildArgs a{};
    a.out = Kt; a.ldo = Np; a.R = N; a.C = mt; a.Rp = Np; a.Cp = mtp;
    a.x1 = m->d_x; a.x2 = d_xp; a.D = m->D; a.hp = m->d_hp; a.spec = m->spec;
    a.eps = m->eps_host; a.same = same_x; a.add_noise = 0; a.pad_identity = 0; a.sigma_one = 0; a.row_scale = nullptr;
    a.diag_shift = m0;          // training point r is test point c of this tile when r == m0 + c (xp === md.x)
    // vector y: mu = K* wt is reduced inside the build (per-CTA partial sums over 64 training points), so the tile is
    // not re-read; without a variance request it is not even stored
    const bool fuse_mean = (m->ny == 1);
    const int64_t rt = kbuild_rows_per_cta(ctx, a);
    const int64_t nrow_tiles = (Np + rt - 1) / rt;
    if (fuse_mean) {
      rc = ensure(ctx, m->w_part, (size_t)nrow_tiles * mtp);
      if (rc) return rc;
      a.mean_w_rows = m->d_wt; a.mean_partial = m->w_part.p;
      if (!d_var) a.out = nullptr;
    }
    rc = launch_kbuild(ctx, DM_EUCLID, a, m->d_x);
    if (rc) return rc;
    if (fuse_mean) {
      rowreduce_finalize_kernel<<<(unsigned)((mt + 255) / 256), 256, 0, ctx->stream>>>(m->w_part.p, (int)nrow_tiles, mtp, mt, 0.0, 1.0, d_mean);
      ctx->launches++;
      CK(cudaGetLastError());
    }
  }
  if (m->ny > 1) {
    // matrix y: mu = Kt^T wt for all columns at once, one T,N GEMM on the zero-padded weights (mtp x nyp)
    Scope s(m->tm, GPR_T_PRED_MEAN, ctx->stream);
    rc = ensure(ctx, m->w_part, (size_t)mtp * m->nyp);
    if (rc) return rc;
    be.gemm('T', 'N', mtp, m->nyp, Np, 1.0, Kt, Np, m->d_wt, Np, 0.0, m->w_part.p, mtp, 0);
    CK(cudaMemcpy2DAsync(d_mean, sizeof(double) * ldmean, m->w_part.p, sizeof(double) * mtp, sizeof(double) * mt, m->ny,
                         cudaMemcpyDeviceToDevice, ctx->stream));
  }
  if (d_var) {
    Blocked<CudaBE> blk(be, m->d_dinv);
    {
      Scope s(m->tm, GPR_T_PRED_TRSM, ctx->stream);
      blk.trsm_LUT(m->d_U, Np, Np, 0, Kt, Np, mtp, 1.0);   // Kt <- U^-T Kt = (Kxp U^-1)^T  (rdiv!, src/predict.jl:90)
    }
    {
      Scope s(m->tm, GPR_T_PRED_ROWNORM, ctx->stream);
      colsumsq_kernel<<<(unsigned)mt, 256, 0, ctx->stream>>>(Kt, Np, Np, mt, prior_var(m->spec, m->hp_host.data()), d_var);   // predict.jl:91-93
      ctx->launches++;
      CK(cudaGetLastError());
    }
  }
  return check_pending(ctx, "predict_tile");
}

// One tile of boxes resident on the device: d_a, d_b are D x mt (mt boxes).  k1 of every box is a column of the transposed
// tile, as Kt in predict_tile, but there is no covariance build to fuse the mean into.  Writes Iout = k1^T wt to the host
// (mt x ny, column stride ldI) and, when h_sq is given, h_sq[i] = -|U^-T k1_i|^2 (mt entries, host).
int integrate_tile(gpr_model* m, const double* d_a, const double* d_b, int64_t mt, double* Iout, int64_t ldI, double* h_sq) {
  gpr_ctx* ctx = m->ctx;
  const int64_t Np = m->Np;
  const int64_t mtp = round_up(mt, 128);
  ctx->oz_active = m->oz;
  int rc = ensure(ctx, m->w_kxp, (size_t)mtp * Np);
  if (!rc) rc = ensure(ctx, m->w_part, (size_t)mtp * m->nyp);
  if (!rc && h_sq) rc = ensure(ctx, m->w_var, (size_t)mtp);
  if (rc) return rc;
  double* k1 = m->w_kxp.p;
  double* d_I = m->w_part.p;     // mtp x ny
  CudaBE be{ctx};
  {
    Scope s(m->tm, GPR_T_PRED_KSTAR, ctx->stream);
    rc = launch_antideriv(ctx, m->d_x, m->D, m->N, Np, m->d_hp, d_a, d_b, mt, mtp, k1, Np);   // antideriv!  (:15-31)
    if (rc) return rc;
  }
  {
    Scope s(m->tm, GPR_T_PRED_MEAN, ctx->stream);
    if (m->ny == 1) {
      CK(cudaMemsetAsync(d_I, 0, sizeof(double) * mt, ctx->stream));
      be.gemv('T', mt, Np, 1.0, k1, Np, m->d_wt, d_I);                                          // Iout = k1' wt  (:118-121)
    } else {
      be.gemm('T', 'N', mtp, m->nyp, Np, 1.0, k1, Np, m->d_wt, Np, 0.0, d_I, mtp, 0);
    }
    CK(cudaMemcpy2DAsync(Iout, sizeof(double) * ldI, d_I, sizeof(double) * mtp, sizeof(double) * mt, m->ny,
                         cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (h_sq) {
    Blocked<CudaBE> blk(be, m->d_dinv);
    {
      Scope s(m->tm, GPR_T_PRED_TRSM, ctx->stream);
      blk.trsm_LUT(m->d_U, Np, Np, 0, k1, Np, mtp, 1.0);          // ldiv!(kchol.L, tt), L = U^T, every box at once  (:133-134)
    }
    {
      Scope s(m->tm, GPR_T_PRED_ROWNORM, ctx->stream);
      colsumsq_kernel<<<(unsigned)mt, 256, 0, ctx->stream>>>(k1, Np, Np, mt, 0.0, m->w_var.p);
      ctx->launches++;
      CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(h_sq, m->w_var.p, sizeof(double) * mt, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return check_pending(ctx, "integrate_tile");
}

}  // namespace

extern "C" {

int gpr_predict_device(gpr_model* m, const double* d_xp, int64_t M, int same_x, double* d_mean, double* d_var) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!d_xp || !d_mean || M < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  if (!m->have_factor || m->factor_destroyed) return fail(ctx, GPR_ERR_STATE, "predict: call gpr_update_cache first");
  if (same_x && M != m->N) return fail(ctx, GPR_ERR_ARG, "same_x requires M == N");
  CK(cudaSetDevice(ctx->device));
  timer_reset_predict(m->tm);
  const int64_t MT = ctx->predict_tile;
  for (int64_t m0 = 0; m0 < M; m0 += MT) {
    const int64_t mt = std::min(MT, M - m0);
    int rc = predict_tile(m, d_xp + m0 * m->D, mt, m0, same_x, d_mean + m0, M, d_var ? d_var + m0 : nullptr);
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return GPR_OK;
}

int gpr_predict(gpr_model* m, const double* xp, int64_t M, int same_x, double* mean, double* var_diag, double* cov_full) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!xp || !mean || M < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  if (!m->have_factor || m->factor_destroyed) return fail(ctx, GPR_ERR_STATE, "predict: call gpr_update_cache first");
  if (same_x && M != m->N) return fail(ctx, GPR_ERR_ARG, "same_x requires M == N");
  CK(cudaSetDevice(ctx->device));
  timer_reset_predict(m->tm);
  const int64_t Np = m->Np, N = m->N;
  const int D = m->D, ny = m->ny;

  if (cov_full) {
    // dense path (src/predict.jl:42-49,83-87): needs V = K* U^-1 for all test points at once
    const int64_t Mp = round_up(M, 128);
    int rc = ensure(ctx, m->w_xp, (size_t)D * M); if (rc) return rc;
    rc = ensure(ctx, m->w_mean, (size_t)Mp * ny); if (rc) return rc;
    rc = ensure(ctx, m->w_var, (size_t)Mp); if (rc) return rc;
    double* d_sigma = nullptr;
    CK(cudaMalloc(&d_sigma, sizeof(double) * Mp * Mp));
    cudaError_t e = cudaMemcpyAsync(m->w_xp.p, xp, sizeof(double) * D * M, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { cudaFree(d_sigma); return fail_cuda(ctx, e, "upload xp", __LINE__); }
    rc = predict_tile(m, m->w_xp.p, M, 0, same_x, m->w_mean.p, Mp, m->w_var.p);   // leaves V^T in w_kxp (Np x Mp)
    if (!rc) {
      KBuildArgs a{};
      a.out = d_sigma; a.ldo = Mp; a.R = M; a.C = M; a.Rp = Mp; a.Cp = Mp;
      a.x1 = m->w_xp.p; a.x2 = m->w_xp.p; a.D = D; a.hp = m->d_hp; a.spec = m->spec;
      a.eps = m->eps_host; a.same = 1; a.add_noise = 1; a.pad_identity = 0; a.sigma_one = 0; a.row_scale = nullptr; a.diag_shift = 0;
      rc = launch_kbuild(ctx, DM_EUCLID, a, m->w_xp.p);   // kernel!(Sigma, covar, params, xp)  (src/predict.jl:45)
    }
    if (!rc) {
      CudaBE be{ctx};
      be.gemm('T', 'N', Mp, Mp, Np, -1.0, m->w_kxp.p, Np, m->w_kxp.p, Np, 1.0, d_sigma, Mp, 0);   // Sigma -= V V^T = (V^T)^T V^T
      rc = check_pending(ctx, "predict cov");
    }
    if (!rc) {
      e = cudaMemcpy2DAsync(cov_full, sizeof(double) * M, d_sigma, sizeof(double) * Mp, sizeof(double) * M, M, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaMemcpy2DAsync(mean, sizeof(double) * M, m->w_mean.p, sizeof(double) * Mp, sizeof(double) * M, ny, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess && var_diag) e = cudaMemcpyAsync(var_diag, m->w_var.p, sizeof(double) * M, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      if (e != cudaSuccess) rc = fail_cuda(ctx, e, "download cov", __LINE__);
    }
    cudaStreamSynchronize(ctx->stream);
    cudaFree(d_sigma);
    (void)N;
    return rc;
  }

  const int64_t MT = std::min<int64_t>(ctx->predict_tile, round_up(M, 128));
  int rc = ensure(ctx, m->w_xp, (size_t)D * MT); if (rc) return rc;
  rc = ensure(ctx, m->w_mean, (size_t)MT * ny); if (rc) return rc;
  rc = ensure(ctx, m->w_var, (size_t)MT); if (rc) return rc;
  for (int64_t m0 = 0; m0 < M; m0 += MT) {
    const int64_t mt = std::min(MT, M - m0);
    CK(cudaMemcpyAsync(m->w_xp.p, xp + m0 * D, sizeof(double) * D * mt, cudaMemcpyHostToDevice, ctx->stream));
    rc = predict_tile(m, m->w_xp.p, mt, m0, same_x, m->w_mean.p, MT, var_diag ? m->w_var.p : nullptr);
    if (rc) return rc;
    CK(cudaMemcpy2DAsync(mean + m0, sizeof(double) * M, m->w_mean.p, sizeof(double) * MT, sizeof(double) * mt, ny, cudaMemcpyDeviceToHost, ctx->stream));
    if (var_diag) CK(cudaMemcpyAsync(var_diag + m0, m->w_var.p, sizeof(double) * mt, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return GPR_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// split kernel / split predict
// ---------------------------------------------------------------------------
namespace {

struct SplitBufs {
  double *A = nullptr, *B = nullptr, *C = nullptr;   // per non-noise component slices
  double *Bt = nullptr, *Cu = nullptr;               // variance path: B transposed (Np x nep x k), C unscaled (Np x nqp x k)
  const double* C_row_scale = nullptr;               // rows of C scaled by it (device, Np; nullptr: unscaled)
  double *d_xe = nullptr, *d_xq = nullptr;
  int64_t nep = 0, nqp = 0;
  void release() {
    cudaFree(A); cudaFree(B); cudaFree(C); cudaFree(Bt); cudaFree(Cu); cudaFree(d_xe); cudaFree(d_xq);
    A = B = C = Bt = Cu = d_xe = d_xq = nullptr;
  }
};

// Builds each of A (nep x nqp x k), B (nep x Np x k), C (Np x nqp x k; rows scaled by sb.C_row_scale if set) and, for the
// variance, Bt (Np x nep x k) and the unscaled Cu (Np x nqp x k) whose buffer in sb is not NULL: Bt and Cu with the training
// index fastest, the layout the transposed tile assembly reads coalesced.  d_hp: device global hp.  x: D x N device.
int split_build(gpr_ctx* ctx, const KSpec& spec, int D, const double* d_hp, const double* d_xe, int64_t ne,
                const double* d_xq, int64_t nq, const double* d_x, int64_t N, int64_t Np, const SplitBufs& sb) {
  const int64_t nep = sb.nep, nqp = sb.nqp;
  int k = 0;
  for (int c = 0; c < spec.ncomp; ++c) {
    if (spec.type[c] == KT_NOISE) continue;
    KSpec one{};
    one.ncomp = 1; one.type[0] = spec.type[c]; one.hp_off[0] = spec.hp_off[c];
    KBuildArgs a{};
    a.D = D; a.hp = d_hp; a.spec = one; a.eps = 0.0; a.same = 0; a.add_noise = 0; a.pad_identity = 0; a.diag_shift = 0;
    // A[:, :, k] = exp(-sum (l xq)^2 - 2 sum l^2 xe xq), sigma := 1   (split_kernel.jl:152-155)
    int rc = GPR_OK;
    if (sb.A) {
      a.out = sb.A + (int64_t)k * nep * nqp; a.ldo = nep; a.R = ne; a.C = nq; a.Rp = nep; a.Cp = nqp;
      a.x1 = d_xe; a.x2 = d_xq; a.sigma_one = 1; a.row_scale = nullptr;
      rc = launch_kbuild(ctx, DM_SPLIT_A, a); if (rc) return rc;
    }
    // B[:, :, k] = exp(-|l (xe - xs)|^2), sigma := 1                    (split_kernel.jl:156)
    if (sb.B) {
      a.out = sb.B + (int64_t)k * nep * Np; a.ldo = nep; a.R = ne; a.C = N; a.Rp = nep; a.Cp = Np;
      a.x1 = d_xe; a.x2 = d_x; a.sigma_one = 1;
      rc = launch_kbuild(ctx, DM_EUCLID, a, d_x); if (rc) return rc;
    }
    // C[:, :, k] = sigma^2 exp(+2 sum l^2 xs xq)                         (split_kernel.jl:157)
    if (sb.C) {
      a.out = sb.C + (int64_t)k * Np * nqp; a.ldo = Np; a.R = N; a.C = nq; a.Rp = Np; a.Cp = nqp;
      a.x1 = d_x; a.x2 = d_xq; a.sigma_one = 0; a.row_scale = sb.C_row_scale;
      rc = launch_kbuild(ctx, DM_SPLIT_C, a); if (rc) return rc;
    }
    if (sb.Cu) {
      a.out = sb.Cu + (int64_t)k * Np * nqp; a.ldo = Np; a.R = N; a.C = nq; a.Rp = Np; a.Cp = nqp;
      a.x1 = d_x; a.x2 = d_xq; a.sigma_one = 0; a.row_scale = nullptr;
      rc = launch_kbuild(ctx, DM_SPLIT_C, a); if (rc) return rc;
    }
    if (sb.Bt) {
      a.out = sb.Bt + (int64_t)k * Np * nep; a.ldo = Np; a.R = N; a.C = ne; a.Rp = Np; a.Cp = nep;
      a.x1 = d_x; a.x2 = d_xe; a.sigma_one = 1; a.row_scale = nullptr;
      rc = launch_kbuild(ctx, DM_EUCLID, a, d_x); if (rc) return rc;   // B is symmetric in its two point sets: Bt[s, e] = B[e, s]
    }
    ++k;
  }
  return GPR_OK;
}

}  // namespace

extern "C" {

int gpr_split_kernel(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, const double* hp, const double* xe,
                     int64_t ne, const double* xq, int64_t nq, const double* x, int64_t N, double* A, double* B,
                     double* C) {
  if (!ctx) return GPR_ERR_ARG;
  if (!hp || !xe || !xq || !x || !A || !B || !C || ne < 1 || nq < 1 || N < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  CK(cudaSetDevice(ctx->device));
  KSpec spec; int P = 0, nk = 0;
  int rc = make_spec(ctx, comp_types, ncomp, D, &spec, &P, &nk);
  if (rc) return rc;
  SplitBufs sb; sb.nep = ne; sb.nqp = nq;   // unpadded: plain host-shaped outputs
  double *d_x = nullptr, *d_hp = nullptr;
  cudaError_t e = cudaMalloc(&sb.A, sizeof(double) * ne * nq * nk);
  if (e == cudaSuccess) e = cudaMalloc(&sb.B, sizeof(double) * ne * N * nk);
  if (e == cudaSuccess) e = cudaMalloc(&sb.C, sizeof(double) * N * nq * nk);
  if (e == cudaSuccess) e = cudaMalloc(&sb.d_xe, sizeof(double) * D * ne);
  if (e == cudaSuccess) e = cudaMalloc(&sb.d_xq, sizeof(double) * D * nq);
  if (e == cudaSuccess) e = cudaMalloc(&d_x, sizeof(double) * D * N);
  if (e == cudaSuccess) e = cudaMalloc(&d_hp, sizeof(double) * P);
  if (e == cudaSuccess) e = cudaMemcpyAsync(sb.d_xe, xe, sizeof(double) * D * ne, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(sb.d_xq, xq, sizeof(double) * D * nq, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_x, x, sizeof(double) * D * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_hp, hp, sizeof(double) * P, cudaMemcpyHostToDevice, ctx->stream);
  rc = GPR_OK;
  if (e == cudaSuccess) {
    rc = split_build(ctx, spec, D, d_hp, sb.d_xe, ne, sb.d_xq, nq, d_x, N, N, sb);
    if (!rc) e = cudaMemcpyAsync(A, sb.A, sizeof(double) * ne * nq * nk, cudaMemcpyDeviceToHost, ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(B, sb.B, sizeof(double) * ne * N * nk, cudaMemcpyDeviceToHost, ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(C, sb.C, sizeof(double) * N * nq * nk, cudaMemcpyDeviceToHost, ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  cudaStreamSynchronize(ctx->stream);
  sb.release(); cudaFree(d_x); cudaFree(d_hp);
  if (rc) return rc;
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_split_kernel", __LINE__);
  return GPR_OK;
}

int gpr_split_predict(gpr_model* m, const double* xe, int64_t ne, const double* xq, int64_t nq, int64_t e_lo,
                      int64_t e_hi, double* mean, double* var) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!xe || !xq || !mean || ne < 1 || nq < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  if (!m->have_factor || m->factor_destroyed) return fail(ctx, GPR_ERR_STATE, "split predict: call gpr_update_cache first");
  if (m->ny != 1) return fail(ctx, GPR_ERR_UNSUPPORTED, "split predict needs a vector y (Diagonal(wt), src/split_predict.jl:13)");
  if (var && (e_lo < 1 || e_hi > ne || e_lo > e_hi + 1)) return fail(ctx, GPR_ERR_ARG, "var_range out of bounds");
  CK(cudaSetDevice(ctx->device));
  timer_reset_predict(m->tm);
  ctx->oz_active = m->oz;
  const int D = m->D, nk = m->nk;
  const int64_t N = m->N, Np = m->Np;
  const bool want_var = var != nullptr && e_hi >= e_lo;
  // Workspaces live in the model handle (the reference's GPRSplitPredictCache, src/caches/split_kernel.jl:1-30, is
  // allocated once per cache as well): no cudaMalloc / cudaFree on the path after the first call of a given shape.
  SplitBufs sb; sb.nep = round_up(ne, 128); sb.nqp = round_up(nq, 128);
  const int64_t nep = sb.nep, nqp = sb.nqp;
  int rc = ensure(ctx, m->w_sA, (size_t)nep * nqp * nk);
  if (!rc) rc = ensure(ctx, m->w_sBt, (size_t)Np * nep * nk);
  if (!rc) rc = ensure(ctx, m->w_sC, (size_t)Np * nqp * nk);
  if (!rc && want_var) rc = ensure(ctx, m->w_sCu, (size_t)Np * nqp * nk);
  if (!rc) rc = ensure(ctx, m->w_sx, (size_t)D * (ne + nq));
  if (!rc) rc = ensure(ctx, m->w_smu, (size_t)nep * nqp);
  if (rc) return rc;
  sb.A = m->w_sA.p; sb.Bt = m->w_sBt.p; sb.C = m->w_sC.p; sb.Cu = want_var ? m->w_sCu.p : nullptr; sb.C_row_scale = m->d_wt;
  sb.d_xe = m->w_sx.p; sb.d_xq = m->w_sx.p + (size_t)D * ne;
  double* d_mu = m->w_smu.p;
  CK(cudaMemcpyAsync(sb.d_xe, xe, sizeof(double) * D * ne, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(sb.d_xq, xq, sizeof(double) * D * nq, cudaMemcpyHostToDevice, ctx->stream));
  {
    // A, Bt = B^T (training index fastest), Cw = Diagonal(wt) * C[:, :, k] (split_predict.jl:13), and Cu for the variance
    Scope s(m->tm, GPR_T_SPLIT_BUILD, ctx->stream);
    rc = split_build(ctx, m->spec, D, m->d_hp, sb.d_xe, ne, sb.d_xq, nq, m->d_x, N, Np, sb);
    if (rc) return rc;
  }
  CudaBE be{ctx};
  // mu = sum_k A_k .* (B_k Cw_k)  (split_predict.jl:14-16): per component ONE T,N product Bt_k^T Cw_k whose epilogue
  // multiplies by A_k and accumulates into mu -- no BCw buffer, no separate Hadamard pass.  The columns are processed in
  // up to 4 chunks: the device -> host copy of a finished chunk (pageable destination: ~4 GB/s, it would otherwise add
  // 35 ms to a 64 ms product at ne = nq = 4096) runs on the side queue while the next chunk is being computed.
  const int nch = (nqp >= 1024 && (nqp / 128) % 4 == 0) ? 4 : 1;
  const int64_t cw = nqp / nch;
  if (!ctx->ev_chunk[0])
    for (int i = 0; i < 4; ++i) CK(cudaEventCreateWithFlags(&ctx->ev_chunk[i], cudaEventDisableTiming));
  {
    Scope s(m->tm, GPR_T_SPLIT_GEMM, ctx->stream);
    for (int ch = 0; ch < nch; ++ch) {
      const int64_t q0 = ch * cw;
      for (int k = 0; k < nk; ++k)
        be.gemm_hadamard(nep, cw, Np, sb.Bt + (int64_t)k * Np * nep, Np, sb.C + (int64_t)k * Np * nqp + q0 * Np, Np,
                         sb.A + (int64_t)k * nep * nqp + q0 * nep, nep, k == 0 ? 0.0 : 1.0, d_mu + q0 * nep, nep);
      CK(cudaEventRecord(ctx->ev_chunk[ch], ctx->stream));
    }
  }
  rc = check_pending(ctx, "split mean");
  if (rc) return rc;
  // Download: the caller's array is pageable (2-4 GB/s through the driver's bounce buffer -- 75 ms for 134 MB, longer than the
  // products since they moved to the INT8 tensor cores), so the chunks land in a pinned staging buffer of the context at PCIe speed
  // and the host copies each finished chunk on while the GPU computes the next one.  Falls back to the direct copy if the pinned
  // allocation fails or would exceed 1 GB.
  double* stage = ctx->host_stage((size_t)ne * (size_t)nq);
  if (stage && !ctx->ev_d2h[0])
    for (int i = 0; i < 4; ++i) CK(cudaEventCreateWithFlags(&ctx->ev_d2h[i], cudaEventDisableTiming));
  double* dst = stage ? stage : mean;
  int nsent = 0;
  {
    Scope s(m->tm, GPR_T_SPLIT_D2H, ctx->side_stream);
    for (int ch = 0; ch < nch; ++ch) {
      const int64_t q0 = ch * cw, qn = std::min<int64_t>(cw, nq - q0);
      if (qn <= 0) break;
      CK(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_chunk[ch], 0));
      CK(cudaMemcpy2DAsync(dst + q0 * ne, sizeof(double) * ne, d_mu + q0 * nep, sizeof(double) * nep, sizeof(double) * ne, qn,
                           cudaMemcpyDeviceToHost, ctx->side_stream));
      if (stage) CK(cudaEventRecord(ctx->ev_d2h[ch], ctx->side_stream));
      ++nsent;
    }
  }
  if (stage)
    for (int ch = 0; ch < nsent; ++ch) {
      const int64_t q0 = ch * cw, qn = std::min<int64_t>(cw, nq - q0);
      CK(cudaEventSynchronize(ctx->ev_d2h[ch]));
      memcpy(mean + q0 * ne, stage + q0 * ne, sizeof(double) * (size_t)ne * (size_t)qn);
    }
  CK(cudaStreamSynchronize(ctx->side_stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const double prior = prior_var(m->spec, m->hp_host.data());
  if (var) for (int64_t i = 0; i < ne * nq; ++i) var[i] = prior;   // fill!(Sigma.diag, sum sigma^2)  (src/predict.jl:55-58)
  if (want_var) {
    const int64_t EB = std::max<int64_t>(1, ctx->predict_tile / nqp);
    rc = ensure(ctx, m->w_kxp, (size_t)EB * nqp * Np);
    if (!rc) rc = ensure(ctx, m->w_var, (size_t)EB * nqp);
    if (rc) return rc;
    double* d_var = m->w_var.p;
    Blocked<CudaBE> blk(be, m->d_dinv);
    for (int64_t e0 = e_lo - 1; e0 < e_hi; e0 += EB) {
      const int64_t ec = std::min<int64_t>(EB, e_hi - e0);
      const int64_t rows = ec * nqp;
      {
        Scope s(m->tm, GPR_T_PRED_KSTAR, ctx->stream);
        // Kxq^T for the rows e0 .. e0+ec-1, training index fastest (split_predict.jl:44-47, transposed)
        split_assemble_t_kernel<<<(unsigned)std::min<int64_t>((rows * Np + 255) / 256, (int64_t)ctx->sm_count * 32), 256, 0, ctx->stream>>>(
            m->w_kxp.p, Np, sb.A, sb.Bt, sb.Cu, nep, nqp, Np, nk, e0, ec, ne, nq, N);
        ctx->launches++;
      }
      {
        Scope s(m->tm, GPR_T_PRED_TRSM, ctx->stream);
        blk.trsm_LUT(m->d_U, Np, Np, 0, m->w_kxp.p, Np, rows, 1.0);     // V^T = U^-T Kxq^T, T,N products
      }
      {
        Scope s(m->tm, GPR_T_PRED_ROWNORM, ctx->stream);
        colsumsq_kernel<<<(unsigned)rows, 256, 0, ctx->stream>>>(m->w_kxp.p, Np, Np, rows, prior, d_var);
        ctx->launches++;
      }
      rc = check_pending(ctx, "split variance");
      if (rc) return rc;
      // var[(e-1)*nq + q]  (q fastest within e: split_predict.jl:48)
      CK(cudaMemcpy2DAsync(var + e0 * nq, sizeof(double) * nq, d_var, sizeof(double) * nqp, sizeof(double) * nq, ec, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
    }
  }
  return GPR_OK;
}

// ---------------------------------------------------------------------------
// analytic integration over a box (src/integrate.jl, noise-free path)
// ---------------------------------------------------------------------------
int gpr_integrate(gpr_model* m, const double* a, const double* b, double* Iout, double* var_out) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!a || !b || !Iout) return fail(ctx, GPR_ERR_ARG, "NULL argument");
  if (!m->have_factor || m->factor_destroyed) return fail(ctx, GPR_ERR_STATE, "integrate: call gpr_update_cache first");
  if (m->spec.type[0] == KT_NOISE) return fail(ctx, GPR_ERR_UNSUPPORTED, "integrate: the first component must be a SquaredExp (antideriv!, src/integrate.jl:15)");
  CK(cudaSetDevice(ctx->device));
  const int D = m->D;
  const int64_t N = m->N, Np = m->Np;
  int rc = ensure(ctx, m->w_part, (size_t)Np + 2 * D + 2 + m->nyp);
  if (rc) return rc;
  double* d_k1 = m->w_part.p;
  double* d_ab = d_k1 + Np;            // a[D], b[D]
  double* d_sq = d_ab + 2 * D;         // |U^-T k1|^2
  double* d_I = d_sq + 2;              // nyp
  CK(cudaMemcpyAsync(d_ab, a, sizeof(double) * D, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_ab + D, b, sizeof(double) * D, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_I, 0, sizeof(double) * m->nyp, ctx->stream));
  rc = launch_antideriv(ctx, m->d_x, D, N, Np, m->d_hp, d_ab, d_ab + D, 1, 1, d_k1, Np);
  if (rc) return rc;
  CudaBE be{ctx};
  be.gemv('T', m->nyp, Np, 1.0, m->d_wt, Np, d_k1, d_I);          // Iout = wt' * k1   (mean_integ_impl!, :118-121)
  std::vector<double> hI((size_t)m->ny);
  CK(cudaMemcpyAsync(hI.data(), d_I, sizeof(double) * m->ny, cudaMemcpyDeviceToHost, ctx->stream));
  double hsq = 0.0;
  if (var_out) {
    Blocked<CudaBE> blk(be, m->d_dinv);
    blk.trsv_LUT(m->d_U, Np, Np, 0, d_k1, 1.0);                     // ldiv!(kchol.L, tt), L = U^T   (:133-134)
    sumsq_kernel<<<1, 1024, 0, ctx->stream>>>(d_k1, Np, d_sq);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&hsq, d_sq, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  rc = check_pending(ctx, "gpr_integrate");
  if (rc) return rc;
  for (int e = 0; e < m->ny; ++e) Iout[e] = hI[e];
  if (var_out) var_out[0] = antideriv2_se(m->hp_host.data(), a, b, D) - hsq;
  return GPR_OK;
}

// nbox boxes in tiles of predict_tile: one triangular solve with all of a tile's k1 columns instead of one trsv per box
int gpr_integrate_batch(gpr_model* m, int64_t nbox, const double* a, const double* b, double* Iout, double* var_out) {
  if (!m) return GPR_ERR_ARG;
  gpr_ctx* ctx = m->ctx;
  if (!a || !b || !Iout || nbox < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  if (!m->have_factor || m->factor_destroyed) return fail(ctx, GPR_ERR_STATE, "integrate: call gpr_update_cache first");
  if (m->spec.type[0] == KT_NOISE) return fail(ctx, GPR_ERR_UNSUPPORTED, "integrate: the first component must be a SquaredExp (antideriv!, src/integrate.jl:15)");
  CK(cudaSetDevice(ctx->device));
  timer_reset_predict(m->tm);
  const int D = m->D;
  const int64_t MT = std::min<int64_t>(ctx->predict_tile, round_up(nbox, 128));
  int rc = ensure(ctx, m->w_xp, (size_t)2 * D * MT);
  if (rc) return rc;
  double* d_a = m->w_xp.p;
  double* d_b = d_a + (size_t)D * MT;
  std::vector<double> hsq(var_out ? (size_t)MT : 0);
  for (int64_t m0 = 0; m0 < nbox; m0 += MT) {
    const int64_t mt = std::min(MT, nbox - m0);
    CK(cudaMemcpyAsync(d_a, a + m0 * D, sizeof(double) * D * mt, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_b, b + m0 * D, sizeof(double) * D * mt, cudaMemcpyHostToDevice, ctx->stream));
    rc = integrate_tile(m, d_a, d_b, mt, Iout + m0, nbox, var_out ? hsq.data() : nullptr);
    if (rc) return rc;
    if (var_out)   // k2 - |U^-T k1|^2, hsq holding the negated sum  (:131-136)
      for (int64_t i = 0; i < mt; ++i) var_out[m0 + i] = antideriv2_se(m->hp_host.data(), a + (m0 + i) * D, b + (m0 + i) * D, D) + hsq[i];
  }
  return GPR_OK;
}

// ---------------------------------------------------------------------------
// prior sampling (src/distributions.jl)
// ---------------------------------------------------------------------------
int gpr_sample_mvn(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, const double* hp, const double* x, int64_t N,
                   double shift, const double* z, const double* mu, double* out, int64_t* info) {
  if (!ctx) return GPR_ERR_ARG;
  if (!hp || !x || !z || !out || N < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  CK(cudaSetDevice(ctx->device));
  if (info) *info = 0;
  KSpec spec; int P = 0, nk = 0;
  int rc = make_spec(ctx, comp_types, ncomp, D, &spec, &P, &nk);
  if (rc) return rc;
  const int64_t Np = round_up(N, 128);
  double *d_x = nullptr, *d_hp = nullptr, *d_S = nullptr, *d_dinv = nullptr, *d_z = nullptr, *d_o = nullptr;
  cudaError_t e = cudaMalloc(&d_x, sizeof(double) * D * N);
  if (e == cudaSuccess) e = cudaMalloc(&d_hp, sizeof(double) * P);
  if (e == cudaSuccess) e = cudaMalloc(&d_S, sizeof(double) * Np * Np);
  if (e == cudaSuccess) e = cudaMalloc(&d_dinv, sizeof(double) * Np * 128);
  if (e == cudaSuccess) e = cudaMalloc(&d_z, sizeof(double) * Np);
  if (e == cudaSuccess) e = cudaMalloc(&d_o, sizeof(double) * Np);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_x, x, sizeof(double) * D * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_hp, hp, sizeof(double) * P, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_z, 0, sizeof(double) * Np, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_o, 0, sizeof(double) * Np, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_z, z, sizeof(double) * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && mu) e = cudaMemcpyAsync(d_o, mu, sizeof(double) * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_info, 0, sizeof(long long), ctx->stream);
  long long h_info = 0;
  rc = GPR_OK;
  if (e == cudaSuccess) {
    // Sigma (upper triangle, zero below: the product U^T z below then is a plain transposed matrix-vector product)
    KBuildArgs a{};
    a.out = d_S; a.ldo = Np; a.R = N; a.C = N; a.Rp = Np; a.Cp = Np;
    a.x1 = d_x; a.x2 = d_x; a.D = D; a.hp = d_hp; a.spec = spec;
    a.eps = 1e-8; a.same = 1; a.add_noise = 1; a.pad_identity = 1; a.zero_lower = 1; a.all_shift = shift;   // kernel(cov, theta, x): src/distributions.jl:43
    rc = launch_kbuild(ctx, DM_EUCLID, a, d_x);
    if (!rc) {
      CudaBE be{ctx};
      Blocked<CudaBE> blk(be, d_dinv);
      ctx->oz_active = ctx->ozaki > 0 ? ctx->ozaki : 0;
      blk.potrf(d_S, Np, Np, 0);                                  // Sigma = U^T U, L = U^T  (cholesky(Sigma .+ 1e-7), :25)
      be.gemv('T', Np, Np, 1.0, d_S, Np, d_z, d_o);               // out = mu + U^T z              (:32)
      e = cudaMemcpyAsync(&h_info, ctx->d_info, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_o, sizeof(double) * N, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      if (e == cudaSuccess) rc = check_pending(ctx, "gpr_sample_mvn");
    }
  }
  cudaStreamSynchronize(ctx->stream);
  cudaFree(d_x); cudaFree(d_hp); cudaFree(d_S); cudaFree(d_dinv); cudaFree(d_z); cudaFree(d_o);
  if (rc) return rc;
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_sample_mvn", __LINE__);
  if (info) *info = h_info;
  if (h_info != 0) return fail(ctx, GPR_ERR_NOT_POSDEF, "matrix is not positive definite; Cholesky failed at pivot " + std::to_string(h_info));
  return GPR_OK;
}

// ---------------------------------------------------------------------------
// diagnostics
// ---------------------------------------------------------------------------
int gpr_dbg_dgemm(gpr_ctx* ctx, char transA, char transB, int M, int N, int K, double alpha, const double* A,
                  int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int reps,
                  double* ms) {
  if (!ctx) return GPR_ERR_ARG;
  if (!A || !B || !C) return fail(ctx, GPR_ERR_ARG, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  const bool aT = (transA == 'T'), bT = (transB == 'T');
  const int64_t a_cols = aT ? M : K, b_cols = bT ? K : N;
  double *dA = nullptr, *dB = nullptr, *dC = nullptr, *dC0 = nullptr;
  cudaError_t e = cudaMalloc(&dA, sizeof(double) * lda * a_cols);
  if (e == cudaSuccess) e = cudaMalloc(&dB, sizeof(double) * ldb * b_cols);
  if (e == cudaSuccess) e = cudaMalloc(&dC, sizeof(double) * ldc * N);
  if (e == cudaSuccess) e = cudaMalloc(&dC0, sizeof(double) * ldc * N);
  // every copy goes through the library stream: a pageable cudaMemcpy on the legacy stream may still be
  // in flight when work on a non-blocking stream starts
  if (e == cudaSuccess) e = cudaMemcpyAsync(dA, A, sizeof(double) * lda * a_cols, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dB, B, sizeof(double) * ldb * b_cols, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dC0, C, sizeof(double) * ldc * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  float total = 0.f;
  if (e == cudaSuccess) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    if (reps < 1) reps = 1;
    for (int r = 0; r < reps && e == cudaSuccess; ++r) {
      e = cudaMemcpyAsync(dC, dC0, sizeof(double) * ldc * N, cudaMemcpyDeviceToDevice, ctx->stream);
      cudaEventRecord(e0, ctx->stream);
      if (e == cudaSuccess) {
        if (ctx->gemm_tma && gemm_tma_supported(transA, transB, M, N, K, dA, dB, dC, flags, 1, 0, 0))
          e = launch_dgemm128_tma(ctx->stream, M, N, K, alpha, dA, lda, dB, ldb, beta, dC, ldc, flags, 1, 0, 0, 0);
        else
          e = launch_dgemm128(ctx->stream, transA, transB, M, N, K, alpha, dA, lda, dB, ldb, beta, dC, ldc, flags, 1, 0, 0, 0,
                              nullptr, 0, 0, ctx->gemm_cfg);
      }
      ctx->launches++;
      cudaEventRecord(e1, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      float t = 0.f; cudaEventElapsedTime(&t, e0, e1);
      if (r > 0 || reps == 1) total += t;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e == cudaSuccess) e = cudaMemcpyAsync(C, dC, sizeof(double) * ldc * N, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  if (ms) *ms = total / (float)(reps > 1 ? reps - 1 : 1);
  cudaFree(dA); cudaFree(dB); cudaFree(dC); cudaFree(dC0);
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_dbg_dgemm", __LINE__);
  return GPR_OK;
}

int gpr_dbg_ozaki_dgemm(gpr_ctx* ctx, int M, int N, int K, int S, double alpha, const double* A, int64_t lda, const double* B, int64_t ldb,
                        double beta, double* C, int64_t ldc, int flags, int reps, double* ms) {
  if (!ctx) return GPR_ERR_ARG;
  if (!A || !B || !C) return fail(ctx, GPR_ERR_ARG, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  double *dA = nullptr, *dB = nullptr, *dC = nullptr, *dC0 = nullptr;
  void* ws = nullptr;
  cudaError_t e = cudaMalloc(&dA, sizeof(double) * lda * M);
  if (e == cudaSuccess) e = cudaMalloc(&dB, sizeof(double) * ldb * N);
  if (e == cudaSuccess) e = cudaMalloc(&dC, sizeof(double) * ldc * N);
  if (e == cudaSuccess) e = cudaMalloc(&dC0, sizeof(double) * ldc * N);
  if (e == cudaSuccess) e = cudaMalloc(&ws, oz_workspace_bytes(M, N, K, S));
  if (e == cudaSuccess) e = cudaMemcpyAsync(dA, A, sizeof(double) * lda * M, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dB, B, sizeof(double) * ldb * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dC0, C, sizeof(double) * ldc * N, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  float total = 0.f;
  if (e == cudaSuccess) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    if (reps < 1) reps = 1;
    for (int r = 0; r < reps && e == cudaSuccess; ++r) {
      e = cudaMemcpyAsync(dC, dC0, sizeof(double) * ldc * N, cudaMemcpyDeviceToDevice, ctx->stream);
      cudaEventRecord(e0, ctx->stream);
      if (e == cudaSuccess) e = launch_ozaki_dgemm(ctx->stream, M, N, K, S, alpha, dA, lda, dB, ldb, beta, dC, ldc, flags, ws);
      ctx->launches += 3;
      cudaEventRecord(e1, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      float t = 0.f; cudaEventElapsedTime(&t, e0, e1);
      if (r > 0 || reps == 1) total += t;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e == cudaSuccess) e = cudaMemcpyAsync(C, dC, sizeof(double) * ldc * N, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  if (ms) *ms = total / (float)(reps > 1 ? reps - 1 : 1);
  cudaFree(dA); cudaFree(dB); cudaFree(dC); cudaFree(dC0); cudaFree(ws);
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_dbg_ozaki_dgemm", __LINE__);
  return GPR_OK;
}

int gpr_dbg_factor(gpr_ctx* ctx, double* A, int64_t N, int mode, int64_t* info, double* ms) {
  if (!ctx) return GPR_ERR_ARG;
  if (!A || N < 1) return fail(ctx, GPR_ERR_ARG, "NULL or empty argument");
  CK(cudaSetDevice(ctx->device));
  const int64_t Np = round_up(N, 128);
  double *dA = nullptr, *dinv = nullptr;
  cudaError_t e = cudaMalloc(&dA, sizeof(double) * Np * Np);
  if (e == cudaSuccess) e = cudaMalloc(&dinv, sizeof(double) * Np * 128);
  int rc = GPR_OK;
  long long h_info = 0;
  float t = 0.f;
  if (e == cudaSuccess) {
    // identity padding
    std::vector<double> pad;
    if (Np != N) {
      pad.assign((size_t)Np * Np, 0.0);
      for (int64_t j = 0; j < N; ++j) memcpy(&pad[(size_t)j * Np], A + j * N, sizeof(double) * N);
      for (int64_t j = N; j < Np; ++j) pad[(size_t)j * Np + j] = 1.0;
      e = cudaMemcpyAsync(dA, pad.data(), sizeof(double) * Np * Np, cudaMemcpyHostToDevice, ctx->stream);
    } else {
      e = cudaMemcpyAsync(dA, A, sizeof(double) * Np * Np, cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_info, 0, sizeof(long long), ctx->stream);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    CudaBE be{ctx};
    Blocked<CudaBE> blk(be, dinv);
    blk.leaf_lookahead = ctx->leaf_lookahead != 0;
    ctx->oz_active = ctx->ozaki > 0 ? ctx->ozaki : 0;     // diagnostics: only a forced digit count
    double *dW = nullptr, *dC = nullptr;
    if (mode == 3) {
      if (e == cudaSuccess) e = cudaMalloc(&dW, sizeof(double) * Np * Np);
      if (e == cudaSuccess) e = cudaMalloc(&dC, sizeof(double) * Np * Np);
    }
    cudaEventRecord(e0, ctx->stream);
    blk.potrf(dA, Np, Np, 0);
    if (mode == 3 && e == cudaSuccess) {   // out-of-place inverse: W = U^-1 with clean diagonal blocks, C = W W^T, upper(C) -> upper(A)
      blk.trtri_t(dA, Np, dW, Np, Np, 0);
      blk.lauum_oop_t(dW, Np, Np, dC, Np);
    } else {
      if (mode >= 1) blk.trtri(dA, Np, Np, 0);
      if (mode >= 2) blk.lauum(dA, Np, Np, 0);
    }
    cudaEventRecord(e1, ctx->stream);
    if (mode == 3 && e == cudaSuccess) {
      dim3 grid((unsigned)((Np + 31) / 32), (unsigned)((Np + 31) / 32)), block(32, 8);
      copy_upper_kernel<<<grid, block, 0, ctx->stream>>>(dA, Np, dC, Np, Np);
      ctx->launches++;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_info, ctx->d_info, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaEventElapsedTime(&t, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(dW); cudaFree(dC);
    rc = check_pending(ctx, "gpr_dbg_factor");
    if (e == cudaSuccess && !rc) {
      e = cudaMemcpy2DAsync(A, sizeof(double) * N, dA, sizeof(double) * Np, sizeof(double) * N, N, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
  }
  cudaFree(dA); cudaFree(dinv);
  if (info) *info = h_info;
  if (ms) *ms = t;
  if (rc) return rc;
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gpr_dbg_factor", __LINE__);
  return h_info ? GPR_ERR_NOT_POSDEF : GPR_OK;
}

}  // extern "C"

#include "mgpu_api.inl"
