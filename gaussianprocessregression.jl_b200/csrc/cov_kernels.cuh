// Covariance-side kernels: fused covariance build (all components, jitter,
// noise, padding in one pass), dense dK/dtheta_i (API parity only), the
// split-kernel A/B/C builders, and the fused all-hyperparameter gradient
// reduction that replaces the reference's per-hyperparameter
// {materialise dK, dgemv, ddot} loop.
//
// Reference semantics restated here (parameterisation: SURVEY.md A.1-A.4):
//   /root/reference/src/covariance.jl:29-58,72-95     SE kernel, jitter iff x === xp
//   /root/reference/src/compose_covar.jl:47-77        sum over non-noise components, noise on the diagonal
//   /root/reference/src/deriv_covar.jl:20-32          dK/dsigma = (2/|sigma|) K (incl. jitter), dK/dl_d = -2 l_d K (x_d - x'_d)^2
//   /root/reference/src/loss_grad.jl:43-52            g_i = -1/2 (alpha^T dK alpha - <K^-1, dK>)
//   /root/reference/src/split_kernel.jl:108-123,151-159  split distances A / C and the A, B, C factors
// Matern-5/2 is an extension that does not exist in the reference (parity unpinned).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "fastexp.cuh"

namespace gpr {

constexpr int KSPEC_MAXC = 8;
enum KernType : int { KT_SE = 1, KT_NOISE = 2, KT_MATERN52 = 3 };
enum DistMode : int { DM_EUCLID = 0, DM_SPLIT_A = 1, DM_SPLIT_C = 2 };

struct KSpec {
  int ncomp;
  int type[KSPEC_MAXC];
  int hp_off[KSPEC_MAXC];   // offset of the component's first hyper-parameter in the global hp vector
};

struct KBuildArgs {
  double* out; long long ldo;
  long long R, C;        // valid rows / cols (rows index x1 points, cols index x2 points)
  long long Rp, Cp;      // padded extents actually written
  const double* x1; const double* x2;   // D x R, D x C column major (one point = D contiguous doubles)
  int D;
  const double* hp;      // device, global hp vector
  KSpec spec;
  double eps;            // jitter added per non-noise component where global row == global col (only if same != 0)
  int same;              // x1 and x2 are the same object (reference: x === xp)
  int add_noise;         // add sigma_n^2 (first noise component) on the diagonal (self covariance)
  int pad_identity;      // padded diagonal entries (row == col >= R) get 1.0
  int sigma_one;         // force sigma := 1 (split A and B factors)
  const double* row_scale;   // optional: multiply row r by row_scale[r] (Cw = diag(wt) C), may be null
  long long diag_shift;  // row r is "the same point" as col r + diag_shift (tiles of a larger problem)
  int zero_lower;        // entries strictly below that diagonal are written as 0 and not evaluated (block-cyclic
                         // multi-GPU layout: only the upper triangle is referenced, csrc/dist_blocked.hpp)
  // Fused posterior mean (mu = K* wt, src/predict.jl:73-76): when mean_w != nullptr every CTA also writes
  //   mean_partial[blockIdx.y * Rp + r] = sum over its 64 columns of out(r, c) * mean_w[c]
  // so the K* tile is never re-read for the mean (the partials are 1/64 of the tile).  out may then be nullptr
  // (mean-only prediction: K* is not stored at all).
  const double* mean_w;
  double* mean_partial;
  // The same for the TRANSPOSED layout out = K(x, xp) (rows = training points): mean_w_rows != nullptr makes every CTA
  // write mean_partial[blockIdx.x * Cp + c] = sum over its 64 rows of out(r, c) * mean_w_rows[r].
  const double* mean_w_rows;
  double all_shift;      // added to EVERY valid entry (prior sampling: `Sigma .+ 1e-7`, src/distributions.jl:25)
  int lower_only;        // write only the entries strictly below the diagonal (fills in what a zero_lower build left out)
};

constexpr int KB_TILE = 64;
constexpr int KB_THREADS = 256;

__device__ __forceinline__ double kern_value(int type, double sig2, double dist) {
  if (type == KT_SE) return sig2 * exp(-dist);
  const double r = sqrt(dist > 0.0 ? dist : 0.0);
  const double s5r = 2.23606797749978969640917366873128 * r;
  return sig2 * (1.0 + s5r + (5.0 / 3.0) * dist) * exp(-s5r);
}

// Coordinates per chunk of the wide covariance build and the pitch of its d-major point tiles (odd in doubles: the
// staging stores, consecutive coordinates of one point, fall in distinct banks).
constexpr int KBW_DC = 32;
constexpr int KBW_P = KB_TILE + 1;

// out[r + c*ldo] = sum_comp k_comp(x1[:,r], x2[:,c]) (+ jitter, + noise, padding)
// WIDE = false: smem xs1[nk][D][64], xs2[nk][D][64] = inverse-length-scaled coordinates (the reference
// scales x by l before taking differences: covariance.jl:90-92), all staged at once.
// WIDE = true (the wide build): one component at a time, its scaled coordinates staged KBW_DC at a time
// (smem xs1[KBW_DC][KBW_P], xs2[KBW_DC][KBW_P]), distances accumulated in registers in the same order over d, so any D
// and any number of components fit.
template <int MODE, bool WIDE = false>
__global__ void __launch_bounds__(KB_THREADS) kbuild_kernel(const KBuildArgs a) {
  extern __shared__ __align__(16) double kb_smem[];
  const int D = a.D;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long r0 = (long long)blockIdx.x * KB_TILE, c0 = (long long)blockIdx.y * KB_TILE;

  if (a.lower_only && r0 + (KB_TILE - 1) <= c0 + a.diag_shift) return;   // tile entirely on / above the diagonal
  if (a.zero_lower && r0 > c0 + a.diag_shift + (KB_TILE - 1)) {   // tile entirely below the diagonal
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long r = r0 + tx + 16 * i, c = c0 + ty + 16 * j;
        if (r < a.Rp && c < a.Cp) a.out[r + c * a.ldo] = 0.0;
      }
    return;
  }

  // non-noise components
  int kidx[KSPEC_MAXC]; int nk = 0;
#pragma unroll
  for (int c = 0; c < KSPEC_MAXC; ++c)
    if (c < a.spec.ncomp && a.spec.type[c] != KT_NOISE) kidx[nk++] = c;

  double* xs1 = kb_smem;
  double* xs2 = WIDE ? kb_smem + (size_t)KBW_DC * KBW_P : kb_smem + (size_t)nk * D * KB_TILE;
  if constexpr (!WIDE) {
    for (int idx = tid; idx < nk * D * KB_TILE; idx += KB_THREADS) {
      const int p = idx % KB_TILE, d = (idx / KB_TILE) % D, k = idx / (KB_TILE * D);
      const double l = a.hp[a.spec.hp_off[kidx[k]] + 1 + d];
      const long long r = r0 + p, c = c0 + p;
      xs1[idx] = (r < a.R) ? a.x1[d + r * D] * l : 0.0;
      xs2[idx] = (c < a.C) ? a.x2[d + c * D] * l : 0.0;
    }
    __syncthreads();
  }

  double sum[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) sum[i][j] = 0.0;

  for (int k = 0; k < nk; ++k) {
    const int comp = kidx[k];
    const double sg = a.sigma_one ? 1.0 : a.hp[a.spec.hp_off[comp]];
    const double sig2 = sg * sg;
    double dist[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dist[i][j] = 0.0;
    if constexpr (!WIDE) {
      const double* p1 = xs1 + (size_t)k * D * KB_TILE;
      const double* p2 = xs2 + (size_t)k * D * KB_TILE;
      for (int d = 0; d < D; ++d) {
        double u[4], v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) u[i] = p1[d * KB_TILE + tx + 16 * i];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = p2[d * KB_TILE + ty + 16 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (MODE == DM_EUCLID) { const double df = u[i] - v[j]; dist[i][j] += df * df; }
            else if (MODE == DM_SPLIT_A) dist[i][j] += v[j] * v[j] + 2.0 * u[i] * v[j];   // split_kernel.jl:114
            else dist[i][j] += -2.0 * u[i] * v[j];                                       // split_kernel.jl:121
          }
      }
    } else {
      const double* lsc = a.hp + a.spec.hp_off[comp] + 1;
      for (int d0 = 0; d0 < D; d0 += KBW_DC) {
        const int nd = D - d0 < KBW_DC ? D - d0 : KBW_DC;
        __syncthreads();   // the previous chunk has been read
        // consecutive threads read consecutive coordinates of one point (coalesced)
        for (int idx = tid; idx < 2 * KB_TILE * KBW_DC; idx += KB_THREADS) {
          const int d = idx % KBW_DC, p = (idx / KBW_DC) % KB_TILE;
          if (d >= nd) continue;
          if (idx < KB_TILE * KBW_DC) {
            const long long r = r0 + p;
            xs1[d * KBW_P + p] = (r < a.R) ? a.x1[d0 + d + r * D] * lsc[d0 + d] : 0.0;
          } else {
            const long long c = c0 + p;
            xs2[d * KBW_P + p] = (c < a.C) ? a.x2[d0 + d + c * D] * lsc[d0 + d] : 0.0;
          }
        }
        __syncthreads();
        for (int d = 0; d < nd; ++d) {   // the same arithmetic as above, in the same order over d
          double u[4], v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) u[i] = xs1[d * KBW_P + tx + 16 * i];
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = xs2[d * KBW_P + ty + 16 * j];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (MODE == DM_EUCLID) { const double df = u[i] - v[j]; dist[i][j] += df * df; }
              else if (MODE == DM_SPLIT_A) dist[i][j] += v[j] * v[j] + 2.0 * u[i] * v[j];
              else dist[i][j] += -2.0 * u[i] * v[j];
            }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        double kv = kern_value(a.spec.type[comp], sig2, dist[i][j]);
        const long long r = r0 + tx + 16 * i, c = c0 + ty + 16 * j;
        if (a.same && r == c + a.diag_shift) kv += a.eps;
        sum[i][j] += kv;
      }
  }

  double noise2 = 0.0;
  if (a.add_noise) {
    for (int c = 0; c < a.spec.ncomp; ++c)
      if (a.spec.type[c] == KT_NOISE) { const double s = a.hp[a.spec.hp_off[c]]; noise2 = s * s; break; }   // findfirst: compose_covar.jl:65
  }
  double msum[4] = {0.0, 0.0, 0.0, 0.0};   // per row (mean_w) or per column (mean_w_rows) of this thread's 4 x 4 patch
  double wr[4] = {0.0, 0.0, 0.0, 0.0};
  if (a.mean_w_rows) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { const long long r = r0 + tx + 16 * i; wr[i] = (r < a.R) ? a.mean_w_rows[r] : 0.0; }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long long c = c0 + ty + 16 * j;
    const double wc = (a.mean_w && c < a.C) ? a.mean_w[c] : 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long r = r0 + tx + 16 * i;
      if (r >= a.Rp || c >= a.Cp) continue;
      if (a.lower_only && r <= c + a.diag_shift) continue;
      double v;
      if (r < a.R && c < a.C) {
        v = sum[i][j];
        if (a.add_noise && r == c + a.diag_shift) v += noise2;
        if (a.row_scale) v *= a.row_scale[r];
        v += a.all_shift;
      } else {
        v = (a.pad_identity && r == c + a.diag_shift) ? 1.0 : 0.0;
      }
      if (a.zero_lower && r > c + a.diag_shift) v = 0.0;
      if (a.out) a.out[r + c * a.ldo] = v;
      if (a.mean_w_rows) msum[j] += v * wr[i]; else msum[i] += v * wc;
    }
  }
  if (a.mean_w_rows) {
    // 16 threads (tx = 0..15) hold partial sums of the same column: reduce through shared memory in a fixed order
    __syncthreads();
    double* red = kb_smem;                 // [16][65]: the 16 writers of one column differ in tx -> odd row stride, no bank conflict
#pragma unroll
    for (int j = 0; j < 4; ++j) red[tx * (KB_TILE + 1) + ty + 16 * j] = msum[j];
    __syncthreads();
    if (tid < KB_TILE) {
      double sacc = 0.0;
#pragma unroll
      for (int q = 0; q < 16; ++q) sacc += red[q * (KB_TILE + 1) + tid];
      const long long c = c0 + tid;
      if (c < a.Cp) a.mean_partial[(long long)blockIdx.x * a.Cp + c] = sacc;
    }
    return;
  }
  if (a.mean_w) {
    // 16 threads (ty = 0..15) hold partial sums of the same row: reduce through shared memory in a fixed order
    __syncthreads();                       // xs1 / xs2 are dead from here on
    double* red = kb_smem;                 // [16][64]
#pragma unroll
    for (int i = 0; i < 4; ++i) red[ty * KB_TILE + tx + 16 * i] = msum[i];
    __syncthreads();
    if (tid < KB_TILE) {
      double s = 0.0;
#pragma unroll
      for (int q = 0; q < 16; ++q) s += red[q * KB_TILE + tid];
      const long long r = r0 + tid;
      if (r < a.Rp) a.mean_partial[(long long)blockIdx.y * a.Rp + r] = s;
    }
  }
}

// dynamic shared memory of kbuild_kernel<MODE, true> (the fused-mean reductions reuse the point tiles)
constexpr size_t KBW_SMEM_BYTES = (size_t)2 * KBW_DC * KBW_P * sizeof(double);
static_assert(KBW_SMEM_BYTES >= (size_t)16 * (KB_TILE + 1) * sizeof(double), "fused-mean reduction buffer");

// Dense dK/dtheta for ONE non-noise component (API parity with grad(cov,i,hp,x):
// /root/reference/src/deriv_covar.jl:2-29).  li = local hyper-parameter index
// (0 = sigma, d+1 = l_d).  The product path never materialises this matrix.
struct KGradArgs {
  double* out; long long ldo; long long N;
  const double* x; int D;
  const double* hp;   // device, hp of this component only: [sigma, l_1..l_D]
  int type; int li; double eps;
};

__global__ void __launch_bounds__(256) kgrad_dense_kernel(const KGradArgs a) {
  const long long total = a.N * a.N;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx % a.N, c = idx / a.N;
    double dist = 0.0;
    for (int d = 0; d < a.D; ++d) {
      const double l = a.hp[1 + d];
      const double df = a.x[d + r * a.D] * l - a.x[d + c * a.D] * l;
      dist += df * df;
    }
    const double sg = a.hp[0];
    double v;
    if (a.li == 0) {
      double kv = kern_value(a.type, sg * sg, dist);
      if (r == c) kv += a.eps;
      v = (2.0 / fabs(sg)) * kv;
    } else {
      const int d = a.li - 1;
      const double dx = a.x[d + r * a.D] - a.x[d + c * a.D];
      if (a.type == KT_SE) {
        double kv = sg * sg * exp(-dist);
        if (r == c) kv += a.eps;
        v = -2.0 * a.hp[a.li] * kv * (dx * dx);
      } else {
        const double rr = sqrt(dist);
        const double s5r = 2.23606797749978969640917366873128 * rr;
        v = -(5.0 / 3.0) * sg * sg * (1.0 + s5r) * exp(-s5r) * a.hp[a.li] * (dx * dx);
      }
    }
    a.out[r + c * a.ldo] = v;
  }
}

// ---------------------------------------------------------------------------
// Fused gradient reduction.  One pass over the upper triangle of K^-1:
//   acc_sigma[c]   = sum_{a,b} (alpha_a alpha_b - Kinv_ab) * Kc_ab            (Kc incl. jitter on the diagonal)
//   acc_len[c][d]  = sum_{a,b} (alpha_a alpha_b - Kinv_ab) * KL_ab (x_da - x_db)^2,  dKc/dl_d = -2 l_d KL (x_da-x_db)^2
//   acc_diag       = sum_a     (alpha_a^2 - Kinv_aa)
// with every off-diagonal pair counted twice (symmetry).  dK is never
// materialised.  Per-thread accumulators live in shared memory
// (slot-major, thread-minor: conflict free) so that P is a run-time value.
// Output: partial[block][slot], slot in [0, P] (slot P = acc_diag), reduced by
// grad_finalize_kernel in a fixed order.
// ---------------------------------------------------------------------------
struct GradArgs {
  const double* Kinv; long long ld;
  const double* alpha; const double* x; int D; long long N;
  const double* hp; KSpec spec; int P; double eps;
  double* partial;   // gridDim.x * (P+1)
  // DIST form (block-cyclic multi-GPU layout): Kinv holds this rank's block columns only
  int G, rank;           // local block column lb is global block column DistLayout::gblock(rank, lb)
  int nbt;               // 64-tiles per block column (nb / 64)
  long long lcol_tiles;  // local 64-tile columns (matrix columns only)
};

constexpr int GR_TILE = 64;
constexpr int GR_THREADS = 256;

template <bool DIST>
__global__ void __launch_bounds__(GR_THREADS) grad_reduce_kernel(const GradArgs a) {
  extern __shared__ __align__(16) double gr_smem[];
  const int D = a.D, P = a.P;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  double* acc = gr_smem;                                   // (P+1) * 256
  double* x1 = gr_smem + (size_t)(P + 1) * GR_THREADS;     // D * 64
  double* x2 = x1 + (size_t)D * GR_TILE;                   // D * 64
  double* al1 = x2 + (size_t)D * GR_TILE;                  // 64
  double* al2 = al1 + GR_TILE;                             // 64
  double* etab = al2 + GR_TILE;                            // 32: 2^(j/32) (fastexp.cuh)
  if (tid < 32) etab[tid] = kg_exp2_tab[tid];
  for (int s = 0; s <= P; ++s) acc[s * GR_THREADS + tid] = 0.0;

  const long long T = (a.N + GR_TILE - 1) / GR_TILE;
  const long long ntiles = DIST ? T * a.lcol_tiles : T * (T + 1) / 2;
  for (long long lin = blockIdx.x; lin < ntiles; lin += gridDim.x) {
    long long ti, tj, lc0;   // tile row, GLOBAL tile column, first column of the tile inside Kinv
    if (DIST) {
      const long long ltj = lin / T;
      ti = lin % T;
      const long long lb = ltj / a.nbt;   // local block column -> global block column (DistLayout::gblock, snake order)
      tj = (lb * a.G + ((lb & 1) ? a.G - 1 - a.rank : a.rank)) * a.nbt + ltj % a.nbt;
      lc0 = ltj * GR_TILE;
      if (ti > tj || tj >= T) continue;   // block uniform
    } else {
      tj = (long long)((sqrt(8.0 * (double)lin + 1.0) - 1.0) * 0.5);
      while (tj * (tj + 1) / 2 > lin) --tj;
      while ((tj + 1) * (tj + 2) / 2 <= lin) ++tj;
      ti = lin - tj * (tj + 1) / 2;
      lc0 = tj * GR_TILE;
    }
    const long long r0 = ti * GR_TILE, c0 = tj * GR_TILE;
    __syncthreads();
    for (int idx = tid; idx < D * GR_TILE; idx += GR_THREADS) {
      const int p = idx % GR_TILE, d = idx / GR_TILE;
      x1[idx] = (r0 + p < a.N) ? a.x[d + (r0 + p) * D] : 0.0;
      x2[idx] = (c0 + p < a.N) ? a.x[d + (c0 + p) * D] : 0.0;
    }
    if (tid < GR_TILE) al1[tid] = (r0 + tid < a.N) ? a.alpha[r0 + tid] : 0.0;
    else if (tid < 2 * GR_TILE) al2[tid - GR_TILE] = (c0 + tid - GR_TILE < a.N) ? a.alpha[c0 + tid - GR_TILE] : 0.0;
    __syncthreads();

    double wm[4][4];   // weight * (alpha_a alpha_b - Kinv_ab)
    double dsum = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long r = r0 + tx + 16 * i, c = c0 + ty + 16 * j;
        double v = 0.0;
        if (r < a.N && c < a.N && r <= c) {
          const double m = al1[tx + 16 * i] * al2[ty + 16 * j] - a.Kinv[r + (lc0 + ty + 16 * j) * a.ld];
          if (r == c) { v = m; dsum += m; } else v = 2.0 * m;
        }
        wm[i][j] = v;
      }
    acc[P * GR_THREADS + tid] += dsum;

    for (int comp = 0; comp < a.spec.ncomp; ++comp) {
      const int type = a.spec.type[comp];
      if (type == KT_NOISE) continue;
      const int off = a.spec.hp_off[comp];
      const double sg = a.hp[off];
      const double sig2 = sg * sg;
      double dist[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dist[i][j] = 0.0;
      for (int d = 0; d < D; ++d) {
        const double l = a.hp[off + 1 + d];
        double u[4], v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) u[i] = x1[d * GR_TILE + tx + 16 * i] * l;
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = x2[d * GR_TILE + ty + 16 * j] * l;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) { const double df = u[i] - v[j]; dist[i][j] += df * df; }
      }
      // valL reuses dist's registers: dist -> wm * KL ; the sigma sum is reduced on the fly
      double ssum = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const long long r = r0 + tx + 16 * i, c = c0 + ty + 16 * j;
          double kc, kl;
          if (type == KT_SE) {
            kc = sig2 * exp_tab32(-dist[i][j], etab);
            if (r == c) kc += a.eps;        // dK/dsigma and dK/dl both use the jittered K (deriv_covar.jl:23,26)
            kl = kc;
          } else {
            const double rr = sqrt(dist[i][j]);
            const double s5r = 2.23606797749978969640917366873128 * rr;
            const double e = exp_tab32(-s5r, etab);
            kc = sig2 * (1.0 + s5r + (5.0 / 3.0) * dist[i][j]) * e;
            if (r == c) kc += a.eps;
            kl = (5.0 / 6.0) * sig2 * (1.0 + s5r) * e;
          }
          ssum += wm[i][j] * kc;
          dist[i][j] = wm[i][j] * kl;
        }
      acc[off * GR_THREADS + tid] += ssum;
      for (int d = 0; d < D; ++d) {
        double u[4], v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) u[i] = x1[d * GR_TILE + tx + 16 * i];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = x2[d * GR_TILE + ty + 16 * j];
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) { const double df = u[i] - v[j]; s += dist[i][j] * (df * df); }
        acc[(off + 1 + d) * GR_THREADS + tid] += s;
      }
    }
  }
  __syncthreads();
  // block reduction per slot (fixed order), one warp per slot round-robin
  const int lane = tid & 31, warp = tid >> 5;
  for (int s = warp; s <= P; s += GR_THREADS / 32) {
    double v = 0.0;
    for (int q = lane; q < GR_THREADS; q += 32) v += acc[s * GR_THREADS + q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) a.partial[(size_t)blockIdx.x * (P + 1) + s] = v;
  }
}

// G[p] from the block partials.  sigma: -acc/|sigma| ; l_d: +l_d * acc ; noise: -sigma_n * acc_diag
// (loss_grad.jl:43-52 with deriv_covar.jl:23,26,31).  log_scale: G .*= hp (cost.jl:65).
// Every thread sums the slots it needs over the blocks in block order, so any P is taken.
__global__ void grad_finalize_kernel(const double* __restrict__ partial, int nblocks, int P, const double* __restrict__ hp,
                                     KSpec spec, int D, int log_scale, double* __restrict__ G) {
  auto tot = [&](int s) {
    double v = 0.0;
    for (int b = 0; b < nblocks; ++b) v += partial[(size_t)b * (P + 1) + s];
    return v;
  };
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    int c = 0;
    while (c + 1 < spec.ncomp && spec.hp_off[c + 1] <= p) ++c;
    const int off = spec.hp_off[c];
    double v;
    if (spec.type[c] == KT_NOISE) v = -hp[off] * tot(P);
    else if (p == off) v = -tot(off) / fabs(hp[off]);
    else v = hp[p] * tot(p);
    if (log_scale) v *= hp[p];
    G[p] = v;
  }
}

// ---------------------------------------------------------------------------
// Streaming reductions of the prediction path.
// ---------------------------------------------------------------------------
// out[r*ostride] = base - sign * sum_split partial[split][r]  (r < rows_valid)
__global__ void rowreduce_finalize_kernel(const double* __restrict__ partial, int nsplit, long long rows_pad,
                                          long long rows_valid, double base, double sign, double* __restrict__ out) {
  const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (r >= rows_valid) return;
  double s = 0.0;
  for (int q = 0; q < nsplit; ++q) s += partial[(size_t)q * rows_pad + r];
  out[r] = base + sign * s;
}

// out[c] = base - sum_r V[r + c*ld]^2 for the columns of an (rows x cols) column-major matrix (V^T = U^-T K*^T: the
// posterior variance of test point c, predict.jl:91-93).  One CTA per column, 16-byte streaming loads, fixed order.
__global__ void __launch_bounds__(256) colsumsq_kernel(const double* __restrict__ V, long long ld, long long rows,
                                                       long long cols_valid, double base, double* __restrict__ out) {
  __shared__ double red[256];
  const long long c = blockIdx.x;
  if (c >= cols_valid) return;
  const double2* p = reinterpret_cast<const double2*>(V + c * ld);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  const long long n2 = rows >> 1;
  long long i = threadIdx.x;
  for (; i + 768 < n2; i += 1024) {
    const double2 a = __ldcs(p + i), b = __ldcs(p + i + 256), cc = __ldcs(p + i + 512), d = __ldcs(p + i + 768);
    s0 += a.x * a.x + a.y * a.y; s1 += b.x * b.x + b.y * b.y; s2 += cc.x * cc.x + cc.y * cc.y; s3 += d.x * d.x + d.y * d.y;
  }
  for (; i < n2; i += 256) { const double2 a = __ldcs(p + i); s0 += a.x * a.x + a.y * a.y; }
  red[threadIdx.x] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[c] = base - red[0];
}

// mu[r + c*ldm] += A[r + c*lda] * T[r + c*ldt]   (split mean: BCw .*= A ; mu .+= BCw, split_predict.jl:15-16)
__global__ void hadamard_acc_kernel(double* __restrict__ mu, long long ldm, const double* __restrict__ A, long long lda,
                                    const double* __restrict__ T, long long ldt, long long rows, long long cols, int first) {
  const long long total = rows * cols;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx % rows, c = idx / rows;
    const double v = A[r + c * lda] * T[r + c * ldt];
    if (first) mu[r + c * ldm] = v; else mu[r + c * ldm] += v;
  }
}

// Kxq[(e - e0)*nqp + q, s] = sum_k A[e,q,k] * B[e,s,k] * Ct[q,s,k]
// (split_predict.jl:44-47).  A: nep x nqp x k, B: nep x Np x k, Ct: nqp x Np x k (C transposed).
__global__ void split_assemble_kernel(double* __restrict__ out, long long ldo, const double* __restrict__ A,
                                      const double* __restrict__ B, const double* __restrict__ Ct, long long nep,
                                      long long nqp, long long Np, int nk, long long e0, long long ecount,
                                      long long ne_valid, long long nq_valid, long long N_valid) {
  const long long rows = ecount * nqp;
  const long long total = rows * Np;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx % rows, s = idx / rows;
    const long long q = r % nqp, e = e0 + r / nqp;
    double v = 0.0;
    if (e < ne_valid && q < nq_valid && s < N_valid) {
      for (int k = 0; k < nk; ++k)
        v += A[e + q * nep + (long long)k * nep * nqp] * B[e + s * nep + (long long)k * nep * Np] *
             Ct[q + s * nqp + (long long)k * nqp * Np];
    }
    out[r + s * ldo] = v;
  }
}

// The same block TRANSPOSED (training index fastest), which is what the T,N triangular solve wants:
//   out[s + ((e - e0)*nqp + q)*ldo] = sum_k A[e,q,k] * Bt[s,e,k] * Cu[s,q,k]
// Bt: Np x nep x k (B transposed), Cu: Np x nqp x k (C, not scaled by wt).  All three reads and the write are coalesced in s.
__global__ void split_assemble_t_kernel(double* __restrict__ out, long long ldo, const double* __restrict__ A,
                                        const double* __restrict__ Bt, const double* __restrict__ Cu, long long nep,
                                        long long nqp, long long Np, int nk, long long e0, long long ecount,
                                        long long ne_valid, long long nq_valid, long long N_valid) {
  const long long rows = ecount * nqp;
  const long long total = rows * Np;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long s = idx % Np, r = idx / Np;
    const long long q = r % nqp, e = e0 + r / nqp;
    double v = 0.0;
    if (e < ne_valid && q < nq_valid && s < N_valid) {
      for (int k = 0; k < nk; ++k)
        v += A[e + q * nep + (long long)k * nep * nqp] * Bt[s + e * Np + (long long)k * Np * nep] *
             Cu[s + q * Np + (long long)k * Np * nqp];
    }
    out[s + r * ldo] = v;
  }
}

// ---------------------------------------------------------------------------
// Analytic integration of the posterior over a box (SURVEY.md 8f row 3, noise-free path):
//   k1[j] = sigma^2 (sqrt(pi)/2)^D prod_i (1/l_i) * prod_i erf(l_i (a_i - x_ij), l_i (b_i - x_ij))
// (antideriv!, /root/reference/src/integrate.jl:15-31).  erf(x, y) = erf(y) - erf(x) evaluated the way
// SpecialFunctions.jl does (erfc differences when both arguments lie on the same side, no cancellation).
// ---------------------------------------------------------------------------
__device__ __forceinline__ double erf_between(double x, double y) {
  const double r = 0.70710678118654752440;
  if (fabs(x) <= r && fabs(y) <= r) return erf(y) - erf(x);
  if (x >= 0.0 && y >= 0.0) return erfc(x) - erfc(y);
  if (x <= 0.0 && y <= 0.0) return erfc(-y) - erfc(-x);
  return erf(y) - erf(x);
}

// hp: [sigma, l_1..l_D] (the first D + 1 hyper-parameters of the model, as the reference reads them).
// k1 tile (np x mtp, ld ldk, training index fastest): column c is k1 of box c, bounds a[i + c D], b[i + c D] (D x nbox);
// rows >= n (padding of the factor) and columns >= nbox (padding of the tile) are zero.  Threads run along the training
// index (coalesced stores); each CTA stages ANTIDERIV_BOXES boxes' bounds in shared memory (2 D ANTIDERIV_BOXES doubles of
// dynamic shared memory) and walks the box chunks blockIdx.y, blockIdx.y + gridDim.y, ...
// CHUNKED: the bounds are staged ANTIDERIV_DCH coordinates at a time (2 ANTIDERIV_DCH ANTIDERIV_BOXES doubles), the
// products carried in registers across the chunks in the same order over i, for D whose bounds exceed shared memory.
constexpr int ANTIDERIV_BOXES = 8;
constexpr int ANTIDERIV_DCH = 1024;
template <bool CHUNKED = false>
__global__ void __launch_bounds__(256) antideriv_se_kernel(const double* __restrict__ x, int D, long long n, long long np,
                                                           const double* __restrict__ hp, const double* __restrict__ a,
                                                           const double* __restrict__ b, long long nbox, long long mtp,
                                                           double* __restrict__ k1, long long ldk) {
  extern __shared__ double sab[];   // [a | b] of the chunk, D x ANTIDERIV_BOXES each
  const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if constexpr (!CHUNKED) {
    const int nab = D * ANTIDERIV_BOXES;
    for (long long c0 = (long long)blockIdx.y * ANTIDERIV_BOXES; c0 < mtp; c0 += (long long)gridDim.y * ANTIDERIV_BOXES) {
      __syncthreads();
      for (int t = threadIdx.x; t < 2 * nab; t += blockDim.x) {
        const long long o = c0 * D + (t % nab);
        sab[t] = o < nbox * D ? (t < nab ? a[o] : b[o]) : 0.0;
      }
      __syncthreads();
      if (j >= np) continue;
      for (int cc = 0; cc < ANTIDERIV_BOXES && c0 + cc < mtp; ++cc) {
        const long long c = c0 + cc;
        double out = 0.0;
        if (j < n && c < nbox) {
          const double* ac = sab + cc * D;
          const double* bc = sab + nab + cc * D;
          double prefac = hp[0] * hp[0], v = 1.0;
          for (int i = 0; i < D; ++i) {
            const double l = hp[1 + i], xij = x[i + j * D];
            prefac *= 0.88622692545275801365 / l;
            v *= erf_between(l * (ac[i] - xij), l * (bc[i] - xij));
          }
          out = v * prefac;
        }
        k1[j + c * ldk] = out;
      }
    }
  } else {
    const int nab = ANTIDERIV_DCH * ANTIDERIV_BOXES;   // sab: a[cc][i], b[cc][i] of coordinates d0 + i
    for (long long c0 = (long long)blockIdx.y * ANTIDERIV_BOXES; c0 < mtp; c0 += (long long)gridDim.y * ANTIDERIV_BOXES) {
      double prefac[ANTIDERIV_BOXES], v[ANTIDERIV_BOXES];
#pragma unroll
      for (int cc = 0; cc < ANTIDERIV_BOXES; ++cc) { prefac[cc] = hp[0] * hp[0]; v[cc] = 1.0; }
      for (int d0 = 0; d0 < D; d0 += ANTIDERIV_DCH) {
        const int nd = D - d0 < ANTIDERIV_DCH ? D - d0 : ANTIDERIV_DCH;
        __syncthreads();
        for (int t = threadIdx.x; t < 2 * nab; t += blockDim.x) {
          const int cc = (t % nab) / ANTIDERIV_DCH, i = t % ANTIDERIV_DCH;
          const long long c = c0 + cc;
          sab[t] = (i < nd && c < nbox) ? (t < nab ? a : b)[c * D + d0 + i] : 0.0;
        }
        __syncthreads();
        if (j >= n) continue;
#pragma unroll
        for (int cc = 0; cc < ANTIDERIV_BOXES; ++cc) {
          if (c0 + cc >= nbox) continue;
          const double* ac = sab + cc * ANTIDERIV_DCH;
          const double* bc = sab + nab + cc * ANTIDERIV_DCH;
          for (int i = 0; i < nd; ++i) {
            const double l = hp[1 + d0 + i], xij = x[d0 + i + j * D];
            prefac[cc] *= 0.88622692545275801365 / l;
            v[cc] *= erf_between(l * (ac[i] - xij), l * (bc[i] - xij));
          }
        }
      }
      if (j >= np) continue;
#pragma unroll
      for (int cc = 0; cc < ANTIDERIV_BOXES; ++cc) {
        const long long c = c0 + cc;
        if (c >= mtp) break;
        k1[j + c * ldk] = (j < n && c < nbox) ? v[cc] * prefac[cc] : 0.0;
      }
    }
  }
}

// out[0] = sum_i v[i]^2 over n entries; one CTA, fixed order
__global__ void __launch_bounds__(1024, 1) sumsq_kernel(const double* __restrict__ v, long long n, double* __restrict__ out) {
  __shared__ double red[1024];
  double s = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s += v[i] * v[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}

}  // namespace gpr
