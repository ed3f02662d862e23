// Fused gradient reduction for wide models: the contract of grad_reduce_kernel (same tile enumeration, same
// partial[block][P+1] output) with O(P) state per CTA instead of one shared-memory accumulator per hyper-parameter and
// thread, and without a whole point tile in shared memory, so that any D and any number of components fit.
//
// Per 64 x 64 tile (rows a of the tile row, columns b of the tile column, upper triangle of K^-1 only) and per non-noise
// component, with u_a = x_a - x_0 and v_b = x_b - x_0 the coordinates centred on the first training point and l the
// component's inverse length scales:
//   W_ab  = w_ab (alpha_a alpha_b - Kinv_ab)      w = 1 on the diagonal, 2 above it, 0 below it and in the padding
//   r2_ab = |l u_a|^2 + |l v_b|^2 - 2 (l u_a).(l v_b)   Gram product on the DMMA pipe over D in chunks (r2_aa := 0)
//   sigma sum  += sum_ab W_ab Kc_ab ;  M_ab = W_ab KL_ab  (Kc, KL as in grad_reduce_kernel)
//   s_d = sum_ab M_ab (u_ad - v_bd)^2 = sum_a u_ad^2 R_a + sum_b v_bd^2 C_b - 2 sum_a u_ad (M V)_ad
// with R, C the row and column sums of M (M is not symmetric: the tile holds one triangle only) and M V on the DMMA
// pipe over D in chunks.  The translation-invariant form needs the centring: without it the three terms are each of
// the size of |x|^2 and cancel.  Each s_d goes into partial[block][slot] through the one thread that owns coordinate
// d of the chunk; the sigma and diagonal sums are per-thread shared-memory accumulators reduced at the end, both in a
// fixed order, so the result is deterministic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "cov_kernels.cuh"
#include "dgemm_sm100.cuh"

namespace gpr {

constexpr int GW_DC = 32;             // coordinates per chunk
constexpr int GW_P = GR_TILE + 4;     // pitch of the d-major tiles and of M: pitch mod 16 == 4 -> conflict-free fragment loads
constexpr int GW_NACC = KSPEC_MAXC + 1;   // per-thread accumulators: one sigma sum per component, the diagonal sum

// smem carve-up (doubles): xc1, xc2: GW_DC x GW_P (centred coordinates of the tile's rows / columns, d-major),
// ms: GR_TILE x GW_P (M, column b at ms + b * GW_P), nrm: 128, rs: 64, cs: 64, lsc: GW_DC, red: 2 x GW_DC, al1, al2: 64,
// etab: 32, acc: GW_NACC x GR_THREADS
constexpr size_t GW_SMEM_DOUBLES = (size_t)2 * GW_DC * GW_P + (size_t)GR_TILE * GW_P + 128 + 2 * GR_TILE + GW_DC + 2 * GW_DC +
                                   2 * GR_TILE + 32 + (size_t)GW_NACC * GR_THREADS;
constexpr size_t GW_SMEM_BYTES = GW_SMEM_DOUBLES * sizeof(double);

template <bool DIST>
__global__ void __launch_bounds__(GR_THREADS) grad_reduce_wide_kernel(const GradArgs a) {
  extern __shared__ __align__(16) double gw_smem[];
  const int D = a.D, P = a.P;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp & 1, wn = warp >> 1;   // W / Gram / M: the warp's rows 32 wm .. +32, columns 16 wn .. +16;
                                             // M V: the same rows, coordinates 8 wn .. +8 of the chunk
  double* xc1 = gw_smem;
  double* xc2 = xc1 + (size_t)GW_DC * GW_P;
  double* ms = xc2 + (size_t)GW_DC * GW_P;
  double* nrm = ms + (size_t)GR_TILE * GW_P;
  double* rs = nrm + 128;
  double* cs = rs + GR_TILE;
  double* lsc = cs + GR_TILE;
  double* red = lsc + GW_DC;
  double* al1 = red + 2 * GW_DC;
  double* al2 = al1 + GR_TILE;
  double* etab = al2 + GR_TILE;
  double* acc = etab + 32;
  double* part = a.partial + (size_t)blockIdx.x * (P + 1);
  if (tid < 32) etab[tid] = kg_exp2_tab[tid];
  for (int s = 0; s < GW_NACC; ++s) acc[s * GR_THREADS + tid] = 0.0;
  for (int s = tid; s <= P; s += GR_THREADS) part[s] = 0.0;

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
    if (tid < GR_TILE) al1[tid] = (r0 + tid < a.N) ? a.alpha[r0 + tid] : 0.0;
    else if (tid < 2 * GR_TILE) al2[tid - GR_TILE] = (c0 + tid - GR_TILE < a.N) ? a.alpha[c0 + tid - GR_TILE] : 0.0;
    __syncthreads();

    // W in the accumulator layout of the m8n8k4 product: entry (32 wm + g + 8 i, 16 wn + 8 jj + 2 t + v)
    double w[4][2][2];
    double dsum = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int jj = 0; jj < 2; ++jj)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int il = 32 * wm + g + 8 * i, jl = 16 * wn + 8 * jj + 2 * t + v;
          const long long r = r0 + il, c = c0 + jl;
          double x = 0.0;
          if (r < a.N && c < a.N && r <= c) {
            const double m = al1[il] * al2[jl] - a.Kinv[r + (lc0 + jl) * a.ld];
            if (r == c) { x = m; dsum += m; } else x = 2.0 * m;
          }
          w[i][jj][v] = x;
        }
    acc[KSPEC_MAXC * GR_THREADS + tid] += dsum;

    // centred coordinates d0 .. d0 + GW_DC of the tile's rows (xc1) and columns (xc2); zero beyond D and beyond N.
    // Consecutive threads read consecutive coordinates of one point (coalesced).
    auto stage = [&](int d0) {
      for (int idx = tid; idx < 2 * GR_TILE * GW_DC; idx += GR_THREADS) {
        const int d = idx % GW_DC, p = (idx / GW_DC) % GR_TILE;
        const bool second = idx >= GR_TILE * GW_DC;
        const long long pt = (second ? c0 : r0) + p;
        const double x = (d0 + d < D && pt < a.N) ? a.x[d0 + d + pt * D] - a.x[d0 + d] : 0.0;
        (second ? xc2 : xc1)[d * GW_P + p] = x;
      }
    };

    for (int comp = 0; comp < a.spec.ncomp; ++comp) {
      const int type = a.spec.type[comp];
      if (type == KT_NOISE) continue;
      const int off = a.spec.hp_off[comp];
      const double sg = a.hp[off];
      const double sig2 = sg * sg;

      // ---- pass 1: Gram product of the scaled centred coordinates and the squared norms, over D in chunks
      double gm[4][2][2];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) gm[i][jj][0] = gm[i][jj][1] = 0.0;
      double nacc = 0.0;   // thread p < 128: squared norm of point p (rows, then columns)
      for (int d0 = 0; d0 < D; d0 += GW_DC) {
        __syncthreads();
        stage(d0);
        if (tid < GW_DC) lsc[tid] = (d0 + tid < D) ? a.hp[off + 1 + d0 + tid] : 0.0;
        __syncthreads();
        if (tid < 2 * GR_TILE) {
          const double* src = tid < GR_TILE ? xc1 + tid : xc2 + (tid - GR_TILE);
#pragma unroll 8
          for (int d = 0; d < GW_DC; ++d) { const double u = src[d * GW_P] * lsc[d]; nacc = fma(u, u, nacc); }
        }
#pragma unroll 2
        for (int s = 0; s < GW_DC; s += 4) {
          const double l = lsc[s + t];
          double fa[4], fb[2];
#pragma unroll
          for (int i = 0; i < 4; ++i) fa[i] = xc1[(s + t) * GW_P + 32 * wm + 8 * i + g] * l;
#pragma unroll
          for (int jj = 0; jj < 2; ++jj) fb[jj] = xc2[(s + t) * GW_P + 16 * wn + 8 * jj + g] * l;
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) dmma884(gm[i][jj][0], gm[i][jj][1], fa[i], fb[jj]);
        }
      }
      if (tid < 2 * GR_TILE) nrm[tid] = nacc;
      __syncthreads();

      // ---- Kc (sigma sum) and M = W o KL into shared memory
      double ssum = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jj = 0; jj < 2; ++jj)
#pragma unroll
          for (int v = 0; v < 2; ++v) {
            const int il = 32 * wm + g + 8 * i, jl = 16 * wn + 8 * jj + 2 * t + v;
            const bool diag = r0 + il == c0 + jl;
            double d2 = fmax(fma(-2.0, gm[i][jj][v], nrm[il] + nrm[GR_TILE + jl]), 0.0);
            if (diag) d2 = 0.0;
            double kc, kl;
            if (type == KT_SE) {
              kc = sig2 * exp_tab32(-d2, etab);
              if (diag) kc += a.eps;        // dK/dsigma and dK/dl both use the jittered K (deriv_covar.jl:23,26)
              kl = kc;
            } else {
              const double rr = sqrt(d2);
              const double s5r = 2.23606797749978969640917366873128 * rr;
              const double e = exp_tab32(-s5r, etab);
              kc = sig2 * (1.0 + s5r + (5.0 / 3.0) * d2) * e;
              if (diag) kc += a.eps;
              kl = (5.0 / 6.0) * sig2 * (1.0 + s5r) * e;
            }
            ssum += w[i][jj][v] * kc;
            ms[jl * GW_P + il] = w[i][jj][v] * kl;
          }
      acc[comp * GR_THREADS + tid] += ssum;
      __syncthreads();
      if (tid < GR_TILE) {                    // row sums R
        double s = 0.0;
        for (int b = 0; b < GR_TILE; ++b) s += ms[b * GW_P + tid];
        rs[tid] = s;
      } else if (tid < 2 * GR_TILE) {         // column sums C
        const double* col = ms + (tid - GR_TILE) * GW_P;
        double s = 0.0;
        for (int q = 0; q < GR_TILE; ++q) s += col[q];
        cs[tid - GR_TILE] = s;
      }

      // ---- pass 2: s_d = sum_a u_ad^2 R_a + sum_b v_bd^2 C_b - 2 sum_a u_ad (M V)_ad, over D in chunks
      for (int d0 = 0; d0 < D; d0 += GW_DC) {
        __syncthreads();
        stage(d0);
        __syncthreads();
        double mv[4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i) mv[i][0] = mv[i][1] = 0.0;
#pragma unroll 4
        for (int s = 0; s < GR_TILE; s += 4) {
          const double fb = xc2[(8 * wn + g) * GW_P + s + t];   // V(b = s + t, d = 8 wn + g)
#pragma unroll
          for (int i = 0; i < 4; ++i) dmma884(mv[i][0], mv[i][1], ms[(s + t) * GW_P + 32 * wm + 8 * i + g], fb);
        }
        // sum over the warp's 32 rows a of u_ad (u_ad R_a - 2 (M V)_ad) + v_ad^2 C_a, coordinates d = 8 wn + 2 t + v
        // (the column sum over b runs over the same 64 indices, so the two halves of the tile share one reduction)
        double q[2];
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const double* ucol = xc1 + (8 * wn + 2 * t + v) * GW_P + 32 * wm + g;
          const double* vcol = xc2 + (8 * wn + 2 * t + v) * GW_P + 32 * wm + g;
          double s = 0.0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int ra = 32 * wm + g + 8 * i;
            const double u = ucol[8 * i], w = vcol[8 * i];
            s = fma(u, fma(u, rs[ra], -2.0 * mv[i][v]), s);
            s = fma(w * w, cs[ra], s);
          }
          s += __shfl_xor_sync(0xffffffffu, s, 4);
          s += __shfl_xor_sync(0xffffffffu, s, 8);
          s += __shfl_xor_sync(0xffffffffu, s, 16);
          q[v] = s;
        }
        if (g == 0) {
          red[wm * GW_DC + 8 * wn + 2 * t] = q[0];
          red[wm * GW_DC + 8 * wn + 2 * t + 1] = q[1];
        }
        __syncthreads();
        if (tid < GW_DC && d0 + tid < D) part[off + 1 + d0 + tid] += red[tid] + red[GW_DC + tid];
      }
    }
  }
  __syncthreads();
  // sigma and diagonal slots: one warp per accumulator round-robin, fixed order
  for (int s = warp; s < GW_NACC; s += GR_THREADS / 32) {
    int slot = -1;
    if (s == KSPEC_MAXC) slot = P;
    else if (s < a.spec.ncomp && a.spec.type[s] != KT_NOISE) slot = a.spec.hp_off[s];
    if (slot < 0) continue;   // warp uniform
    double v = 0.0;
    for (int q = lane; q < GR_THREADS; q += 32) v += acc[s * GR_THREADS + q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) part[slot] = v;
  }
}

}  // namespace gpr
