// Block-cyclic multi-GPU drivers for the factor / inverse path at sizes where one factorization no longer
// fits (or is too slow on) a single device: BASELINE.json config 5 (N = 131072, 137 GB of FP64 K), SURVEY.md 8e.
//
// Replaces, across G ranks, the same LAPACK calls as csrc/blocked.hpp:
//   dpotrf('U') + dpotrs on y     /root/reference/src/cost.jl:104-106
//   K^-1 (dpotrs on the identity) /root/reference/src/cost.jl:107-109   (here trtri + lauum, 2N^3/3)
//
// Layout.  The padded Np x Np matrix is cut into block columns of width nb (a multiple of 128); block column J
// lives on one rank as its local block J / G (1-D block-cyclic; the order of the ranks alternates from round to
// round, see DistLayout::owner).  The right-hand sides y (padded to nyp columns)
// form one more, narrower block column with index nblk, owned by owner(nblk) and stored after that rank's
// matrix columns.  Every rank keeps its columns in ONE column-major array L (Np rows, leading dimension ld), so
// the row panel U(k, :) of step k is a contiguous-by-column slab of every rank's L and all trailing updates of a
// step are a single GEMM launch per rank.  Only the upper triangle is ever referenced; the strict lower
// triangle of L must be zero (the distributed covariance build writes it that way).
//
// Algorithms (U^T U = K, upper factor, all in place in L):
//   potrf   right-looking over block rows k: owner factors the nb x nb diagonal block (recursive panel code of
//           blocked.hpp, which also applies U_kk^-T to the owner's part of the row panel) -> U_kk and its Dinv
//           leaves go to every rank -> every rank finishes its part of the row panel -> the row panel is
//           gathered on every rank -> one rank-nb update of the local trailing columns (tiles above the
//           diagonal only).  The y columns ride along, so z = U^-T y falls out of the same updates.
//   trtri   bottom-up over block rows k: W(k, j) = -U_kk^-1 * sum_{k < m <= j} U(k, m) W(m, j) for the local
//           columns j > k (row panel of U gathered, one GEMM with a per-column contraction limit).  In the y
//           columns the same recurrence with the old content added is the back substitution: they end up
//           holding -alpha = -K^-1 y.
//   lauum   K^-1 = W W^T accumulated column panel by column panel: step k sends W(0:k, k) to every rank, which
//           adds W(i, k) W(j, k)^T to its columns j <= k (rows i <= j).
// Communication per phase and rank: 4 N^2 bytes received in total (SURVEY.md 8e), in N / nb steps.
//
// The drivers are lock-step SPMD over the ranks held by THIS process: `ranks` holds all G ranks in the
// single-process multi-device mode (gpr_mgpu_*, peer copies over NVLink) and exactly one rank when every GPU
// has its own process.  All cross-rank data movement goes through COMM; all arithmetic through BE
// (the CUDA backend in the product, a plain-loop CPU backend in tests/hostlogic).
//
//   BE (in addition to the members blocked.hpp needs):
//     be.gemm_map(tA, tB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, flags, map)
//        flags: BLK_MAP_UPPER  element (m, n) exists iff (map.row_gtile0 + m/128, m%128) <= (gt(n), n%128),
//                              gt(n) = map.col_gtile[n / 128]  (global 128-tile column of local tile n/128)
//               BLK_MAP_KUPTO  column tile contracts over k < (gt(n) - map.k_gtile0 + 1) * 128 only
//               BLK_MAP_BROWS  the op(B) columns of column tile n/128 start at gt(n) * 128 instead of n
//     be.activate()          select the rank's device
//     be.fork() / be.join()  side queue waits for everything queued on the main queue so far / vice versa
//     be.side(on)            route the following launches (and the rank's part of collectives) to the side queue
//   COMM (collective: called once per step, acts on every local rank, on the rank's CURRENT queue; b = 0/1
//   selects one of the two panel / Ukk buffers):
//     comm.bcast_diag(k, with_owner, b)   Ukk[b] (nb x nb, ld nb) and dinv blocks k*tpb.. <- owner's diagonal block k
//     comm.gather_rowpanel(k, b)          panel[b][p + ((J-k-1)*nb + c)*nb] <- U(k*nb + p, J*nb + c), J = k+1 .. nblk-1
//     comm.gather_rowpanel_t(k, b)        the same panel TRANSPOSED: panel[b][((J-k-1)*nb + c) + p*Krem], Krem = Np - (k+1)*nb
//                                         (trtri contracts over the panel's columns: transposed, the product is T,N)
//     comm.bcast_colpanel(k, b)           panel[b][c + i*nb] <- L_owner(i, block k col c), i < (k+1)*nb  (TRANSPOSED: both
//                                         operands of the lauum update are then contraction-contiguous, the fastest GEMM form)
//     comm.barrier()                      every rank's main-queue work so far is ordered before every rank's later
//                                         main-queue work
//   The collectives themselves do not synchronise: the drivers place a barrier between producing a block on
//   one rank and reading it from another, and between the last remote read of a block and overwriting it.
//
// Overlap.  potrf looks one block ahead: right after the owner of block k+1 has updated that block column in
// step k it factors the diagonal block on its side queue while the main queue finishes the trailing update, so
// the only serial work per step is the row-panel solve and its gather.  trtri and lauum read data that is
// already final (U, resp. W), so the copies for step k -+ 1 are issued on the side queue during step k (two
// panel buffers) and never wait for arithmetic; the barrier of step k only orders "every rank holds its copy"
// before "the source is overwritten".
#pragma once
#include <stdint.h>

#include <vector>

#include "blocked.hpp"

namespace gpr {

constexpr int BLK_MAP_UPPER = 8;    // == GEMM_MAP_UPPER
constexpr int BLK_MAP_KUPTO = 16;   // == GEMM_MAP_KUPTO
constexpr int BLK_MAP_BROWS = 32;   // == GEMM_MAP_BROWS
constexpr int GTILE_RHS = 1 << 22;  // global tile index of the y columns: beyond every matrix tile

struct TileMap {
  const int* col_gtile;   // device (or host, CPU backend) array: global 128-tile column of each local 128-tile column
  int row_gtile0;         // global 128-tile row of the first row of C
  int k_gtile0;           // global 128-tile row of the first contraction index
};

struct DistLayout {
  int G = 1;
  int64_t Np = 0, nb = 0, nblk = 0, nyp = 0;
  int tpb() const { return (int)(nb / LEAF); }
  // Block column J belongs to round q = J / G.  Even rounds deal the blocks to ranks 0..G-1, odd rounds to
  // G-1..0 ("snake" order), which evens out the TOTAL work and memory per rank (with the plain cyclic order the
  // last rank owns the longest column of every round).  Every rank owns exactly one block per round, so the local
  // block index is still q.  Measured (2 x B200, N = 32768): no change in run time -- the steps are globally
  // ordered by the panel exchange, so what counts is the per-step maximum (one block of nb columns more on
  // some rank), which no 1-D order can remove.
  int owner(int64_t J) const { const int p = (int)(J % G); return ((J / G) & 1) ? G - 1 - p : p; }
  int64_t gblock(int r, int64_t lb) const { return lb * G + ((lb & 1) ? G - 1 - r : r); }   // global block of local block lb
  int y_owner() const { return owner(nblk); }
  int64_t count_le(int r, int64_t k) const {     // owned matrix blocks J <= k
    if (k < 0) return 0;
    const int64_t q = (k + 1) / G, rem = (k + 1) % G;
    const int64_t pos = (q & 1) ? G - 1 - r : r;   // position of rank r inside the partial round q
    return q + (pos < rem ? 1 : 0);
  }
  int64_t nloc(int r) const { return count_le(r, nblk - 1); }          // matrix blocks owned by r
  int64_t ycol0(int r) const { return nloc(r) * nb; }
  int64_t lcols(int r) const { return nloc(r) * nb + (r == y_owner() ? nyp : 0); }
  int64_t ltiles(int r) const { return lcols(r) / LEAF; }
  int gtile(int r, int64_t jt) const {
    const int64_t t = tpb();
    if (jt >= nloc(r) * t) return GTILE_RHS + (int)(jt - nloc(r) * t);
    return (int)(gblock(r, jt / t) * t + jt % t);
  }
};

template <class BE>
struct DistRank {
  int r = 0;
  BE* be = nullptr;
  double* L = nullptr;       // Np x lcols(r), ld
  int64_t ld = 0;
  double* dinv = nullptr;    // Np/128 leaves, global leaf index (every rank holds all leaves it ever needs)
  double* Ukk[2] = {nullptr, nullptr};     // nb x nb each
  double* panel[2] = {nullptr, nullptr};   // Np * nb doubles each: row panel (nb x Np) or column panel (Np x nb)
  const int* gtile = nullptr;   // ltiles(r) entries, readable by BE
};

template <class BE, class COMM>
struct DistBlocked {
  DistLayout lay;
  std::vector<DistRank<BE>>& ranks;
  COMM& comm;
  bool prefetch_trtri = true, prefetch_lauum = true;   // issue the copies for the next step on the side queue

  DistBlocked(const DistLayout& l, std::vector<DistRank<BE>>& rk, COMM& c) : lay(l), ranks(rk), comm(c) {}

  void all_join() { for (auto& R : ranks) { R.be->activate(); R.be->join(); } }
  void all_side(bool on) {
    for (auto& R : ranks) {
      R.be->activate();
      if (on) R.be->fork();
      R.be->side(on);
    }
  }

  // L(upper) <- U, y columns <- U^-T y
  void potrf() {
    const int64_t nb = lay.nb, Np = lay.Np;
    const int tpb = lay.tpb();
    for (auto& R : ranks)
      if (R.r == lay.owner(0)) {
        R.be->activate();
        Blocked<BE> blk(*R.be, R.dinv);
        blk.potrf_panel(R.L, R.ld, nb, 0, 0);
      }
    for (int64_t k = 0; k < lay.nblk; ++k) {
      const int o = lay.owner(k);
      // diagonal block k was factored on its owner's side queue during step k-1 (main queue for k = 0)
      for (auto& R : ranks)
        if (R.r == o) { R.be->activate(); R.be->join(); }
      if (lay.G > 1) {
        comm.barrier();
        comm.bcast_diag(k, false, 0);
      }
      for (auto& R : ranks) {
        const int64_t c0 = lay.count_le(R.r, k) * nb, m = lay.lcols(R.r) - c0;
        if (m <= 0) continue;
        R.be->activate();
        Blocked<BE> blk(*R.be, R.dinv);
        if (R.r == o) blk.trsm_LUT(R.L + k * nb + (c0 - nb) * R.ld, R.ld, nb, k * tpb, R.L + k * nb + c0 * R.ld, R.ld, m, 1.0);
        else blk.trsm_LUT(R.Ukk[0], nb, nb, k * tpb, R.L + k * nb + c0 * R.ld, R.ld, m, 1.0);
      }
      const int64_t Mrows = Np - (k + 1) * nb;
      if (Mrows <= 0) break;   // last block row: nothing below it
      comm.barrier();
      comm.gather_rowpanel(k, 0);
      const int o2 = lay.owner(k + 1);
      for (auto& R : ranks) {
        const int64_t c0 = lay.count_le(R.r, k) * nb, m = lay.lcols(R.r) - c0;
        if (m <= 0) continue;
        R.be->activate();
        const double* rowp = R.L + k * nb + c0 * R.ld;
        double* C = R.L + (k + 1) * nb + c0 * R.ld;
        TileMap map{R.gtile + c0 / LEAF, (int)((k + 1) * tpb), 0};
        if (R.r == o2) {
          // block column k+1 first, then its diagonal block is factored while the rest of the update runs
          R.be->gemm_map('T', 'N', Mrows, nb, nb, -1.0, R.panel[0], nb, rowp, R.ld, 1.0, C, R.ld, BLK_MAP_UPPER, map);
          R.be->fork();
          R.be->side(true);
          Blocked<BE> blk(*R.be, R.dinv);
          blk.potrf_panel(C, R.ld, nb, 0, (k + 1) * tpb);
          R.be->side(false);
          if (m > nb) {
            TileMap map2{R.gtile + (c0 + nb) / LEAF, (int)((k + 1) * tpb), 0};
            R.be->gemm_map('T', 'N', Mrows, m - nb, nb, -1.0, R.panel[0], nb, rowp + nb * R.ld, R.ld, 1.0, C + nb * R.ld, R.ld,
                           BLK_MAP_UPPER, map2);
          }
        } else {
          R.be->gemm_map('T', 'N', Mrows, m, nb, -1.0, R.panel[0], nb, rowp, R.ld, 1.0, C, R.ld, BLK_MAP_UPPER, map);
        }
      }
    }
    all_join();
  }

  // L(upper) <- W = U^-1 (diagonal 128-blocks with explicit zeros below the diagonal), y columns <- -U^-1 (y columns)
  void trtri() {
    const int64_t nb = lay.nb, Np = lay.Np;
    const int tpb = lay.tpb();
    comm.barrier();
    comm.bcast_diag(lay.nblk - 1, true, (int)((lay.nblk - 1) & 1));   // copies for the first step (no row panel: nothing right of it)
    for (int64_t k = lay.nblk - 1; k >= 0; --k) {
      const int o = lay.owner(k);
      const int b = (int)(k & 1);
      const int64_t Krem = Np - (k + 1) * nb;
      all_join();       // the copies for step k (side queue of step k+1)
      comm.barrier();   // every rank holds its copies: row panel k and diagonal block k may be overwritten
      if (prefetch_trtri) all_side(true);
      if (k > 0) {      // copies for step k-1: U is final there, so they only wait for the buffers
        comm.bcast_diag(k - 1, true, b ^ 1);
        comm.gather_rowpanel_t(k - 1, b ^ 1);
      }
      for (auto& R : ranks)
        if (R.r == o) {
          R.be->activate();
          Blocked<BE> blk(*R.be, R.dinv);
          blk.trtri(R.L + k * nb + (k / lay.G) * nb * R.ld, R.ld, nb, k * tpb, true);
        }
      all_side(false);
      for (auto& R : ranks) {
        const int64_t c0 = lay.count_le(R.r, k) * nb;
        const int64_t mreg = lay.nloc(R.r) * nb - c0, m = lay.lcols(R.r) - c0;
        R.be->activate();
        double* rowp = R.L + k * nb + c0 * R.ld;
        const double* below = R.L + (k + 1) * nb + c0 * R.ld;
        if (Krem > 0 && mreg > 0) {
          TileMap map{R.gtile + c0 / LEAF, 0, (int)((k + 1) * tpb)};
          R.be->gemm_map('T', 'N', nb, mreg, Krem, 1.0, R.panel[b], Krem, below, R.ld, 0.0, rowp, R.ld, BLK_MAP_KUPTO, map);
        }
        if (Krem > 0 && m > mreg)
          R.be->gemm('T', 'N', nb, m - mreg, Krem, 1.0, R.panel[b], Krem, below + mreg * R.ld, R.ld, 1.0, rowp + mreg * R.ld, R.ld, 0, 1, 0, 0, 0);
        if (m > 0) {
          Blocked<BE> blk(*R.be, R.dinv);
          blk.trsm_LUN(R.Ukk[b], nb, nb, k * tpb, rowp, R.ld, m, -1.0);
        }
      }
    }
    all_join();
  }

  // L(upper) <- W W^T (matrix columns only)
  void lauum() {
    const int64_t nb = lay.nb;
    comm.barrier();
    comm.bcast_colpanel(0, 0);
    for (int64_t k = 0; k < lay.nblk; ++k) {
      const int o = lay.owner(k);
      const int b = (int)(k & 1);
      all_join();       // column panel k (side queue of step k-1)
      comm.barrier();   // every rank holds it: the owner may overwrite block column k
      if (k + 1 < lay.nblk) {
        if (prefetch_lauum) all_side(true);
        comm.bcast_colpanel(k + 1, b ^ 1);   // W is final: only waits for the buffer
        all_side(false);
      }
      for (auto& R : ranks) {
        const int64_t cnt = lay.count_le(R.r, k);
        const int64_t nacc = (R.r == o) ? cnt - 1 : cnt;
        const int64_t Mrows = (k + 1) * nb;
        R.be->activate();
        if (nacc > 0) {
          TileMap map{R.gtile, 0, 0};
          R.be->gemm_map('T', 'N', Mrows, nacc * nb, nb, 1.0, R.panel[b], nb, R.panel[b], nb, 1.0, R.L, R.ld,
                         BLK_MAP_UPPER | BLK_MAP_BROWS, map);
        }
        if (R.r == o) {
          TileMap map{R.gtile + (cnt - 1) * lay.tpb(), 0, 0};
          R.be->gemm_map('T', 'N', Mrows, nb, nb, 1.0, R.panel[b], nb, R.panel[b], nb, 0.0, R.L + (cnt - 1) * nb * R.ld, R.ld,
                         BLK_MAP_UPPER | BLK_MAP_BROWS, map);
        }
      }
    }
    all_join();
  }
};

// Posterior prediction (predict_mean! / predict!, src/predict.jl:36-102) from the K^-1 that lauum leaves block-cyclic in L.
// A distributed triangular solve with U^T would be sequential over the ranks; the explicit inverse needs no solve.
// Uu = upper triangle of K^-1 including its diagonal (L of every rank, zeros below), d = diag(K^-1), so
// K^-1 = Uu + Uu^T - diag(d).  For one tile of mtp test points with Kt = K(x, xp) (Np x mtp, training index fastest,
// padded rows zero) held by every rank, and g(b) = global row of local column b:
//   T(i, b)  = sum_a Kt(a, i) Uu(a, b)                one T,N product per rank (column tile n contracts up to its global tile)
//   T~(i, b) = T(i, b) - 1/2 d_b Kt(g(b), i)
//   quad_i   = 2 sum_r sum_{b in r} T~(i, b) Kt(g(b), i)       = (Kt^T K^-1 Kt)(i, i)
//   X        = sum_r T~_r Kt(g(local columns of r), :)      Kt^T K^-1 Kt = X + X^T   (dense covariance only)
//   mean     = -Kt^T (y columns of the y owner, which hold -K^-1 Y after trtri)
// Every rank writes its share into `red` = [quad partial (mtp) | mean (mtp x ny) | X (mtp x mtp, dense only)] (ranks
// without the y columns or without blocks contribute zeros) and one sum over the ranks completes the tile.  Cost per
// rank ~ mtp Np^2 / G flop, the single-device solve split G ways; communication is the one sum of `red`.
//   BE (in addition to gemm / gemm_map / activate):
//     be.pred_fixup(T, ldt, ncols, Kt, ldk, L, ld, lay, r, mtp, part, out, write_back)
//                         out[i] = sum_b T~(i, b) Kt(g(b), i) over the ncols local columns (fixed order), T <- T~ if write_back
//     be.copy2d(dst, ldd, src, lds, rows, cols)   be.zero(p, n)
//   COMM:
//     comm.sum_vec(count)  red of the FIRST local rank <- sum over all G ranks of red[0 .. count), in a fixed order
template <class BE>
struct DistPredRank {
  int r = 0;
  BE* be = nullptr;
  const double* L = nullptr;   // Np x lcols(r), ld
  int64_t ld = 0;
  const int* gtile = nullptr;
  const double* Kt = nullptr;  // Np x mtp, ld Np
  double* T = nullptr;         // mtp x nloc(r) * nb
  double* Ktl = nullptr;       // nloc(r) * nb x mtp: the rows of Kt at the rank's global blocks (dense only)
  double* mscr = nullptr;      // mtp x nyp (y owner)
  double* part = nullptr;      // per-CTA partial sums of the fix-up (backend-defined size)
  double* red = nullptr;
};

template <class BE, class COMM>
struct DistPredict {
  DistLayout lay;
  std::vector<DistPredRank<BE>>& ranks;
  COMM& comm;
  int64_t mtp = 0;
  int ny = 1;
  bool want_quad = true, dense = false;
  bool quad_only = false;   // red = [quad partial (mtp)] only, mean() is not called (split-predict variance rows)

  DistPredict(const DistLayout& l, std::vector<DistPredRank<BE>>& rk, COMM& c, int64_t mtp_, int ny_, bool quad, bool dense_)
      : lay(l), ranks(rk), comm(c), mtp(mtp_), ny(ny_), want_quad(quad || dense_), dense(dense_) {}

  int64_t count() const { return quad_only ? mtp : mtp * (1 + ny) + (dense ? mtp * mtp : 0); }
  int64_t ncols(int r) const { return lay.nloc(r) * lay.nb; }

  void product() {
    if (!want_quad) return;
    for (auto& R : ranks) {
      const int64_t n = ncols(R.r);
      if (n <= 0) continue;
      R.be->activate();
      TileMap map{R.gtile, 0, 0};
      R.be->gemm_map('T', 'N', mtp, n, lay.Np, 1.0, R.Kt, lay.Np, R.L, R.ld, 0.0, R.T, mtp, BLK_MAP_KUPTO, map);
    }
  }
  void fixup() {
    for (auto& R : ranks) {
      R.be->activate();
      const int64_t n = ncols(R.r);
      if (!want_quad || n <= 0) R.be->zero(R.red, mtp);
      else R.be->pred_fixup(R.T, mtp, n, R.Kt, lay.Np, R.L, R.ld, lay, R.r, mtp, R.part, R.red, dense);
    }
  }
  void mean() {
    for (auto& R : ranks) {
      R.be->activate();
      if (R.r == lay.y_owner()) {
        R.be->gemm('T', 'N', mtp, lay.nyp, lay.Np, -1.0, R.Kt, lay.Np, R.L + lay.ycol0(R.r) * R.ld, R.ld, 0.0, R.mscr, mtp, 0);
        R.be->copy2d(R.red + mtp, mtp, R.mscr, mtp, mtp, ny);
      } else {
        R.be->zero(R.red + mtp, mtp * ny);
      }
    }
  }
  void dense_product() {
    if (!dense) return;
    for (auto& R : ranks) {
      R.be->activate();
      const int64_t n = ncols(R.r);
      double* X = R.red + mtp * (1 + ny);
      if (n <= 0) { R.be->zero(X, mtp * mtp); continue; }
      for (int64_t lb = 0; lb < lay.nloc(R.r); ++lb)
        R.be->copy2d(R.Ktl + lb * lay.nb, n, R.Kt + lay.gblock(R.r, lb) * lay.nb, lay.Np, lay.nb, mtp);
      R.be->gemm('N', 'N', mtp, mtp, n, 1.0, R.T, mtp, R.Ktl, n, 0.0, X, mtp, 0);
    }
  }
  void reduce() { comm.sum_vec(count()); }
};

// Split prediction (predict_mean! / predict!(mu, Sigma::Diagonal, md, Cmap(+, xe, xq), pc), src/split_predict.jl:5-53).
// The mean mu = sum_k A_k .* (B_k diag(alpha) C_k) never touches K^-1, and every rank holds x and alpha: the q columns are
// SHARDED.  A chunk of `cols` padded q columns (a multiple of 128) is cut into contiguous slabs of whole 128-column tiles, one
// per rank (split_slab; with fewer tiles than ranks the last ranks get none).  Rank r builds A and Cw = diag(alpha) C for its
// slab only and runs per component the T,N product with the Hadamard epilogue against its Bt (all e rows) -- the call the
// single-device path makes for the same columns.  It writes its slab into `red` (nep x cols, zeros elsewhere) and one sum over
// the ranks assembles the chunk: adding zeros is exact, so the chunk is what one rank computing it alone would give.
// The var_range rows are ordinary test points: DistPredict with quad_only, in tiles of ec rows x w q columns (split_var_tile).
//   BE (in addition to zero / activate):
//     be.split_slab(q0, qn, A, Cw)   A (nep x qn x nk, ld nep) and Cw (Np x qn x nk, ld Np) of the padded q columns q0 .. q0+qn-1
//     be.gemm_hadamard(M, N, K, A, lda, B, ldb, E, lde, beta, C, ldc)    C = (A^T B) .* E + beta C
//   COMM: comm.sum_vec(count) as for DistPredict (`red` of the first local rank)
inline void split_slab(int64_t cols, int G, int r, int64_t& q0, int64_t& qn) {
  const int64_t tiles = cols / LEAF, base = tiles / G, extra = tiles % G;
  q0 = (r * base + std::min<int64_t>(r, extra)) * LEAF;
  qn = (base + (r < extra ? 1 : 0)) * LEAF;
}

// variance tile of at most mt points (mt: a multiple of 128): w q columns (every one when a whole row fits, else a multiple of
// 128 of them) of up to eb of the erows variance rows
inline void split_var_tile(int64_t mt, int64_t nqp, int64_t erows, int64_t& w, int64_t& eb) {
  w = std::min<int64_t>(nqp, mt);
  eb = std::min<int64_t>(erows, std::max<int64_t>(1, mt / w));
}

template <class BE>
struct DistSplitRank {
  int r = 0;
  BE* be = nullptr;
  const double* Bt = nullptr;   // Np x nep x nk: B^T of every e row (training index fastest)
  double* A = nullptr;          // nep x (slab width) x nk
  double* Cw = nullptr;         // Np x (slab width) x nk
  double* red = nullptr;        // nep x cols
};

template <class BE, class COMM>
struct DistSplitMean {
  int G = 1, nk = 1;
  int64_t Np = 0, nep = 0, nqp = 0;
  std::vector<DistSplitRank<BE>>& ranks;
  COMM& comm;

  DistSplitMean(int G_, int nk_, int64_t Np_, int64_t nep_, int64_t nqp_, std::vector<DistSplitRank<BE>>& rk, COMM& c)
      : G(G_), nk(nk_), Np(Np_), nep(nep_), nqp(nqp_), ranks(rk), comm(c) {}

  // chunk width for slabs of at most `slab` columns per rank (slab: a multiple of 128)
  int64_t chunk_cols(int64_t slab) const { return std::min<int64_t>(nqp, slab * G); }
  // widest slab of a chunk of `cols` columns: what A and Cw must hold
  int64_t max_slab(int64_t cols) const { return (cols / LEAF + G - 1) / G * LEAF; }

  // chunk = padded q columns c0 .. c0 + cols - 1
  void build(int64_t c0, int64_t cols) {
    for (auto& R : ranks) {
      int64_t q0, qn;
      split_slab(cols, G, R.r, q0, qn);
      if (qn <= 0) continue;
      R.be->activate();
      R.be->split_slab(c0 + q0, qn, R.A, R.Cw);
    }
  }
  void product(int64_t cols) {
    for (auto& R : ranks) {
      int64_t q0, qn;
      split_slab(cols, G, R.r, q0, qn);
      R.be->activate();
      if (q0 > 0) R.be->zero(R.red, q0 * nep);
      for (int k = 0; k < nk; ++k)
        if (qn > 0)
          R.be->gemm_hadamard(nep, qn, Np, R.Bt + (int64_t)k * Np * nep, Np, R.Cw + (int64_t)k * Np * qn, Np, R.A + (int64_t)k * nep * qn,
                              nep, k == 0 ? 0.0 : 1.0, R.red + q0 * nep, nep);
      if (q0 + qn < cols) R.be->zero(R.red + (q0 + qn) * nep, (cols - q0 - qn) * nep);
    }
  }
  void reduce(int64_t cols) { comm.sum_vec(nep * cols); }
};

}  // namespace gpr
