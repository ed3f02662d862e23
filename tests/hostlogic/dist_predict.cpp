// TEST INFRASTRUCTURE ONLY -- never linked into libgpr_sm100a.so.
// Runs the block-cyclic prediction driver (gpr::DistPredict, csrc/dist_blocked.hpp) on G simulated ranks with the
// plain-loop CPU backend of hostlogic.cpp, after the distributed factorization of the same file.
#include "hostlogic.cpp"

namespace {

struct CpuPredBE : CpuBE {
  void pred_fixup(double* T, int64_t ldt, int64_t ncols, const double* Kt, int64_t ldk, const double* L, int64_t ld,
                  const gpr::DistLayout& lay, int r, int64_t mtp, double*, double* out, bool write_back) {
    for (int64_t i = 0; i < mtp; ++i) {
      double s = 0.0;
      for (int64_t b = 0; b < ncols; ++b) {
        const int64_t g = lay.gblock(r, b / lay.nb) * lay.nb + b % lay.nb;
        const double k = Kt[g + i * ldk];
        const double t = T[i + b * ldt] - 0.5 * L[g + b * ld] * k;
        if (write_back) T[i + b * ldt] = t;
        s += t * k;
      }
      out[i] = s;
    }
  }
  void copy2d(double* dst, int64_t ldd, const double* src, int64_t lds, int64_t rows, int64_t cols) {
    for (int64_t c = 0; c < cols; ++c) memcpy(dst + c * ldd, src + c * lds, sizeof(double) * rows);
  }
  void zero(double* p, int64_t n) { std::fill(p, p + n, 0.0); }
};

struct CpuPredComm {
  std::vector<gpr::DistPredRank<CpuPredBE>>* ranks = nullptr;
  long long sums = 0;
  void sum_vec(int64_t count) {
    sums++;
    auto& rk = *ranks;
    for (int64_t i = 0; i < count; ++i) {
      double s = rk[0].red[i];
      for (size_t g = 1; g < rk.size(); ++g) s += rk[g].red[i];
      rk[0].red[i] = s;
    }
  }
};

}  // namespace

extern "C" {

// K: N x N SPD (the training covariance), Y: N x ny, Kt: N x M = K(x, xp).  K^-1 and -K^-1 Y come from the block-cyclic
// potrf / trtri / lauum over G ranks (hl_dist_factor); the test points then go through DistPredict in tiles of `tile`.
// Outputs: mean (M x ny) = Kt^T K^-1 Y, quad (M, nullable) = diag(Kt^T K^-1 Kt), XX (M x M, nullable: the dense path)
// = Kt^T K^-1 Kt.  Returns the factorization info, or -1 for tiles that do not fit the arguments.
long long hl_dist_predict(const double* K, int64_t N, int64_t nb, int G, const double* Y, int ny, const double* Kt, int64_t M,
                          int64_t tile, double* mean, double* quad, double* XX, long long* sums) {
  const int64_t Np = (N + nb - 1) / nb * nb, nyp = (ny + 127) / 128 * 128;
  if (XX && tile < M) return -1;
  std::vector<double> A((size_t)Np * Np, 0.0), Yp((size_t)Np * nyp, 0.0);
  for (int64_t j = 0; j < Np; ++j) {
    if (j >= N) { A[j + j * Np] = 1.0; continue; }
    for (int64_t i = 0; i <= j; ++i) A[i + j * Np] = K[i + j * N];
  }
  for (int c = 0; c < ny; ++c) memcpy(&Yp[(size_t)c * Np], Y + (int64_t)c * N, sizeof(double) * N);
  const long long info = hl_dist_factor(A.data(), Np, nb, G, Yp.data(), nyp, 2);   // upper(A) = K^-1, Yp = -K^-1 Y
  if (info) return info;

  gpr::DistLayout lay;
  lay.G = G; lay.Np = Np; lay.nb = nb; lay.nblk = Np / nb; lay.nyp = nyp;
  const int64_t MT = (tile + 127) / 128 * 128;
  const bool dense = XX != nullptr;
  std::vector<CpuPredBE> bes(G);
  std::vector<std::vector<double>> Ls(G), Ts(G), Ktls(G), mscrs(G), reds(G), Kts(G);
  std::vector<std::vector<int>> gts(G);
  std::vector<gpr::DistPredRank<CpuPredBE>> ranks(G);
  for (int r = 0; r < G; ++r) {
    const int64_t nc = lay.nloc(r) * nb;
    Ls[r].assign((size_t)Np * std::max<int64_t>(lay.lcols(r), 1), 0.0);
    for (int64_t lb = 0; lb < lay.nloc(r); ++lb)
      memcpy(&Ls[r][(size_t)lb * nb * Np], &A[(size_t)lay.gblock(r, lb) * nb * Np], sizeof(double) * Np * nb);
    if (r == lay.y_owner()) memcpy(&Ls[r][(size_t)lay.ycol0(r) * Np], Yp.data(), sizeof(double) * Np * nyp);
    gts[r].resize(std::max<int64_t>(lay.ltiles(r), 1));
    for (int64_t t = 0; t < lay.ltiles(r); ++t) gts[r][t] = lay.gtile(r, t);
    Kts[r].assign((size_t)Np * MT, 0.0);
    Ts[r].assign((size_t)MT * std::max<int64_t>(nc, 1), 0.0);
    Ktls[r].assign((size_t)std::max<int64_t>(nc, 1) * MT, 0.0);
    mscrs[r].assign((size_t)MT * nyp, 0.0);
    reds[r].assign((size_t)(MT * (1 + ny) + (dense ? MT * MT : 0)), std::nan(""));   // every entry must be written
    ranks[r] = gpr::DistPredRank<CpuPredBE>{r, &bes[r], Ls[r].data(), Np, gts[r].data(), Kts[r].data(), Ts[r].data(),
                                           Ktls[r].data(), mscrs[r].data(), nullptr, reds[r].data()};
  }
  CpuPredComm comm;
  comm.ranks = &ranks;
  for (int64_t m0 = 0; m0 < M; m0 += MT) {
    const int64_t mt = std::min(MT, M - m0), mtp = (mt + 127) / 128 * 128;
    for (int r = 0; r < G; ++r) {   // every rank holds the tile of K(x, xp): padded rows and columns zero
      std::fill(Kts[r].begin(), Kts[r].end(), 0.0);
      for (int64_t c = 0; c < mt; ++c) memcpy(&Kts[r][(size_t)c * Np], Kt + (m0 + c) * N, sizeof(double) * N);
    }
    gpr::DistPredict<CpuPredBE, CpuPredComm> dp(lay, ranks, comm, mtp, ny, quad != nullptr, dense);
    dp.product();
    dp.fixup();
    dp.mean();
    dp.dense_product();
    dp.reduce();
    const double* red = reds[0].data();
    for (int c = 0; c < ny; ++c)
      for (int64_t i = 0; i < mt; ++i) mean[m0 + i + c * M] = red[mtp + i + c * mtp];
    if (quad)
      for (int64_t i = 0; i < mt; ++i) quad[m0 + i] = 2.0 * red[i];
    if (dense) {
      const double* X = red + mtp * (1 + ny);
      for (int64_t j = 0; j < mt; ++j)
        for (int64_t i = 0; i < mt; ++i) XX[i + j * M] = X[i + j * mtp] + X[j + i * mtp];
    }
  }
  if (sums) *sums = comm.sums;
  return 0;
}

}  // extern "C"
