// TEST INFRASTRUCTURE ONLY -- never linked into libgpr_sm100a.so.
// Runs the split-prediction drivers of csrc/dist_blocked.hpp (gpr::split_slab, gpr::DistSplitMean, gpr::DistPredict in its
// quad-only mode) on G simulated ranks with the plain-loop CPU backends of dist_predict.cpp / hostlogic.cpp.
#include "dist_predict.cpp"

namespace {

// The CUDA backend builds the slab operands from x, hp and alpha; here they are cut out of the full arrays the test passes.
struct CpuSplitBE : CpuPredBE {
  const double* Afull = nullptr;    // nep x nqp x nk
  const double* Cwfull = nullptr;   // Np x nqp x nk
  int64_t nep = 0, nqp = 0, Np = 0;
  int nk = 0;
  void split_slab(int64_t q0, int64_t qn, double* A, double* Cw) {
    for (int k = 0; k < nk; ++k)
      for (int64_t c = 0; c < qn; ++c) {
        memcpy(A + (k * qn + c) * nep, Afull + (k * nqp + q0 + c) * nep, sizeof(double) * nep);
        memcpy(Cw + (k * qn + c) * Np, Cwfull + (k * nqp + q0 + c) * Np, sizeof(double) * Np);
      }
  }
  // C = (A^T B) .* E + beta C
  void gemm_hadamard(int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B, int64_t ldb, const double* E,
                     int64_t lde, double beta, double* C, int64_t ldc) {
    for (int64_t n = 0; n < N; ++n)
      for (int64_t m = 0; m < M; ++m) {
        double s = 0.0;
        for (int64_t k = 0; k < K; ++k) s += A[k + m * lda] * B[k + n * ldb];
        const double v = s * E[m + n * lde];
        C[m + n * ldc] = beta != 0.0 ? v + beta * C[m + n * ldc] : v;
      }
  }
};

// sum_vec over plain vectors, rank order; remembers how many sums and how many entries the last one covered
struct CpuSumComm {
  std::vector<double*> reds;
  long long sums = 0, last = 0;
  void sum_vec(int64_t count) {
    sums++;
    last = count;
    for (int64_t i = 0; i < count; ++i) {
      double s = reds[0][i];
      for (size_t g = 1; g < reds.size(); ++g) s += reds[g][i];
      reds[0][i] = s;
    }
  }
};

}  // namespace

extern "C" {

void hl_split_slab(int64_t cols, int G, int r, int64_t* q0, int64_t* qn) { gpr::split_slab(cols, G, r, *q0, *qn); }

// mean (nep x nqp) = sum_k A_k .* (Bt_k^T Cw_k): chunks of slabs of at most `slab` columns over G ranks.
// Bt: Np x nep x nk, A: nep x nqp x nk, Cw: Np x nqp x nk.  Returns the number of sums over the ranks.
long long hl_split_mean(int G, int nk, int64_t Np, int64_t nep, int64_t nqp, const double* Bt, const double* A, const double* Cw,
                        int64_t slab, double* mean) {
  std::vector<CpuSplitBE> bes(G);
  std::vector<gpr::DistSplitRank<CpuSplitBE>> ranks(G);
  CpuSumComm comm;
  gpr::DistSplitMean<CpuSplitBE, CpuSumComm> dm(G, nk, Np, nep, nqp, ranks, comm);
  const int64_t cols = dm.chunk_cols(slab), qmax = dm.max_slab(cols);
  std::vector<std::vector<double>> As(G), Cws(G), reds(G);
  for (int r = 0; r < G; ++r) {
    CpuSplitBE& b = bes[r];
    b.Afull = A; b.Cwfull = Cw; b.nep = nep; b.nqp = nqp; b.Np = Np; b.nk = nk;
    As[r].assign((size_t)(nep * qmax * nk), std::nan(""));   // slab buffers sized as the CUDA driver sizes them
    Cws[r].assign((size_t)(Np * qmax * nk), std::nan(""));
    reds[r].assign((size_t)(nep * cols), std::nan(""));      // every entry must be written
    ranks[r] = gpr::DistSplitRank<CpuSplitBE>{r, &b, Bt, As[r].data(), Cws[r].data(), reds[r].data()};
    comm.reds.push_back(reds[r].data());
  }
  for (int64_t q0 = 0; q0 < nqp; q0 += cols) {
    const int64_t cw = std::min(cols, nqp - q0);
    dm.build(q0, cw);
    dm.product(cw);
    dm.reduce(cw);
    if (comm.last != nep * cw) return -1;
    memcpy(mean + q0 * nep, reds[0].data(), sizeof(double) * nep * cw);
  }
  return comm.sums;
}

// quad[(e-1)*nq + q] = (Kt^T K^-1 Kt) of the grid point (e, q) for the rows e in [e_lo, e_hi] (1-based), others untouched, with
// Kt(s, (e, q)) = sum_k A[e,q,k] Bt[s,e,k] Cu[s,q,k] and K^-1 from the block-cyclic factorization of K (N x N) over G ranks.
// Tiles of at most mt points as gpr_mgpu_split_predict cuts them (gpr::split_var_tile): the operands of the variance rows and of
// the tile's q columns are cut out of the full arrays (what the CUDA driver builds), Kt is assembled with the index formula of
// split_assemble_t_kernel.  A: nep x nqp x nk, Bt: Np x nep x nk, Cu: Np x nqp x nk, Np = N rounded up to nb.
// Returns the number of tiles (one sum over the ranks each), -2 if a sum did not cover exactly one tile, or the factorization info.
long long hl_split_var(const double* K, int64_t N, int64_t nb, int G, int64_t ne, int64_t nq, int nk, const double* A,
                       const double* Bt, const double* Cu, int64_t e_lo, int64_t e_hi, int64_t mt, double* quad) {
  const int64_t Np = (N + nb - 1) / nb * nb, nyp = 128, nep = (ne + 127) / 128 * 128, nqp = (nq + 127) / 128 * 128;
  std::vector<double> Kf((size_t)Np * Np, 0.0), Yp((size_t)Np * nyp, 0.0);
  for (int64_t j = 0; j < Np; ++j) {
    if (j >= N) { Kf[j + j * Np] = 1.0; continue; }
    for (int64_t i = 0; i <= j; ++i) Kf[i + j * Np] = K[i + j * N];
  }
  const long long info = hl_dist_factor(Kf.data(), Np, nb, G, Yp.data(), nyp, 2);   // upper(Kf) = K^-1
  if (info) return info;

  gpr::DistLayout lay;
  lay.G = G; lay.Np = Np; lay.nb = nb; lay.nblk = Np / nb; lay.nyp = nyp;
  const int64_t erows = e_hi - e_lo + 1, nevp = (erows + 127) / 128 * 128;
  int64_t W, EB;
  gpr::split_var_tile(mt, nqp, erows, W, EB);
  const int64_t MT = EB * W;
  std::vector<CpuPredBE> bes(G);
  std::vector<std::vector<double>> Ls(G), Ts(G), reds(G);
  std::vector<std::vector<int>> gts(G);
  std::vector<double> Kt((size_t)Np * MT), Btv((size_t)Np * nevp * nk, 0.0), Av((size_t)nevp * W * nk), Cuv((size_t)Np * W * nk);
  std::vector<gpr::DistPredRank<CpuPredBE>> ranks(G);
  CpuPredComm comm;
  comm.ranks = &ranks;
  for (int r = 0; r < G; ++r) {
    const int64_t nc = lay.nloc(r) * nb;
    Ls[r].assign((size_t)Np * std::max<int64_t>(lay.lcols(r), 1), 0.0);
    for (int64_t lb = 0; lb < lay.nloc(r); ++lb)
      memcpy(&Ls[r][(size_t)lb * nb * Np], &Kf[(size_t)lay.gblock(r, lb) * nb * Np], sizeof(double) * Np * nb);
    gts[r].resize(std::max<int64_t>(lay.ltiles(r), 1));
    for (int64_t t = 0; t < lay.ltiles(r); ++t) gts[r][t] = lay.gtile(r, t);
    Ts[r].assign((size_t)MT * std::max<int64_t>(nc, 1), 0.0);
    reds[r].assign((size_t)(2 * MT), std::nan(""));
    ranks[r] = gpr::DistPredRank<CpuPredBE>{r, &bes[r], Ls[r].data(), Np, gts[r].data(), Kt.data(), Ts[r].data(), nullptr, nullptr,
                                           nullptr, reds[r].data()};
  }
  for (int k = 0; k < nk; ++k)   // B^T of the variance rows only
    for (int64_t e = 0; e < erows; ++e)
      memcpy(&Btv[(size_t)(k * nevp + e) * Np], Bt + (k * nep + e_lo - 1 + e) * Np, sizeof(double) * Np);
  long long tiles = 0;
  for (int64_t qa = 0; qa < nqp; qa += W) {
    const int64_t wq = std::min(W, nqp - qa), qv = std::min(wq, nq - qa);
    std::fill(Av.begin(), Av.end(), 0.0);
    for (int k = 0; k < nk; ++k)
      for (int64_t q = 0; q < wq; ++q) {
        for (int64_t e = 0; e < erows; ++e) Av[e + q * nevp + k * nevp * wq] = A[(e_lo - 1 + e) + (qa + q) * nep + k * nep * nqp];
        memcpy(&Cuv[(size_t)(k * wq + q) * Np], Cu + (k * nqp + qa + q) * Np, sizeof(double) * Np);
      }
    for (int64_t e0 = 0; e0 < erows; e0 += EB) {
      const int64_t ec = std::min(EB, erows - e0), rows = ec * wq;
      for (int64_t rr = 0; rr < rows; ++rr)   // index formula of split_assemble_t_kernel (csrc/cov_kernels.cuh)
        for (int64_t s = 0; s < Np; ++s) {
          const int64_t q = rr % wq, e = e0 + rr / wq;
          double v = 0.0;
          if (e < erows && q < qv && s < N)
            for (int k = 0; k < nk; ++k)
              v += Av[e + q * nevp + k * nevp * wq] * Btv[s + e * Np + k * Np * nevp] * Cuv[s + q * Np + k * Np * wq];
          Kt[s + rr * Np] = v;
        }
      for (int r = 0; r < G; ++r) std::fill(reds[r].begin(), reds[r].end(), std::nan(""));
      gpr::DistPredict<CpuPredBE, CpuPredComm> dp(lay, ranks, comm, rows, 1, true, false);
      dp.quad_only = true;
      if (dp.count() != rows) return -2;
      dp.product();
      dp.fixup();
      dp.reduce();
      tiles++;
      if (!std::isnan(reds[0][rows])) return -2;   // nothing beyond the quad partials is written or summed
      for (int64_t j = 0; j < ec; ++j)
        for (int64_t q = 0; q < qv; ++q) quad[(e_lo - 1 + e0 + j) * nq + qa + q] = 2.0 * reds[0][j * wq + q];
    }
  }
  return tiles == comm.sums ? tiles : -2;
}

}  // extern "C"
