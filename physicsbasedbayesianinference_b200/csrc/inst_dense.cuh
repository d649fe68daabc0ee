// Instantiations of the dense-Gaussian fused kernel for one dtype.
#pragma once

#include "host_defs.h"
#include "k_dense.cuh"

namespace ehmc {

template <typename T, int TN, int MINB>
static int launch_dense_tn(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc,
                           cudaStream_t st) {
  typedef DenseShape<T, TN> S;
  const size_t sm = S::smem_bytes(A.D);
  if (sm > 227 * 1024) return fail(EHMC_ERR_UNSUPPORTED, "dense kernel needs %zu B shared memory", sm);
  CUDA_TRY(cudaFuncSetAttribute(k_dense<T, TN, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  DenseArgs<T> pa;
  pa.Ls = static_cast<const T*>(p->dense.ls);
  pa.mu = static_cast<const T*>(p->dense.mu);
  const unsigned grid = (unsigned)((A.P + S::PT - 1) / S::PT);
  k_dense<T, TN, MINB><<<grid, K2_THREADS, sm, st>>>(A, pa, integ, hmc ? 1 : 0);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

template <typename T>
int launch_dense(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st) {
  const bool two = sizeof(T) == 4 && c->dense_occupancy >= 2;
  switch (p->dense.tn) {
    case 4: return launch_dense_tn<T, 4, 1>(c, p, A, integ, hmc, st);
    case 8: return launch_dense_tn<T, 8, 1>(c, p, A, integ, hmc, st);
    case 13:
      if constexpr (sizeof(T) == 4) {
        if (two) return launch_dense_tn<T, 13, 2>(c, p, A, integ, hmc, st);
      }
      return launch_dense_tn<T, 13, 1>(c, p, A, integ, hmc, st);
    case 16: return launch_dense_tn<T, 16, 1>(c, p, A, integ, hmc, st);
  }
  return fail(EHMC_ERR_INVALID, "dense potential not packed (TN = %d)", p->dense.tn);
}

template <typename T>
int dense_particles_per_cta() {
  return 32 * DenseTile<T>::TM;
}

template <typename T>
int dense_tnp(int TN) {
  const int VW = 16 / (int)sizeof(T);
  return (TN + VW - 1) / VW * VW;
}

template <typename T>
int build_dense(ehmc_potential* p, std::vector<double>& lambda, std::vector<double>& mu) {
  DenseState& s = p->dense;
  const int D = p->D;
  TRY(upload<T>(lambda, &s.lambda));
  if (D <= 16) {
    TRY(upload<T>(mu, &s.mu));
    s.h_lambda.swap(lambda);
    s.h_mu.swap(mu);
    return EHMC_OK;
  }
  // k_dense: warp w owns rows w TN .. w TN + TN - 1 of Lambda, stored per column k as [k][w][TNP]
  const int TN = dense_tn(D), TNP = dense_tnp<T>(TN);
  s.tn = TN;
  std::vector<double> Ls((size_t)D * K2_WARPS_HOST * TNP, 0.0), mu_pad((size_t)K2_WARPS_HOST * TN, 0.0);
  for (int k = 0; k < D; ++k)
    for (int w = 0; w < K2_WARPS_HOST; ++w)
      for (int j = 0; j < TN; ++j) {
        const int i = w * TN + j;
        if (i < D) Ls[((size_t)k * K2_WARPS_HOST + w) * TNP + j] = lambda[(size_t)i * D + k];
      }
  for (int d = 0; d < D; ++d) mu_pad[d] = mu[d];
  TRY(upload<T>(Ls, &s.ls));
  TRY(upload<T>(mu_pad, &s.mu));
  if constexpr (sizeof(T) == 4) TRY(pack_dense_tc3(p, lambda, mu));
  return EHMC_OK;
}

}  // namespace ehmc
