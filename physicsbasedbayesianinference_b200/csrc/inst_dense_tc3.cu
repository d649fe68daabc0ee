// 3xFP16 persistent tensor-core kernel of the dense Gaussian family (its own translation unit: the
// fully unrolled epilogues make it the slowest file of the build).
#include <algorithm>

#include "host_defs.h"
#include "k_dense_tc3.cuh"

namespace ehmc {

// Operands of k_dense_tc3: Lambda scaled by a power of two so that max |Lambda| lands in [2^13, 2^14), hi = rn16,
// lo = rn16(remainder); canonical K-major no-swizzle layout [KP/8][NP][8].
int pack_dense_tc3(ehmc_potential* p, const std::vector<double>& lambda, const std::vector<double>& mu) {
  const int D = p->D, C8 = (D + 7) / 8, KP = (C8 + 1) / 2 * 16, NP = KP, KCH = KP / 8;
  const Fp16Split split(lambda, 14);
  std::vector<__half> bhi((size_t)KCH * NP * 8, __float2half_rn(0.f)), blo(bhi.size(), __float2half_rn(0.f));
  // Guard of the split (auto path only; dense_path = 4 overrides).  fp16 has 5 exponent bits: entries more
  // than ~2^27 below max |Lambda| lose bits (hi subnormal, lo flushed).  What that does to the gradient is
  // measured in the units the target itself sets: x_k ~ Lambda_kk^-1/2 and (grad U)_n ~ Lambda_nn^1/2, so the
  // relative gradient error of row n is rss_k( dLambda_nk / sqrt(Lambda_nn Lambda_kk) ).  The same argument on
  // the x side (one power-of-two scale per particle row, 2^7 headroom) bounds the spread of the coordinate
  // scales: sqrt(max Lambda_kk / min Lambda_kk) <= 2^10.  Otherwise the exact CUDA-core kernel runs.
  double dmin = INFINITY, dmax = 0.0;
  for (int d = 0; d < D; ++d) {
    dmin = std::min(dmin, lambda[(size_t)d * D + d]);
    dmax = std::max(dmax, lambda[(size_t)d * D + d]);
  }
  bool ok = dmin > 0 && std::isfinite(dmax) && dmax <= dmin * 1048576.0;
  double worst = 0.0;
  for (int n = 0; n < D; ++n) {
    double rss = 0.0;
    for (int k = 0; k < D; ++k) {
      const size_t o = ((size_t)(k / 8) * NP + n) * 8 + (k % 8);
      double rem;
      split(lambda[(size_t)n * D + k], &bhi[o], &blo[o], &rem);
      if (ok) {
        const double err = rem / split.scale;
        rss += err * err / (lambda[(size_t)n * D + n] * lambda[(size_t)k * D + k]);
      }
    }
    worst = std::max(worst, rss);
  }
  DenseState& s = p->dense;
  s.tc3.exact = ok && std::sqrt(worst) <= 9.5367431640625e-7;  // 2^-20
  s.tc3.c8 = C8;
  s.tc3.inv_scale = (float)std::ldexp(1.0, -split.shift);
  std::vector<float> mu3(128, 0.f);
  for (int d = 0; d < D; ++d) mu3[d] = (float)mu[d];
  TRY(upload_raw(bhi.data(), sizeof(__half) * bhi.size(), &s.tc3.hi));
  TRY(upload_raw(blo.data(), sizeof(__half) * blo.size(), &s.tc3.lo));
  return upload_raw(mu3.data(), sizeof(float) * mu3.size(), &s.tc3.mu);
}

template <int C8>
static int launch_tc3_c8(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<float>& A, int integ, bool hmc,
                         cudaStream_t st) {
  constexpr size_t sm = Tc3Shape<C8>::smem_bytes();
  static_assert(sm <= 227 * 1024, "dense tensor-core kernel (fp16 split): shared memory");
  CUDA_TRY(cudaFuncSetAttribute(k_dense_tc3<C8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  DenseTc3Args pa;
  pa.Bhi = static_cast<const __half*>(p->dense.tc3.hi);
  pa.Blo = static_cast<const __half*>(p->dense.tc3.lo);
  pa.mu = static_cast<const float*>(p->dense.tc3.mu);
  pa.inv_lscale = p->dense.tc3.inv_scale;
  pa.dbg = c->tc_debug;
  pa.prof = c->tc_prof ? static_cast<long long*>(c->tc_prof_buf.ptr) : nullptr;
  if (!hmc && c->overflow.ptr == nullptr) {
    TRY(c->overflow.ensure(sizeof(unsigned)));
    CUDA_TRY(cudaMemsetAsync(c->overflow.ptr, 0, sizeof(unsigned), st));
  }
  pa.overflow = static_cast<unsigned*>(c->overflow.ptr);
  // persistent: one CTA per SM (the CTA takes the whole TMEM), tiles dealt in contiguous ranges
  const long long ntiles = (A.P + TC_M - 1) / TC_M;
  const unsigned grid = (unsigned)std::min<long long>(c->prop.multiProcessorCount, ntiles);
  k_dense_tc3<C8><<<grid, TC3_THREADS, sm, st>>>(A, pa, hmc ? 1 : 0, integ);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

int launch_dense_tc3(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<float>& A, int integ, bool hmc, cudaStream_t st) {
  switch (p->dense.tc3.c8) {
    case 3: return launch_tc3_c8<3>(c, p, A, integ, hmc, st);
    case 4: return launch_tc3_c8<4>(c, p, A, integ, hmc, st);
    case 5: return launch_tc3_c8<5>(c, p, A, integ, hmc, st);
    case 6: return launch_tc3_c8<6>(c, p, A, integ, hmc, st);
    case 7: return launch_tc3_c8<7>(c, p, A, integ, hmc, st);
    case 8: return launch_tc3_c8<8>(c, p, A, integ, hmc, st);
    case 9: return launch_tc3_c8<9>(c, p, A, integ, hmc, st);
    case 10: return launch_tc3_c8<10>(c, p, A, integ, hmc, st);
    case 11: return launch_tc3_c8<11>(c, p, A, integ, hmc, st);
    case 12: return launch_tc3_c8<12>(c, p, A, integ, hmc, st);
    case 13: return launch_tc3_c8<13>(c, p, A, integ, hmc, st);
    case 14: return launch_tc3_c8<14>(c, p, A, integ, hmc, st);
    case 15: return launch_tc3_c8<15>(c, p, A, integ, hmc, st);
    case 16: return launch_tc3_c8<16>(c, p, A, integ, hmc, st);
  }
  return fail(EHMC_ERR_UNSUPPORTED, "dense tensor-core kernel (fp16 split): D = %d not packed", p->D);
}

}  // namespace ehmc
