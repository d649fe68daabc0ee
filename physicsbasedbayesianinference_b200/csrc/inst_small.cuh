// Instantiations of the small-D fused kernels for one dtype (included by inst_small_f32/f64.cu).
#pragma once

#include <algorithm>
#include <type_traits>

#include "host_defs.h"
#include "k_misc.cuh"
#include "k_small.cuh"

namespace ehmc {

template <typename T, int DT>
static DiagPot<T, DT> make_diag(const ehmc_potential* p) {
  DiagPot<T, DT> f;
  for (int d = 0; d < DT; ++d) f.k[d] = d < p->D ? (T)p->diag.k[d] : T(0);
  return f;
}
template <typename T, int DT>
static DenseSmallPot<T, DT> make_dense_small(const ehmc_potential* p) {
  DenseSmallPot<T, DT> f;
  for (int i = 0; i < DT; ++i) {
    f.mu[i] = i < p->D ? (T)p->dense.h_mu[i] : T(0);
    for (int j = 0; j < DT; ++j) f.lam[i * DT + j] = (i < p->D && j < p->D) ? (T)p->dense.h_lambda[(size_t)i * p->D + j] : T(0);
  }
  return f;
}
template <typename T, int DT>
static FunnelPot<T, DT> make_funnel(const ehmc_potential* p) {
  const FunnelState& s = p->funnel;
  FunnelPot<T, DT> f;
  f.inv_s2 = (T)(s.scaleV * s.scaleV / (s.sigmaV * s.sigmaV));
  f.half_dm1 = (T)(0.5 * s.scaleV * (p->D - 1));
  f.a = (T)s.scaleV;
  f.lnb = (T)(2.0 * std::log(s.scaleX));
  return f;
}

// `small_waves` resident waves of CTAs (the kernel walks the particles with a grid-stride loop)
template <class K>
static int small_grid(ehmc_ctx* c, K kernel, size_t sm, long long P, unsigned* grid) {
  int occ = 0;
  if (sm > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, K1_THREADS, sm));
  const long long need = (P + K1_THREADS - 1) / K1_THREADS;
  const long long wave = (long long)std::max(occ, 1) * c->prop.multiProcessorCount;
  // measured at config 5 (profiles/k1_probe.py): without statistics 4+ waves are ~8 % faster than one
  // (CTAs drift out of lockstep); with statistics the per-CTA reduction favours few, long-lived CTAs
  const int waves = sm > 0 ? std::min(2, c->small_waves) : c->small_waves;
  *grid = (unsigned)std::max<long long>(1, std::min<long long>(need, wave * std::max(1, waves)));
  return EHMC_OK;
}

template <typename T, int DT>
static CoinPot<T, DT> make_coin(const ehmc_potential* p) {
  const CoinState& s = p->coin;
  CoinPot<T, DT> f;
  for (int d = 0; d < DT; ++d) {
    f.k[d] = d < p->D ? (T)s.k[d] : T(0);
    f.nk[d] = d < p->D ? (T)(s.n[d] - s.k[d]) : T(0);
  }
  return f;
}

// the hierarchical normal model; centred or not is part of the functor's type (HierPot)
template <typename T, int DT, bool CENTERED>
static HierPot<T, DT, CENTERED> make_hier(const ehmc_potential* p) {
  const HierarchicalState& h = p->hier;
  HierPot<T, DT, CENTERED> f;
  for (int d = 0; d < DT; ++d) {
    const bool theta = d >= 2 && d < p->D;
    f.s[d] = d < p->D ? (T)h.scale[d] : T(0);
    f.m[d] = theta ? T(1) : T(0);
    f.w[d] = theta ? (T)h.w[d - 2] : T(0);
    f.y[d] = theta ? (T)h.y[d - 2] : T(0);
    f.nwy[d] = theta ? (T)(-h.w[d - 2] * h.y[d - 2]) : T(0);
  }
  f.muLoc = (T)h.muLoc;
  f.invMuS2 = (T)(1.0 / (h.muScale * h.muScale));
  f.lnTau2 = (T)(2.0 * std::log(h.tauScale));
  f.invTau2 = (T)(1.0 / (h.tauScale * h.tauScale));
  f.J = (T)(p->D - 2);
  f.scaled = false;
  for (int d = 2; d < p->D; ++d) f.scaled = f.scaled || h.scale[d] != 1.0;
  return f;
}

template <typename T, int DT>
static MixturePot<T, DT> make_mixture(const ehmc_potential* p) {
  const MixtureState& s = p->mixture;
  MixturePot<T, DT> f;
  f.K = s.K;
  for (int k = 0; k < MIX_KMAX; ++k) {
    f.c[k] = k < s.K ? (T)s.c[k] : T(0);
    for (int d = 0; d < DT; ++d) {
      const bool on = k < s.K && d < p->D;
      f.mu[k][d] = on ? (T)s.mu[(size_t)k * p->D + d] : T(0);
      f.iv[k][d] = on ? (T)s.iv[(size_t)k * p->D + d] : T(0);
    }
  }
  return f;
}

// The register-resident functor of p at its kernel width DT, the least of 2, 4, 8, 10, 16, 32 that holds p->D, handed
// to f(std::integral_constant<int, DT>(), pot).  The dense family has one up to DT = 16 (above, k_dense), the
// hierarchical model from DT = 4 (D = J + 2 >= 3).  Without one: EHMC_ERR_UNSUPPORTED, with the message "family F has
// no <what> for D = N" unless `what` is null.
template <typename T, class F>
static int with_small_pot(const ehmc_potential* p, const char* what, F&& f) {
  auto none = [&]() -> int {
    return what ? fail(EHMC_ERR_UNSUPPORTED, "family %d has no %s for D = %d", p->family, what, p->D) : EHMC_ERR_UNSUPPORTED;
  };
  auto at = [&](auto dt) -> int {
    constexpr int DT = decltype(dt)::value;
    switch (p->family) {
      case EHMC_FAMILY_DIAG_GAUSSIAN: return f(dt, make_diag<T, DT>(p));
      case EHMC_FAMILY_FUNNEL: return f(dt, make_funnel<T, DT>(p));
      case EHMC_FAMILY_COIN_TOSS: return f(dt, make_coin<T, DT>(p));
      case EHMC_FAMILY_DENSE_GAUSSIAN:
        if constexpr (DT <= 16) return f(dt, make_dense_small<T, DT>(p));
        break;
      case EHMC_FAMILY_HIERARCHICAL_NORMAL:
        if constexpr (DT >= 4) return p->hier.centered ? f(dt, make_hier<T, DT, true>(p)) : f(dt, make_hier<T, DT, false>(p));
        break;
      case EHMC_FAMILY_GAUSSIAN_MIXTURE: return f(dt, make_mixture<T, DT>(p));
      default: break;
    }
    return none();
  };
  const int D = p->D;
  if (D <= 2) return at(std::integral_constant<int, 2>());
  if (D <= 4) return at(std::integral_constant<int, 4>());
  if (D <= 8) return at(std::integral_constant<int, 8>());
  if (D <= 10) return at(std::integral_constant<int, 10>());
  if (D <= 16) return at(std::integral_constant<int, 16>());
  if (D <= 32) return at(std::integral_constant<int, 32>());
  return none();
}

template <typename T>
int launch_small(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st) {
  static_assert(K1_THREADS == K1_THREADS_HOST, "K1 block size");
  return with_small_pot<T>(p, "small-D kernel", [&](auto dt, const auto& pot) -> int {
    constexpr int DT = decltype(dt)::value;
    using Pot = std::decay_t<decltype(pot)>;
    // statistics: per-warp value tiles + per-warp rows (WarpStats, k_small.cuh)
    const size_t sm = A.partials != nullptr ? WarpStats<T, DT>::kSmemBytes : 0;
    unsigned grid = 1;
    auto go = [&](auto kernel) -> int {
      TRY(small_grid(c, kernel, sm, A.P, &grid));
      kernel<<<grid, K1_THREADS, sm, st>>>(A, pot);
      return EHMC_OK;
    };
    const bool exact = A.D == DT;  // no padded dimensions: the kernel without the per-dimension bounds tests
    if (hmc) {
      if (integ == INTEG_LEAPFROG)
        TRY(exact ? go(k_small<T, DT, Pot, INTEG_LEAPFROG, true, true>) : go(k_small<T, DT, Pot, INTEG_LEAPFROG, true, false>));
      else
        TRY(exact ? go(k_small<T, DT, Pot, INTEG_STORMER, true, true>) : go(k_small<T, DT, Pot, INTEG_STORMER, true, false>));
    } else {
      if (integ == INTEG_LEAPFROG)
        TRY(exact ? go(k_small<T, DT, Pot, INTEG_LEAPFROG, false, true>) : go(k_small<T, DT, Pot, INTEG_LEAPFROG, false, false>));
      else
        TRY(exact ? go(k_small<T, DT, Pot, INTEG_STORMER, false, true>) : go(k_small<T, DT, Pot, INTEG_STORMER, false, false>));
    }
    c->launches++;
    c->last_rows = grid;  // statistics partials: one row per CTA actually launched
    CUDA_TRY(cudaGetLastError());
    return EHMC_OK;
  });
}

template <typename T>
int run_small(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, const RunArgs<T>& R, cudaStream_t st) {
  return with_small_pot<T>(p, "fused multi-iteration kernel", [&](auto dt, const auto& pot) -> int {
    constexpr int DT = decltype(dt)::value;
    using Pot = std::decay_t<decltype(pot)>;
    const unsigned grid = (unsigned)std::max<long long>(1, (A.P + K1_THREADS - 1) / K1_THREADS);
    if (integ == INTEG_LEAPFROG)
      k_small_run<T, DT, Pot, INTEG_LEAPFROG><<<grid, K1_THREADS, 0, st>>>(A, pot, R, TemperRun());
    else
      k_small_run<T, DT, Pot, INTEG_STORMER><<<grid, K1_THREADS, 0, st>>>(A, pot, R, TemperRun());
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return EHMC_OK;
  });
}

template <typename T>
int run_small_tempered(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, const RunArgs<T>& R,
                       const TemperRun& X, cudaStream_t st) {
  return with_small_pot<T>(p, "tempered multi-iteration kernel", [&](auto dt, const auto& pot) -> int {
    constexpr int DT = decltype(dt)::value;
    using Pot = std::decay_t<decltype(pot)>;
    // one thread per particle: the kernel's lane mask covers exactly the warp's particles
    const unsigned grid = (unsigned)std::max<long long>(1, (A.P + K1_THREADS - 1) / K1_THREADS);
    if (integ == INTEG_LEAPFROG)
      k_small_run<T, DT, Pot, INTEG_LEAPFROG, true><<<grid, K1_THREADS, 0, st>>>(A, pot, R, X);
    else
      k_small_run<T, DT, Pot, INTEG_STORMER, true><<<grid, K1_THREADS, 0, st>>>(A, pot, R, X);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return EHMC_OK;
  });
}

template <typename T>
int eval_small(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
               long long g_ld, cudaStream_t st) {
  return with_small_pot<T>(p, "eval kernel", [&](auto dt, const auto& pot) -> int {
    constexpr int DT = decltype(dt)::value;
    // dense potentials are evaluated by k_eval_dense at every D (eval_device): k_eval_small has no dense instance
    if constexpr (std::is_same_v<std::decay_t<decltype(pot)>, DenseSmallPot<T, DT>>) {
      return fail(EHMC_ERR_UNSUPPORTED, "eval: dense potentials are evaluated by k_eval_dense");
    } else {
      k_eval_small<T, DT><<<(unsigned)((P + 127) / 128), 128, 0, st>>>(q, q_ld, P, p->D, e, g, g_ld, pot);
      c->launches++;
      CUDA_TRY(cudaGetLastError());
      return EHMC_OK;
    }
  });
}

}  // namespace ehmc
