// Instantiations of the small-D fused kernels for one dtype (included by inst_small_f32/f64.cu).
#pragma once

#include <algorithm>

#include "host_defs.h"
#include "k_misc.cuh"
#include "k_small.cuh"

namespace ehmc {

template <typename T, int DT>
static DiagPot<T, DT> make_diag(const ehmc_potential* p) {
  DiagPot<T, DT> f;
  for (int d = 0; d < DT; ++d) f.k[d] = d < p->D ? (T)p->diag_k[d] : T(0);
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
  FunnelPot<T, DT> f;
  // scalars {D, sigma_v [, scaleV, scaleX]}: the funnel of v = scaleV q[0], x_k = scaleX q[k]
  const double a = p->scalars.size() >= 4 ? p->scalars[2] : 1.0, cx = p->scalars.size() >= 4 ? p->scalars[3] : 1.0;
  f.inv_s2 = (T)(a * a / (p->scalars[1] * p->scalars[1]));
  f.half_dm1 = (T)(0.5 * a * (p->D - 1));
  f.a = (T)a;
  f.lnb = (T)(2.0 * std::log(cx));
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
  CoinPot<T, DT> f;
  for (int d = 0; d < DT; ++d) {
    f.k[d] = d < p->D ? (T)p->coin_k[d] : T(0);
    f.nk[d] = d < p->D ? (T)(p->coin_n[d] - p->coin_k[d]) : T(0);
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

template <typename T, int DT, class Pot>
static int launch_small_pot(ehmc_ctx* c, const IterArgs<T>& A, const Pot& pot, int integ, bool hmc, cudaStream_t st) {
  static_assert(K1_THREADS == K1_THREADS_HOST, "K1 block size");
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
}

template <typename T, int DT>
static int launch_small_dt(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc,
                           cudaStream_t st) {
  switch (p->family) {
    case EHMC_FAMILY_DIAG_GAUSSIAN:
      return launch_small_pot<T, DT>(c, A, make_diag<T, DT>(p), integ, hmc, st);
    case EHMC_FAMILY_FUNNEL:
      return launch_small_pot<T, DT>(c, A, make_funnel<T, DT>(p), integ, hmc, st);
    case EHMC_FAMILY_COIN_TOSS:
      return launch_small_pot<T, DT>(c, A, make_coin<T, DT>(p), integ, hmc, st);
    case EHMC_FAMILY_DENSE_GAUSSIAN:
      if constexpr (DT <= 16) return launch_small_pot<T, DT>(c, A, make_dense_small<T, DT>(p), integ, hmc, st);
      break;
    case EHMC_FAMILY_HIERARCHICAL_NORMAL:  // D = J + 2 >= 3
      if constexpr (DT >= 4)
        return p->hier.centered ? launch_small_pot<T, DT>(c, A, make_hier<T, DT, true>(p), integ, hmc, st)
                                : launch_small_pot<T, DT>(c, A, make_hier<T, DT, false>(p), integ, hmc, st);
      break;
    default:
      break;
  }
  return fail(EHMC_ERR_UNSUPPORTED, "family %d has no small-D kernel for D = %d", p->family, p->D);
}

template <typename T>
int launch_small(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st) {
  const int D = p->D;
  if (D <= 2) return launch_small_dt<T, 2>(c, p, A, integ, hmc, st);
  if (D <= 4) return launch_small_dt<T, 4>(c, p, A, integ, hmc, st);
  if (D <= 8) return launch_small_dt<T, 8>(c, p, A, integ, hmc, st);
  if (D <= 10) return launch_small_dt<T, 10>(c, p, A, integ, hmc, st);
  if (D <= 16) return launch_small_dt<T, 16>(c, p, A, integ, hmc, st);
  if (D <= 32) return launch_small_dt<T, 32>(c, p, A, integ, hmc, st);
  return fail(EHMC_ERR_UNSUPPORTED, "small-D kernel: D = %d > 32", D);
}

template <typename T, int DT, class Pot>
static int run_small_pot(ehmc_ctx* c, const IterArgs<T>& A, const Pot& pot, int integ, const RunArgs<T>& R, cudaStream_t st) {
  const unsigned grid = (unsigned)std::max<long long>(1, (A.P + K1_THREADS - 1) / K1_THREADS);
  if (integ == INTEG_LEAPFROG)
    k_small_run<T, DT, Pot, INTEG_LEAPFROG><<<grid, K1_THREADS, 0, st>>>(A, pot, R);
  else
    k_small_run<T, DT, Pot, INTEG_STORMER><<<grid, K1_THREADS, 0, st>>>(A, pot, R);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

template <typename T, int DT>
static int run_small_dt(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, const RunArgs<T>& R,
                        cudaStream_t st) {
  switch (p->family) {
    case EHMC_FAMILY_DIAG_GAUSSIAN: return run_small_pot<T, DT>(c, A, make_diag<T, DT>(p), integ, R, st);
    case EHMC_FAMILY_FUNNEL: return run_small_pot<T, DT>(c, A, make_funnel<T, DT>(p), integ, R, st);
    case EHMC_FAMILY_COIN_TOSS: return run_small_pot<T, DT>(c, A, make_coin<T, DT>(p), integ, R, st);
    case EHMC_FAMILY_DENSE_GAUSSIAN:
      if constexpr (DT <= 16) return run_small_pot<T, DT>(c, A, make_dense_small<T, DT>(p), integ, R, st);
      break;
    case EHMC_FAMILY_HIERARCHICAL_NORMAL:
      if constexpr (DT >= 4)
        return p->hier.centered ? run_small_pot<T, DT>(c, A, make_hier<T, DT, true>(p), integ, R, st)
                                : run_small_pot<T, DT>(c, A, make_hier<T, DT, false>(p), integ, R, st);
      break;
    default: break;
  }
  return fail(EHMC_ERR_UNSUPPORTED, "family %d has no fused multi-iteration kernel for D = %d", p->family, p->D);
}

template <typename T>
int run_small(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, const RunArgs<T>& R, cudaStream_t st) {
  const int D = p->D;
  if (D <= 2) return run_small_dt<T, 2>(c, p, A, integ, R, st);
  if (D <= 4) return run_small_dt<T, 4>(c, p, A, integ, R, st);
  if (D <= 8) return run_small_dt<T, 8>(c, p, A, integ, R, st);
  if (D <= 10) return run_small_dt<T, 10>(c, p, A, integ, R, st);
  if (D <= 16) return run_small_dt<T, 16>(c, p, A, integ, R, st);
  if (D <= 32) return run_small_dt<T, 32>(c, p, A, integ, R, st);
  return fail(EHMC_ERR_UNSUPPORTED, "small-D kernel: D = %d > 32", D);
}

template <typename T, int DT>
static int eval_small_dt(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
                         long long g_ld, cudaStream_t st) {
  const unsigned grid = (unsigned)((P + 127) / 128);
  switch (p->family) {
    case EHMC_FAMILY_DIAG_GAUSSIAN:
      k_eval_small<T, DT><<<grid, 128, 0, st>>>(q, q_ld, P, p->D, e, g, g_ld, make_diag<T, DT>(p));
      break;
    case EHMC_FAMILY_FUNNEL:
      k_eval_small<T, DT><<<grid, 128, 0, st>>>(q, q_ld, P, p->D, e, g, g_ld, make_funnel<T, DT>(p));
      break;
    case EHMC_FAMILY_COIN_TOSS:
      k_eval_small<T, DT><<<grid, 128, 0, st>>>(q, q_ld, P, p->D, e, g, g_ld, make_coin<T, DT>(p));
      break;
    case EHMC_FAMILY_HIERARCHICAL_NORMAL:
      if constexpr (DT >= 4) {
        if (p->hier.centered)
          k_eval_small<T, DT><<<grid, 128, 0, st>>>(q, q_ld, P, p->D, e, g, g_ld, make_hier<T, DT, true>(p));
        else
          k_eval_small<T, DT><<<grid, 128, 0, st>>>(q, q_ld, P, p->D, e, g, g_ld, make_hier<T, DT, false>(p));
        break;
      }
      return fail(EHMC_ERR_UNSUPPORTED, "eval: family %d", p->family);
    default:
      return fail(EHMC_ERR_UNSUPPORTED, "eval: family %d", p->family);
  }
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

template <typename T>
int eval_small(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
               long long g_ld, cudaStream_t st) {
  const int D = p->D;
  if (D <= 2) return eval_small_dt<T, 2>(c, p, q, q_ld, P, e, g, g_ld, st);
  if (D <= 4) return eval_small_dt<T, 4>(c, p, q, q_ld, P, e, g, g_ld, st);
  if (D <= 8) return eval_small_dt<T, 8>(c, p, q, q_ld, P, e, g, g_ld, st);
  if (D <= 10) return eval_small_dt<T, 10>(c, p, q, q_ld, P, e, g, g_ld, st);
  if (D <= 16) return eval_small_dt<T, 16>(c, p, q, q_ld, P, e, g, g_ld, st);
  if (D <= 32) return eval_small_dt<T, 32>(c, p, q, q_ld, P, e, g, g_ld, st);
  return fail(EHMC_ERR_UNSUPPORTED, "eval: D = %d", D);
}

}  // namespace ehmc
