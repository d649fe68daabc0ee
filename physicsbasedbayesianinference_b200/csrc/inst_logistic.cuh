#pragma once

#include <algorithm>

#include "host_defs.h"
#include "k_logistic.cuh"

namespace ehmc {

template <typename T>
static LogisticArgs<T> logistic_args(const ehmc_potential* p) {
  LogisticArgs<T> pa;
  pa.X = static_cast<const T*>(p->logistic.x);
  pa.y = static_cast<const T*>(p->logistic.y);
  pa.N = p->logistic.n;
  pa.D = p->D;
  pa.inv_s2 = (T)(1.0 / (p->logistic.priorScale * p->logistic.priorScale));
  return pa;
}

template <typename T>
static int logistic_grad(ehmc_ctx* c, const ehmc_potential* p, const T* theta, long long t_ld, long long P, T* g,
                         long long g_ld, T* e, double* e64, cudaStream_t st) {
  if constexpr (sizeof(T) == 4) {
    const LogisticState& s = p->logistic;
    if (s.kernel == LOGISTIC_FP16X3 && s.chunks.buf) return logistic_grad_tcs(c, p, theta, t_ld, P, g, g_ld, e, e64, st);
    if (s.kernel == LOGISTIC_BF16 && s.chunks.buf) return logistic_grad_tc(c, p, theta, t_ld, P, g, g_ld, e, e64, st);
  }
  constexpr int PT = LogiTile<T>::PT;
  const int D = p->D, DS = (D + 3) & ~3;
  if (D > LG_DMAX) return fail(EHMC_ERR_UNSUPPORTED, "logistic: D = %d > %d", D, LG_DMAX);
  const size_t sm = sizeof(T) * ((size_t)D * PT + (size_t)LG_NC * DS + (size_t)LG_NC * PT + LG_THREADS);
  CUDA_TRY(cudaFuncSetAttribute(k_logistic_grad<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  k_logistic_grad<T><<<(unsigned)((P + PT - 1) / PT), LG_THREADS, sm, st>>>(theta, t_ld, P, g, g_ld, e, e64,
                                                                             logistic_args<T>(p));
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

// precision: the selector ehmc_potential_create checked (1 and 2 need float32 state; auto falls back to the exact
// kernel for float64 state or where the fp16 split of X loses accuracy).  X and y go to the device as they are only
// for the exact kernel.
template <typename T>
int build_logistic(ehmc_potential* p, const std::vector<double>& X, const std::vector<double>& y, int precision) {
  LogisticState& s = p->logistic;
  if constexpr (sizeof(T) == 4) {
    if (precision != LOGISTIC_EXACT) TRY(pack_logistic_tc(p, X, y, precision));
  }
  if (s.kernel != LOGISTIC_EXACT) return EHMC_OK;
  TRY(upload<T>(X, &s.x));
  return upload<T>(y, &s.y);
}

template <typename T>
int eval_logistic(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
                  long long g_ld, cudaStream_t st) {
  return logistic_grad<T>(c, p, q, q_ld, P, g, g_ld, e, nullptr, st);
}

// One HMC iteration / one integrate() call as a sequence of launches on `st`.
// Endpoint cache (device path, leapfrog, HMC): the gradient and energy at the position every particle keeps
// are saved by the final kernel; with EHMC_FLAG_REUSE_ENDPOINT the next iteration starts from them instead
// of re-evaluating (L instead of L + 1 gradient launches, the energy variant only once).
template <typename T>
int launch_logistic(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st,
                    int slot) {
  const long long P = A.P;
  const int D = A.D, L = A.L;
  // scratch: U0, U1 [P] double (first: alignment) | w, v, g [D][P] | K0 [P]
  TRY(c->uf[slot].ensure(sizeof(double) * 2 * (size_t)P + sizeof(T) * ((size_t)3 * D * P + (size_t)P)));
  double* U0 = static_cast<double*>(c->uf[slot].ptr);
  double* U1 = U0 + P;
  T* w = reinterpret_cast<T*>(U1 + P);
  T* v = w + (size_t)D * P;
  T* g = v + (size_t)D * P;
  T* K0 = g + (size_t)D * P;
  const unsigned grid = (unsigned)((P + 127) / 128);
  // kick/drift: enough CTAs to fill the GPU (particles x dimension slices)
  const unsigned ysplit = (unsigned)std::max(1, std::min(D, (int)((8 * c->prop.multiProcessorCount + grid - 1) / grid)));
  const dim3 kgrid(grid, ysplit);
  const T h = A.h, h2 = A.h2;
  // ep_enabled is set by the device path only (one call = the whole resident ensemble)
  const bool cacheable = hmc && integ == INTEG_LEAPFROG && slot == 0 && c->ep_enabled && L > 0;
  const bool hit = cacheable && (A.flags & FLAG_REUSE_ENDPOINT) && c->ep_valid && c->ep_q == (const void*)A.q &&
                   c->ep_pot == p && c->ep_P == P && c->ep_bits == (int)sizeof(T) * 8;
  T *g_start = g, *g_keep = nullptr;
  double *u_start = U0, *u_keep = nullptr;
  if (cacheable) {
    for (int k = 0; k < 2; ++k) {
      TRY(c->ep_grad[k].ensure(sizeof(T) * (size_t)D * P));
      TRY(c->ep_energy[k].ensure(sizeof(double) * (size_t)P));
    }
    const int cur = hit ? c->ep_cur : 0;
    g_start = static_cast<T*>(c->ep_grad[cur].ptr);
    u_start = static_cast<double*>(c->ep_energy[cur].ptr);
    g_keep = static_cast<T*>(c->ep_grad[cur ^ 1].ptr);
    u_keep = static_cast<double*>(c->ep_energy[cur ^ 1].ptr);
    c->ep_cur = cur ^ 1;
  }
  c->ep_valid = false;  // re-established below on success
  k_uf_init<T><<<grid, 128, 0, st>>>(A, w, v, hmc ? K0 : nullptr, hmc ? 1 : 0);
  c->launches++;
  if (!hit) TRY(logistic_grad<T>(c, p, w, P, P, g_start, P, nullptr, hmc ? u_start : nullptr, st));
  if (integ == INTEG_LEAPFROG) {
    if (L > 0) {
      k_uf_kick_drift<T><<<kgrid, 128, 0, st>>>(w, v, g_start, A.mass, P, D, T(0.5) * h, h);
      c->launches++;
    }
    for (int s = 0; s < L; ++s) {
      const bool last = s == L - 1;
      TRY(logistic_grad<T>(c, p, w, P, P, g, P, nullptr, (hmc && last) ? U1 : nullptr, st));
      k_uf_kick_drift<T><<<kgrid, 128, 0, st>>>(w, v, g, A.mass, P, D, last ? T(0.5) * h : h, last ? T(0) : h);
      c->launches++;
    }
    if (L == 0 && hmc) CUDA_TRY(cudaMemcpyAsync(U1, u_start, sizeof(double) * P, cudaMemcpyDeviceToDevice, st));
  } else {
    k_uf_sv_step<T><<<grid, 128, 0, st>>>(w, v, g_start, A.mass, P, D, h, h2, 1);
    c->launches++;
    for (int s = 0; s < L; ++s) {
      TRY(logistic_grad<T>(c, p, w, P, P, g, P, nullptr, nullptr, st));
      k_uf_sv_step<T><<<grid, 128, 0, st>>>(w, v, g, A.mass, P, D, h, h2, 0);
      c->launches++;
    }
    k_uf_sv_finish<T><<<grid, 128, 0, st>>>(w, v, P, D, h);
    c->launches++;
    if (hmc) TRY(logistic_grad<T>(c, p, w, P, P, nullptr, 0, nullptr, U1, st));
  }
  k_uf_final<T><<<grid, 128, 0, st>>>(A, w, v, K0, u_start, U1, hmc ? 1 : 0, A.partials, g_start, g, g_keep, u_keep);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  if (cacheable) {
    c->ep_valid = true;
    c->ep_q = A.q;
    c->ep_pot = p;
    c->ep_P = P;
    c->ep_bits = (int)sizeof(T) * 8;
  }
  return EHMC_OK;
}

}  // namespace ehmc
