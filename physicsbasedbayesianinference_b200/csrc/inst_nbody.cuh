#pragma once

#include "host_defs.h"
#include "k_nbody.cuh"

namespace ehmc {

static int nbody_threads(int B, int ti) {
  int nt = 32;
  while (nt * ti < B && nt < 1024) nt <<= 1;
  return nt;
}

template <typename T>
static NBodyArgs<T> nbody_args(const ehmc_potential* p) {
  NBodyArgs<T> pa;
  pa.bmass = static_cast<const T*>(p->nbody.body_mass);
  pa.B = p->nbody.b;
  pa.G = (T)p->nbody.G;
  pa.eps2 = (T)(p->nbody.eps * p->nbody.eps);
  pa.fcache = nullptr;
  pa.ucache = nullptr;
  pa.cache_read = 0;
  return pa;
}

template <typename T, int TI>
static int launch_nbody_ti(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc,
                           cudaStream_t st) {
  const int B = p->nbody.b, nt = nbody_threads(B, TI);
  if (nt * TI < B) return fail(EHMC_ERR_UNSUPPORTED, "nbody: B = %d > %d bodies", B, 1024 * TI);
  const size_t sm = (size_t)B * BodyRec<T>::VECS * 4 * sizeof(T) + 40 * sizeof(T);
  if (sm > 227 * 1024) return fail(EHMC_ERR_UNSUPPORTED, "nbody: B = %d needs %zu B shared memory", B, sm);
  NBodyArgs<T> pa = nbody_args<T>(p);
  // endpoint cache (device path of ehmc_hmc_iter, leapfrog): see EHMC_FLAG_REUSE_ENDPOINT
  const bool cacheable = hmc && integ == INTEG_LEAPFROG && c->ep_enabled && A.L > 0;
  if (cacheable) {
    const bool hit = (A.flags & FLAG_REUSE_ENDPOINT) && c->ep_valid && c->ep_q == (const void*)A.q && c->ep_pot == p &&
                     c->ep_P == A.P && c->ep_bits == (int)sizeof(T) * 8;
    TRY(c->ep_grad[0].ensure(sizeof(T) * (size_t)A.D * A.P));
    TRY(c->ep_energy[0].ensure(sizeof(T) * (size_t)A.P));
    pa.fcache = static_cast<T*>(c->ep_grad[0].ptr);
    pa.ucache = static_cast<T*>(c->ep_energy[0].ptr);
    pa.cache_read = hit ? 1 : 0;
  }
  c->ep_valid = false;
  const bool eps0 = p->nbody.eps == 0.0;
  void (*k)(const IterArgs<T>, const NBodyArgs<T>, const int, const int);
  if (nt <= 128)
    k = eps0 ? k_nbody<T, true, 128, TI> : k_nbody<T, false, 128, TI>;
  else if (nt <= 512)
    k = eps0 ? k_nbody<T, true, 512, TI> : k_nbody<T, false, 512, TI>;
  else
    k = eps0 ? k_nbody<T, true, 1024, TI> : k_nbody<T, false, 1024, TI>;
  CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  k<<<(unsigned)A.P, nt, sm, st>>>(A, pa, integ, hmc ? 1 : 0);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  if (cacheable) {
    c->ep_valid = true;
    c->ep_q = A.q;
    c->ep_pot = p;
    c->ep_P = A.P;
    c->ep_bits = (int)sizeof(T) * 8;
  }
  return EHMC_OK;
}

template <typename T>
int launch_nbody(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st) {
  // 4 bodies per thread (twice the warps per SM) while that covers B, else 8
  const int ti = c->nbody_ti ? c->nbody_ti : (p->nbody.b <= 4096 ? 4 : 8);
  if (ti == 4 && p->nbody.b <= 4096) return launch_nbody_ti<T, 4>(c, p, A, integ, hmc, st);
  return launch_nbody_ti<T, 8>(c, p, A, integ, hmc, st);
}

template <typename T>
int eval_nbody(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
               long long g_ld, cudaStream_t st) {
  const int B = p->nbody.b;
  int nt = 32;
  while (nt < B && nt < 256) nt <<= 1;
  const size_t sm = (size_t)B * 4 * sizeof(T) + 40 * sizeof(T);
  if (sm > 227 * 1024) return fail(EHMC_ERR_UNSUPPORTED, "nbody: B = %d needs %zu B shared memory", B, sm);
  const NBodyArgs<T> pa = nbody_args<T>(p);
  auto k = p->nbody.eps == 0.0 ? k_nbody_eval<T, true> : k_nbody_eval<T, false>;
  CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  k<<<(unsigned)P, nt, sm, st>>>(q, q_ld, e, g, g_ld, pa);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

template <typename T>
int build_nbody(ehmc_potential* p, const std::vector<double>& body_mass) {
  p->nbody.b = (int)body_mass.size();
  return upload<T>(body_mass, &p->nbody.body_mass);
}

template <typename T>
int colstats(ehmc_ctx* c, const T* q, long long q_ld, long long P, int D, double* out, cudaStream_t st) {
  k_colstats<T><<<D, 256, 0, st>>>(q, q_ld, P, D, out);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

}  // namespace ehmc
