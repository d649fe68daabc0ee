// Small support kernels: statistics finalisation, potential evaluation, Philox
// fills (Ensemble.setPosition / setMomentum), FP32 peak probe, and the reference's
// bodies-as-particles N-body mode.
#pragma once

#include "common.cuh"
#include "k_small.cuh"

namespace ehmc {

// partials[nblocks][NS] -> out[NS]; one block per 32 statistics, deterministic order.
static __global__ void k_stats_finalize(const double* __restrict__ partials, int nblocks, int NS, double* __restrict__ out) {
  const int j = blockIdx.x;
  double s = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) s += partials[(size_t)b * NS + j];
  __shared__ double sm[32];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0;
    t = warp_sum(t);
    if (threadIdx.x == 0) out[j] = t;
  }
}

// Ensemble statistics of the families that report per-particle scalars (pstats [P][3] = accepted, acceptance
// probability, H of the kept state): CTA b sums its contiguous slice of particles -- the three scalars and, straight
// from q, sum_i q[d, i] and sum_i q[d, i]^2 of every coordinate -- into row b of rows[gridDim.x][2D+3];
// k_stats_finalize adds the rows.  Fixed slicing, float64 sums: deterministic and shard-additive.
template <typename T>
__global__ void __launch_bounds__(256) k_ens_stats_partial(const double* __restrict__ pstats, const T* __restrict__ q,
                                                           long long q_ld, long long P, int D, double* __restrict__ rows) {
  const long long lo = P * blockIdx.x / gridDim.x, hi = P * (blockIdx.x + 1) / gridDim.x;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  __shared__ double sm[2][8];
  double* row = rows + (size_t)blockIdx.x * (2 * D + 3);
  auto block_sum2 = [&](double a, double b, double* oa, double* ob) {
    a = warp_sum(a);
    b = warp_sum(b);
    __syncthreads();
    if (lane == 0) {
      sm[0][w] = a;
      sm[1][w] = b;
    }
    __syncthreads();
    if (tid == 0) {
      double x = 0.0, y = 0.0;
      for (int k = 0; k < 8; ++k) {
        x += sm[0][k];
        y += sm[1][k];
      }
      *oa = x;
      if (ob) *ob = y;
    }
  };
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (long long i = lo + tid; i < hi; i += 256) {
    s0 += pstats[i * 3 + 0];
    s1 += pstats[i * 3 + 1];
    s2 += pstats[i * 3 + 2];
  }
  block_sum2(s0, s1, &row[0], &row[1]);
  block_sum2(s2, 0.0, &row[2], nullptr);
  for (int d = 0; d < D; ++d) {
    const T* qd = q + (long long)d * q_ld;
    double a = 0.0, b = 0.0;
    for (long long i = lo + tid; i < hi; i += 256) {
      const double v = (double)qd[i];
      a += v;
      b = fma(v, v, b);
    }
    block_sum2(a, b, &row[3 + d], &row[3 + D + d]);
  }
}

// U and/or grad U for the register-resident families (vectorised potential(q[:, i])).
template <typename T, int DT, class Pot>
__global__ void k_eval_small(const T* __restrict__ q, long long q_ld, long long P, int D, T* energy, T* grad,
                             long long g_ld, const Pot pot) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  T x[DT], g[DT];
#pragma unroll
  for (int d = 0; d < DT; ++d) x[d] = d < D ? q[d * q_ld + i] : T(0);
  const T U = pot.grad(x, g, true);
  if (energy) energy[i] = U;
  if (grad) {
#pragma unroll
    for (int d = 0; d < DT; ++d)
      if (d < D) grad[d * g_ld + i] = g[d];
  }
}

// Dense Gaussian, any D: one thread per (particle, output dim); not a hot path.
// lam is the plain row-major Lambda[D][D].
template <typename T>
__global__ void k_eval_dense(const T* __restrict__ q, long long q_ld, long long P, int D, const T* __restrict__ lam,
                             const T* __restrict__ mu, T* energy, T* grad, long long g_ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  T U = T(0);
  for (int r = 0; r < D; ++r) {
    T s = T(0);
    for (int c = 0; c < D; ++c) s += lam[r * D + c] * (q[c * q_ld + i] - mu[c]);
    if (grad) grad[r * g_ld + i] = s;
    U += (q[r * q_ld + i] - mu[r]) * s;
  }
  if (energy) energy[i] = T(0.5) * U;
}

// mode 0: out = z * scale                    (Ensemble.setPosition, src/ensemble.py:72-74)
// mode 1: out = z * sqrt((m * kB) * T)       (Ensemble.setMomentum, src/ensemble.py:88-91)
// u (optional): Metropolis uniforms of the same (seed, iteration).
template <typename T>
__global__ void k_philox_fill(T* out, long long ld, long long P, int D, T* u, const T* mass, int mode, double scale,
                              double kB, double temp, u64 seed, u64 iter, u64 offset) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const PhiloxKey K(seed, iter);
  if (out != nullptr) {
    T s = (T)scale;
    if (mode == 1) s = momentum_std<T>(mass[i], kB, temp, sqrt(kB * temp));
    constexpr int NB = NormalBlock<T>::N;
    for (int b = 0; b * NB < D; ++b) {
      T zz[NB];
      NormalBlock<T>::draw(K, offset + (u64)i, (uint32_t)b, zz);
#pragma unroll
      for (int t = 0; t < NB; ++t)
        if (b * NB + t < D) out[(long long)(b * NB + t) * ld + i] = Ar<T>::mul(zz[t], s);
    }
  }
  // (u without z: D = 0, the dedicated uniform block)
  if (u != nullptr) u[i] = NormalBlock<T>::uniform(K, offset + (u64)i, out != nullptr ? D : 0);
}

// Per-chain moments of the host loop (HMC.run outside the fused launch): the n-th draw q[D, P] of every chain enters its
// running mean / m2 (chain_moments_update, the same bits as the fused run's epilogue).  One pass, coalesced along P.
template <typename T>
__global__ void __launch_bounds__(256) k_chain_moments(const T* __restrict__ q, long long q_ld, long long P, int D,
                                                      T* mean, T* m2, long long ld, long long n, T rn) {
  for (int d = blockIdx.y; d < D; d += gridDim.y)
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x)
      chain_moments_update(&mean[d * ld + i], &m2[d * ld + i], q[d * q_ld + i], n, rn);
}

// Register-only FFMA chain: 8 independent accumulators x ITER FMAs per thread.
static __global__ void k_fma_peak(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  const float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 123.456f) out[0] = s;  // never true in practice; keeps the chain live
}

// Reference N-body mode (Integrator(..., gradient=None)): the P particles are the
// bodies; body i completes all its steps before body i+1 starts while every
// acceleration reads the shared q (src/integrator.py:105-120 with getAccel rebound to
// getAccelNBody, src/potential.py:30-53).  One CTA; the sum over j is block-parallel.
// D <= 4 (the reference uses 3).
template <typename T, int NT>
__device__ __forceinline__ void nbody_accel(const T* q, long long ld, const T* mass, int P, int D, int i, T G,
                                            const T (&qi)[4], T (&a)[4], T (*red)[4]) {
  T s[4] = {T(0), T(0), T(0), T(0)};
  for (int j = threadIdx.x; j < P; j += NT) {
    if (j == i) continue;
    T r[4], n2 = T(0);
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      r[d] = d < D ? q[d * ld + j] - qi[d] : T(0);
      n2 += r[d] * r[d];
    }
    const T n = sqrt(n2);
    const T den = n * n * n;  // norm(r) ** 3
#pragma unroll
    for (int d = 0; d < 4; ++d) s[d] += G * mass[j] * r[d] / den;
  }
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    T v = s[d];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][d] = v;
  }
  __syncthreads();
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    T v = T(0);
    for (int ww = 0; ww < NT / 32; ++ww) v += red[ww][d];
    a[d] = v;
  }
  __syncthreads();
}

template <typename T>
__device__ __forceinline__ void store4(T* base, long long ld, int i, int D, const T (&val)[4]) {
  if (threadIdx.x == 0) {
#pragma unroll
    for (int d = 0; d < 4; ++d)
      if (d < D) base[d * ld + i] = val[d];
  }
}

template <typename T>
__global__ void __launch_bounds__(128) k_nbody_mode(T* q, long long q_ld, T* p, long long p_ld, const T* mass, int P,
                                                    int D, T G, T h, T h2, int L, int integ) {
  constexpr int NT = 128;
  __shared__ T red[NT / 32][4];
  typedef Ar<T> R;
  for (int i = 0; i < P; ++i) {
    const T m = mass[i];
    T qi[4], v[4], a[4], a2[4], qp[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      qi[d] = d < D ? q[d * q_ld + i] : T(0);
      v[d] = d < D ? p[d * p_ld + i] / m : T(0);
    }
    nbody_accel<T, NT>(q, q_ld, mass, P, D, i, G, qi, a, red);
    if (integ == INTEG_LEAPFROG) {
      for (int s = 0; s < L; ++s) {
#pragma unroll
        for (int d = 0; d < 4; ++d)
          qi[d] = R::add(qi[d], R::add(R::mul(v[d], h), R::mul(R::mul(T(0.5), a[d]), h2)));
        __syncthreads();
        store4(q, q_ld, i, D, qi);
        __syncthreads();
        nbody_accel<T, NT>(q, q_ld, mass, P, D, i, G, qi, a2, red);
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          v[d] = R::add(v[d], R::mul(R::mul(T(0.5), R::add(a[d], a2[d])), h));
          a[d] = a2[d];
        }
      }
    } else {
#pragma unroll
      for (int d = 0; d < 4; ++d) {
        qp[d] = qi[d];
        qi[d] = R::add(R::add(qi[d], R::mul(v[d], h)), R::mul(R::mul(T(0.5), a[d]), h2));
      }
      __syncthreads();
      store4(q, q_ld, i, D, qi);
      __syncthreads();
      for (int s = 0; s < L; ++s) {
        nbody_accel<T, NT>(q, q_ld, mass, P, D, i, G, qi, a, red);
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          const T t = qi[d];
          qi[d] = R::add(R::sub(R::mul(T(2), qi[d]), qp[d]), R::mul(a[d], h2));
          qp[d] = t;
        }
        __syncthreads();
        store4(q, q_ld, i, D, qi);
        __syncthreads();
      }
#pragma unroll
      for (int d = 0; d < 4; ++d) v[d] = R::sub(qi[d], qp[d]) / h;
    }
    __syncthreads();
    {
      T pv[4];
#pragma unroll
      for (int d = 0; d < 4; ++d) pv[d] = R::mul(v[d], m);
      store4(p, p_ld, i, D, pv);
    }
    __syncthreads();
  }
}

}  // namespace ehmc
