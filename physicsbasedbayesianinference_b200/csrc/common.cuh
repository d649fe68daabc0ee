// Shared device-side definitions for the ehmc kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace ehmc {

typedef unsigned long long u64;

// ---------------------------------------------------------------------------
// Arithmetic traits.
// float : plain operators, nvcc may contract to FFMA (tolerance 1e-5, north_star).
// double: explicit round-to-nearest mul/add so nothing is contracted -- the fp64
//         mode evaluates the reference's expressions (src/integrator.py:112-118) in
//         the reference's order and is bit-identical to NumPy for element-wise work.
// ---------------------------------------------------------------------------
template <typename T>
struct Ar;

template <>
struct Ar<float> {
  static __device__ __forceinline__ float add(float a, float b) { return a + b; }
  static __device__ __forceinline__ float sub(float a, float b) { return a - b; }
  static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
  // x / m with a precomputed reciprocal (1 ulp off a true divide; fp32 tolerance 1e-5)
  static __device__ __forceinline__ float divm(float x, float m, float inv_m) { return x * inv_m; }
  static __device__ __forceinline__ float exp_(float x) { return expf(x); }
  static __device__ __forceinline__ float rsqrt_(float x) { return rsqrtf(x); }
  // 1 / m as one MUFU.RCP (<= 1 ulp, exact for powers of two such as the reference's unit masses): the IEEE
  // divide carries a slow-path branch, and a branch right after the mass load pins every later instruction
  // (the whole momentum draw) behind that load
  static __device__ __forceinline__ float rcp_(float x) {
    float r;
    asm("rcp.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
  }
};

template <>
struct Ar<double> {
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dadd_rn(a, -b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double divm(double x, double m, double) { return x / m; }
  static __device__ __forceinline__ double exp_(double x) { return exp(x); }
  static __device__ __forceinline__ double rsqrt_(double x) { return 1.0 / sqrt(x); }
  static __device__ __forceinline__ double rcp_(double x) { return 1.0 / x; }
};

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Bit-level spec: oracle/hmc_oracle.py.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

// NW independent Philox blocks advanced in lock step: the rounds of different blocks interleave,
// which hides the multiply latency of the (strictly serial) rounds of one block.
template <int NW>
__device__ __forceinline__ void philox4x32_10_multi(uint4 (&c)[NW], uint2 k) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      const uint32_t hi0 = __umulhi(M0, c[w].x), lo0 = M0 * c[w].x;
      const uint32_t hi1 = __umulhi(M1, c[w].z), lo1 = M1 * c[w].z;
      c[w] = make_uint4(hi1 ^ c[w].y ^ k.x, lo1, hi0 ^ c[w].w ^ k.y, lo0);
    }
    k.x += W0;
    k.y += W1;
  }
}

#define EHMC_UNIFORM_BLOCK 0xFFFFFFFFu
#define EHMC_SWAP_BLOCK 0xFFFFFFFEu  // replica-exchange uniforms of the tempered run (k_small_run_tempered)

struct PhiloxKey {
  uint2 key;
  uint32_t it;
  __device__ __forceinline__ PhiloxKey(u64 seed, u64 iteration) {
    key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(iteration >> 32));
    it = (uint32_t)iteration;
  }
  __device__ __forceinline__ uint4 block(u64 pid, uint32_t blk) const {
    return philox4x32_10(make_uint4((uint32_t)pid, (uint32_t)(pid >> 32), blk, it), key);
  }
};

// MUFU.SQRT (max relative error 2^-23): one instruction instead of sqrtf's rsqrt + Newton step + slow-path branch
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// bare MUFU forms (flush-to-zero: no denormal rescue code around the instruction)
__device__ __forceinline__ float sqrt_ftz(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float lg2_ftz(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ex2_ftz(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sin_ftz(float x) {
  float r;
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float cos_ftz(float x) {
  float r;
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Standard normals of one Philox block.
// float : 4 normals (dims 4b .. 4b+3);  double: 2 normals (dims 2b, 2b+1).
template <typename T>
struct NormalBlock;

template <>
struct NormalBlock<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void draw(const PhiloxKey& K, u64 pid, uint32_t blk, float* z) {
    transform(K.block(pid, blk), z);
  }
  // NW consecutive blocks blk .. blk+NW-1 -> z[4*NW]
  template <int NW>
  static __device__ __forceinline__ void draw_multi(const PhiloxKey& K, u64 pid, uint32_t blk, float* z) {
    uint4 c[NW];
#pragma unroll
    for (int w = 0; w < NW; ++w) c[w] = make_uint4((uint32_t)pid, (uint32_t)(pid >> 32), blk + w, K.it);
    philox4x32_10_multi<NW>(c, K.key);
#pragma unroll
    for (int w = 0; w < NW; ++w) transform(c[w], z + 4 * w);
  }
  static __device__ __forceinline__ void transform(const uint4 r, float* z) {
    const float s = 5.9604644775390625e-8f;  // 2^-24
    const float u1a = (float)((r.x >> 8) + 1u) * s, u1b = (float)((r.z >> 8) + 1u) * s;
    // Box-Muller on the SFU: r = sqrt(-2 ln u1) via lg2.approx (clamped: u1 -> 1 may give a tiny
    // positive lg2 error), angle via sin/cos.approx on [-pi, pi).  Absolute error ~5e-7, far below
    // the sampling noise; the integer stream (and therefore u) stays exact.
    // The .ftz forms are bare MUFU instructions: u1 >= 2^-24 and -2 ln u1 is 0 or >= 1.19e-7, never denormal, and
    // the plain forms wrap each MUFU.LG2 / MUFU.SQRT in a denormal rescue (FSETP + 2 predicated FMUL / FADD each:
    // 30 of the ~110 instructions of five pairs).  The angle 2 pi (u2 - 1/2) is ONE FFMA on the integer.
    const float c = -1.3862943611198906f;  // -2 ln 2
    const float ra = sqrt_ftz(fmaxf(c * lg2_ftz(u1a), 0.0f)), rb = sqrt_ftz(fmaxf(c * lg2_ftz(u1b), 0.0f));
    const float k2pi = 3.7450702829317378e-7f;  // 2 pi 2^-24
    const float ta = fmaf((float)(r.y >> 8), k2pi, -3.14159265358979f), tb = fmaf((float)(r.w >> 8), k2pi, -3.14159265358979f);
    // cos(2 pi u) = -cos(2 pi (u - 1/2)), sin likewise
    const float sa = -sin_ftz(ta), ca = -cos_ftz(ta), sb = -sin_ftz(tb), cb = -cos_ftz(tb);
    z[0] = ra * ca;
    z[1] = ra * sa;
    z[2] = rb * cb;
    z[3] = rb * sb;
  }
  // Metropolis uniform of a D-dimensional state (stream version 2): for D mod 4 in {1, 2} the last normal block
  // (block D / 4) leaves its words z, w unused and the uniform is (z >> 8) 2^-24 of THAT block -- the kernels that
  // have just drawn it keep the word instead of running a fourth Philox block (D = 10: 3 blocks instead of 4, D = 2:
  // 1 instead of 2); otherwise word x of the dedicated block 0xFFFFFFFF as before.
  static __host__ __device__ __forceinline__ bool uniform_in_normal_block(int D) { return ((D - 1) & 3) < 2; }
  static __device__ __forceinline__ float uniform_from_word(uint32_t w) { return (float)(w >> 8) * 5.9604644775390625e-8f; }
  static __device__ __forceinline__ float uniform(const PhiloxKey& K, u64 pid, int D) {
    const bool spare = uniform_in_normal_block(D);
    const uint4 r = K.block(pid, spare ? (uint32_t)(D >> 2) : EHMC_UNIFORM_BLOCK);
    return uniform_from_word(spare ? r.z : r.x);
  }
};

template <>
struct NormalBlock<double> {
  static constexpr int N = 2;
  static __device__ __forceinline__ u64 u53(uint32_t a, uint32_t b) {
    return ((u64)(a >> 6) << 27) | (u64)(b >> 5);
  }
  static __device__ __forceinline__ void draw(const PhiloxKey& K, u64 pid, uint32_t blk, double* z) {
    const uint4 r = K.block(pid, blk);
    const double s = 1.1102230246251565e-16;  // 2^-53
    const double u1 = ((double)u53(r.x, r.y) + 1.0) * s, u2 = (double)u53(r.z, r.w) * s;
    const double rr = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    z[0] = rr * cs;
    z[1] = rr * sn;
  }
  // (float64 normal blocks use all four words: the uniform always has its own block)
  static __host__ __device__ __forceinline__ bool uniform_in_normal_block(int) { return false; }
  static __device__ __forceinline__ double uniform_from_word(uint32_t) { return 0.0; }
  static __device__ __forceinline__ double uniform(const PhiloxKey& K, u64 pid, int /*D*/) {
    const uint4 r = K.block(pid, EHMC_UNIFORM_BLOCK);
    return (double)u53(r.x, r.y) * 1.1102230246251565e-16;
  }
};

// Zero unless `on`: a predicated load INTO a zeroed register.  Written as `on ? *p : 0` the compiler loads into a
// temporary and selects, and the select is a consumer of the load: with ten of them at the top of k_small every
// warp waited for HBM before it started its RNG work (and ran out of predicate registers: 14 instructions per
// element).  This form is setp + mov + @p ld and the register has no reader until the state is used.
__device__ __forceinline__ float ld_if(const float* p, bool on) {
  float v;
  asm volatile("{\n .reg .pred q;\n setp.ne.s32 q, %2, 0;\n mov.f32 %0, 0f00000000;\n @q ld.global.f32 %0, [%1];\n}"
               : "=f"(v) : "l"(p), "r"((int)on));
  return v;
}
__device__ __forceinline__ double ld_if(const double* p, bool on) {
  double v;
  asm volatile("{\n .reg .pred q;\n setp.ne.s32 q, %2, 0;\n mov.f64 %0, 0d0000000000000000;\n @q ld.global.f64 %0, [%1];\n}"
               : "=d"(v) : "l"(p), "r"((int)on));
  return v;
}

// ---------------------------------------------------------------------------
// Kernel argument block shared by every fused trajectory kernel.
// (D,P) arrays: element [d, i] at base[d * ld + i].
// ---------------------------------------------------------------------------
struct DynArgs {  // == ehmc_dynamic (include/ehmc.h)
  double stepSize, logStepSize;
  u64 iteration, updates, row;
};

template <typename T>
struct IterArgs {
  T* q;
  long long q_ld;
  T* p;  // integrate: momentum in/out.  hmc: optional momentum_hmc output (may be null)
  long long p_ld;
  const T* mass;
  const T* z;  // optional fed standard normals (null -> Philox)
  long long z_ld;
  const T* u;              // optional fed uniforms (null -> Philox)
  unsigned char* accept;   // optional
  double* partials;        // optional [gridDim.x][2D+3] block partial sums
  long long P;
  int D;
  int L;
  unsigned flags;
  T h, h2;
  double kB, temp;
  double pscale;  // sqrt(kB * temp), host-computed
  u64 seed, iter, offset;
  const DynArgs* dyn;  // optional device-resident step size / iteration (ehmc_dynamic)
};

// kernel-side copy of the arguments with the dynamic fields resolved
template <typename T>
__device__ __forceinline__ IterArgs<T> resolve_dynamic(const IterArgs<T>& in) {
  IterArgs<T> A = in;
  if (in.dyn != nullptr) {
    A.h = (T)in.dyn->stepSize;
    A.h2 = A.h * A.h;
    A.iter = in.dyn->iteration;
  }
  return A;
}

// output side of the fused multi-iteration kernel (k_small_run)
template <typename T>
struct RunArgs {
  T* samples;       // [D*P][S] (element (d, i, s) at (d*P + i)*S + s) or null
  T* momenta;       // same layout or null
  int* accepted;    // [P] number of accepted proposals, or null
  long long S;      // samples per particle in the arrays
  long long s0;     // first sample slot written by this launch
  int nIter;
};

// Replica exchange of the tempered run (k_small_run_tempered, ehmc_hmc_run_tempered): particle i is replica
// r = i mod R of system i / R, R a power of two <= 32, so a system is R adjacent lanes of one warp and a swap is a
// few register shuffles.  Slot r always runs at inverse temperature betas[r]; the STATES move between the lanes.
struct TemperRun {
  const double* betas;  // [R] device, betas[0] = 1 > betas[1] > ... > 0
  int R;
  int* swaps;           // [P] or null: accepted swaps of slot r with slot r + 1
  int* roundtrips;      // [P / R] or null: states labelled "hottest" that reached slot 0
  unsigned lanes;       // the warp's lanes that hold a particle (set by the kernel)
};

constexpr unsigned FLAG_BUGCOMPAT = 1u;
constexpr unsigned FLAG_REJECT_NONFINITE = 2u;
constexpr unsigned FLAG_REUSE_ENDPOINT = 4u;

constexpr int INTEG_LEAPFROG = 0;
constexpr int INTEG_STORMER = 1;

// momentum std of one particle: sqrt((m * kB) * T) in double (src/ensemble.py:88);
// double because m*kB underflows float for molecular masses (tests/test_ensemble.py:74-80).
template <typename T>
__device__ __forceinline__ T momentum_std(T m, double kB, double temp, double pscale);
template <>
__device__ __forceinline__ double momentum_std<double>(double m, double kB, double temp, double) {
  return sqrt(__dmul_rn(__dmul_rn(m, kB), temp));
}
// float32 mode: sqrt(m) * sqrt(kB T), the scalar factor pscale = sqrt(kB T) formed in double on the
// host; 3 ulp (float) from the reference expression, no double-precision work per particle and no
// branch (sqrtf's slow path) between the mass load and the momentum draw.
template <>
__device__ __forceinline__ float momentum_std<float>(float m, double, double, double pscale) {
  return sqrt_approx(m) * (float)pscale;
}

// Metropolis rule of src/HMC.py:168-173: reject iff u > min(1, exp(oldH - newH)).
// np.minimum propagates NaN and (u > NaN) is False -> the reference ACCEPTS NaN ratios.
template <typename T>
__device__ __forceinline__ bool metropolis_reject(T oldH, T newH, T u, unsigned flags, T* accp_out) {
  const T ratio = Ar<T>::exp_(Ar<T>::sub(oldH, newH));
  const T accp = ratio < T(1) ? ratio : T(1);  // NaN -> 1 -> never rejected, as in the reference
  *accp_out = accp;
  bool rej = u > accp;
  if ((flags & FLAG_REJECT_NONFINITE) && !(ratio == ratio)) rej = true;
  return rej;
}

// ---- packed float32 pairs (sm_100 FFMA2 / FADD2 / FMUL2: two lanes of work per issue slot) ----
// Measured (profiles/microbench/op_rates.cu): the packed instructions issue at 0.5 / clk / SM
// sub-partition, i.e. the same flop rate as the scalar ones for HALF the issue slots.  Kernels that
// are issue bound in scalar form (the all-pairs N-body loop: 13 slots + loop overhead per interaction
// against 12 cycles of FMA pipe; the small-D trajectory loop) become pipe bound when packed.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
  return ((f32x2)__float_as_uint(hi) << 32) | (f32x2)__float_as_uint(lo);
}
__device__ __forceinline__ float pk_lo(f32x2 v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float pk_hi(f32x2 v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// ---------------------------------------------------------------------------
// Per-chain moments (nested R-hat, diagnostics.py): Welford's streaming update of one chain's mean and sum of squared
// deviations m2 with its n-th draw q; rn = 1/n rounded to T, computed on the host (an IEEE reciprocal on the device is
// a slow-path subroutine call, and a call changes the register allocation of the whole trajectory kernel).  n = 1
// writes (q, 0) and reads nothing, so the buffers need no initialisation.  Every operation is an explicitly rounded
// intrinsic: the fused run (k_small_ens) and the host loop's k_chain_moments call this in different kernels and must
// produce the same bits.
// ---------------------------------------------------------------------------
template <typename T>
struct WelfordOps;
template <>
struct WelfordOps<float> {
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
};
template <>
struct WelfordOps<double> {
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double fma(double a, double b, double c) { return __fma_rn(a, b, c); }
};

template <typename T>
__device__ __forceinline__ void chain_moments_update(T* mean, T* m2, T q, long long n, T rn) {
  typedef WelfordOps<T> W;
  if (n <= 1) {
    *mean = q;
    *m2 = T(0);
    return;
  }
  const T m0 = *mean;
  const T d = W::sub(q, m0);
  const T m1 = W::fma(d, rn, m0);
  *mean = m1;
  *m2 = W::fma(d, W::sub(q, m1), *m2);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace ehmc
