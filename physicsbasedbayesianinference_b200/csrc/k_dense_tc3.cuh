// K2-TC3: dense-precision Gaussian trajectory kernel, tensor cores, fp16 split operands,
// persistent CTAs.
//
// Kick-drift-kick trajectory with G = X Lambda^T re-issued L+1 times on on-chip state.  Two choices
// (against the 3xTF32 kernels this replaced, 4.84 ms -> 2.6 ms per iteration at config 2):
//
//  * 3xFP16 split instead of 3xTF32.  tf32 and fp16 carry the same 11 significant bits, but
//    tcgen05.mma kind::f16 consumes K = 16 per instruction where kind::tf32 consumes K = 8, at the
//    same M*N/256 cycles per instruction: 3*K16 = 21 MMAs per evaluation at D = 100 instead of 39.
//    The split is round-to-nearest:  hi = rn16(x), lo = rn16(x - hi)  ->  |x - hi - lo| <= 2^-24 |x|,
//    i.e. the (hi, lo) pair is as accurate as the float32 it came from, so the pair IS the master
//    copy of the row's position (no separate fp32 x anywhere).  fp16's narrow exponent range is
//    handled by exact power-of-two scalings: Lambda by `lscale` on the host (max |Lambda| -> 2^13),
//    each particle row by 2^e chosen in the prologue from max(|x|, h L |v|) (-> 2^7, 256x headroom);
//    both are undone in the kick coefficient.  G ~= hi L_hi + lo L_hi + hi L_lo, fp32 accumulate.
//  * every operand of the tile lives in TENSOR MEMORY (all three products are TS-mode MMAs):
//        per tile (256 columns):  [0, NP) D fp32 | [NP, NP + KP/2) hi (fp16 pairs) | [.., NP + KP) lo
//    shared memory only holds Lambda_hi / Lambda_lo (fp16, canonical K-major no-swizzle layout
//    [KP/8][NP][8]), loaded ONCE per CTA: the kernel is persistent (grid = #SMs), each of the two
//    4-warp groups of a CTA walks its own list of 128-particle tiles.  Tiles are dealt to CTAs in
//    contiguous ranges and alternately to the two groups, so when the tile count per SM is odd the
//    last tile runs alone at full tensor-pipe rate (tail = ~0.6 of a paired round, not a full one).
//
// Thread <-> particle row <-> TMEM lane; the row's D velocities stay in registers for the whole
// trajectory.  One group's epilogue (tcgen05.ld G/hi/lo -> kick, drift, re-split -> tcgen05.st)
// overlaps the other group's MMAs.
//
// Reference arithmetic replaced: src/integrator.py:105-120 with gradient = Lambda (q - mu),
// src/HMC.py:106-116,168-176, src/ensemble.py:88-91.
#pragma once

#include <cuda_fp16.h>

#include "k_dense.cuh"  // one_normal
#include "tc_common.cuh"

namespace ehmc {

constexpr int TC3_THREADS = 384;       // 2 consumer groups x 4 warps + 1 producer warpgroup (Philox normals)
constexpr int TC3_CONSUMERS = 256;

// C8 = ceil(D / 8): 8-dim chunks the epilogue touches.  MMA K = N = KP = C8 rounded up to 16 dims.
template <int C8>
struct Tc3Shape {
  static constexpr int K16 = (C8 + 1) / 2;
  static constexpr int KP = 16 * K16;
  static constexpr int NP = KP;
  static constexpr int DC = 8 * C8;
  static constexpr int KCH = KP / 8;  // 16-byte chunks along K
  static constexpr int HI_COL = NP, LO_COL = NP + KP / 2;
  static_assert(NP + KP <= 256, "tile does not fit 256 TMEM columns");
  // Lambda hi / lo + mean + barriers + the two groups' stashes of standard normals [DC][128]
  static constexpr size_t smem_bytes() {
    return (size_t)2 * KCH * NP * 16 + (size_t)KP * 4 + 64 + (size_t)2 * DC * TC_M * 4;
  }
};

struct DenseTc3Args {
  const __half* Bhi;  // [KP/8][NP][8]  rn16(lscale * Lambda)
  const __half* Blo;  //                rn16(lscale * Lambda - hi)
  const float* mu;    // [128] zero padded
  float inv_lscale;   // 1 / lscale (power of two)
  int dbg;            // 1: issue no MMAs (commit only); 2: skip the epilogue arithmetic
  long long* prof;    // optional clock64() trace of the second tile of CTA 0 / group 0 (ctx option "tc_prof")
  unsigned* overflow; // counter of integrate() rows whose position saturated the fp16 operand range
};

// ---- software-pipelined epilogue: batches of 16 dims (a trailing batch of 8 when C8 is odd) ----
struct Tc3Batch {
  uint32_t g[16], hi[8], lo[8];
};

template <int NCOL>
__device__ __forceinline__ void tc3_issue(Tc3Batch& b, uint32_t t_d, uint32_t t_hi, uint32_t t_lo, int col0) {
  tm_ld<NCOL>(t_d + (uint32_t)col0, b.g);
  tm_ld<NCOL / 2>(t_hi + (uint32_t)(col0 / 2), b.hi);
  tm_ld<NCOL / 2>(t_lo + (uint32_t)(col0 / 2), b.lo);
}
template <int NCOL>
__device__ __forceinline__ void tc3_wait(Tc3Batch& b) {
  tm_wait<NCOL>(b.g);
  tm_wait<NCOL / 2>(b.hi);
  tm_wait<NCOL / 2>(b.lo);
}

// One code path for every evaluation (first / middle / last differ only in ck and `store`).
// w = (h 2^e) v is the row's velocity in drift units, so the drift is two additions:
//   kick  w -= ck G            (ck carries h 2^e * h/m * 2^-e / lscale)
//   drift x' = hi + (lo + w)   (5 issue slots per dim including the re-split)
template <int NCOL>
__device__ __forceinline__ void tc3_compute(float* w, Tc3Batch& b, uint32_t t_hi, uint32_t t_lo, int col0, float ck,
                                            bool store) {
#pragma unroll
  for (int i = 0; i < NCOL / 2; ++i) {
    w[2 * i] = fmaf(-ck, __uint_as_float(b.g[2 * i]), w[2 * i]);
    w[2 * i + 1] = fmaf(-ck, __uint_as_float(b.g[2 * i + 1]), w[2 * i + 1]);
    const float x0 = add_h(h_lo(b.hi[i]), add_h(h_lo(b.lo[i]), w[2 * i]));
    const float x1 = add_h(h_hi(b.hi[i]), add_h(h_hi(b.lo[i]), w[2 * i + 1]));
    split16_sat(x0, x1, b.hi[i], b.lo[i]);
  }
  if (store) {
    tm_st<NCOL / 2>(t_hi + (uint32_t)(col0 / 2), b.hi);
    tm_st<NCOL / 2>(t_lo + (uint32_t)(col0 / 2), b.lo);
  }
}

template <int C8, int B>
__device__ __forceinline__ void tc3_pipe(float (&w)[8 * C8], Tc3Batch (&bb)[2], uint32_t t_d, uint32_t t_hi,
                                         uint32_t t_lo, float ck, bool store) {
  constexpr int NB = (C8 + 1) / 2;
  constexpr int NCOL = (B == NB - 1 && (C8 % 2) == 1) ? 8 : 16;
  constexpr int cur = B & 1;
  tc3_wait<NCOL>(bb[cur]);
  if constexpr (B + 1 < NB) {
    constexpr int NCOL_N = (B + 1 == NB - 1 && (C8 % 2) == 1) ? 8 : 16;
    tc3_issue<NCOL_N>(bb[cur ^ 1], t_d, t_hi, t_lo, 16 * (B + 1));
  }
  tc3_compute<NCOL>(&w[16 * B], bb[cur], t_hi, t_lo, 16 * B, ck, store);
  if constexpr (B + 1 < NB) tc3_pipe<C8, B + 1>(w, bb, t_d, t_hi, t_lo, ck, store);
}

template <int C8>
__device__ __forceinline__ void tc3_epilogue(float (&w)[8 * C8], uint32_t t_d, uint32_t t_hi, uint32_t t_lo, float ck,
                                             bool store) {
  Tc3Batch bb[2];
  constexpr int NCOL0 = (C8 == 1) ? 8 : 16;
  tc3_issue<NCOL0>(bb[0], t_d, t_hi, t_lo, 0);
  tc3_pipe<C8, 0>(w, bb, t_d, t_hi, t_lo, ck, store);
  if (store) tmem_wait_st();
}

// L2 prefetch of one warp's 32 rows of the next tile, all D coordinates (out of line: inlined, the compiler
// folds its lane / D tests into the branch of EVERY evaluation, an S2R and an LDC in the serial chain)
static __device__ __noinline__ void tc3_prefetch_rows(const float* row0, long long ld, int D) {
  for (int d = (int)(threadIdx.x & 31); d < D; d += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(row0 + (long long)d * ld));
}

// sum_d xs_d G_d of this row (first and last evaluation only: a rolled loop, kept out of the
// unrolled epilogue so that the 49 middle evaluations do not pay for it)
// Also reports whether a coordinate of the row sits at the fp16 saturation value (see split16_sat).
template <int C8>
__device__ __noinline__ float tc3_energy(uint32_t t_d, uint32_t t_hi, uint32_t t_lo, uint32_t* sat) {
  float2 acc = make_float2(0.f, 0.f);
  uint32_t s = 0u;
#pragma unroll 1
  for (int c = 0; c < C8; ++c) {
    uint32_t g[8], hh[4], ll[4];
    tmem_ld8_issue2(t_d + (uint32_t)(8 * c), g);
    tmem_ld4_issue(t_hi + (uint32_t)(4 * c), hh);
    tmem_ld4_issue(t_lo + (uint32_t)(4 * c), ll);
    tmem_wait_ld8(g);
    tmem_wait_ld4(hh);
    tmem_wait_ld4(ll);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 xh = h2_unpack(hh[i]);
      acc.x = fmaf(add_h(h_lo(ll[i]), xh.x), __uint_as_float(g[2 * i]), acc.x);
      acc.y = fmaf(add_h(h_hi(ll[i]), xh.y), __uint_as_float(g[2 * i + 1]), acc.y);
      s |= h16_saturated(hh[i]);
    }
  }
  *sat = s;
  return acc.x + acc.y;
}

template <int C8>
__global__ void __launch_bounds__(TC3_THREADS, 1) k_dense_tc3(const IterArgs<float> Ain, const DenseTc3Args pa,
                                                              const int hmc, const int integ) {
  const IterArgs<float> A = resolve_dynamic(Ain);
  typedef Tc3Shape<C8> S;
  constexpr int NP = S::NP, KP = S::KP, K16 = S::K16, DC = S::DC, KCH = S::KCH;
  extern __shared__ __align__(128) unsigned char tc3_smem_raw[];
  const int D = A.D;
  uint4* Bhi = reinterpret_cast<uint4*>(tc3_smem_raw);  // [KCH][NP] x 16 bytes
  uint4* Blo = Bhi + (size_t)KCH * NP;
  float* mus = reinterpret_cast<float*>(Blo + (size_t)KCH * NP);  // [KP]
  uint64_t* mbar = reinterpret_cast<uint64_t*>(mus + KP);         // [2] MMA done, per group
  uint64_t* zfull = mbar + 2;                                     // [2] the group's stash of normals is complete
  uint64_t* zempty = mbar + 4;                                    // [2] ... has been consumed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 6);
  float* zstash_all = reinterpret_cast<float*>(tc3_smem_raw + (size_t)2 * KCH * NP * 16 + (size_t)KP * 4 + 64);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform by construction
  const int grp = warp >> 2, quarter = warp & 3;
  const int row = quarter * 32 + lane;

  // ---- CTA setup (once) ------------------------------------------------------------------
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    if (lane == 0) {
      mbar_init(&mbar[0], 1);
      mbar_init(&mbar[1], 1);
      for (int g = 0; g < 2; ++g) {
        mbar_init(&zfull[g], 128);
        mbar_init(&zempty[g], 128);
      }
      fence_barrier_init();
    }
  }
  {
    const uint4* s0 = reinterpret_cast<const uint4*>(pa.Bhi);
    const uint4* s1 = reinterpret_cast<const uint4*>(pa.Blo);
    for (int i = tid; i < KCH * NP; i += TC3_THREADS) {
      Bhi[i] = s0[i];
      Blo[i] = s1[i];
    }
    if (tid < KP) mus[tid] = pa.mu[tid];
  }
  fence_proxy_async();  // Lambda written through the generic proxy, read by the tensor core
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
  const uint32_t t_d = tmem_base + (uint32_t)(grp * 256) + lane_off;  // this row's accumulator
  const uint32_t t_hi = t_d + (uint32_t)S::HI_COL, t_lo = t_d + (uint32_t)S::LO_COL;
  uint32_t idesc = umma_idesc_f16(TC_M, NP);
  uint64_t db_hi = umma_desc(smem_u32(Bhi), NP), db_lo = umma_desc(smem_u32(Blo), NP);
  uint32_t mbar_a = smem_u32(&mbar[grp < 2 ? grp : 0]);
  pin(idesc);
  pin(db_hi);
  pin(db_lo);
  pin(mbar_a);
  // kernel parameters tested in every evaluation: one constant-bank load each, here, instead of an LDC -> use
  // latency in the serial chain of every evaluation
  uint32_t k_dbg = (uint32_t)pa.dbg, k_hmc = (uint32_t)hmc, k_sv = integ == INTEG_STORMER ? 1u : 0u;
  pin(k_dbg);
  pin(k_hmc);
  pin(k_sv);
  constexpr uint64_t b_step = (2u * NP * 16u) >> 4;
  const uint32_t mma_d = tmem_base + (uint32_t)(grp * 256);
  const uint32_t mma_hi = mma_d + (uint32_t)S::HI_COL, mma_lo = mma_d + (uint32_t)S::LO_COL;

  // h == 0 is a fixed point (q, p, H unchanged, accepted): run it as L = 0 so that 1 / h never appears.  That holds
  // for Leapfrog only: Stormer-Verlet's start-up evaluation would still kick and drift a full step of the stand-in
  // h = 1, so launch_tc3_c8 runs Stormer-Verlet at h == 0 as Leapfrog.  (k_dense follows the reference there instead:
  // q unchanged, p = (q - q) / 0 = NaN, accepted unless EHMC_FLAG_REJECT_NONFINITE.)
  const int L = A.h == 0.f ? 0 : A.L;
  const float h = A.h == 0.f ? 1.f : A.h;
  const long long ntiles = (A.P + TC_M - 1) / TC_M;
  const long long tile0 = ntiles * blockIdx.x / gridDim.x, tile1 = ntiles * (blockIdx.x + 1) / gridDim.x;
  uint32_t phase = 0;

  // Momentum refresh off the critical path: a PRODUCER warpgroup (warps 8..11, one thread per particle
  // row, 56 registers after setmaxnreg) draws the standard normals of the tiles ahead of the two consumer
  // groups into shared-memory stashes zst[g][d][row]; full / empty mbarriers per group.  Measured history:
  // Philox + Box-Muller at the start of a tile cost 11.6k of the tile's 154k cycles with the tensor pipe idle;
  // drawn by the consumer threads themselves in the shadow of their MMAs the L = 50 iteration was as fast as
  // with this warpgroup (same-box A/B within the +-4 % run-to-run noise) but the first tile of every group
  // still paid for it (L = 0: 0.54 ms against 0.39 ms); a separate warpgroup spreads the ~3k instructions
  // per row over the whole tile.
  const bool philox = hmc && A.z == nullptr;
  if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (philox) {
      const PhiloxKey PK(A.seed, A.iter);
      const int prow = tid - TC3_CONSUMERS;  // 0 .. 127
      uint32_t par0 = 0u, par1 = 0u;
      for (long long t = tile0; t < tile1; ++t) {
        const int g = (int)((t - tile0) & 1);
        float* zs = zstash_all + (size_t)g * DC * TC_M + prow;
        // first pass: a fresh barrier reads as "previous phase complete".  The producer is ~8x faster than a
        // tile, so it mostly waits here: back off instead of spinning on the consumers' sub-partitions
        const uint32_t want = g == 0 ? par0 ^ 1u : par1 ^ 1u;
        while (!mbar_try_wait(&zempty[g], want)) __nanosleep(2000);
        if (g == 0) par0 ^= 1u; else par1 ^= 1u;
        const long long r = t * TC_M + prow;
        const u64 pid = A.offset + (u64)(r < A.P ? r : 0);
#pragma unroll 1
        for (int c = 0; c < C8; ++c) {
          float zz[8];
          NormalBlock<float>::draw_multi<2>(PK, pid, (uint32_t)(2 * c), zz);
#pragma unroll
          for (int e = 0; e < 8; ++e) zs[(8 * c + e) * TC_M] = zz[e];
        }
        mbar_arrive(&zfull[g]);  // release: the stash writes above are visible to the waiting consumers
      }
    }
    tc_fence_before();
    __syncthreads();
    return;
  }
  asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
  float* zst = zstash_all + (size_t)grp * DC * TC_M + row;
  uint32_t zpar = 0;

  for (long long tile = tile0 + grp; tile < tile1; tile += 2) {
    // phase trace of one steady-state tile (the second of CTA 0 / group 0), thread 0
    const bool prof = pa.prof != nullptr && blockIdx.x == 0 && tid == 0 && tile == tile0 + 2;
    int pi = 0;
    auto stamp = [&]() {
      if (prof && pi < 62) pa.prof[pi++] = clock64();
    };
    stamp();  // 0: tile start
    const long long prow = tile * TC_M + row;
    const bool valid = prow < A.P;
    const long long pc = valid ? prow : 0;

    float v[DC];
    const float m = valid ? A.mass[pc] : 1.f;
    const float inv_m = 1.f / m;
    const float pstd = hmc ? momentum_std<float>(m, A.kB, A.temp, A.pscale) : 0.f;
    float K0 = 0.f, amax = 0.f, vmax = 0.f;
    // The per-tile prologue runs once per L + 1 evaluations but its code must stay SMALL: straight-line
    // code executed once per tile is fetched from L2 every time.  (Measured at config 2: with the 26
    // Philox blocks and the general write-back unrolled the kernel was 390 KB of SASS and an L = 0
    // iteration took 1.06 ms; with the rolled loops below, 84 KB and 0.47 ms.)  Everything that can be
    // indexed dynamically (tensor-memory columns) runs in rolled loops; only register-array traffic
    // is unrolled.
    // ---- positions: all loads in flight (v[] doubles as the staging array) ----------------------
    // (rows past the end of the ensemble replay row 0 and are never written; only the last 8-dim
    // chunk can hold dims >= D, so every other load is unconditional)
    auto col = [&](const float* base, long long ld, int d) -> float {
      return (d < DC - 8 || d < D) ? base[(long long)d * ld] : 0.f;
    };
    const float* qcol = A.q + pc;
#pragma unroll
    for (int d = 0; d < DC; ++d) v[d] = col(qcol, A.q_ld, d);
    stamp();  // 1: position loads issued
    stamp();  // 2
    // x = q - mu parked in the (idle) accumulator columns
#pragma unroll
    for (int c = 0; c < C8; ++c) {
      uint32_t xx[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float x = v[8 * c + e] - mus[8 * c + e];  // dims >= D: 0 - 0
        amax = fmaxf(amax, fabsf(x));
        xx[e] = __float_as_uint(x);
      }
      tmem_st8(t_d + (uint32_t)(8 * c), xx);
    }
    if (philox) {
      mbar_wait(&zfull[grp], zpar);
      zpar ^= 1u;
#pragma unroll
      for (int d = 0; d < DC; ++d) v[d] = (d < DC - 8 || d < D) ? zst[d * TC_M] * pstd : 0.f;
      mbar_arrive(&zempty[grp]);  // (the loads above have returned: v[] is consumed by the arithmetic below)
    } else {
      // fed momenta (parity mode) or integrate()
      const float* mcol = (hmc ? A.z : A.p) + pc;
      const long long mld = hmc ? A.z_ld : A.p_ld;
      const float msc = hmc ? pstd : 1.f;
#pragma unroll
      for (int d = 0; d < DC; ++d) v[d] = col(mcol, mld, d) * msc;
    }
#pragma unroll
    for (int d = 0; d < DC; ++d) {
      K0 = fmaf(v[d], v[d], K0);
      v[d] *= inv_m;
      vmax = fmaxf(vmax, fabsf(v[d]));
    }
    K0 *= 0.5f * inv_m;
    stamp();  // 3: positions landed and parked, momenta in registers
    // ---- row scale 2^e: max(|x|, reach of the ballistic drift) -> [2^7, 2^8) ----------------------
    amax = fmaxf(amax, fabsf(h) * (float)L * vmax);
    uint32_t eb = (__float_as_uint(amax) >> 23) & 0xffu;
    eb = eb < 16u ? 134u : eb;  // zero / tiny rows: no scaling
    const float sc = __uint_as_float((261u - eb) << 23);   // 2^(7 - (eb - 127))
    const float isc = __uint_as_float((eb - 7u) << 23);    // 1 / sc
    tmem_wait_st();
#pragma unroll 1
    for (int c = 0; c < C8; ++c) {
      uint32_t xx[8], hh[4], ll[4];
      tmem_ld8_issue2(t_d + (uint32_t)(8 * c), xx);
      tmem_wait_ld8(xx);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        split16_sat(__uint_as_float(xx[2 * i]) * sc, __uint_as_float(xx[2 * i + 1]) * sc, hh[i], ll[i]);
      tmem_st4(t_hi + (uint32_t)(4 * c), hh);
      tmem_st4(t_lo + (uint32_t)(4 * c), ll);
    }
    if constexpr (DC < KP) {
      // operand columns of the padded dims [DC, KP): finite zeros
      uint32_t zero[4] = {0u, 0u, 0u, 0u};
      tmem_st4(t_hi + (uint32_t)(DC / 2), zero);
      tmem_st4(t_lo + (uint32_t)(DC / 2), zero);
    }
    tmem_wait_st();

    stamp();  // 4: operands split and stored
    // velocities in drift units: w = (h 2^e) v;  g_true = G * isc * inv_lscale
    const float hs = h * sc, gs = isc * pa.inv_lscale;
#pragma unroll
    for (int d = 0; d < DC; ++d) v[d] *= hs;
    float ckf = (h * inv_m) * (h * pa.inv_lscale), ckh = 0.5f * ckf;  // hs * (h / m) * gs
    pin(ckf);
    pin(ckh);
    float U0 = 0.f, U1 = 0.f;
    uint32_t sat = 0u;  // the trajectory left the fp16 range of its row scale (diverged): never accepted

    // Leapfrog (src/integrator.py:105-120): evaluations 0 .. L; half kick, (L - 1) x [drift, kick], drift, half kick.
    // Stormer-Verlet (src/integrator.py:142-163) in displacement form d_n = q_n - q_{n-1} (w IS sc d_n):
    //   start-up q_1 = q_0 + v h + a_0 h^2 / 2  = half kick + drift;  q_{n+1} = 2 q_n - q_{n-1} + a_n h^2 = kick + drift,
    //   L + 1 drifts in all, v = d_{L+1} / h (backward difference, no closing half kick); one more evaluation
    //   (no kick, no drift) only for the energy at q_{L+1}.
    // first row of this warp in the group's next tile (null: no next tile / past the end)
    const float* pf_row = (tile + 2 < tile1 && (tile + 2) * TC_M + quarter * 32 < A.P)
                              ? A.q + (tile + 2) * TC_M + quarter * 32 : nullptr;
    const bool sv = k_sv != 0u;
    const int Lend = (sv && k_hmc) ? L + 1 : L;
    for (int ev = 0; ev <= Lend; ++ev) {
      // the tile's operands are complete once all 128 rows arrive
      tc_fence_before();
      asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
      if (quarter == 0 && elect_one()) {
        tc_fence_after();
        if (!(k_dbg & 1u)) {
#pragma unroll
          for (int j = 0; j < K16; ++j) umma_f16_ts(mma_d, mma_hi + 8u * j, db_hi + j * b_step, idesc, j > 0);
#pragma unroll
          for (int j = 0; j < K16; ++j) umma_f16_ts(mma_d, mma_lo + 8u * j, db_hi + j * b_step, idesc, 1);
#pragma unroll
          for (int j = 0; j < K16; ++j) umma_f16_ts(mma_d, mma_hi + 8u * j, db_lo + j * b_step, idesc, 1);
        }
        umma_commit_a(mbar_a);
      }
      // in the shadow of the MMAs: L2 prefetch of the next tile's positions
      if (ev == 1 && pf_row != nullptr) tc3_prefetch_rows(pf_row, A.q_ld, D);
      mbar_wait_a(mbar_a, phase);
      phase ^= 1u;
      tc_fence_after();
      const bool first = ev == 0;
      const bool last = sv ? ev == L + 1 : ev == L;  // the evaluation that neither drifts nor stores
      if (k_hmc && (first || last)) {
        uint32_t sat_ev;
        const float Uev = tc3_energy<C8>(t_d, t_hi, t_lo, &sat_ev);
        if (first) U0 = Uev;
        if (last) {
          U1 = Uev;
          sat = sat_ev;
        }
      }
      const float ck = sv ? (first ? ckh : (last ? 0.f : ckf)) : (L == 0 ? 0.f : ((first || last) ? ckh : ckf));
      if (!(k_dbg & 2u)) tc3_epilogue<C8>(v, t_d, t_hi, t_lo, ck, !last);
      if (ev < 2 || ev >= L - 1) stamp();  // 5, 6: first two evaluations; then the last two
    }
    // U = 1/2 x . g_true = 1/2 (xs isc) . (G gs)
    U0 = (U0 * isc) * (0.5f * gs);
    U1 = (U1 * isc) * (0.5f * gs);

    // ---- Metropolis + write back -------------------------------------------------------------
    float K1 = 0.f;
    const float w2p = m / hs;  // p = v * m = w * m / (h 2^e)
#pragma unroll
    for (int d = 0; d < DC; ++d) {
      v[d] *= w2p;
      K1 = fmaf(v[d], v[d], K1);
    }
    bool rej = false;
    float accp = 1.f, oldH = 0.f, newH = 0.f;
    if (hmc) {
      oldH = K0 + U0;
      newH = 0.5f * K1 * inv_m + U1;
      float u = 0.f;
      if (valid)
        u = A.u != nullptr ? A.u[pc] : NormalBlock<float>::uniform(PhiloxKey(A.seed, A.iter), A.offset + (u64)pc, A.D);
      rej = metropolis_reject<float>(oldH, newH, u, A.flags, &accp);
      // A row whose position ran more than 256x past its prologue scale saturates its fp16 operands (finite, but no
      // longer the trajectory).  The exact kernels carry such a divergent trajectory to |q| ~ 1e38 and reject it
      // with ratio exp(-huge) = 0; here it is rejected outright, whatever EHMC_FLAG_REJECT_NONFINITE says, so
      // that nothing but a genuine trajectory end is ever written to q.
      if (sat) {
        rej = true;
        accp = 0.f;
      }
    }
    stamp();  // Metropolis decided
    const bool fast = A.p == nullptr;  // statistics are per-particle scalars here (A.partials = [P][3]), see below
    const bool wr = valid && !rej;  // HMC.py:175: rejected rows keep the value in HBM
    // tcgen05.ld is warp-collective (.sync.aligned): every lane loads, only accepted rows store.
    // Rolled loops (see the prologue note on code size).
    if (fast) {
#pragma unroll 1
      for (int c = 0; c < C8; ++c) {
        uint32_t hh[4], ll[4];
        tmem_ld4_issue(t_hi + (uint32_t)(4 * c), hh);
        tmem_ld4_issue(t_lo + (uint32_t)(4 * c), ll);
        tmem_wait_ld4(hh);
        tmem_wait_ld4(ll);
        if (!hmc) sat |= h16_saturated(hh[0]) | h16_saturated(hh[1]) | h16_saturated(hh[2]) | h16_saturated(hh[3]);
        float* qd = A.q + (long long)(8 * c) * A.q_ld + pc;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 xh = h2_unpack(hh[i]);
          const float q0 = fmaf(add_h(h_lo(ll[i]), xh.x), isc, mus[8 * c + 2 * i]);
          const float q1 = fmaf(add_h(h_hi(ll[i]), xh.y), isc, mus[8 * c + 2 * i + 1]);
          if (8 * c + 2 * i < D && wr) qd[(long long)(2 * i) * A.q_ld] = q0;
          if (8 * c + 2 * i + 1 < D && wr) qd[(long long)(2 * i + 1) * A.q_ld] = q1;
        }
      }
    } else {
      // general path (momentum output and / or statistics): park p in the accumulator columns so that
      // the rolled loop can index it
#pragma unroll
      for (int c = 0; c < C8; ++c) {
        uint32_t pk[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) pk[e] = __float_as_uint(v[8 * c + e]);
        tmem_st8(t_d + (uint32_t)(8 * c), pk);
      }
      tmem_wait_st();
      const bool need_old = rej && (A.flags & FLAG_BUGCOMPAT);
#pragma unroll 1
      for (int c = 0; c < C8; ++c) {
        uint32_t hh[4], ll[4], pk[8];
        tmem_ld4_issue(t_hi + (uint32_t)(4 * c), hh);
        tmem_ld4_issue(t_lo + (uint32_t)(4 * c), ll);
        tmem_ld8_issue2(t_d + (uint32_t)(8 * c), pk);
        tmem_wait_ld4(hh);
        tmem_wait_ld4(ll);
        tmem_wait_ld8(pk);
        if (!hmc) sat |= h16_saturated(hh[0]) | h16_saturated(hh[1]) | h16_saturated(hh[2]) | h16_saturated(hh[3]);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int d = 8 * c + e;
          if (d >= D) continue;  // uniform
          const float xh = (e & 1) ? h2_unpack(hh[e / 2]).y : h2_unpack(hh[e / 2]).x;
          const float xl = (e & 1) ? h2_unpack(ll[e / 2]).y : h2_unpack(ll[e / 2]).x;
          const float qn = fmaf(xl + xh, isc, mus[d]);
          float qold = 0.f;
          if (valid && need_old) qold = A.q[d * A.q_ld + pc];
          if (wr) A.q[d * A.q_ld + pc] = qn;
          if (A.p != nullptr && valid) {
            float pv = __uint_as_float(pk[e]);
            if (rej) {
              if (A.flags & FLAG_BUGCOMPAT)
                pv = qold;  // HMC.py:176 (sic)
              else if (A.z != nullptr)
                pv = A.z[d * A.z_ld + pc] * pstd;
              else
                pv = one_normal<float>(A.seed, A.iter, A.offset + (u64)pc, d) * pstd;
            }
            A.p[d * A.p_ld + pc] = pv;
          }
        }
      }
    }
    // integrate() has no Metropolis step to absorb a saturated row: count it (ehmc_ctx_overflow_count)
    if (!hmc && valid && sat && pa.overflow != nullptr) atomicAdd(pa.overflow, 1u);
    if (hmc && valid && A.accept != nullptr) A.accept[pc] = rej ? 0 : 1;
    // ensemble statistics: this kernel only reports the per-particle scalars; the coordinate sums are taken
    // from q by k_ens_stats_partial afterwards (a warp reduction of 2 D doubles per tile cost 1.3 ms per
    // iteration at config 2, a streaming pass over q costs 0.1 ms)
    if (hmc && valid && A.partials != nullptr) {
      A.partials[pc * 3 + 0] = rej ? 0.0 : 1.0;
      A.partials[pc * 3 + 1] = (double)accp;
      A.partials[pc * 3 + 2] = (double)(rej ? oldH : newH);
    }
    stamp();  // write-back issued
    if (prof) pa.prof[63] = (long long)pi;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

}  // namespace ehmc
