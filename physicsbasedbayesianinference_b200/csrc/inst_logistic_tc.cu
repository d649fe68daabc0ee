#include <algorithm>
#include <cstring>

#include "host_defs.h"
#include "k_logistic_tc.cuh"
#include "k_logistic_tcs.cuh"

namespace ehmc {

// X [N][D] and y [N] of a float32 potential in 64-row chunks for the tensor-core gradients; precision 1 (bf16), 2 (fp16
// split) or 3 (auto: the fp16 split where it represents X to float32 accuracy, else the exact kernel).  Sets
// p->logistic.kernel; the chunks are uploaded only for a tensor-core kernel.
int pack_logistic_tc(ehmc_potential* p, const std::vector<double>& X, const std::vector<double>& y, int precision) {
  LogisticState& s = p->logistic;
  const int D = p->D, N = s.n, DP = (D + 15) / 16 * 16, NB = LT_NB, NC = (N + NB - 1) / NB;
  size_t bytes = 0;
  std::vector<unsigned char> buf;
  if (precision >= LOGISTIC_FP16X3) {
    // float32-accurate path (k_logistic_tcs): X * 2^a as fp16 (hi, lo) pairs, half-chunk ring entries
    // [DP/8][64][8] fp16 + 64 floats (2^10 y in the hi entry).  Guard (auto only): one power-of-two scale serves
    // the whole matrix, so a column whose entries sit more than ~2^10 below max |X| has its lo parts in fp16's
    // subnormal range; if any column's worst split error exceeds 2^-20 of the column's own max, auto selects the
    // exact CUDA-core kernel instead.
    const Fp16Split split(X, 8);
    bytes = (size_t)DP * NB * 2 + NB * 4;
    buf.assign(bytes * 2 * NC, 0);
    std::vector<double> colmax(D, 0.0), colerr(D, 0.0);
    for (int c = 0; c < NC; ++c) {
      // ring order: entry 2c = Xl, entry 2c + 1 = Xh followed by 2^10 y (the small products run first)
      __half* xl = reinterpret_cast<__half*>(buf.data() + bytes * (2 * c));
      __half* xh = reinterpret_cast<__half*>(buf.data() + bytes * (2 * c + 1));
      float* ky = reinterpret_cast<float*>(buf.data() + bytes * (2 * c + 1) + (size_t)DP * NB * 2);
      for (int r = 0; r < NB; ++r) {
        const int n = c * NB + r;
        ky[r] = 1024.f * (n < N ? (float)y[n] : 0.5f);
        if (n >= N) continue;
        for (int d = 0; d < D; ++d) {
          const size_t o = ((size_t)(d / 8) * NB + r) * 8 + (d % 8);
          double rem;
          const float x = split(X[(size_t)n * D + d], &xh[o], &xl[o], &rem);
          colmax[d] = std::max(colmax[d], (double)std::fabs(x));
          colerr[d] = std::max(colerr[d], std::fabs(rem));
        }
      }
    }
    bool ok = std::isfinite(split.amax);
    for (int d = 0; d < D && ok; ++d) ok = colerr[d] <= colmax[d] * 9.5367431640625e-7;  // 2^-20
    if (precision == 3 && !ok) return EHMC_OK;  // auto: s.kernel stays LOGISTIC_EXACT
    s.kernel = LOGISTIC_FP16X3;
    s.chunks.x_iscale = (float)std::ldexp(1.0, -split.shift);
  } else {
    // bf16 chunks of 64 data rows in the canonical UMMA layout [DP/8][64][8] + y[64] (float) (k_logistic_tc)
    bytes = (size_t)DP * NB * 2 + NB * 4 + NB * 2;  // X | y float | (1/2 - y) half
    buf.assign(bytes * NC, 0);
    auto bf16 = [](float f) -> uint16_t {
      uint32_t b;
      memcpy(&b, &f, 4);
      b += 0x7FFFu + ((b >> 16) & 1u);  // round to nearest even
      return (uint16_t)(b >> 16);
    };
    for (int c = 0; c < NC; ++c) {
      uint16_t* xs = reinterpret_cast<uint16_t*>(buf.data() + bytes * c);
      float* ys = reinterpret_cast<float*>(buf.data() + bytes * c + (size_t)DP * NB * 2);
      __half* cs = reinterpret_cast<__half*>(buf.data() + bytes * c + (size_t)DP * NB * 2 + NB * 4);
      for (int r = 0; r < NB; ++r) {
        const int n = c * NB + r;
        ys[r] = n < N ? (float)y[n] : 0.5f;
        cs[r] = __float2half_rn(0.5f - ys[r]);
        if (n >= N) continue;
        for (int d = 0; d < D; ++d) xs[((size_t)(d / 8) * NB + r) * 8 + (d % 8)] = bf16((float)X[(size_t)n * D + d]);
      }
    }
    s.kernel = LOGISTIC_BF16;
  }
  s.chunks.nc = NC;
  s.chunks.dp = DP;
  s.chunks.npad = NC * NB - N;
  s.chunks.bytes = (unsigned)bytes;
  return upload_raw(buf.data(), buf.size(), &s.chunks.buf);
}

// One launch of a tensor-core gradient kernel, with or without the energy (WITH_E = true / false), on `sm` bytes of
// shared memory.  Wave quantisation: T tiles on S SMs take ceil(T / S) rounds; splitting every tile over two halves
// of the data rows doubles the units of work (config 3: 512 tiles, 148 SMs: 4 rounds for 3.46 -> 7 for 6.92).
template <class Args, class Kernel>
static int launch_grad_tc(ehmc_ctx* c, const ehmc_potential* p, Args pa, size_t sm, int threads, Kernel with_e,
                          Kernel without_e, const float* theta, long long t_ld, long long P, float* g, long long g_ld,
                          float* e, double* e64, cudaStream_t st) {
  const long long tiles = (P + LT_M - 1) / LT_M;
  const int sms = c->prop.multiProcessorCount;
  auto waste = [&](long long units) { return (double)((units + sms - 1) / sms) * sms / (double)units; };
  pa.split = (pa.NC >= 2 && waste(2 * tiles) + 0.03 < waste(tiles)) ? 2 : 1;
  if (pa.split == 2) {
    if (g != nullptr) CUDA_TRY(cudaMemset2DAsync(g, (size_t)g_ld * sizeof(float), 0, (size_t)P * sizeof(float), (size_t)p->D, st));
    if (e != nullptr) CUDA_TRY(cudaMemsetAsync(e, 0, (size_t)P * sizeof(float), st));
    if (e64 != nullptr) CUDA_TRY(cudaMemsetAsync(e64, 0, (size_t)P * sizeof(double), st));
  }
  const unsigned grid = (unsigned)(tiles * pa.split);
  auto k = (e != nullptr || e64 != nullptr) ? with_e : without_e;
  CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  k<<<grid, threads, sm, st>>>(theta, t_ld, P, g, g_ld, e, e64, pa);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

int logistic_grad_tc(ehmc_ctx* c, const ehmc_potential* p, const float* theta, long long t_ld, long long P, float* g,
                     long long g_ld, float* e, double* e64, cudaStream_t st) {
  const LogisticState& s = p->logistic;
  LogisticTcArgs pa;
  pa.chunks = static_cast<const unsigned char*>(s.chunks.buf);
  pa.NC = s.chunks.nc;
  pa.DP = s.chunks.dp;
  pa.D = p->D;
  pa.n_pad = s.chunks.npad;
  pa.chunk_bytes = s.chunks.bytes;
  pa.inv_s2 = (float)(1.0 / (s.priorScale * s.priorScale));
  const size_t fixed = 2 * LT_M * 8 + (2 * LT_MAX_STAGES + 5) * 8 + 16;
  pa.stages = (int)std::min<size_t>(LT_MAX_STAGES, (227 * 1024 - fixed) / pa.chunk_bytes);
  if (pa.stages < 2) return fail(EHMC_ERR_UNSUPPORTED, "logistic tensor-core kernel: chunk of %u B does not fit twice", pa.chunk_bytes);
  const size_t sm = (size_t)pa.stages * pa.chunk_bytes + fixed;
  return launch_grad_tc(c, p, pa, sm, LT_THREADS, k_logistic_tc<true>, k_logistic_tc<false>, theta, t_ld, P, g, g_ld, e,
                        e64, st);
}

// float32-accurate variant: 3-pass fp16 split of both GEMMs (k_logistic_tcs.cuh)
int logistic_grad_tcs(ehmc_ctx* c, const ehmc_potential* p, const float* theta, long long t_ld, long long P, float* g,
                      long long g_ld, float* e, double* e64, cudaStream_t st) {
  const LogisticState& s = p->logistic;
  LogisticTcsArgs pa;
  pa.entries = static_cast<const unsigned char*>(s.chunks.buf);
  pa.NC = s.chunks.nc;
  pa.DP = s.chunks.dp;
  pa.D = p->D;
  pa.n_pad = s.chunks.npad;
  pa.entry_bytes = s.chunks.bytes;
  pa.inv_s2 = (float)(1.0 / (s.priorScale * s.priorScale));
  pa.x_iscale = s.chunks.x_iscale;
  const size_t fixed = (size_t)pa.DP * LT_M * 2 + (2 * LT_MAX_STAGES + 6) * 8 + 16;  // Theta_lo + barriers + TMEM slot
  pa.stages = (int)std::min<size_t>(LT_MAX_STAGES, (227 * 1024 - fixed) / pa.entry_bytes);
  if (pa.stages < LTS_MIN_STAGES)
    return fail(EHMC_ERR_UNSUPPORTED, "logistic tensor-core kernel (fp16 split): %d ring entries of %u B fit, %d needed",
                pa.stages, pa.entry_bytes, LTS_MIN_STAGES);
  const size_t sm = (size_t)pa.stages * pa.entry_bytes + fixed;
  return launch_grad_tc(c, p, pa, sm, LTS_THREADS, k_logistic_tcs<true>, k_logistic_tcs<false>, theta, t_ld, P, g,
                        g_ld, e, e64, st);
}

}  // namespace ehmc
