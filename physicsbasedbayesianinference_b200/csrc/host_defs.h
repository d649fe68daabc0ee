// Host-side definitions shared by the translation units of _ehmc.so.
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <vector>

#include "../../include/ehmc.h"
#include "common.cuh"

// ---- errors ------------------------------------------------------------------
int ehmc_fail(int code, const char* fmt, ...);
#define fail ehmc_fail

#define CUDA_TRY(expr)                                                                                         \
  do {                                                                                                         \
    cudaError_t e__ = (expr);                                                                                  \
    if (e__ != cudaSuccess)                                                                                    \
      return fail(EHMC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

#define TRY(expr)                     \
  do {                                \
    int rc__ = (expr);                \
    if (rc__ != EHMC_OK) return rc__; \
  } while (0)

// ---- context / potential objects ------------------------------------------------
struct DevBuf {
  void* ptr = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes);
  void release();
};

constexpr int N_STAGE = 3;  // host path: chunks in flight

struct ehmc_ctx {
  int device = 0;
  cudaDeviceProp prop;
  uint64_t launches = 0;
  long long last_rows = 0;  // rows of statistics partials the last trajectory launch wrote
  DevBuf partials;        // block partial sums for the statistics
  DevBuf stage[N_STAGE];  // host path staging (one slab per in-flight chunk)
  DevBuf stage_stats;
  DevBuf pstats;          // per-particle statistics rows [P][3] (CTA-per-particle / unfused families)
  DevBuf uf[N_STAGE];     // scratch of the unfused path: w, v, g [D][P] + K0, U0, U1 [P]
  // endpoint cache of the unfused (logistic) family: grad U and U at the position the last ehmc_hmc_iter kept
  DevBuf ep_grad[2], ep_energy[2];
  int ep_cur = 0;                  // slot holding the valid cache
  bool ep_valid = false;
  bool ep_enabled = false;         // set by the device path of ehmc_hmc_iter only (the host path stages chunks)
  const void* ep_q = nullptr;      // identity of the cached call: q pointer, potential, P, dtype
  const ehmc_potential* ep_pot = nullptr;
  long long ep_P = 0;
  int ep_bits = 0;
  cudaStream_t streams[N_STAGE] = {nullptr, nullptr, nullptr};
  // tuning options (ehmc_ctx_set_option)
  int small_waves = 8;            // k_small grid = this many resident waves of CTAs (grid-stride over particles)
  int nbody_ti = 0;               // bodies per thread of k_nbody: 0 auto, 4 or 8
  int dense_occupancy = 2;        // CTAs/SM the float32 dense kernel is compiled for (1 or 2)
  int dense_path = 0;             // 0 auto (3xFP16 tensor cores when eligible), 1 CUDA cores (exact fp32 FMA),
                                  // 4 force 3xFP16 (even when the split of Lambda loses accuracy)
  long long host_chunk_bytes = 32LL << 20;
  int tc_prof = 0;                // 1: record a clock64 trace of CTA 0 into tc_prof_buf (64 x int64)
  DevBuf tc_prof_buf;
  int ens_groups = 0;             // fused ensemble run: groups of batches per iteration at most (one float64 row each); 0 = auto
  int ens_sshift = -1;            // fused ensemble run: log2(sub-batches per queue item), -1 = by shard size
  int ens_debug = 0;              // iterations of the fused ensemble run whose phase stamps are recorded
  DevBuf ens_dbg_buf;
  DevBuf ens_ctl;                 // control block of the fused ensemble run: step-size schedule, tickets, partial rows
  DevBuf overflow;                // unsigned: integrate() rows that saturated the fp16 operand range of k_dense_tc3
  int tc_debug = 0;               // profiling knobs of the tensor-core kernels (see DenseTcArgs::dbg)
};

// Per-family state of a potential: what that family's launchers and eval read.  Device arrays hold the dtype of the
// potential (float / double) unless noted.
struct DenseState {                 // dense Gaussian (and the diagonal family for 32 < D <= 128)
  void* lambda = nullptr;           // Lambda [D][D] row-major (k_eval_dense)
  void* mu = nullptr;               // mu [D]; D > 16: zero padded to 8 TN
  void* ls = nullptr;               // D > 16: Lambda transposed and padded for k_dense [D][8][TNP]
  int tn = 0;                       // D > 16: rows of Lambda per warp of k_dense
  std::vector<double> h_lambda, h_mu;  // D <= 16: host copies (make_dense_small)
  struct {                          // float32, D > 16: 3xFP16 tensor-core operands (pack_dense_tc3)
    void* hi = nullptr;             // fp16 [KP/8][NP][8] rn16(scale * Lambda)
    void* lo = nullptr;             // fp16 [KP/8][NP][8] rn16(scale * Lambda - hi)
    void* mu = nullptr;             // float [128], zero padded
    int c8 = 0;                     // ceil(D / 8) (0 = not packed)
    bool exact = false;             // the (hi, lo) split represents Lambda to float32 accuracy (the auto guard)
    float inv_scale = 1.f;          // 1 / scale (power of two)
  } tc3;
};

// gradient kernel of the logistic family: the values of the precision selector (its second scalar) but auto (3)
enum LogisticKernel { LOGISTIC_EXACT = 0, LOGISTIC_BF16 = 1, LOGISTIC_FP16X3 = 2 };

struct LogisticState {
  int n = 0;                        // data rows
  double priorScale = 1.0;          // s of the Gaussian prior N(0, s^2 I) on the coefficients
  LogisticKernel kernel = LOGISTIC_EXACT;  // resolved from the selector (auto decides here, once)
  void* x = nullptr;                // exact kernel: X [N][D]
  void* y = nullptr;                // exact kernel: y [N]
  struct {                          // tensor-core kernels: X and y in 64-row chunks (pack_logistic_tc)
    void* buf = nullptr;            // bf16: NC chunks; fp16 split: 2 NC ring entries (lo, hi)
    int nc = 0, dp = 0, npad = 0;   // chunks, D rounded up to 16, zero rows appended to the last chunk
    unsigned bytes = 0;             // one chunk / ring entry
    float x_iscale = 1.f;           // fp16 split: 1 / (power-of-two scale of X)
  } chunks;
};

struct NBodyState {
  void* body_mass = nullptr;        // [B]
  int b = 0;                        // bodies per particle
  double G = 0.0, eps = 0.0;        // gravitational constant, softening length (eps = 0: the unsoftened kernel)
};

struct DiagState {                  // diagonal Gaussian, D <= 32 (make_diag)
  std::vector<double> k;
};

struct CoinState {                  // coin toss (make_coin)
  std::vector<double> k, n;         // successes, trials
};

struct FunnelState {                // the funnel of v = scaleV q[0], x_k = scaleX q[k] (make_funnel)
  double sigmaV = 1.0, scaleV = 1.0, scaleX = 1.0;
};

struct HierarchicalState {          // hierarchical normal model (make_hier), float64 host tables
  std::vector<double> y, w;         // y [J], w = 1 / sigma^2 [J]
  std::vector<double> scale;        // coordinate scale [J + 2] (ones without rescaling)
  double muLoc = 0.0, muScale = 1.0, tauScale = 1.0;
  bool centered = false;
};

struct ehmc_potential {
  ehmc_ctx* ctx = nullptr;
  int family = 0;
  int D = 0;
  int bits = 32;
  DiagState diag;
  CoinState coin;
  FunnelState funnel;
  DenseState dense;
  LogisticState logistic;
  NBodyState nbody;
  HierarchicalState hier;
};

// peer-memory mailboxes of the fused ensemble run (comm.cu)
struct ehmc_comm {
  ehmc_ctx* ctx = nullptr;
  int rank = 0, world = 1;
  size_t bytes = 0;
  void* mailbox = nullptr;                       // [2][world][ENS_MB_STRIDE] doubles, local
  double* peers[EHMC_COMM_MAX_RANKS] = {};       // every rank's mailbox as mapped into this process
  bool opened[EHMC_COMM_MAX_RANKS] = {};
  double** peers_dev = nullptr;                  // device copy of peers[]
  bool connected = false;
  unsigned long long seq = 0;                    // iterations reduced so far (identical on all ranks)
};

// ---- potential builders and launchers (explicitly instantiated for float / double in inst_*.cu) ----------
namespace ehmc {

constexpr int K1_THREADS_HOST = 128;
constexpr int K2_WARPS_HOST = 8;

// new device array holding `bytes` host bytes (*dptr = nullptr, nothing allocated, for 0 bytes)
int upload_raw(const void* src, size_t bytes, void** dptr);
// new device array of T holding h converted entry by entry
template <typename T>
int upload(const std::vector<double>& h, void** dptr) {
  const std::vector<T> t(h.begin(), h.end());
  return upload_raw(t.data(), sizeof(T) * t.size(), dptr);
}

// Builders: the device state of a potential whose parameters ehmc_potential_create has checked (host, float64).
// On failure the buffers allocated so far stay in the state for ehmc_potential_destroy.
template <typename T>
int build_dense(ehmc_potential* p, std::vector<double>& lambda, std::vector<double>& mu);  // takes the vectors at D <= 16
int pack_dense_tc3(ehmc_potential* p, const std::vector<double>& lambda, const std::vector<double>& mu);
template <typename T>
int build_logistic(ehmc_potential* p, const std::vector<double>& X, const std::vector<double>& y, int precision);
int pack_logistic_tc(ehmc_potential* p, const std::vector<double>& X, const std::vector<double>& y, int precision);
template <typename T>
int build_nbody(ehmc_potential* p, const std::vector<double>& body_mass);

// whether p has a register-resident kernel (with_small_pot, inst_small.cuh): the only potentials the fused
// multi-iteration runs cover
bool has_small_kernel(const ehmc_potential* p);
// fused trajectory kernels, D <= 32 register-resident families
template <typename T>
int launch_small(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st);
// getSamples' whole loop in one launch (small-D families, Philox draws)
template <typename T>
int run_small(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, const RunArgs<T>& R, cudaStream_t st);
// the adaptive ensemble run as one persistent launch (k_small_ens.cuh)
template <typename T>
struct EnsRunArgs;
template <typename T>
int run_small_ens(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, const EnsRunArgs<T>& R, cudaStream_t st);
// dense Gaussian, 16 < D <= 128
template <typename T>
int launch_dense(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st);
// float32 3xFP16 persistent tensor-core variant (leapfrog and Stormer-Verlet; the default)
int launch_dense_tc3(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<float>& A, int integ, bool hmc, cudaStream_t st);
template <typename T>
int dense_particles_per_cta();
int dense_tn(int D);
template <typename T>
int dense_tnp(int TN);
// potential evaluation for the register-resident families
template <typename T>
int eval_small(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
               long long g_ld, cudaStream_t st);

// pairwise gravitational family (one CTA per ensemble particle)
template <typename T>
int launch_nbody(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st);
template <typename T>
int eval_nbody(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
               long long g_ld, cudaStream_t st);
// sum_i q[d,i], sum_i q[d,i]^2 -> out[3 + d], out[3 + D + d]
template <typename T>
int colstats(ehmc_ctx* c, const T* q, long long q_ld, long long P, int D, double* out, cudaStream_t st);
// logistic regression: unfused trajectory driver (gradient kernel + kick/drift kernels)
template <typename T>
int launch_logistic(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc, cudaStream_t st,
                    int slot);
// bf16 tensor-core gradient (float32 state only)
int logistic_grad_tc(ehmc_ctx* c, const ehmc_potential* p, const float* theta, long long t_ld, long long P, float* g,
                     long long g_ld, float* e, double* e64, cudaStream_t st);
// float32-accurate tensor-core gradient: 3-pass fp16 split (float32 state only)
int logistic_grad_tcs(ehmc_ctx* c, const ehmc_potential* p, const float* theta, long long t_ld, long long P, float* g,
                      long long g_ld, float* e, double* e64, cudaStream_t st);
template <typename T>
int eval_logistic(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
                  long long g_ld, cudaStream_t st);

}  // namespace ehmc
