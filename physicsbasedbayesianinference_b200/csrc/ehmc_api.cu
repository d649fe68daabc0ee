// C-ABI of the ehmc engine (include/ehmc.h): argument validation, kernel dispatch, host-buffer staging.  The device
// state of each potential family is built beside that family's launchers (build_* / pack_* in inst_*).  No torch
// types, no exceptions.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only (dlopens the tools library only when a profiler is attached)

#include "host_defs.h"
#include "k_misc.cuh"
#include "k_small_ens.cuh"

// NVTX range around a C-ABI call (SURVEY section 5: the reference's only tracing is cProfile around integrate())
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

using namespace ehmc;

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";
// CUDA device of the device tensors parsed since the last entry point bound its context (-1: none yet), and whether
// two of them disagreed; checked and cleared by enter_device(), cleared by every failure
static thread_local int g_dev_seen = -1;
static thread_local bool g_dev_mixed = false;

int ehmc_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  g_dev_seen = -1;
  g_dev_mixed = false;
  va_end(ap);
  return code;
}

int DevBuf::ensure(size_t bytes) {
  if (bytes <= cap) return EHMC_OK;
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
  const size_t want = bytes + bytes / 8;
  if (cudaMalloc(&ptr, want) != cudaSuccess) {
    cudaGetLastError();
    return fail(EHMC_ERR_NOMEM, "cudaMalloc(%zu) failed", want);
  }
  cap = want;
  return EHMC_OK;
}

void DevBuf::release() {
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
}

// ---------------------------------------------------------------------------
// DLTensor views
// ---------------------------------------------------------------------------
struct View {
  char* data = nullptr;
  int bits = 0;
  int code = 0;
  bool host = false;
  int ndim = 0;
  long long shape[2] = {1, 1};
  long long ld = 0;  // elements between rows (2-D) ; 1-D: unused
};

static int parse(const DLTensor* t, const char* name, int ndim, View* v) {
  if (t == nullptr) return fail(EHMC_ERR_INVALID, "%s: NULL tensor", name);
  if (t->ndim != ndim) return fail(EHMC_ERR_INVALID, "%s: expected %d-D tensor, got %d-D", name, ndim, t->ndim);
  if (t->dtype.lanes != 1) return fail(EHMC_ERR_INVALID, "%s: vector dtypes unsupported", name);
  v->bits = t->dtype.bits;
  v->code = t->dtype.code;
  v->ndim = ndim;
  switch (t->device.device_type) {
    case kDLCUDA:
    case kDLCUDAManaged:
      v->host = false;
      if (g_dev_seen >= 0 && g_dev_seen != t->device.device_id) g_dev_mixed = true;
      g_dev_seen = t->device.device_id;
      break;
    case kDLCPU:
    case kDLCUDAHost:
      v->host = true;
      break;
    default:
      return fail(EHMC_ERR_INVALID, "%s: unsupported device type %d", name, t->device.device_type);
  }
  for (int i = 0; i < ndim; ++i) {
    v->shape[i] = t->shape[i];
    if (t->shape[i] < 0) return fail(EHMC_ERR_INVALID, "%s: negative extent", name);
  }
  const long long inner = t->strides ? t->strides[ndim - 1] : 1;
  if (inner != 1 && v->shape[ndim - 1] > 1)
    return fail(EHMC_ERR_INVALID, "%s: innermost (particle) stride must be 1, got %lld", name, inner);
  if (ndim == 2) {
    v->ld = t->strides ? t->strides[0] : t->shape[1];
    if (v->shape[0] > 1 && v->ld < v->shape[1])
      return fail(EHMC_ERR_INVALID, "%s: row stride %lld < row length %lld", name, v->ld, v->shape[1]);
    if (v->shape[0] <= 1 && v->ld < v->shape[1]) v->ld = v->shape[1];
  }
  v->data = static_cast<char*>(t->data) + t->byte_offset;
  if (v->data == nullptr && v->shape[0] * v->shape[1] > 0) return fail(EHMC_ERR_INVALID, "%s: NULL data", name);
  return EHMC_OK;
}

static int parse_float(const DLTensor* t, const char* name, int ndim, int bits, View* v) {
  TRY(parse(t, name, ndim, v));
  if (v->code != kDLFloat || (v->bits != 32 && v->bits != 64))
    return fail(EHMC_ERR_INVALID, "%s: dtype must be float32 or float64", name);
  if (bits && v->bits != bits)
    return fail(EHMC_ERR_INVALID, "%s: dtype float%d does not match float%d of the call", name, v->bits, bits);
  return EHMC_OK;
}

// Binds the calling thread to the context's device -- after checking that every device tensor parsed for this call
// lives there: a kernel launched on the context's device with another device's pointers is an illegal address at
// best and silent peer access at worst.
static int enter_device(const ehmc_ctx* ctx) {
  const int seen = g_dev_seen;
  const bool mixed = g_dev_mixed;
  g_dev_seen = -1;
  g_dev_mixed = false;
  if (mixed) return fail(EHMC_ERR_INVALID, "the device tensors of the call live on different CUDA devices");
  if (seen >= 0 && seen != ctx->device)
    return fail(EHMC_ERR_INVALID, "tensor on cuda:%d handed to a context bound to cuda:%d", seen, ctx->device);
  CUDA_TRY(cudaSetDevice(ctx->device));
  return EHMC_OK;
}

// ---------------------------------------------------------------------------
// library / context
// ---------------------------------------------------------------------------
extern "C" int ehmc_version(void) { return EHMC_VERSION; }

extern "C" const char* ehmc_last_error(const ehmc_ctx*) { return g_err; }

extern "C" int ehmc_ctx_create(int device, ehmc_ctx** out) {
  if (out == nullptr) return fail(EHMC_ERR_INVALID, "ehmc_ctx_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(EHMC_ERR_CUDA, "no usable CUDA device (%s); ehmc has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  }
  if (device < 0) CUDA_TRY(cudaGetDevice(&device));
  if (device >= n) return fail(EHMC_ERR_INVALID, "device %d out of range (%d devices)", device, n);
  ehmc_ctx* c = new (std::nothrow) ehmc_ctx();
  if (!c) return fail(EHMC_ERR_NOMEM, "out of host memory");
  c->device = device;
  if (cudaGetDeviceProperties(&c->prop, device) != cudaSuccess) {
    delete c;
    return fail(EHMC_ERR_CUDA, "cudaGetDeviceProperties failed");
  }
  if (c->prop.major < 10) {
    const int major = c->prop.major, minor = c->prop.minor;
    delete c;
    return fail(EHMC_ERR_CUDA, "device is sm_%d%d; this library is built for sm_100a (B200) only", major, minor);
  }
  *out = c;
  return EHMC_OK;
}

extern "C" int ehmc_ctx_destroy(ehmc_ctx* c) {
  if (!c) return EHMC_OK;
  cudaSetDevice(c->device);
  c->partials.release();
  c->stage_stats.release();
  c->pstats.release();
  c->tc_prof_buf.release();
  c->overflow.release();
  c->ens_ctl.release();
  c->ens_dbg_buf.release();
  for (int k = 0; k < 2; ++k) {
    c->ep_grad[k].release();
    c->ep_energy[k].release();
  }
  for (int i = 0; i < N_STAGE; ++i) {
    c->stage[i].release();
    c->uf[i].release();
    if (c->streams[i]) cudaStreamDestroy(c->streams[i]);
  }
  delete c;
  return EHMC_OK;
}

extern "C" int ehmc_ctx_launch_count(const ehmc_ctx* c, uint64_t* out) {
  if (!c || !out) return fail(EHMC_ERR_INVALID, "ehmc_ctx_launch_count: NULL argument");
  *out = c->launches;
  return EHMC_OK;
}

extern "C" int ehmc_ctx_overflow_count(ehmc_ctx* c, uint64_t* out, int reset) {
  if (!c || !out) return fail(EHMC_ERR_INVALID, "ehmc_ctx_overflow_count: NULL argument");
  *out = 0;
  if (c->overflow.ptr == nullptr) return EHMC_OK;
  CUDA_TRY(cudaSetDevice(c->device));
  unsigned v = 0;
  CUDA_TRY(cudaMemcpy(&v, c->overflow.ptr, sizeof(v), cudaMemcpyDeviceToHost));  // synchronises the device
  if (reset && v) CUDA_TRY(cudaMemset(c->overflow.ptr, 0, sizeof(v)));
  *out = v;
  return EHMC_OK;
}

extern "C" int ehmc_ctx_device_info(const ehmc_ctx* c, double out[4]) {
  if (!c || !out) return fail(EHMC_ERR_INVALID, "ehmc_ctx_device_info: NULL argument");
  int clk = 0;
  cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, c->device);
  out[0] = c->prop.multiProcessorCount;
  out[1] = clk / 1000.0;
  out[2] = (double)c->prop.totalGlobalMem;
  out[3] = (double)c->prop.l2CacheSize;
  return EHMC_OK;
}

extern "C" int ehmc_ctx_set_option(ehmc_ctx* c, const char* name, double value) {
  if (!c || !name) return fail(EHMC_ERR_INVALID, "ehmc_ctx_set_option: NULL argument");
  if (!strcmp(name, "dense_occupancy")) {
    if (value != 1 && value != 2) return fail(EHMC_ERR_INVALID, "dense_occupancy must be 1 or 2");
    c->dense_occupancy = (int)value;
  } else if (!strcmp(name, "dense_path")) {
    if (value != 0 && value != 1 && value != 4)
      return fail(EHMC_ERR_INVALID, "dense_path must be 0 (auto), 1 (CUDA cores) or 4 (force the 3xFP16 tensor-core kernel)");
    c->dense_path = (int)value;
  } else if (!strcmp(name, "tc_prof")) {
    c->tc_prof = (int)value;
    if (c->tc_prof) {
      TRY(c->tc_prof_buf.ensure(64 * sizeof(long long)));
      CUDA_TRY(cudaMemset(c->tc_prof_buf.ptr, 0, 64 * sizeof(long long)));
    }
  } else if (!strcmp(name, "tc_prof_dump")) {
    // debugging aid: print the trace to stderr
    if (c->tc_prof_buf.ptr) {
      long long h[64];
      CUDA_TRY(cudaMemcpy(h, c->tc_prof_buf.ptr, sizeof(h), cudaMemcpyDeviceToHost));
      // k_dense_tc3 stores the number of stamps in h[63] (absolute clocks); the older kernels store the start clock
      const bool counted = h[63] > 0 && h[63] < 63;
      const long long base = counted ? h[0] : h[63];
      fprintf(stderr, "tc_prof:");
      for (int i = 0; i < (counted ? (int)h[63] : 62) && h[i]; ++i) fprintf(stderr, " %lld", h[i] - base);
      fprintf(stderr, "\n");
    }
  } else if (!strcmp(name, "small_waves")) {
    if (!(value >= 1 && value <= 1e6)) return fail(EHMC_ERR_INVALID, "small_waves must be in [1, 1e6]");
    c->small_waves = (int)value;
  } else if (!strcmp(name, "nbody_ti")) {
    if (value != 0 && value != 4 && value != 8) return fail(EHMC_ERR_INVALID, "nbody_ti must be 0, 4 or 8");
    c->nbody_ti = (int)value;
  } else if (!strcmp(name, "ens_groups")) {
    if (!(value >= 0 && value <= 8192)) return fail(EHMC_ERR_INVALID, "ens_groups must be in [0, 8192] (0 = auto)");
    c->ens_groups = (int)value;
  } else if (!strcmp(name, "ens_sshift")) {
    if (!(value >= -1 && value <= 4)) return fail(EHMC_ERR_INVALID, "ens_sshift must be in [-1, 4]");
    c->ens_sshift = (int)value;
  } else if (!strcmp(name, "ens_debug")) {
    if (!(value >= 0 && value <= 65536)) return fail(EHMC_ERR_INVALID, "ens_debug must be in [0, 65536]");
    c->ens_debug = (int)value;
  } else if (!strcmp(name, "ens_debug_dump")) {
    // debugging aid: phase stamps of the last fused ensemble run (ns relative to the first), to stderr
    if (c->ens_dbg_buf.ptr && c->ens_debug > 0) {
      std::vector<long long> hbuf((size_t)8 * (c->ens_debug + 1));
      CUDA_TRY(cudaMemcpy(hbuf.data(), c->ens_dbg_buf.ptr, sizeof(long long) * hbuf.size(), cudaMemcpyDeviceToHost));
      const int first = (int)value;
      {
        const long long* t = &hbuf[(size_t)8 * c->ens_debug];  // totals over the compute warps of the launch
        fprintf(stderr, "ens_debug totals: %lld compute warps; mean wait per warp: %.1f us for the group mark, %.1f us "
                "for the step size\n", t[2], t[2] ? 1e-3 * (double)t[0] / (double)t[2] : 0.0,
                t[2] ? 1e-3 * (double)t[1] / (double)t[2] : 0.0);
      }
      for (int it = first; it < c->ens_debug && hbuf[(size_t)8 * it]; ++it) {
        const long long* r = &hbuf[(size_t)8 * it];
        fprintf(stderr, "ens_debug it %d: master: tickets of it at %lld, +reduce %lld +push %lld +peers %lld +publish %lld | "
                "cta0: start %lld, waited %lld for h, end %lld | master period %lld\n", it, r[0] - hbuf[0], r[1] - r[0],
                r[2] ? r[2] - r[1] : 0LL, r[2] ? r[3] - r[2] : 0LL, r[4] - (r[2] ? r[3] : r[1]), r[5] - hbuf[0], r[6],
                r[7] - hbuf[0], it > 0 ? r[0] - r[-8] : 0LL);
      }
    }
  } else if (!strcmp(name, "tc_debug")) {
    c->tc_debug = (int)value;
  } else if (!strcmp(name, "host_chunk_mb")) {
    if (!(value >= 1 && value <= 4096)) return fail(EHMC_ERR_INVALID, "host_chunk_mb must be in [1, 4096]");
    c->host_chunk_bytes = (long long)value << 20;
  } else {
    return fail(EHMC_ERR_INVALID, "unknown option '%s'", name);
  }
  return EHMC_OK;
}

extern "C" int ehmc_measure_fp32_peak(ehmc_ctx* c, double millis, double* tflops_out) {
  if (!c || !tflops_out) return fail(EHMC_ERR_INVALID, "ehmc_measure_fp32_peak: NULL argument");
  CUDA_TRY(cudaSetDevice(c->device));
  float* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, 4));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  const int blocks = c->prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  const double flop_per_launch = (double)blocks * threads * iters * 16.0 * 8.0 * 2.0;
  double best = 0.0, elapsed = 0.0;
  k_fma_peak<<<blocks, threads>>>(d, 64, 0.999f, 0.001f);  // warm-up
  c->launches++;
  while (elapsed < millis) {
    cudaEventRecord(e0);
    k_fma_peak<<<blocks, threads>>>(d, iters, 0.999f, 0.001f);
    c->launches++;
    cudaEventRecord(e1);
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    elapsed += ms;
    best = std::max(best, flop_per_launch / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  CUDA_TRY(cudaGetLastError());
  *tflops_out = best;
  return EHMC_OK;
}

// ---------------------------------------------------------------------------
// potentials
// ---------------------------------------------------------------------------
static int fetch_param(const DLTensor* t, const char* name, int ndim, std::vector<double>* out, View* v) {
  TRY(parse_float(t, name, ndim, 0, v));
  const long long rows = ndim == 2 ? v->shape[0] : 1, cols = v->shape[ndim - 1];
  const size_t es = v->bits / 8;
  std::vector<char> tmp((size_t)rows * cols * es);
  const size_t pitch = (ndim == 2 ? v->ld : cols) * es;
  if (rows * cols > 0)
    CUDA_TRY(cudaMemcpy2D(tmp.data(), cols * es, v->data, pitch, cols * es, rows,
                          v->host ? cudaMemcpyHostToHost : cudaMemcpyDeviceToHost));
  out->resize((size_t)rows * cols);
  for (size_t i = 0; i < out->size(); ++i)
    (*out)[i] = v->bits == 32 ? (double)reinterpret_cast<float*>(tmp.data())[i] : reinterpret_cast<double*>(tmp.data())[i];
  return EHMC_OK;
}

int ehmc::upload_raw(const void* src, size_t bytes, void** dptr) {
  *dptr = nullptr;
  if (bytes == 0) return EHMC_OK;
  if (cudaMalloc(dptr, bytes) != cudaSuccess) {
    cudaGetLastError();
    *dptr = nullptr;
    return fail(EHMC_ERR_NOMEM, "cudaMalloc(%zu) failed", bytes);
  }
  CUDA_TRY(cudaMemcpy(*dptr, src, bytes, cudaMemcpyHostToDevice));
  return EHMC_OK;
}

extern "C" int ehmc_potential_create(ehmc_ctx* ctx, int family, const DLTensor* const* params, int nparams,
                                     const double* scalars, int nscalars, int dtype_bits, ehmc_potential** out) {
  if (!ctx || !out) return fail(EHMC_ERR_INVALID, "ehmc_potential_create: NULL argument");
  *out = nullptr;
  if (dtype_bits != 32 && dtype_bits != 64) return fail(EHMC_ERR_INVALID, "dtype_bits must be 32 or 64");
  if (nparams < 0 || nscalars < 0 || (nparams > 0 && !params) || (nscalars > 0 && !scalars))
    return fail(EHMC_ERR_INVALID, "ehmc_potential_create: bad params/scalars");
  TRY(enter_device(ctx));
  ehmc_potential* p = new (std::nothrow) ehmc_potential();
  if (!p) return fail(EHMC_ERR_NOMEM, "out of host memory");
  p->ctx = ctx;
  p->family = family;
  p->bits = dtype_bits;
  const bool f32 = dtype_bits == 32;
  int rc = EHMC_OK;
  View v;
  std::vector<double> a, b;  // the float64 host copies of params[0], params[1]
  switch (family) {
    case EHMC_FAMILY_DIAG_GAUSSIAN: {
      if (nparams != 1) { rc = fail(EHMC_ERR_INVALID, "diag gaussian: params = {k[D]}"); break; }
      rc = fetch_param(params[0], "k", 1, &a, &v);
      if (rc) break;
      p->D = (int)a.size();
      if (p->D < 1) { rc = fail(EHMC_ERR_INVALID, "diag gaussian: empty k"); break; }
      if (p->D > 32 && p->D <= 128) {
        // route through the dense kernel with Lambda = diag(k)
        std::vector<double> lam((size_t)p->D * p->D, 0.0);
        for (int d = 0; d < p->D; ++d) lam[(size_t)d * p->D + d] = a[d];
        a.swap(lam);
        b.assign(p->D, 0.0);
        p->family = EHMC_FAMILY_DENSE_GAUSSIAN;
      } else if (p->D > 128) {
        rc = fail(EHMC_ERR_UNSUPPORTED, "diag gaussian: D = %d > 128 not built", p->D);
      } else {
        p->diag.k.swap(a);
      }
      break;
    }
    case EHMC_FAMILY_DENSE_GAUSSIAN: {
      if (nparams < 1 || nparams > 2) { rc = fail(EHMC_ERR_INVALID, "dense gaussian: params = {Lambda[D,D], mu[D]?}"); break; }
      rc = fetch_param(params[0], "Lambda", 2, &a, &v);
      if (rc) break;
      if (v.shape[0] != v.shape[1] || v.shape[0] < 1) { rc = fail(EHMC_ERR_INVALID, "Lambda must be square"); break; }
      p->D = (int)v.shape[0];
      if (nparams == 2 && params[1] != nullptr) {
        rc = fetch_param(params[1], "mu", 1, &b, &v);
        if (rc) break;
        if ((int)b.size() != p->D) { rc = fail(EHMC_ERR_INVALID, "mu must have D entries"); break; }
      } else {
        b.assign(p->D, 0.0);
      }
      if (p->D > 128) rc = fail(EHMC_ERR_UNSUPPORTED, "dense gaussian: D = %d > 128 not built", p->D);
      break;
    }
    case EHMC_FAMILY_FUNNEL: {
      if (nscalars != 2 && nscalars != 4) { rc = fail(EHMC_ERR_INVALID, "funnel: scalars = {D, sigma_v [, scaleV, scaleX]}"); break; }
      p->D = (int)scalars[0];
      if (p->D < 2 || p->D > 32) { rc = fail(EHMC_ERR_UNSUPPORTED, "funnel: 2 <= D <= 32 (got %d)", p->D); break; }
      FunnelState& s = p->funnel;
      s.sigmaV = scalars[1];
      if (nscalars == 4) {
        s.scaleV = scalars[2];
        s.scaleX = scalars[3];
      }
      if (!(s.sigmaV > 0)) rc = fail(EHMC_ERR_INVALID, "funnel: sigma_v must be > 0");
      else if (!(s.scaleV > 0 && s.scaleX > 0)) rc = fail(EHMC_ERR_INVALID, "funnel: scales must be > 0");
      break;
    }
    case EHMC_FAMILY_COIN_TOSS: {
      if (nparams != 2) { rc = fail(EHMC_ERR_INVALID, "coin toss: params = {successes[D], trials[D]}"); break; }
      CoinState& s = p->coin;
      rc = fetch_param(params[0], "successes", 1, &s.k, &v);
      if (rc) break;
      rc = fetch_param(params[1], "trials", 1, &s.n, &v);
      if (rc) break;
      p->D = (int)s.k.size();
      if (p->D < 1 || p->D > 32) { rc = fail(EHMC_ERR_UNSUPPORTED, "coin toss: 1 <= D <= 32 (got %d)", p->D); break; }
      if ((int)s.n.size() != p->D) { rc = fail(EHMC_ERR_INVALID, "coin toss: trials must have D entries"); break; }
      for (int d = 0; d < p->D && rc == EHMC_OK; ++d)
        if (!(s.k[d] >= 0 && s.n[d] >= s.k[d])) rc = fail(EHMC_ERR_INVALID, "coin toss: need 0 <= successes <= trials");
      break;
    }
    case EHMC_FAMILY_NBODY: {
      if (nparams != 1 || nscalars != 2) { rc = fail(EHMC_ERR_INVALID, "nbody: params = {bodyMass[B]}, scalars = {G, eps}"); break; }
      rc = fetch_param(params[0], "bodyMass", 1, &a, &v);
      if (rc) break;
      const int B = (int)a.size();
      p->D = 3 * B;
      if (B < 1) { rc = fail(EHMC_ERR_INVALID, "nbody: empty bodyMass"); break; }
      if (B > 7000) { rc = fail(EHMC_ERR_UNSUPPORTED, "nbody: B = %d > 7000 bodies", B); break; }
      p->nbody.G = scalars[0];
      p->nbody.eps = scalars[1];
      if (!(p->nbody.eps >= 0)) { rc = fail(EHMC_ERR_INVALID, "nbody: eps must be >= 0"); break; }
      rc = f32 ? build_nbody<float>(p, a) : build_nbody<double>(p, a);
      break;
    }
    case EHMC_FAMILY_LOGISTIC: {
      if (nparams != 2 || nscalars < 1 || nscalars > 2) { rc = fail(EHMC_ERR_INVALID, "logistic: params = {X[N,D], y[N]}, scalars = {priorScale, precision?}"); break; }
      rc = fetch_param(params[0], "X", 2, &a, &v);
      if (rc) break;
      p->logistic.n = (int)v.shape[0];
      p->D = (int)v.shape[1];
      rc = fetch_param(params[1], "y", 1, &b, &v);
      if (rc) break;
      if ((int)b.size() != p->logistic.n) { rc = fail(EHMC_ERR_INVALID, "logistic: y must have N entries"); break; }
      if (p->D < 1 || p->D > 256) { rc = fail(EHMC_ERR_UNSUPPORTED, "logistic: 1 <= D <= 256 (got %d)", p->D); break; }
      p->logistic.priorScale = scalars[0];
      if (!(p->logistic.priorScale > 0)) { rc = fail(EHMC_ERR_INVALID, "logistic: priorScale must be > 0"); break; }
      const int precision = nscalars == 2 ? (int)scalars[1] : 0;
      if (precision < 0 || precision > 3) { rc = fail(EHMC_ERR_INVALID, "logistic: precision selector must be 0 (CUDA cores), 1 (bf16), 2 (fp16 split) or 3 (auto)"); break; }
      if ((precision == 1 || precision == 2) && !f32) { rc = fail(EHMC_ERR_INVALID, "logistic: the tensor-core path needs float32 state"); break; }
      rc = f32 ? build_logistic<float>(p, a, b, precision) : build_logistic<double>(p, a, b, precision);
      break;
    }
    case EHMC_FAMILY_HIERARCHICAL_NORMAL: {
      if ((nparams != 2 && nparams != 3) || nscalars != 4) {
        rc = fail(EHMC_ERR_INVALID, "hierarchical normal: params = {y[J], sigma[J] [, scale[J+2]]}, scalars = {muLoc, muScale, tauScale, centered}");
        break;
      }
      HierarchicalState& h = p->hier;
      rc = fetch_param(params[0], "y", 1, &h.y, &v);
      if (rc) break;
      rc = fetch_param(params[1], "sigma", 1, &b, &v);
      if (rc) break;
      const int J = (int)h.y.size();
      p->D = J + 2;
      if (J < 1) { rc = fail(EHMC_ERR_INVALID, "hierarchical normal: empty y"); break; }
      if (J > 30) { rc = fail(EHMC_ERR_UNSUPPORTED, "hierarchical normal: 1 <= J <= 30 groups (got %d)", J); break; }
      if ((int)b.size() != J) { rc = fail(EHMC_ERR_INVALID, "hierarchical normal: sigma must have J entries"); break; }
      h.w.resize(J);
      for (int j = 0; j < J && rc == EHMC_OK; ++j) {
        if (!std::isfinite(h.y[j])) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: y must be finite");
        else if (!(b[j] > 0 && std::isfinite(b[j]))) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: sigma must be > 0");
        else h.w[j] = 1.0 / (b[j] * b[j]);
      }
      if (rc) break;
      if (nparams == 3 && params[2] != nullptr) {
        rc = fetch_param(params[2], "scale", 1, &h.scale, &v);
        if (rc) break;
        if ((int)h.scale.size() != p->D) { rc = fail(EHMC_ERR_INVALID, "hierarchical normal: scale must have J + 2 entries"); break; }
        for (double x : h.scale)
          if (!(x > 0 && std::isfinite(x))) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: scales must be > 0");
        if (rc) break;
      } else {
        h.scale.assign(p->D, 1.0);
      }
      h.muLoc = scalars[0];
      h.muScale = scalars[1];
      h.tauScale = scalars[2];
      if (!std::isfinite(h.muLoc)) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: muLoc must be finite");
      else if (!(h.muScale > 0 && std::isfinite(h.muScale))) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: muScale must be > 0");
      else if (!(h.tauScale > 0 && std::isfinite(h.tauScale))) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: tauScale must be > 0");
      else if (scalars[3] != 0.0 && scalars[3] != 1.0) rc = fail(EHMC_ERR_INVALID, "hierarchical normal: centered must be 0 or 1");
      h.centered = scalars[3] == 1.0;
      break;
    }
    default:
      rc = fail(EHMC_ERR_UNSUPPORTED, "potential family %d is not built into this library", family);
  }
  if (rc == EHMC_OK && p->family == EHMC_FAMILY_DENSE_GAUSSIAN)
    rc = f32 ? build_dense<float>(p, a, b) : build_dense<double>(p, a, b);
  if (rc != EHMC_OK) {
    ehmc_potential_destroy(p);
    return rc;
  }
  *out = p;
  return EHMC_OK;
}

extern "C" int ehmc_potential_destroy(ehmc_potential* p) {
  if (!p) return EHMC_OK;
  if (p->ctx) cudaSetDevice(p->ctx->device);
  if (p->ctx && p->ctx->ep_pot == p) p->ctx->ep_valid = false;  // a new potential may reuse this address
  const DenseState& d = p->dense;
  for (void* buf : {d.lambda, d.mu, d.ls, d.tc3.hi, d.tc3.lo, d.tc3.mu, p->logistic.x, p->logistic.y,
                    p->logistic.chunks.buf, p->nbody.body_mass})
    if (buf) cudaFree(buf);
  delete p;
  return EHMC_OK;
}

// the float32 dense family runs on the tensor cores unless told otherwise
static bool use_dense_tc(const ehmc_ctx* c, const ehmc_potential* p) {
  if (!(p->family == EHMC_FAMILY_DENSE_GAUSSIAN && p->bits == 32) || c->dense_path == 1) return false;
  return p->dense.tc3.c8 >= 3 && (p->dense.tc3.exact || c->dense_path == 4);  // 0 (auto), 4 (forced): 3xFP16 persistent kernel
}

// families whose trajectory kernel reports statistics per particle ([P][3]) and needs k_colstats
static bool per_particle_stats(const ehmc_ctx* c, const ehmc_potential* p) {
  if (p->family == EHMC_FAMILY_NBODY || p->family == EHMC_FAMILY_LOGISTIC) return true;
  // the 3xFP16 tensor-core dense kernel reports per-particle scalars too
  return use_dense_tc(c, p);
}

// number of CTAs the trajectory kernel uses for P particles (statistics partials)
template <typename T>
static long long traj_blocks(const ehmc_ctx* c, const ehmc_potential* p, long long P) {
  if (per_particle_stats(c, p)) return P;
  if (p->family == EHMC_FAMILY_DENSE_GAUSSIAN && p->D > 16) {
    const int PT = dense_particles_per_cta<T>();
    return (P + PT - 1) / PT;
  }
  return (P + K1_THREADS_HOST - 1) / K1_THREADS_HOST;
}

template <typename T>
static int launch_traj(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, int integ, bool hmc,
                       cudaStream_t st, int slot = 0) {
  c->last_rows = 0;
  if (A.P == 0) return EHMC_OK;
  c->last_rows = traj_blocks<T>(c, p, A.P);  // upper bound == exact for every kernel but the persistent k_small
  if (p->family == EHMC_FAMILY_NBODY) return launch_nbody<T>(c, p, A, integ, hmc, st);
  if (p->family == EHMC_FAMILY_LOGISTIC) return launch_logistic<T>(c, p, A, integ, hmc, st, slot);
  if constexpr (sizeof(T) == 4) {
    if (use_dense_tc(c, p)) return launch_dense_tc3(c, p, A, integ, hmc, st);
  }
  if (c->dense_path == 4 && p->family == EHMC_FAMILY_DENSE_GAUSSIAN && p->D > 16 && sizeof(T) == 4)
    return fail(EHMC_ERR_UNSUPPORTED, "dense_path = 4 (tensor cores) but this call is not eligible (D = %d, integrator %d)", p->D, integ);
  if (p->family == EHMC_FAMILY_DENSE_GAUSSIAN && p->D > 16) return launch_dense<T>(c, p, A, integ, hmc, st);
  return launch_small<T>(c, p, A, integ, hmc, st);
}

// ---------------------------------------------------------------------------
// argument assembly shared by integrate / hmc_iter
// ---------------------------------------------------------------------------
struct CallViews {
  View q, p, mass, z, u, accept, stats;
  bool has_p = false, has_z = false, has_u = false, has_accept = false, has_stats = false;
  int bits = 0;
  long long D = 0, P = 0;
};

static int check_same_place(const CallViews& v) {
  const bool host = v.q.host;
  if (v.mass.host != host || (v.has_p && v.p.host != host) || (v.has_z && v.z.host != host) ||
      (v.has_u && v.u.host != host) || (v.has_accept && v.accept.host != host) ||
      (v.has_stats && v.stats.host != host))
    return fail(EHMC_ERR_INVALID, "all tensors of a call must live on the same side (all host or all device)");
  return EHMC_OK;
}

template <typename T>
static IterArgs<T> base_args(const CallViews& v, double h, double h2, int L) {
  IterArgs<T> A;
  memset(&A, 0, sizeof(A));
  A.q = reinterpret_cast<T*>(v.q.data);
  A.q_ld = v.q.ld;
  A.p = v.has_p ? reinterpret_cast<T*>(v.p.data) : nullptr;
  A.p_ld = v.has_p ? v.p.ld : 0;
  A.mass = reinterpret_cast<const T*>(v.mass.data);
  A.z = v.has_z ? reinterpret_cast<const T*>(v.z.data) : nullptr;
  A.z_ld = v.has_z ? v.z.ld : 0;
  A.u = v.has_u ? reinterpret_cast<const T*>(v.u.data) : nullptr;
  A.accept = v.has_accept ? reinterpret_cast<unsigned char*>(v.accept.data) : nullptr;
  A.partials = nullptr;
  A.P = v.P;
  A.D = (int)v.D;
  A.L = L;
  A.h = (T)h;
  A.h2 = (T)h2;
  return A;
}

// the IterArgs of an HMC entry point
template <typename T>
static IterArgs<T> hmc_args(const CallViews& v, const ehmc_hmc_args* a) {
  IterArgs<T> A = base_args<T>(v, a->stepSize, a->stepSizeSq, a->numSteps);
  A.flags = a->flags;
  A.kB = a->boltzmann;
  A.temp = a->temperature;
  A.pscale = std::sqrt(a->boltzmann * a->temperature);
  A.seed = a->seed;
  A.iter = a->iteration;
  A.offset = a->particleOffset;
  A.dyn = static_cast<const DynArgs*>(a->dynamic);
  return A;
}

enum class HmcEntry { iter, run, ensemble };

// The checks of ehmc_hmc_args (and of the fused ensemble run's ehmc_adapt_args `ad`) the HMC entry points share, in
// each entry point's own words.  `negative`: one of the call's own counts (iterations, offsets) is below 0.
static int check_hmc_args(HmcEntry e, const char* fn, const ehmc_hmc_args* a, const ehmc_adapt_args* ad, bool negative) {
  if (!a) return fail(EHMC_ERR_INVALID, "%s: args is NULL", fn);
  if (e == HmcEntry::ensemble) {
    if (a->struct_size != sizeof(ehmc_hmc_args) || ad->struct_size != sizeof(ehmc_adapt_args))
      return fail(EHMC_ERR_INVALID, "%s: struct_size mismatch", fn);
  } else if (a->struct_size != sizeof(ehmc_hmc_args)) {
    return fail(EHMC_ERR_INVALID, "%s: args.struct_size %u != %zu", fn, a->struct_size, sizeof(ehmc_hmc_args));
  }
  if (a->numSteps < 0 || negative)
    return fail(EHMC_ERR_INVALID, e == HmcEntry::iter ? "%s: numSteps < 0" : "%s: negative count", fn);
  if (e == HmcEntry::ensemble && a->integrator != EHMC_LEAPFROG) return fail(EHMC_ERR_UNSUPPORTED, "%s: leapfrog only", fn);
  if (a->integrator != EHMC_LEAPFROG && a->integrator != EHMC_STORMER_VERLET)
    return fail(EHMC_ERR_INVALID, "%s: Invalid integration method selected.", fn);
  // ehmc_hmc_iter checks args.dynamic against the potential
  if (e != HmcEntry::iter && a->dynamic != nullptr) return fail(EHMC_ERR_UNSUPPORTED, "%s: args.dynamic is not supported here", fn);
  return EHMC_OK;
}

// Device path of one iteration / integration.  Statistics go to stats_dev (device, 2D+3 doubles).
template <typename T>
static int run_device(ehmc_ctx* c, const ehmc_potential* pot, IterArgs<T> A, int integ, bool hmc, double* stats_dev,
                      cudaStream_t st) {
  const bool pps = per_particle_stats(c, pot);
  const int NS = 2 * A.D + 3;
  long long nblk = 0;
  if (stats_dev != nullptr) {
    if (pps) {
      // per-particle scalars [P][3] from the trajectory kernel; reduced together with the coordinate sums below
      nblk = std::max<long long>(1, std::min<long long>(4LL * c->prop.multiProcessorCount, (A.P + 255) / 256));
      TRY(c->pstats.ensure(sizeof(double) * 3 * (size_t)std::max(1LL, A.P)));
      if (A.P >= 16LL * A.D) TRY(c->partials.ensure(sizeof(double) * (size_t)nblk * NS));
      A.partials = static_cast<double*>(c->pstats.ptr);
    } else {
      nblk = traj_blocks<T>(c, pot, A.P);
      TRY(c->partials.ensure(sizeof(double) * (size_t)std::max(1LL, nblk) * NS));
      A.partials = static_cast<double*>(c->partials.ptr);
    }
  }
  c->ep_enabled = true;  // the endpoint cache is only meaningful when one call covers the resident ensemble
  const int rc_traj = launch_traj<T>(c, pot, A, integ, hmc, st);
  c->ep_enabled = false;
  TRY(rc_traj);
  if (stats_dev != nullptr && A.P > 0) {
    double* rows = static_cast<double*>(c->partials.ptr);
    if (pps && A.P < 16LL * A.D) {
      // few particles, many coordinates (N-body): one CTA per statistic / per coordinate
      k_stats_finalize<<<3, 256, 0, st>>>(A.partials, (int)A.P, 3, stats_dev);
      c->launches++;
      CUDA_TRY(cudaGetLastError());
      TRY(colstats<T>(c, A.q, A.q_ld, A.P, A.D, stats_dev, st));
      return EHMC_OK;
    }
    if (pps) {
      // many particles: one streaming pass over pstats and q, particle slices per CTA
      k_ens_stats_partial<T><<<(unsigned)nblk, 256, 0, st>>>(A.partials, A.q, A.q_ld, A.P, A.D, rows);
      c->launches++;
    } else {
      nblk = c->last_rows;
    }
    k_stats_finalize<<<NS, 256, 0, st>>>(rows, (int)nblk, NS, stats_dev);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
  }
  return EHMC_OK;
}

// Host path: particles are processed in column chunks; chunk k uses stream k % N_STAGE with
// its own staging slab, so H2D of chunk k+1 / kernel of chunk k / D2H of chunk k-1 overlap.
template <typename T>
static int run_host(ehmc_ctx* c, const ehmc_potential* pot, const CallViews& v, IterArgs<T> proto, int integ, bool hmc) {
  const long long D = v.D, P = v.P;
  const int NS = 2 * (int)D + 3;
  for (int i = 0; i < N_STAGE; ++i) {
    if (!c->streams[i]) CUDA_TRY(cudaStreamCreateWithFlags(&c->streams[i], cudaStreamNonBlocking));
  }
  // chunk size: multiple of 512 particles, ~32 MB of state per array, at least 3 chunks when P is large
  long long chunk = std::max<long long>(512, c->host_chunk_bytes / (long long)(sizeof(T) * std::max<long long>(D, 1)));
  chunk = (chunk / 512) * 512;
  if (P > 3 * 512 && chunk * N_STAGE > P) chunk = std::max<long long>(512, ((P / N_STAGE + 511) / 512) * 512);
  chunk = std::min(chunk, std::max<long long>(P, 1));
  const long long nchunks = P == 0 ? 0 : (P + chunk - 1) / chunk;
  // slab layout (elements of T): q[D][chunk] p[D][chunk] z[D][chunk] mass[chunk] u[chunk] | accept bytes
  const size_t arr = (size_t)D * chunk;
  const size_t slab_elems = 3 * arr + 2 * (size_t)chunk;
  const size_t slab_bytes = slab_elems * sizeof(T) + (size_t)chunk + 64;
  for (int i = 0; i < N_STAGE; ++i) TRY(c->stage[i].ensure(slab_bytes));
  long long blocks_total = 0;  // upper bound of the statistics rows (exact count: rows_done below)
  for (long long k = 0; k < nchunks; ++k) blocks_total += traj_blocks<T>(c, pot, std::min(chunk, P - k * chunk));
  const bool pps = per_particle_stats(c, pot);
  if (v.has_stats) {
    // fused families: one row of NS sums per CTA.  per-particle families: [P][3] rows in pstats plus
    // one row of coordinate sums per chunk (k_colstats) in partials.
    TRY(c->partials.ensure(sizeof(double) * (size_t)std::max(1LL, pps ? nchunks : blocks_total) * NS));
    if (pps) TRY(c->pstats.ensure(sizeof(double) * 3 * (size_t)std::max(1LL, P)));
    TRY(c->stage_stats.ensure(sizeof(double) * NS));
  }
  const size_t es = sizeof(T);
  long long rows_done = 0;  // statistics rows written so far (fused families)
  for (long long k = 0; k < nchunks; ++k) {
    const int s = (int)(k % N_STAGE);
    cudaStream_t st = c->streams[s];
    const long long c0 = k * chunk, n = std::min(chunk, P - c0);
    T* base = static_cast<T*>(c->stage[s].ptr);
    T* dq = base;
    T* dp = base + arr;
    T* dz = base + 2 * arr;
    T* dm = base + 3 * arr;
    T* du = dm + chunk;
    unsigned char* dacc = reinterpret_cast<unsigned char*>(du + chunk);
    // the slab is reused every N_STAGE chunks: stream order already serialises the reuse
    CUDA_TRY(cudaMemcpy2DAsync(dq, chunk * es, v.q.data + c0 * es, v.q.ld * es, n * es, D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dm, v.mass.data + c0 * es, n * es, cudaMemcpyHostToDevice, st));
    if (!hmc)
      CUDA_TRY(cudaMemcpy2DAsync(dp, chunk * es, v.p.data + c0 * es, v.p.ld * es, n * es, D, cudaMemcpyHostToDevice, st));
    if (v.has_z)
      CUDA_TRY(cudaMemcpy2DAsync(dz, chunk * es, v.z.data + c0 * es, v.z.ld * es, n * es, D, cudaMemcpyHostToDevice, st));
    if (v.has_u) CUDA_TRY(cudaMemcpyAsync(du, v.u.data + c0 * es, n * es, cudaMemcpyHostToDevice, st));
    IterArgs<T> A = proto;
    A.q = dq;
    A.q_ld = chunk;
    A.p = v.has_p ? dp : nullptr;
    A.p_ld = chunk;
    A.mass = dm;
    A.z = v.has_z ? dz : nullptr;
    A.z_ld = chunk;
    A.u = v.has_u ? du : nullptr;
    A.accept = v.has_accept ? dacc : nullptr;
    A.P = n;
    A.offset = proto.offset + (u64)c0;
    if (!v.has_stats)
      A.partials = nullptr;
    else if (pps)
      A.partials = static_cast<double*>(c->pstats.ptr) + (size_t)c0 * 3;
    else
      A.partials = static_cast<double*>(c->partials.ptr) + (size_t)rows_done * NS;
    TRY(launch_traj<T>(c, pot, A, integ, hmc, st, s));
    rows_done += c->last_rows;
    if (v.has_stats && pps) {
      double* row = static_cast<double*>(c->partials.ptr) + (size_t)k * NS;
      CUDA_TRY(cudaMemsetAsync(row, 0, sizeof(double) * 3, st));
      TRY(colstats<T>(c, dq, chunk, n, (int)D, row, st));
    }
    CUDA_TRY(cudaMemcpy2DAsync(v.q.data + c0 * es, v.q.ld * es, dq, chunk * es, n * es, D, cudaMemcpyDeviceToHost, st));
    if (v.has_p)
      CUDA_TRY(cudaMemcpy2DAsync(v.p.data + c0 * es, v.p.ld * es, dp, chunk * es, n * es, D, cudaMemcpyDeviceToHost, st));
    if (v.has_accept) CUDA_TRY(cudaMemcpyAsync(v.accept.data + c0, dacc, n, cudaMemcpyDeviceToHost, st));
  }
  for (int i = 0; i < N_STAGE; ++i) CUDA_TRY(cudaStreamSynchronize(c->streams[i]));
  if (v.has_stats) {
    cudaStream_t st = c->streams[0];
    k_stats_finalize<<<NS, 256, 0, st>>>(static_cast<double*>(c->partials.ptr), (int)(pps ? nchunks : rows_done), NS,
                                         static_cast<double*>(c->stage_stats.ptr));
    c->launches++;
    if (pps) {
      k_stats_finalize<<<3, 256, 0, st>>>(static_cast<double*>(c->pstats.ptr), (int)P, 3,
                                          static_cast<double*>(c->stage_stats.ptr));
      c->launches++;
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(v.stats.data, c->stage_stats.ptr, sizeof(double) * NS, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  return EHMC_OK;
}

static int common_checks(ehmc_ctx* ctx, const ehmc_potential* pot, const DLTensor* q, const DLTensor* mass,
                         CallViews* v, const char* fn) {
  if (!ctx || !pot) return fail(EHMC_ERR_INVALID, "%s: NULL context or potential", fn);
  if (pot->ctx != ctx) return fail(EHMC_ERR_INVALID, "%s: potential belongs to another context", fn);
  TRY(parse_float(q, "q", 2, 0, &v->q));
  v->bits = v->q.bits;
  v->D = v->q.shape[0];
  v->P = v->q.shape[1];
  if (v->bits != pot->bits)
    return fail(EHMC_ERR_INVALID, "%s: q is float%d but the potential was created for float%d", fn, v->bits, pot->bits);
  if (v->D != pot->D)
    return fail(EHMC_ERR_INVALID, "%s: q has %lld dimensions, the potential has %d", fn, v->D, pot->D);
  TRY(parse_float(mass, "mass", 1, v->bits, &v->mass));
  if (v->mass.shape[0] != v->P) return fail(EHMC_ERR_INVALID, "%s: mass must have P = %lld entries", fn, v->P);
  return EHMC_OK;
}

static int integrate_entry(ehmc_ctx* ctx, const ehmc_potential* pot, int integ, DLTensor* q, DLTensor* p,
                           const DLTensor* mass, double h, double h2, int L, void* stream, const char* fn) {
  CallViews v;
  TRY(common_checks(ctx, pot, q, mass, &v, fn));
  if (L < 0) return fail(EHMC_ERR_INVALID, "%s: numSteps < 0", fn);
  TRY(parse_float(p, "p", 2, v.bits, &v.p));
  v.has_p = true;
  if (v.p.shape[0] != v.D || v.p.shape[1] != v.P) return fail(EHMC_ERR_INVALID, "%s: p must have q's shape", fn);
  TRY(check_same_place(v));
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (v.bits == 32) {
    IterArgs<float> A = base_args<float>(v, h, h2, L);
    return v.q.host ? run_host<float>(ctx, pot, v, A, integ, false) : run_device<float>(ctx, pot, A, integ, false, nullptr, st);
  }
  IterArgs<double> A = base_args<double>(v, h, h2, L);
  return v.q.host ? run_host<double>(ctx, pot, v, A, integ, false) : run_device<double>(ctx, pot, A, integ, false, nullptr, st);
}

extern "C" int ehmc_leapfrog(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, DLTensor* p, const DLTensor* mass,
                             double stepSize, double stepSizeSq, int numSteps, void* stream) {
  if (ctx) ctx->ep_valid = false;  // q is about to change outside ehmc_hmc_iter
  NvtxRange nvtx_range("ehmc_leapfrog");
  return integrate_entry(ctx, pot, INTEG_LEAPFROG, q, p, mass, stepSize, stepSizeSq, numSteps, stream, "ehmc_leapfrog");
}

extern "C" int ehmc_stormer_verlet(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, DLTensor* p,
                                   const DLTensor* mass, double stepSize, double stepSizeSq, int numSteps,
                                   void* stream) {
  if (ctx) ctx->ep_valid = false;  // q is about to change outside ehmc_hmc_iter
  NvtxRange nvtx_range("ehmc_stormer_verlet");
  return integrate_entry(ctx, pot, INTEG_STORMER, q, p, mass, stepSize, stepSizeSq, numSteps, stream,
                         "ehmc_stormer_verlet");
}

extern "C" int ehmc_hmc_iter(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, DLTensor* p_out,
                             const DLTensor* mass, const ehmc_hmc_args* a, const DLTensor* z, const DLTensor* u,
                             DLTensor* accept_out, DLTensor* stats_out, void* stream) {
  NvtxRange nvtx_range("ehmc_hmc_iter");
  const char* fn = "ehmc_hmc_iter";
  CallViews v;
  TRY(common_checks(ctx, pot, q, mass, &v, fn));
  TRY(check_hmc_args(HmcEntry::iter, fn, a, nullptr, false));
  if (p_out) {
    TRY(parse_float(p_out, "p_out", 2, v.bits, &v.p));
    v.has_p = true;
    if (v.p.shape[0] != v.D || v.p.shape[1] != v.P) return fail(EHMC_ERR_INVALID, "%s: p_out must have q's shape", fn);
  }
  if (z) {
    TRY(parse_float(z, "z", 2, v.bits, &v.z));
    v.has_z = true;
    if (v.z.shape[0] != v.D || v.z.shape[1] != v.P) return fail(EHMC_ERR_INVALID, "%s: z must have q's shape", fn);
  }
  if (u) {
    TRY(parse_float(u, "u", 1, v.bits, &v.u));
    v.has_u = true;
    if (v.u.shape[0] != v.P) return fail(EHMC_ERR_INVALID, "%s: u must have P entries", fn);
  }
  if (accept_out) {
    TRY(parse(accept_out, "accept_out", 1, &v.accept));
    v.has_accept = true;
    if (v.accept.bits != 8 || v.accept.shape[0] != v.P)
      return fail(EHMC_ERR_INVALID, "%s: accept_out must be uint8/bool[P]", fn);
  }
  if (stats_out) {
    TRY(parse_float(stats_out, "stats_out", 1, 64, &v.stats));
    v.has_stats = true;
    if (v.stats.shape[0] != 2 * v.D + 3) return fail(EHMC_ERR_INVALID, "%s: stats_out must be float64[2D+3]", fn);
  }
  TRY(check_same_place(v));
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (a->dynamic != nullptr) {
    // only kernels that resolve the block themselves; everything else would silently use the host values
    const bool tc3 = v.bits == 32 && use_dense_tc(ctx, pot);
    if (v.q.host || !(has_small_kernel(pot) || tc3))
      return fail(EHMC_ERR_UNSUPPORTED, "%s: args.dynamic needs device tensors and a small-D or float32 dense (tensor-core) potential", fn);
  }
  if (v.bits == 32) {
    IterArgs<float> A = hmc_args<float>(v, a);
    if (v.q.host) return run_host<float>(ctx, pot, v, A, a->integrator, true);
    return run_device<float>(ctx, pot, A, a->integrator, true,
                             v.has_stats ? reinterpret_cast<double*>(v.stats.data) : nullptr, st);
  }
  IterArgs<double> A = hmc_args<double>(v, a);
  if (v.q.host) return run_host<double>(ctx, pot, v, A, a->integrator, true);
  return run_device<double>(ctx, pot, A, a->integrator, true,
                            v.has_stats ? reinterpret_cast<double*>(v.stats.data) : nullptr, st);
}

// ---------------------------------------------------------------------------
// getSamples' loop in one launch
// ---------------------------------------------------------------------------
template <typename T>
static int hmc_run_typed(ehmc_ctx* ctx, const ehmc_potential* pot, const CallViews& v, const ehmc_hmc_args* a, int nIter,
                         const View* vs, const View* vm, long long s0, long long S, int* accepted, cudaStream_t st) {
  IterArgs<T> A = hmc_args<T>(v, a);
  RunArgs<T> R;
  R.samples = vs ? reinterpret_cast<T*>(vs->data) : nullptr;
  R.momenta = vm ? reinterpret_cast<T*>(vm->data) : nullptr;
  R.accepted = accepted;
  R.S = S;
  R.s0 = s0;
  R.nIter = nIter;
  if (A.P == 0 || nIter == 0) return EHMC_OK;
  return run_small<T>(ctx, pot, A, a->integrator, R, st);
}

extern "C" int ehmc_hmc_run(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, const DLTensor* mass,
                            const ehmc_hmc_args* a, int numIterations, DLTensor* samples_out, DLTensor* momenta_out,
                            int64_t sampleOffset, DLTensor* accepted_out, void* stream) {
  if (ctx) ctx->ep_valid = false;  // q is about to change outside ehmc_hmc_iter
  NvtxRange nvtx_range("ehmc_hmc_run");
  const char* fn = "ehmc_hmc_run";
  CallViews v;
  TRY(common_checks(ctx, pot, q, mass, &v, fn));
  TRY(check_hmc_args(HmcEntry::run, fn, a, nullptr, numIterations < 0 || sampleOffset < 0));
  if (v.q.host || !has_small_kernel(pot))
    return fail(EHMC_ERR_UNSUPPORTED, "%s: device tensors and a small-D potential family are required", fn);
  View vs, vm, va;
  long long S = 0;
  for (int k = 0; k < 2; ++k) {
    DLTensor* t = k == 0 ? samples_out : momenta_out;
    if (!t) continue;
    View* w = k == 0 ? &vs : &vm;
    TRY(parse_float(t, k == 0 ? "samples_out" : "momenta_out", 2, v.bits, w));
    if (w->host || w->shape[0] != v.D * v.P || w->ld != w->shape[1])
      return fail(EHMC_ERR_INVALID, "%s: sample arrays must be contiguous device [D*P, S] views of (D, P, S)", fn);
    if (S && S != w->shape[1]) return fail(EHMC_ERR_INVALID, "%s: samples_out and momenta_out differ in S", fn);
    S = w->shape[1];
  }
  if ((samples_out || momenta_out) && sampleOffset + numIterations > S)
    return fail(EHMC_ERR_INVALID, "%s: sampleOffset + numIterations exceeds S = %lld", fn, S);
  int* accepted = nullptr;
  if (accepted_out) {
    TRY(parse(accepted_out, "accepted_out", 1, &va));
    if (va.host || va.bits != 32 || va.shape[0] != v.P) return fail(EHMC_ERR_INVALID, "%s: accepted_out must be device int32[P]", fn);
    accepted = reinterpret_cast<int*>(va.data);
  }
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (v.bits == 32)
    return hmc_run_typed<float>(ctx, pot, v, a, numIterations, samples_out ? &vs : nullptr, momenta_out ? &vm : nullptr,
                                sampleOffset, S, accepted, st);
  return hmc_run_typed<double>(ctx, pot, v, a, numIterations, samples_out ? &vs : nullptr, momenta_out ? &vm : nullptr,
                               sampleOffset, S, accepted, st);
}

// ---------------------------------------------------------------------------
// the adaptive ensemble run in one launch
// ---------------------------------------------------------------------------
extern "C" int ehmc_hmc_run_ensemble(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, const DLTensor* mass,
                                     const ehmc_hmc_args* a, int numIterations, const ehmc_adapt_args* ad,
                                     ehmc_comm* comm, DLTensor* state, DLTensor* history, DLTensor* moments,
                                     DLTensor* trace, int64_t traceParticles, int64_t traceOffset, void* stream) {
  if (ctx) ctx->ep_valid = false;
  NvtxRange nvtx_range("ehmc_hmc_run_ensemble");
  const char* fn = "ehmc_hmc_run_ensemble";
  CallViews v;
  TRY(common_checks(ctx, pot, q, mass, &v, fn));
  if (!a || !ad || !state) return fail(EHMC_ERR_INVALID, "%s: args, adapt and state are required", fn);
  TRY(check_hmc_args(HmcEntry::ensemble, fn, a, ad, numIterations < 0 || traceParticles < 0 || traceOffset < 0));
  if (v.q.host || !has_small_kernel(pot))
    return fail(EHMC_ERR_UNSUPPORTED, "%s: device tensors and a small-D potential family are required", fn);
  if (!(ad->numParticlesTotal > 0) || !(ad->minStep > 0) || !(ad->maxStep >= ad->minStep))
    return fail(EHMC_ERR_INVALID, "%s: bad adaptation scalars", fn);
  if (comm && (comm->ctx != ctx || !comm->connected)) return fail(EHMC_ERR_INVALID, "%s: communicator not connected on this context", fn);
  if (ad->lag < 0 || ad->lag > ENS_MAX_LAG) return fail(EHMC_ERR_INVALID, "%s: adapt.lag must be 0 (= 1) or 1 .. %d", fn, ENS_MAX_LAG);
  View vs, vh, vm, vt;
  TRY(parse_float(state, "state", 1, 64, &vs));
  if (vs.host || vs.shape[0] != 4) return fail(EHMC_ERR_INVALID, "%s: state must be a device float64[4]", fn);
  if (history) {
    TRY(parse_float(history, "history", 2, 64, &vh));
    if (vh.host || vh.shape[1] != 4 || vh.ld != 4 || vh.shape[0] < numIterations)
      return fail(EHMC_ERR_INVALID, "%s: history must be a contiguous device float64[>= numIterations, 4]", fn);
  }
  if (moments) {
    TRY(parse_float(moments, "moments", 1, 64, &vm));
    if (vm.host || vm.shape[0] != 2 * v.D) return fail(EHMC_ERR_INVALID, "%s: moments must be a device float64[2D]", fn);
  }
  long long S = 0;
  if (trace) {
    TRY(parse_float(trace, "trace", 2, v.bits, &vt));
    if (vt.host || vt.shape[0] != v.D * traceParticles || vt.ld != vt.shape[1] || traceParticles > v.P ||
        traceOffset + numIterations > vt.shape[1])
      return fail(EHMC_ERR_INVALID, "%s: trace must be a contiguous device [D*traceParticles, S] view with room for the iterations", fn);
    S = vt.shape[1];
  }
  TRY(enter_device(ctx));
  if (numIterations == 0 || v.P == 0) return EHMC_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Robbins-Monro gains of this call's updates, k continuing from state[2] (read back: one small synchronous copy)
  double st_host[4];
  CUDA_TRY(cudaMemcpyAsync(st_host, vs.data, sizeof(st_host), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  const int n_adapt = std::max(0, std::min(numIterations, ad->adaptIterations));
  std::vector<double> gains((size_t)std::max(1, n_adapt));
  for (int i = 0; i < n_adapt; ++i) gains[i] = ad->gain0 / std::pow(st_host[2] + 1.0 + i, ad->kappa);
  auto run = [&](auto tag) -> int {
    typedef decltype(tag) T;
    IterArgs<T> A = hmc_args<T>(v, a);
    EnsRunArgs<T> R;
    memset(&R, 0, sizeof(R));
    R.nIter = numIterations;
    R.lag = ad->lag == 0 ? 1 : ad->lag;
    R.adaptIters = n_adapt;
    R.target = ad->targetAccept;
    R.maxMove = ad->maxMove;
    R.gains = gains.data();  // host array; the launcher uploads it
    R.logLo = std::log(ad->minStep);
    R.logHi = std::log(ad->maxStep);
    R.Ptot = ad->numParticlesTotal;
    R.state = reinterpret_cast<double*>(vs.data);
    R.history = history ? reinterpret_cast<double*>(vh.data) : nullptr;
    R.moments = moments ? reinterpret_cast<double*>(vm.data) : nullptr;
    R.trace = (trace && traceParticles > 0) ? reinterpret_cast<T*>(vt.data) : nullptr;
    R.ntrace = traceParticles;
    R.S = S;
    R.s0 = traceOffset;
    R.rank = comm ? comm->rank : 0;
    R.world = comm ? comm->world : 1;
    R.peers = comm ? comm->peers_dev : nullptr;
    R.seq0 = comm ? comm->seq : 0;
    return run_small_ens<T>(ctx, pot, A, R, st);
  };
  const int rc = v.bits == 32 ? run(float()) : run(double());
  if (rc == EHMC_OK && comm) comm->seq += (unsigned long long)numIterations;
  return rc;
}

// ---------------------------------------------------------------------------
// device-side step-size adaptation (ehmc_dynamic)
// ---------------------------------------------------------------------------
static __global__ void k_adapt_step(const double* __restrict__ stats, int D, double P, double target, double gain0,
                                    double kappa, double maxMove, double logLo, double logHi, u64 adaptRows,
                                    DynArgs* dyn, const DynArgs* state, u64 stride, double* history,
                                    long long hist_rows, double* moments) {
  const int t = threadIdx.x;
  if (moments != nullptr)
    for (int j = t; j < 2 * D; j += blockDim.x) moments[j] += stats[3 + j];
  if (t != 0) return;
  const double meanAcc = stats[1] / P;
  const u64 row = dyn->row;
  if (history != nullptr && (long long)row < hist_rows) {
    history[4 * row + 0] = stats[0] / P;
    history[4 * row + 1] = meanAcc;
    history[4 * row + 2] = stats[2] / P;
    history[4 * row + 3] = dyn->stepSize;
  }
  double logh = state->logStepSize;
  u64 k = state->updates;
  if (row < adaptRows) {
    k += 1;
    const double acc = isfinite(meanAcc) ? meanAcc : 0.0;
    double move = gain0 / pow((double)k, kappa) * (acc - target);
    move = fmin(fmax(move, -maxMove), maxMove);
    logh = fmin(fmax(logh + move, logLo), logHi);
  }
  dyn->logStepSize = logh;
  dyn->stepSize = row < adaptRows ? exp(logh) : state->stepSize;
  dyn->updates = k;
  dyn->iteration += stride;
  dyn->row = row + stride;
}

extern "C" int ehmc_adapt_step(ehmc_ctx* ctx, const DLTensor* stats, double numParticlesTotal, double targetAccept,
                               double gain0, double kappa, double maxMove, double minStep, double maxStep,
                               uint64_t adaptRows, void* dynamic, const void* state, uint64_t stride, DLTensor* history,
                               DLTensor* moments, void* stream) {
  NvtxRange nvtx_range("ehmc_adapt_step");
  const char* fn = "ehmc_adapt_step";
  if (!ctx || !stats || !dynamic) return fail(EHMC_ERR_INVALID, "%s: NULL argument", fn);
  View vs, vh, vm;
  TRY(parse_float(stats, "stats", 1, 64, &vs));
  if (vs.host || vs.shape[0] < 5 || ((vs.shape[0] - 3) & 1)) return fail(EHMC_ERR_INVALID, "%s: stats must be a device float64[2D+3]", fn);
  const int D = (int)((vs.shape[0] - 3) / 2);
  if (!(numParticlesTotal > 0) || !(minStep > 0) || !(maxStep >= minStep) || stride < 1)
    return fail(EHMC_ERR_INVALID, "%s: bad scalar arguments", fn);
  double* hist = nullptr;
  long long hist_rows = 0;
  if (history) {
    TRY(parse_float(history, "history", 2, 64, &vh));
    if (vh.host || vh.shape[1] != 4 || vh.ld != 4) return fail(EHMC_ERR_INVALID, "%s: history must be a contiguous device float64[S,4]", fn);
    hist = reinterpret_cast<double*>(vh.data);
    hist_rows = vh.shape[0];
  }
  double* mom = nullptr;
  if (moments) {
    TRY(parse_float(moments, "moments", 1, 64, &vm));
    if (vm.host || vm.shape[0] != 2 * D) return fail(EHMC_ERR_INVALID, "%s: moments must be a device float64[2D]", fn);
    mom = reinterpret_cast<double*>(vm.data);
  }
  TRY(enter_device(ctx));
  k_adapt_step<<<1, 128, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const double*>(vs.data), D, numParticlesTotal,
                                                                targetAccept, gain0, kappa, maxMove, std::log(minStep),
                                                                std::log(maxStep), adaptRows, static_cast<DynArgs*>(dynamic),
                                                                static_cast<const DynArgs*>(state ? state : dynamic), stride,
                                                                hist, hist_rows, mom);
  ctx->launches++;
  CUDA_TRY(cudaGetLastError());
  return EHMC_OK;
}

// ---------------------------------------------------------------------------
// potential evaluation
// ---------------------------------------------------------------------------
template <typename T>
static int eval_device(ehmc_ctx* c, const ehmc_potential* p, const T* q, long long q_ld, long long P, T* e, T* g,
                       long long g_ld, cudaStream_t st) {
  if (P == 0) return EHMC_OK;
  if (p->family == EHMC_FAMILY_DENSE_GAUSSIAN) {
    const T* lambda = static_cast<const T*>(p->dense.lambda);
    const T* mu = static_cast<const T*>(p->dense.mu);
    k_eval_dense<T><<<(unsigned)((P + 127) / 128), 128, 0, st>>>(q, q_ld, P, p->D, lambda, mu, e, g, g_ld);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return EHMC_OK;
  }
  if (p->family == EHMC_FAMILY_NBODY) return eval_nbody<T>(c, p, q, q_ld, P, e, g, g_ld, st);
  if (p->family == EHMC_FAMILY_LOGISTIC) return eval_logistic<T>(c, p, q, q_ld, P, e, g, g_ld, st);
  return eval_small<T>(c, p, q, q_ld, P, e, g, g_ld, st);
}

template <typename T>
static int eval_any(ehmc_ctx* c, const ehmc_potential* p, const View& q, const View* e, const View* g, cudaStream_t st) {
  const long long D = q.shape[0], P = q.shape[1];
  if (!q.host) {
    return eval_device<T>(c, p, reinterpret_cast<const T*>(q.data), q.ld, P, e ? reinterpret_cast<T*>(e->data) : nullptr,
                          g ? reinterpret_cast<T*>(g->data) : nullptr, g ? g->ld : 0, st);
  }
  // host path: one shot through stage[0]/stage[1] (evaluation is not a hot path)
  const size_t es = sizeof(T);
  TRY(c->stage[0].ensure(es * (size_t)(2 * D + 1) * std::max<long long>(P, 1)));
  T* dq = static_cast<T*>(c->stage[0].ptr);
  T* dg = dq + (size_t)D * P;
  T* de = dg + (size_t)D * P;
  if (P > 0) CUDA_TRY(cudaMemcpy2D(dq, P * es, q.data, q.ld * es, P * es, D, cudaMemcpyHostToDevice));
  TRY(eval_device<T>(c, p, dq, P, P, e ? de : nullptr, g ? dg : nullptr, P, nullptr));
  if (e && P > 0) CUDA_TRY(cudaMemcpy(e->data, de, P * es, cudaMemcpyDeviceToHost));
  if (g && P > 0) CUDA_TRY(cudaMemcpy2D(g->data, g->ld * es, dg, P * es, P * es, D, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaDeviceSynchronize());
  return EHMC_OK;
}

extern "C" int ehmc_potential_eval(ehmc_ctx* ctx, const ehmc_potential* pot, const DLTensor* q, DLTensor* energy_out,
                                   DLTensor* grad_out, void* stream) {
  NvtxRange nvtx_range("ehmc_potential_eval");
  const char* fn = "ehmc_potential_eval";
  if (!ctx || !pot) return fail(EHMC_ERR_INVALID, "%s: NULL context or potential", fn);
  View vq, ve, vg;
  TRY(parse_float(q, "q", 2, pot->bits, &vq));
  if (vq.shape[0] != pot->D) return fail(EHMC_ERR_INVALID, "%s: q has %lld dimensions, the potential has %d", fn, vq.shape[0], pot->D);
  if (energy_out) {
    TRY(parse_float(energy_out, "energy_out", 1, pot->bits, &ve));
    if (ve.shape[0] != vq.shape[1] || ve.host != vq.host) return fail(EHMC_ERR_INVALID, "%s: energy_out must be [P] beside q", fn);
  }
  if (grad_out) {
    TRY(parse_float(grad_out, "grad_out", 2, pot->bits, &vg));
    if (vg.shape[0] != vq.shape[0] || vg.shape[1] != vq.shape[1] || vg.host != vq.host)
      return fail(EHMC_ERR_INVALID, "%s: grad_out must be [D,P] beside q", fn);
  }
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pot->bits == 32) return eval_any<float>(ctx, pot, vq, energy_out ? &ve : nullptr, grad_out ? &vg : nullptr, st);
  return eval_any<double>(ctx, pot, vq, energy_out ? &ve : nullptr, grad_out ? &vg : nullptr, st);
}

// ---------------------------------------------------------------------------
// Philox fills
// ---------------------------------------------------------------------------
template <typename T>
static int fill_any(ehmc_ctx* c, const View* out, const View* u, const View* mass, int mode, double scale, double kB,
                    double temp, uint64_t seed, uint64_t iter, uint64_t off, cudaStream_t st) {
  const long long P = out ? out->shape[1] : u->shape[0];
  const int D = out ? (int)out->shape[0] : 0;
  if (P == 0) return EHMC_OK;
  const bool host = out ? out->host : u->host;
  const size_t es = sizeof(T);
  const unsigned grid = (unsigned)((P + 127) / 128);
  if (!host) {
    k_philox_fill<T><<<grid, 128, 0, st>>>(out ? reinterpret_cast<T*>(out->data) : nullptr, out ? out->ld : 0, P, D,
                                           u ? reinterpret_cast<T*>(u->data) : nullptr,
                                           mass ? reinterpret_cast<const T*>(mass->data) : nullptr, mode, scale, kB,
                                           temp, seed, iter, off);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return EHMC_OK;
  }
  TRY(c->stage[0].ensure(es * (size_t)(D + 2) * P));
  T* dout = static_cast<T*>(c->stage[0].ptr);
  T* du = dout + (size_t)D * P;
  T* dm = du + P;
  if (mass) CUDA_TRY(cudaMemcpy(dm, mass->data, P * es, cudaMemcpyHostToDevice));
  k_philox_fill<T><<<grid, 128>>>(out ? dout : nullptr, P, P, D, u ? du : nullptr, mass ? dm : nullptr, mode, scale, kB,
                                  temp, seed, iter, off);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  if (out && D > 0) CUDA_TRY(cudaMemcpy2D(out->data, out->ld * es, dout, P * es, P * es, D, cudaMemcpyDeviceToHost));
  if (u) CUDA_TRY(cudaMemcpy(u->data, du, P * es, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaDeviceSynchronize());
  return EHMC_OK;
}

extern "C" int ehmc_philox_fill(ehmc_ctx* ctx, DLTensor* z, DLTensor* u, uint64_t seed, uint64_t iteration,
                                uint64_t particleOffset, void* stream) {
  if (!ctx || (!z && !u)) return fail(EHMC_ERR_INVALID, "ehmc_philox_fill: NULL argument");
  View vz, vu;
  int bits = 0;
  if (z) {
    TRY(parse_float(z, "z", 2, 0, &vz));
    bits = vz.bits;
  }
  if (u) {
    TRY(parse_float(u, "u", 1, bits, &vu));
    bits = vu.bits;
    if (z && (vu.shape[0] != vz.shape[1] || vu.host != vz.host))
      return fail(EHMC_ERR_INVALID, "ehmc_philox_fill: u must be [P] beside z");
  }
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (bits == 32)
    return fill_any<float>(ctx, z ? &vz : nullptr, u ? &vu : nullptr, nullptr, 0, 1.0, 0, 0, seed, iteration, particleOffset, st);
  return fill_any<double>(ctx, z ? &vz : nullptr, u ? &vu : nullptr, nullptr, 0, 1.0, 0, 0, seed, iteration, particleOffset, st);
}

extern "C" int ehmc_set_position(ehmc_ctx* ctx, DLTensor* q, double qStd, uint64_t seed, uint64_t particleOffset,
                                 void* stream) {
  if (ctx) ctx->ep_valid = false;  // q is about to change outside ehmc_hmc_iter
  if (!ctx) return fail(EHMC_ERR_INVALID, "ehmc_set_position: NULL context");
  View vq;
  TRY(parse_float(q, "q", 2, 0, &vq));
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint64_t it = ~0ULL;
  if (vq.bits == 32) return fill_any<float>(ctx, &vq, nullptr, nullptr, 0, qStd, 0, 0, seed, it, particleOffset, st);
  return fill_any<double>(ctx, &vq, nullptr, nullptr, 0, qStd, 0, 0, seed, it, particleOffset, st);
}

extern "C" int ehmc_set_momentum(ehmc_ctx* ctx, DLTensor* p, const DLTensor* mass, double boltzmann, double temperature,
                                 uint64_t seed, uint64_t iteration, uint64_t particleOffset, void* stream) {
  if (!ctx) return fail(EHMC_ERR_INVALID, "ehmc_set_momentum: NULL context");
  View vp, vm;
  TRY(parse_float(p, "p", 2, 0, &vp));
  TRY(parse_float(mass, "mass", 1, vp.bits, &vm));
  if (vm.shape[0] != vp.shape[1] || vm.host != vp.host)
    return fail(EHMC_ERR_INVALID, "ehmc_set_momentum: mass must be [P] beside p");
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (vp.bits == 32)
    return fill_any<float>(ctx, &vp, nullptr, &vm, 1, 1.0, boltzmann, temperature, seed, iteration, particleOffset, st);
  return fill_any<double>(ctx, &vp, nullptr, &vm, 1, 1.0, boltzmann, temperature, seed, iteration, particleOffset, st);
}

// ---------------------------------------------------------------------------
// reference N-body mode
// ---------------------------------------------------------------------------
template <typename T>
static int nbody_mode_any(ehmc_ctx* c, int integ, const View& q, const View& p, const View& m, double G, double h,
                          double h2, int L, cudaStream_t st) {
  const long long D = q.shape[0], P = q.shape[1];
  if (P == 0) return EHMC_OK;
  const size_t es = sizeof(T);
  if (!q.host) {
    k_nbody_mode<T><<<1, 128, 0, st>>>(reinterpret_cast<T*>(q.data), q.ld, reinterpret_cast<T*>(p.data), p.ld,
                                       reinterpret_cast<const T*>(m.data), (int)P, (int)D, (T)G, (T)h, (T)h2, L, integ);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return EHMC_OK;
  }
  TRY(c->stage[0].ensure(es * (size_t)(2 * D + 1) * P));
  T* dq = static_cast<T*>(c->stage[0].ptr);
  T* dp = dq + (size_t)D * P;
  T* dm = dp + (size_t)D * P;
  CUDA_TRY(cudaMemcpy2D(dq, P * es, q.data, q.ld * es, P * es, D, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy2D(dp, P * es, p.data, p.ld * es, P * es, D, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(dm, m.data, P * es, cudaMemcpyHostToDevice));
  k_nbody_mode<T><<<1, 128>>>(dq, P, dp, P, dm, (int)P, (int)D, (T)G, (T)h, (T)h2, L, integ);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy2D(q.data, q.ld * es, dq, P * es, P * es, D, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy2D(p.data, p.ld * es, dp, P * es, P * es, D, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaDeviceSynchronize());
  return EHMC_OK;
}

extern "C" int ehmc_integrate_nbody_mode(ehmc_ctx* ctx, int integrator, DLTensor* q, DLTensor* p, const DLTensor* mass,
                                         double gravConst, double stepSize, double stepSizeSq, int numSteps,
                                         void* stream) {
  const char* fn = "ehmc_integrate_nbody_mode";
  if (!ctx) return fail(EHMC_ERR_INVALID, "%s: NULL context", fn);
  if (integrator != EHMC_LEAPFROG && integrator != EHMC_STORMER_VERLET)
    return fail(EHMC_ERR_INVALID, "%s: Invalid integration method selected.", fn);
  if (numSteps < 0) return fail(EHMC_ERR_INVALID, "%s: numSteps < 0", fn);
  View vq, vp, vm;
  TRY(parse_float(q, "q", 2, 0, &vq));
  TRY(parse_float(p, "p", 2, vq.bits, &vp));
  TRY(parse_float(mass, "mass", 1, vq.bits, &vm));
  if (vq.shape[0] > 4) return fail(EHMC_ERR_UNSUPPORTED, "%s: numDimensions <= 4 (got %lld)", fn, vq.shape[0]);
  if (vp.shape[0] != vq.shape[0] || vp.shape[1] != vq.shape[1] || vm.shape[0] != vq.shape[1])
    return fail(EHMC_ERR_INVALID, "%s: shape mismatch", fn);
  if (vp.host != vq.host || vm.host != vq.host) return fail(EHMC_ERR_INVALID, "%s: tensors on different sides", fn);
  TRY(enter_device(ctx));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (vq.bits == 32) return nbody_mode_any<float>(ctx, integrator, vq, vp, vm, gravConst, stepSize, stepSizeSq, numSteps, st);
  return nbody_mode_any<double>(ctx, integrator, vq, vp, vm, gravConst, stepSize, stepSizeSq, numSteps, st);
}
