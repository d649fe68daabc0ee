// Instantiations of the fused adaptive ensemble run (k_small_ens) for one dtype (included by inst_small_ens_f32/f64.cu).
#pragma once

#include <algorithm>

#include "inst_small.cuh"
#include "k_small_ens.cuh"

namespace ehmc {

template <typename T, int DT, class Pot, bool EXACT>
static int ens_launch(ehmc_ctx* c, const IterArgs<T>& A, const Pot& pot, EnsRunArgs<T> R, cudaStream_t st) {
  auto kernel = k_small_ens<T, DT, Pot, INTEG_LEAPFROG, EXACT>;
  // service CTAs: two vectors of <= 72 doubles + the received halves [world][2 (2D + 3)]
  const size_t svc = std::max(ENS_SERVICE_SMEM, (size_t)1152 + sizeof(unsigned) * (size_t)std::max(1, R.world) * 2 * (2 * A.D + 3));
  const size_t sm = std::max(WarpStats<T, DT>::kSmemBytes, svc);
  if (sm > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  int occ = 0, coop = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, K1_THREADS, sm));
  CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, c->device));
  if (!coop || occ < 1) return fail(EHMC_ERR_UNSUPPORTED, "fused ensemble run: cooperative launch unavailable");
  // one resident wave: compute CTAs plus the service CTAs
  const long long need = (A.P + K1_THREADS - 1) / K1_THREADS;
  const long long cap = (long long)occ * c->prop.multiProcessorCount;
  if (cap <= ENS_SERVICE_CTAS) return fail(EHMC_ERR_UNSUPPORTED, "fused ensemble run: device too small");
  const unsigned ncompute = (unsigned)std::max<long long>(1, std::min<long long>(need, cap - ENS_SERVICE_CTAS));
  const int NS = 2 * A.D + 3;
  // batches of 32 particles, tied into groups of 2^bshift consecutive batches (one float64 row each): about 2048
  // groups per iteration, at most ENS_MAX_GROUPS
  const long long nrows = (A.P + 31) / 32;  // sub-batches = rows of per-batch statistics
  // queue items of 1 / 2 / 4 sub-batches.  Measured on B200 (profiles/r02_fused_probe_sshift.txt, us per iteration of
  // the funnel, items of 32 | 64 | 128 | 256 particles):   2^19, L = 20: 32 | 44 | 60 | 70     2^19, L = 4: 22 | 25 | 38 | 44
  //   2^20, L = 20: 56 | 69 | 86 | 116    2^20, L = 4: 39 | 35 | 48 | 71    2^22, L = 20: 222 | 207 | 233 | 277
  //   2^22, L = 4: 160 | 135 | 127 | 139.  Small shards need the fine grain (a warp has 3.5 items per iteration at 2^19),
  // large ones gain from paying the queue round per 64 (long trajectories) or 128 (short ones) particles.
  int sshift = c->ens_sshift >= 0 ? c->ens_sshift : (nrows >= (1 << 16) ? (A.L <= 8 ? 2 : 1) : 0);
  const long long nbatch = (nrows + (1LL << sshift) - 1) >> sshift;
  int bshift = 0;
  // (sweep in profiles/r02_fused_probe_groups.txt: fewer, larger groups make the next iteration's batches wait for
  // their group's mark -- 256 groups: 42 us per iteration at 2^19 x L = 20, 2048: 32.3, 4096: 31.1; short trajectories
  // prefer 2048: 21.4 against 22.3 us at L = 4; 8192 groups cost the reducers more than they save: 35.9 us)
  const long long gmax = c->ens_groups > 0 ? c->ens_groups : (A.L > 8 ? 4096 : 2048);
  while ((nbatch >> bshift) > gmax) ++bshift;
  R.bshift = bshift;
  R.sshift = sshift;
  R.nrows = (unsigned)nrows;
  R.nbatch = (unsigned)nbatch;
  R.nvirt = (unsigned)((nbatch + (1LL << bshift) - 1) >> bshift);
  static_assert(ENS_MAX_GROUPS >= 4096, "group count");
  if (nrows > 0x3FFFFFFFLL || ((long long)R.nIter << bshift) > 0x7FFFFFFFLL)
    return fail(EHMC_ERR_UNSUPPORTED, "fused ensemble run: too many particles or iterations for one launch");
  const unsigned V = R.nvirt, ngroups = (V + ENS_GROUP - 1) / ENS_GROUP;
  // control block (every section on a 128-byte line): hsched [nIter + 1 + lag] | published replicas | ticket [ENS_RING]
  // lines, cursor | group tickets [ENS_RING][ngroups] | done [V], arrived [V] | rows [ENS_RING][V][NS] | group rows
  // [ENS_RING][ngroups][NS] | gains [adaptIters] | batch rows [nbatch][2 DT + 3] (state precision)
  auto up = [](size_t n) { return (n + 15) / 16 * 16; };
  const size_t n_h = up((size_t)R.nIter + 1 + ENS_MAX_LAG);
  const size_t n_pub = (size_t)ENS_PUB_COPIES * 16;
  const size_t n_tk = 16 * (ENS_RING + 1);  // the tickets of the ring and the cursor: one line each
  const size_t n_gt = up(((size_t)ENS_RING * ngroups + 1) / 2);   // ENS_RING * ngroups unsigned
  const size_t n_done = 2 * up((size_t)V / 2 + 1);   // done [V], arrived [V] (unsigned)
  const size_t n_rows = up((size_t)ENS_RING * V * NS);
  const size_t n_grows = up((size_t)ENS_RING * ngroups * NS);
  const size_t n_gains = up((size_t)std::max(1, R.adaptIters));
  const size_t n_brows = up(((size_t)nrows * (2 * DT + 3) * sizeof(T) + 7) / 8);
  const size_t bytes = sizeof(double) * (n_h + n_pub + n_tk + n_gt + n_done + n_rows + n_grows + n_gains + n_brows) + 128;
  TRY(c->ens_ctl.ensure(bytes));
  double* base = reinterpret_cast<double*>(((uintptr_t)c->ens_ctl.ptr + 127) & ~(uintptr_t)127);
  R.hsched = base;
  R.published = reinterpret_cast<long long*>(base + n_h);
  R.ticket = reinterpret_cast<unsigned*>(base + n_h + n_pub);  // ticket[par] at R.ticket[32 * par] (see the kernel)
  R.cursor = reinterpret_cast<unsigned long long*>(base + n_h + n_pub + 16 * ENS_RING);
  R.gticket = reinterpret_cast<unsigned*>(base + n_h + n_pub + n_tk);
  R.done = reinterpret_cast<unsigned*>(base + n_h + n_pub + n_tk + n_gt);
  R.arrived = reinterpret_cast<unsigned*>(base + n_h + n_pub + n_tk + n_gt + n_done / 2);
  R.rows = base + n_h + n_pub + n_tk + n_gt + n_done;
  R.grows = R.rows + n_rows;
  double* gains = R.grows + n_grows;
  R.brows = gains + n_gains;
  // published = 0, tickets = 0, cursor = 0, group tickets = 0, done = 0, arrived = 0
  CUDA_TRY(cudaMemsetAsync(base + n_h, 0, (n_pub + n_tk + n_gt + n_done) * sizeof(double), st));
  if (R.adaptIters > 0)  // R.gains arrives as a HOST array
    CUDA_TRY(cudaMemcpyAsync(gains, R.gains, sizeof(double) * R.adaptIters, cudaMemcpyHostToDevice, st));
  R.gains = gains;
  R.dbg = nullptr;
  R.dbg_iters = 0;
  if (c->ens_debug > 0) {
    TRY(c->ens_dbg_buf.ensure(sizeof(long long) * 8 * ((size_t)c->ens_debug + 1)));  // + one row of totals
    CUDA_TRY(cudaMemsetAsync(c->ens_dbg_buf.ptr, 0, sizeof(long long) * 8 * ((size_t)c->ens_debug + 1), st));
    R.dbg = static_cast<long long*>(c->ens_dbg_buf.ptr);
    R.dbg_iters = c->ens_debug;
  }
  IterArgs<T> Ac = A;
  void* args[] = {(void*)&Ac, (void*)&pot, (void*)&R};
  CUDA_TRY(cudaLaunchCooperativeKernel((const void*)kernel, dim3(ncompute + ENS_SERVICE_CTAS), dim3(K1_THREADS), args, sm, st));
  c->launches++;
  return EHMC_OK;
}

template <typename T>
int run_small_ens(ehmc_ctx* c, const ehmc_potential* p, const IterArgs<T>& A, const EnsRunArgs<T>& R, cudaStream_t st) {
  return with_small_pot<T>(p, "fused ensemble-run kernel", [&](auto dt, const auto& pot) -> int {
    constexpr int DT = decltype(dt)::value;
    using Pot = std::decay_t<decltype(pot)>;
    return A.D == DT ? ens_launch<T, DT, Pot, true>(c, A, pot, R, st) : ens_launch<T, DT, Pot, false>(c, A, pot, R, st);
  });
}

}  // namespace ehmc
