// K6: the adaptive ensemble run as ONE persistent launch -- trajectory kernel, ensemble statistics, the all-reduce
// of those statistics across GPUs and the step-size update fused into a single cooperative kernel.
//
// What it replaces: the outer loop of HMC.getSamples (src/HMC.py:150-179) as HMC.run drives it for large ensembles
// (momentum refresh, trajectory, Metropolis per iteration; build-defined: per-iteration ensemble statistics
// {n_accept, sum acceptance probability, sum H, sum q_d, sum q_d^2} summed over ALL GPUs, Robbins-Monro step-size
// adaptation from them).  The iteration-by-iteration form costs two launches, an NCCL all-reduce of 2D+3 doubles, a
// pinned copy and the Python enqueue per iteration: 63 us per iteration at the 8-GPU shard of config 5 (2^19
// particles) against 33 us of kernel (profiles/r01_adapt_probe.txt).
//
// Structure (grid = one resident wave, cooperative launch so that every CTA is co-resident):
//   * the unit of work is a BATCH of 32 consecutive particles run by one warp (of 64 / 128 particles, as two / four
//     sub-batches in a row, when the shard has >= 2^21 particles: EnsRunArgs::sshift).  The warps of the compute CTAs take
//     (iteration, batch) pairs in order from one global cursor; when an iteration's batches are all taken the cursor
//     simply runs on into the next iteration.  A warp runs k_small_body on its batch (q round-trips through HBM / L2)
//     and writes the batch's row of 2D+3 sums in the state's precision.  Batches are tied into GROUPS of 2^k
//     consecutive batches: the warp that arrives last in a group (one acq_rel atomic per batch) adds the group's
//     batch rows in batch order into one float64 row, marks the group's iteration complete (the batches of the next
//     iteration of that group wait for this mark: it orders iteration it + 1 of a particle behind iteration it,
//     whoever ran it) and releases a ticket (fire and forget).  Nothing here waits for the statistics: iteration
//     `it` only needs the step size h[it], published 1 + lag iterations earlier.
//   * 8 SERVICE CTAs = 32 independent reducer warps: warp w adds the rows of 64 consecutive groups (fixed order)
//     when their tickets are in; the master warp adds those, sends the 2D+3 doubles to every peer GPU's mailbox with
//     8-byte stores over NVLink that carry their own flags (peer memory mapped through CUDA IPC), collects the peers'
//     vectors, adds the world's vectors in rank order (every rank computes the same bits), updates log h and
//     publishes h[it + 1 + lag]: with lag = 1 the one-iteration-stale pipeline of HMC.run, so the reductions, the
//     NVLink round trip (368 B out and in per peer, a few microseconds) and the update hide behind iteration it + 1;
//     lag = 2 gives them two iterations, lag = 3 three.  What the lag has to cover is the whole span of an
//     iteration -- its first batch starts, a period later its last ticket is taken, that batch runs, three
//     reduction levels, the slowest of N GPUs, publish -- measured 90-100 us at 2^19 particles per GPU, where a
//     period is ~30 us: with lag = 2 every iteration's first batches waited 5-10 us for their step size and the run
//     advanced at (span + chain) / 3 per iteration (profiles/r02_ens_wait_ranks2_L20.txt: 34.7 us at 2 GPUs, 37.3 us
//     at 8, against 32.4 us without peers); profiles/r02_bench_n8_mid.json was taken with lag = 1.
// Why batches and a queue (measured at 2^19 particles per GPU, the 8-GPU shard of config 5, 28.8 us for the bare
// per-launch kernel): a fixed share per CTA is 3.46 blocks of 128 that round up to 4, and the warp schedulers'
// preference for the oldest warps let the oldest CTAs of every SM finish early and wait ahead of the others (39 us
// per iteration); CTA-wide slices of 128 particles from a queue need three block barriers per slice and expose the
// queue's L2 round trips to four warps at once (41 us); warp-wide slices of 128 particles make an iteration as long
// as one warp needs for four batches in a row, because every slice of an iteration is in flight at once (72 us).
// With single batches a warp has 3.5 of them per iteration and the order of the queue keeps every dependency
// (previous iteration of the same group, step size) a full iteration behind the cursor.
// The statistics are deterministic: rows belong to batches and groups, never to whichever warp ran them.
#pragma once

#include "k_small.cuh"

namespace ehmc {

constexpr int ENS_PUB_COPIES = 32; // replicas of the "step sizes published" counter, one 128-byte line each (one per
                                   // lane of the master warp: a single release store each)
constexpr int ENS_SERVICE_CTAS = 8; // blocks of reducer warps (one of them also runs the all-reduce and the update)
constexpr int ENS_GROUP = 64;      // group rows per first-level reduction of the service warps
constexpr int ENS_MAX_GROUPS = 8192;  // groups per iteration at most (the launcher aims at 2048)
constexpr int ENS_MB_STRIDE = 144;  // 8-byte words per mailbox slot: two per statistic (up to 2 * 32 + 3 statistics)
constexpr int ENS_RING = 8;        // iterations in flight at most (>= lag + 2): rows, tickets and step sizes are rings of 8
constexpr int ENS_MAX_LAG = 4;
constexpr size_t ENS_SERVICE_SMEM = 5632;  // master warp: two vectors of <= 72 doubles + [8 ranks][2 * 67] received halves

template <typename T>
struct EnsRunArgs {
  int nIter;
  int lag;             // the statistics of iteration it set the step size of iteration it + 1 + lag (1 .. ENS_MAX_LAG)
  int adaptIters;      // Robbins-Monro updates during the first adaptIters iterations of this launch
  double target, maxMove, logLo, logHi;
  const double* gains;  // [adaptIters] Robbins-Monro gain of every update, gain0 / k^kappa (host-computed)
  double Ptot;         // particles of all ranks
  double* hsched;      // [nIter + 1 + lag] step size of every iteration (the master's own record)
  long long* published;  // [ENS_PUB_COPIES][16] per replica line: [0] iterations whose step size is published,
                         //   [1 + it % ENS_RING] the step size of iteration it (double bits)
  unsigned long long* cursor;   // [1] next (iteration * nbatch + batch) to hand out
  unsigned* done;      // [nvirt] iterations of every group that are complete AND reduced into the group's row
  unsigned* arrived;   // [nvirt] batches of every group that have finished, ever
  void* brows;         // [nbatch][2 DT + 3] per-batch sums in the state's precision (padded layout)
  unsigned nvirt;      // groups per iteration
  unsigned nbatch;     // batches (32 << sshift particles: the queue's unit of work) per iteration
  int bshift;          // log2(batches per group)
  int sshift;          // log2(sub-batches of 32 particles per batch): 0 for small shards (the 8-GPU shard of config 5
                       // has 3.5 batches per warp and iteration and needs the fine grain), 1 (L > 8) or 2 when an
                       // iteration has >= 2^16 sub-batches, so that the queue round (cursor, group mark, step size,
                       // arrival atomic: ~170 instructions and four L2 round trips) is paid once per 64 / 128 particles
  unsigned nrows;      // sub-batches (rows of brows) per iteration = ceil(P / 32)
  unsigned* ticket;    // [ENS_RING][32] (entry 0 of each 128-byte line) groups of iteration it % ENS_RING that are reduced
  unsigned* gticket;   // [ENS_RING][ngroups] group rows of the reduction group that are written
  double* rows;        // [ENS_RING][nvirt][2D+3] per-group partial sums
  double* grows;       // [ENS_RING][ngroups][2D+3] per-group sums
  double* state;       // [4] in/out: step size, log step size, updates k, iterations run
  double* history;     // [nIter][4] {accept rate, mean acceptance probability, mean H, step size used} or null
  double* moments;     // [2D] += sum q_d, sum q_d^2 of every iteration, or null
  T* trace;            // [D][ntrace][S] kept positions of the first ntrace local particles, or null
  long long ntrace, S, s0;
  T* cmean;            // [D][c_ld] per-chain running mean over iterations windowStart .. (chain_moments_update), or null
  T* cm2;              // [D][c_ld] per-chain sum of squared deviations from that mean
  long long c_ld;
  int windowStart;     // first iteration of this launch whose positions enter the chain moments
  const T* crcp;       // [nIter - windowStart] 1/n of draw n of the window, rounded to T (host-computed)
  int rank, world;
  double* const* peers;   // [world] every rank's mailbox [2][world][ENS_MB_STRIDE] (peers[rank] = the local one)
  unsigned long long seq0;  // iterations this communicator has reduced before this launch
  long long* dbg;      // optional %globaltimer stamps [dbg_iters][8] (ctx option "ens_debug"):
  int dbg_iters;       //   service: 0 tickets complete, 1 reduced, 2 pushed, 3 peers in, 4 published;
                       //   compute CTA 0: 5 waits for h, 6 starts, 7 done
};

__device__ __forceinline__ long long ld_acquire_gpu(const long long* p) {
  long long v;
  asm volatile("ld.acquire.gpu.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(long long* p, long long v) {
  asm volatile("st.release.gpu.global.s64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

template <typename T, int DT, class Pot, int INTEG, bool EXACT>
__global__ void __launch_bounds__(K1_THREADS, 8) k_small_ens(const IterArgs<T> Ain, const Pot pot, const EnsRunArgs<T> R) {
  extern __shared__ __align__(16) double k1_smem[];
  const int Dn = EXACT ? DT : Ain.D;
  const int NS = 2 * Dn + 3;
  const unsigned ncompute = gridDim.x - ENS_SERVICE_CTAS;
  const unsigned V = R.nvirt;  // slices of `chunk` consecutive particles, one statistics row each
  const unsigned ngroups = (V + ENS_GROUP - 1) / ENS_GROUP;
  const int tid = threadIdx.x;
  constexpr int NWARP = K1_THREADS / 32;
  constexpr int NAP = 2 * DT + 3;  // padded row of a batch
  // per compute warp, lane 0's view of the queue (shared memory rather than registers: it lives across the trajectories)
  __shared__ long long s_pub_seen[NWARP];          // newest value of the published counter the warp has seen
  __shared__ double s_hring[NWARP][ENS_RING];      // step sizes read behind s_pub_seen
  __shared__ unsigned s_done_seen[NWARP];          // "done" counter of the next batch's group when last looked at
  __shared__ unsigned long long s_base[NWARP];     // cursor value of batch 0 of iteration s_next_it
  __shared__ int s_next_it[NWARP];                 // the pair after the current one (-1: the queue is empty)
  __shared__ unsigned s_next_b[NWARP];
  __shared__ int s_it[NWARP];                      // the current pair and its step size, lane 0 -> the warp
  __shared__ unsigned s_b[NWARP];
  __shared__ double s_hcur[NWARP];
  __shared__ unsigned long long s_wait[NWARP][2];  // (debug) ns this warp spun for its group's mark / for the step size

  if (blockIdx.x < ncompute) {
    // ===== compute CTAs: four independent warps, each a worker of ONE queue over (iteration, batch) =====
    // Lane 0 owns the warp's queue state: while a batch runs it already holds the cursor value of the NEXT pair, and
    // when the batch is done it looks at that pair's group mark and at the published step sizes, so the top of the
    // loop normally finds both satisfied; it spins only when the warp really is ahead of the pipeline.
    // (replicas of the "published" line: thousands of warps polling ONE line kept its L2 slice busy enough to slow
    // the ticket atomics in its neighbourhood)
    const int lane = tid & 31, w = tid >> 5;
    const long long* pub = R.published + ((blockIdx.x * NWARP + w) % ENS_PUB_COPIES) * 16;
    const unsigned NB = R.nbatch;
    const unsigned long long total = (unsigned long long)NB * (unsigned long long)R.nIter;
    unsigned long long g_next = 0ull;  // (lane 0) the cursor value taken while the current batch runs
    auto take = [&](unsigned long long g) {  // lane 0: pair g, and a non-blocking look at what it will need
      if (g >= total) {
        s_next_it[w] = -1;
        return;
      }
      // (a warp's cursor values only grow: no 64-bit division)
      unsigned long long base = s_base[w];
      int it = s_next_it[w];
      while (g >= base + NB) {
        base += NB;
        ++it;
      }
      s_base[w] = base;
      const unsigned b = (unsigned)(g - base);
      s_next_it[w] = it;
      s_next_b[w] = b;
      s_done_seen[w] = it > 0 ? ld_acquire_gpu_u32(&R.done[b >> R.bshift]) : 0u;
      if (s_pub_seen[w] < it + 1) {
        s_pub_seen[w] = ld_acquire_gpu(pub);
#pragma unroll
        for (int k = 0; k < ENS_RING; ++k) s_hring[w][k] = __longlong_as_double(__ldcg(pub + 1 + k));
      }
    };
    if (lane == 0) {
      s_pub_seen[w] = 0;
      s_base[w] = 0ull;
      s_next_it[w] = 0;
      s_wait[w][0] = s_wait[w][1] = 0ull;
      take(atomicAdd(R.cursor, 1ull));
    }
    for (;;) {
      if (lane == 0) {
        const int it = s_next_it[w];
        s_it[w] = it;
        if (it >= 0) {
          const unsigned b = s_next_b[w];
          s_b[w] = b;
          unsigned long long t0 = 0, t1 = 0;
          const bool dbg = R.dbg != nullptr && it < R.dbg_iters && b == 0;
          if (dbg) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
          // the batch's positions were written by whoever ran it in the previous iteration
          unsigned dn = s_done_seen[w];
          if (dn < (unsigned)it) {
            unsigned long long ta = 0, tb = 0;
            if (R.dbg != nullptr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ta));
            while (dn < (unsigned)it) {
              __nanosleep(100);
              dn = ld_acquire_gpu_u32(&R.done[b >> R.bshift]);
            }
            if (R.dbg != nullptr) {
              asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tb));
              s_wait[w][0] += tb - ta;
            }
          }
          long long ps = s_pub_seen[w];
          if (ps < it + 1) {
            unsigned long long ta = 0, tb = 0;
            if (R.dbg != nullptr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ta));
            while (ps < it + 1) {
              __nanosleep(200);
              ps = ld_acquire_gpu(pub);
              if (ps >= it + 1) {
#pragma unroll
                for (int k = 0; k < ENS_RING; ++k) s_hring[w][k] = __longlong_as_double(__ldcg(pub + 1 + k));
                s_pub_seen[w] = ps;
              }
            }
            if (R.dbg != nullptr) {
              asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tb));
              s_wait[w][1] += tb - ta;
            }
          }
          // (a ring slot is rewritten only after the iteration it belonged to has completed everywhere, and the
          // counter is re-read whenever a newer iteration is needed, so slot it % ENS_RING read behind a counter
          // value >= it + 1 holds the step size of iteration it: a later one of the same slot is published only
          // after iteration it + ENS_RING - 1 - lag >= it + 1 has been reduced, i.e. after every batch of `it` ran)
          s_hcur[w] = s_hring[w][it % ENS_RING];
          if (dbg) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            R.dbg[it * 8 + 5] = (long long)t0;
            R.dbg[it * 8 + 6] = (long long)(t1 - t0);  // time spent waiting for the group and the step size
          }
        }
      }
      __syncwarp();  // (also orders the other lanes' loads behind lane 0's acquires)
      if (s_it[w] < 0) {
        if (lane == 0 && R.dbg != nullptr) {  // totals over all compute warps, behind the per-iteration stamps
          atomicAdd(reinterpret_cast<unsigned long long*>(R.dbg) + 8 * R.dbg_iters + 0, s_wait[w][0]);
          atomicAdd(reinterpret_cast<unsigned long long*>(R.dbg) + 8 * R.dbg_iters + 1, s_wait[w][1]);
          atomicAdd(reinterpret_cast<unsigned long long*>(R.dbg) + 8 * R.dbg_iters + 2, 1ull);
        }
        break;
      }
      // the round trip of the next atomic hides behind this batch (its result is first used after the trajectories)
      if (lane == 0) g_next = atomicAdd(R.cursor, 1ull);
      {
        // (everything about the pair lives in this scope and is re-read from shared memory afterwards: values kept
        // in registers across the trajectory body cost the kernel its eighth resident CTA per SM)
        const int it = s_it[w];
        const unsigned b = s_b[w];
        const long long lo = ((long long)b * 32) << R.sshift;
        IterArgs<T> A = Ain;
        A.h = (T)s_hcur[w];
        A.h2 = A.h * A.h;
        A.P = min(32LL << R.sshift, Ain.P - lo);
        A.q = Ain.q + lo;
        A.mass = Ain.mass + lo;
        A.offset = Ain.offset + (u64)lo;
        if (Ain.accept != nullptr) A.accept = Ain.accept + lo;
        A.iter = Ain.iter + (u64)it;
        A.partials = reinterpret_cast<double*>(static_cast<T*>(R.brows) + ((size_t)b << R.sshift) * NAP);
        k_small_body<T, DT, Pot, INTEG, true, EXACT, NoStepHook, true>(A, pot, k1_smem, 0u, 1u);
      }
      const int it = *(volatile int*)&s_it[w];
      const unsigned b = *(volatile unsigned*)&s_b[w];
      if (R.trace != nullptr) {
        // kept positions of the first ntrace local particles (each thread re-reads what it wrote itself)
        for (int sb = 0; sb < (1 << R.sshift); ++sb) {
          const long long i = ((((long long)b << R.sshift) + sb) * 32) + lane;
          if (i < min(R.ntrace, Ain.P))
            for (int d = 0; d < Dn; ++d) R.trace[((long long)d * R.ntrace + i) * R.S + R.s0 + it] = Ain.q[d * Ain.q_ld + i];
        }
      }
      if (R.cmean != nullptr && it >= R.windowStart) {
        // per-chain moments of the window (nested R-hat), from the positions each thread just wrote; the next
        // iteration of these particles reads the accumulators behind the same release / acquire as their positions
        const long long n = (long long)(it - R.windowStart) + 1;
        const T rn = R.crcp[n - 1];
        // (kept rolled: a handful of registers at this point, next to the trajectory's 64)
#pragma unroll 1
        for (int sb = 0; sb < (1 << R.sshift); ++sb) {
          const long long i = ((((long long)b << R.sshift) + sb) * 32) + lane;
          if (i < Ain.P)
#pragma unroll 1
            for (int d = 0; d < Dn; ++d)
              chain_moments_update(&R.cmean[d * R.c_ld + i], &R.cm2[d * R.c_ld + i], Ain.q[d * Ain.q_ld + i], n, rn);
        }
      }
      __syncwarp();  // positions, chain moments and the batch row are written (memory ordering among the warp's lanes)
      const unsigned grp = b >> R.bshift;
      const unsigned b0 = grp << R.bshift;
      const unsigned cnt = min(1u << R.bshift, NB - b0);  // batches of this group
      int last = 0;
      if (lane == 0) {
        // release: what the whole warp wrote is visible to whoever acquires; acquire: the last arrival sees the
        // rows of every batch of the group
        unsigned old;
        asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(&R.arrived[grp]) : "memory");
        last = (old + 1u == ((unsigned)it + 1u) * cnt) ? 1 : 0;
      }
      last = __shfl_sync(0xffffffffu, last, 0);
      if (last) {
        // the group's row: its batch rows in batch order, float64; padded dimensions are dropped
        const int ring = it % ENS_RING;
        const unsigned r0 = b0 << R.sshift;                           // first sub-batch row of the group
        const unsigned nr = min(cnt << R.sshift, R.nrows - r0);       // (the last batch may be short of sub-batches)
        const T* br = static_cast<const T*>(R.brows) + (size_t)r0 * NAP;
        double* out = R.rows + ((size_t)ring * V + grp) * NS;
        for (int j = lane; j < NAP; j += 32) {
          double sum = 0.0;
#pragma unroll 8
          for (unsigned r = 0; r < nr; ++r) sum += (double)__ldcg(&br[(size_t)r * NAP + j]);
          int o = j;
          if (j >= 3 + DT) {
            const int d = j - 3 - DT;
            o = d < Dn ? 3 + Dn + d : -1;
          } else if (j >= 3) {
            o = (j - 3) < Dn ? j : -1;
          }
          if (o >= 0) out[o] = sum;
        }
        __syncwarp();
        if (lane == 0) {
          asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&R.done[grp]), "r"((unsigned)it + 1u) : "memory");
          asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(&R.gticket[ring * ngroups + grp / ENS_GROUP])
                       : "memory");
        }
      }
      if (lane == 0) {
        if (R.dbg != nullptr && it < R.dbg_iters && b == 0) {
          unsigned long long t;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
          R.dbg[it * 8 + 7] = (long long)t;
        }
        take(g_next);
      }
    }
    return;
  }

  // ===== service CTAs (the last ENS_SERVICE_CTAS blocks): 32 independent warps, no block-wide barrier =====
  // Warp w reduces the rows of groups w, w + 32, ... (ENS_GROUP consecutive slices each; lane j adds column j over
  // the group's rows: independent loads, fixed order) as soon as the group's tickets are in.
  // Warp 0 is also the MASTER: group rows -> this GPU's vector, all-reduce over NVLink, step-size update, publish.
  // Everything that polls or waits for L2 / NVLink latency lives here, off the compute CTAs' path; 190 KB of rows
  // through ONE CTA took longer than an iteration of the 8-GPU shard and set the pace of the whole run.
  const int lane = tid & 31;
  const unsigned sw = (blockIdx.x - ncompute) * (K1_THREADS / 32) + (tid >> 5);  // service warp index, 0 .. 31
  constexpr unsigned NSW = ENS_SERVICE_CTAS * (K1_THREADS / 32);
  double* loc = k1_smem;        // (master) [<= 67] this GPU's vector
  double* tot = k1_smem + 72;   // (master) [<= 67] the world's
  const bool master = sw == 0;
  double s_h = 0.0, s_logh = 0.0;
  unsigned long long s_k = 0ull;
  if (master) {
    if (lane == 0) {
      s_h = R.state[0];
      s_logh = R.state[1];
      s_k = (unsigned long long)R.state[2];
      for (int k = 0; k <= R.lag; ++k) R.hsched[k] = s_h;  // the first 1 + lag iterations run with the incoming step size
    }
    s_h = __shfl_sync(0xffffffffu, s_h, 0);
    for (int c = lane; c < ENS_PUB_COPIES; c += 32) {
      for (int k = 0; k <= R.lag; ++k) R.published[c * 16 + 1 + k] = __double_as_longlong(s_h);
      st_release_gpu(R.published + c * 16, (long long)R.lag + 1);
    }
  }
  auto stamp = [&](int it, int k) {
    if (R.dbg != nullptr && master && lane == 0 && it < R.dbg_iters) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      R.dbg[it * 8 + k] = (long long)t;
    }
  };
  for (int it = 0; it < R.nIter; ++it) {
    const int par = it & 1;          // mailbox slot (the masters of all ranks advance in step)
    const int ring = it % ENS_RING;  // rows and tickets of this iteration
    // ---- first level: my groups ----
    for (unsigned g = sw; g < ngroups; g += NSW) {
      const unsigned gsize = min((unsigned)ENS_GROUP, V - g * ENS_GROUP);
      unsigned* gt = &R.gticket[ring * ngroups + g];
      if (lane == 0) {
        while (ld_acquire_gpu_u32(gt) < gsize) __nanosleep(100);
        *gt = 0u;  // next used ENS_RING iterations later, behind a step size published after this iteration's update
      }
      __syncwarp();
      const double* rows = R.rows + ((size_t)ring * V + (size_t)g * ENS_GROUP) * NS;
      for (int j = lane; j < NS; j += 32) {
        double sum = 0.0;
#pragma unroll 8
        for (unsigned r = 0; r < gsize; ++r) sum += __ldcg(&rows[(size_t)r * NS + j]);
        R.grows[((size_t)ring * ngroups + g) * NS + j] = sum;
      }
      __syncwarp();
      if (lane == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(&R.ticket[32 * ring]) : "memory");
    }
    if (!master) continue;
    // ---- master: second level, all-reduce, update, publish ----
    if (lane == 0) {
      while (ld_acquire_gpu_u32(&R.ticket[32 * ring]) < ngroups) __nanosleep(100);
      R.ticket[32 * ring] = 0u;  // nobody touches this ring slot again before the step size below is published
    }
    __syncwarp();
    stamp(it, 0);
    const double* grows = R.grows + ((size_t)ring * ngroups) * NS;
    for (int j = lane; j < NS; j += 32) {
      double sum = 0.0;
#pragma unroll 8
      for (unsigned r = 0; r < ngroups; ++r) sum += __ldcg(&grows[(size_t)r * NS + j]);
      loc[j] = sum;
    }
    __syncwarp();
    stamp(it, 1);
    if (R.world > 1) {
      // All-reduce, "LL" style: every 8-byte word that crosses NVLink carries its own flag -- {half of a double,
      // 32-bit sequence number} -- so there is no separate flag store and no system-scope fence (remote stores +
      // __threadfence_system + flag took 8-10 us here; this takes one NVLink store latency).  8-byte stores are
      // single transactions; the slot of this parity was last written two iterations ago with sequence - 2.
      const unsigned flag = (unsigned)(R.seq0 + (unsigned long long)it + 1ull);
      const size_t slot = ((size_t)par * R.world + R.rank) * ENS_MB_STRIDE;
      const int NW = 2 * NS;  // words per vector
      for (int w = lane; w < NW; w += 32) {
        const unsigned long long bits = (unsigned long long)__double_as_longlong(loc[w >> 1]);
        const unsigned half = (w & 1) ? (unsigned)(bits >> 32) : (unsigned)bits;
        const unsigned long long word = ((unsigned long long)flag << 32) | half;
        for (int r = 0; r < R.world; ++r)
          if (r != R.rank) st_relaxed_sys(reinterpret_cast<unsigned long long*>(R.peers[r]) + slot + w, word);
      }
      stamp(it, 2);
      // receive: poll every word of every peer's slot in MY mailbox; halves go to shared memory.  The (world - 1) NW
      // words are dealt to the lanes and up to eight are in flight per lane: polled one after the other (a system-
      // scope load is a 1-2 us round trip under load) the 7 x 46 words of an 8-GPU run made the master's period --
      // and with it every iteration of the run -- 10 us longer than the trajectories (profiles/r02_bench_n8.json:
      // 41.8 us per iteration at 8 GPUs against 32.4 us for the same shard without peers).
      unsigned* rx = reinterpret_cast<unsigned*>(k1_smem + 144);  // [world][NW]
      const unsigned long long* mine =
          reinterpret_cast<const unsigned long long*>(R.peers[R.rank]) + (size_t)par * R.world * ENS_MB_STRIDE;
      const int total = (R.world - 1) * NW;
      for (int k0 = lane; k0 < total; k0 += 32 * 8) {
        const unsigned long long* src[8];
        unsigned long long word[8];
        int dst[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = k0 + 32 * j;
          dst[j] = -1;
          src[j] = mine;
          if (k < total) {
            const int pi = k / NW, w = k - pi * NW;
            const int r = pi + (pi >= R.rank ? 1 : 0);
            src[j] = mine + (size_t)r * ENS_MB_STRIDE + w;
            dst[j] = r * NW + w;
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) word[j] = dst[j] >= 0 ? ld_relaxed_sys(src[j]) : 0ull;  // independent loads
        bool pending;
        do {
          pending = false;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (dst[j] >= 0 && (unsigned)(word[j] >> 32) != flag) {
              word[j] = ld_relaxed_sys(src[j]);
              pending = pending || (unsigned)(word[j] >> 32) != flag;
            }
        } while (pending);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (dst[j] >= 0) rx[dst[j]] = (unsigned)word[j];
      }
      __syncwarp();
      stamp(it, 3);
      for (int j = lane; j < NS; j += 32) {
        double s = 0.0;
        for (int r = 0; r < R.world; ++r) {  // rank order: the same bits on every rank
          const unsigned long long bits = ((unsigned long long)rx[r * NW + 2 * j + 1] << 32) | rx[r * NW + 2 * j];
          s += r == R.rank ? loc[j] : __longlong_as_double((long long)bits);
        }
        tot[j] = s;
      }
    } else {
      for (int j = lane; j < NS; j += 32) tot[j] = loc[j];
    }
    __syncwarp();
    if (lane == 0) {
      // Robbins-Monro on log h (parallel.StepSizeAdapter / ehmc_adapt_step): the update computed from iteration
      // `it` is first used by iteration it + 1 + lag.  gains[i] = gain0 / (k0 + 1 + i)^kappa comes from the host.
      const double meanAcc = tot[1] / R.Ptot;
      if (it < R.adaptIters) {
        s_k += 1ull;
        const double acc = isfinite(meanAcc) ? meanAcc : 0.0;
        double move = R.gains[it] * (acc - R.target);
        move = fmin(fmax(move, -R.maxMove), R.maxMove);
        s_logh = fmin(fmax(s_logh + move, R.logLo), R.logHi);
        s_h = exp(s_logh);
      }
      R.hsched[it + 1 + R.lag] = s_h;
    }
    {
      const double hn = __shfl_sync(0xffffffffu, s_h, 0);
      for (int c = lane; c < ENS_PUB_COPIES; c += 32) {
        R.published[c * 16 + 1 + (it + 1 + R.lag) % ENS_RING] = __double_as_longlong(hn);
        st_release_gpu(R.published + c * 16, (long long)it + 2 + R.lag);  // release: behind the step size in the same line
      }
    }
    stamp(it, 4);
    if (lane == 0 && R.history != nullptr) {
      R.history[4 * it + 0] = tot[0] / R.Ptot;
      R.history[4 * it + 1] = tot[1] / R.Ptot;
      R.history[4 * it + 2] = tot[2] / R.Ptot;
      R.history[4 * it + 3] = R.hsched[it];
    }
    if (R.moments != nullptr)
      for (int j = lane; j < 2 * Dn; j += 32) R.moments[j] += tot[3 + j];
    __syncwarp();
  }
  if (master && lane == 0) {
    // the step size the NEXT iteration would use (the host loop's stepSize after the run)
    R.state[0] = s_h;
    R.state[1] = s_logh;
    R.state[2] = (double)s_k;
    R.state[3] += (double)R.nIter;
  }
}

}  // namespace ehmc
