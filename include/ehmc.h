/*
 * ehmc -- B200-native ensemble-HMC engine: C-ABI of the leapfrog hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference
 * (Anton-Le/PhysicsBasedBayesianInference) is pure Python and has no FFI; what
 * a binding for its hot path has to replace is the arithmetic of
 *
 *   Ensemble.setPosition / setMomentum      src/ensemble.py:63-93
 *   Leapfrog.integrate                      src/integrator.py:94-123
 *   StormerVerlet.integrate                 src/integrator.py:126-165
 *   Integrator.getAccel (gradient call)     src/integrator.py:61-73
 *   potential.* (U and grad U)              src/potential.py:18-53
 *   HMC.getWeightsRatio + getSamples body   src/HMC.py:106-116, 150-179
 *
 * Each entry point below names the reference lines it stands in for.  The
 * Python classes in physicsbasedbayesianinference_b200/ (same names and
 * signatures as the reference's) bind these symbols through ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *  - All tensors are borrowed DLTensor views (ehmc_dlpack.h).  State arrays are
 *    (D, P) = (numDimensions, numParticles) with the PARTICLE index contiguous
 *    (stride[1] == 1), exactly the reference's C-order np.zeros((D, P)) layout
 *    (src/ensemble.py:40-41); stride[0] >= P may be larger (a column slice of a
 *    bigger ensemble is a valid shard).  dtype float32 or float64, the same for
 *    every tensor of a call.
 *  - Tensors on kDLCUDA are used in place and all work is enqueued on `stream`
 *    (a cudaStream_t; NULL = legacy default stream) without any host sync.
 *    Tensors on kDLCPU / kDLCUDAHost select the HOST path: the library stages
 *    them through context-owned device buffers (chunked, double-buffered H2D /
 *    kernel / D2H) and returns after the results are back in host memory.
 *  - Every function returns EHMC_OK (0) or a negative ehmc_status; the message is
 *    available from ehmc_last_error().  No C++ exception crosses this boundary.
 *  - A context is bound to one CUDA device and is not thread-safe.
 *  - There is NO CPU implementation behind this interface: without a CUDA device
 *    ehmc_ctx_create fails with EHMC_ERR_CUDA.
 *
 * RNG stream (production mode, z == NULL / u == NULL): Philox4x32-10 with
 *    counter = (particle id lo, particle id hi, block, iteration lo)
 *    key     = (seed lo, seed hi ^ iteration hi)
 *  where "particle id" is the GLOBAL index (particleOffset + column), so results
 *  do not depend on how the ensemble is sharded over GPUs.  float32: block b
 *  gives the standard normals of dimensions 4b..4b+3 (two Box-Muller pairs);
 *  float64: block b gives dimensions 2b, 2b+1 from 53-bit uniforms.
 *  Metropolis uniform, stream version EHMC_RNG_STREAM_VERSION = 2: float32 state with D mod 4 in {1, 2} (the last
 *  normal block, D / 4, leaves its words z and w unused): (z >> 8) 2^-24 of that block, so that a kernel which has
 *  just drawn the momentum needs no further Philox block (D = 10: 3 blocks instead of 4); every other case: word x
 *  (float64: x, y) of block 0xFFFFFFFF.  Version 1 (library versions < 110) always used block 0xFFFFFFFF.
 *  oracle/hmc_oracle.py::philox_stream is the bit-level specification used by the tests.
 *  Replica-exchange uniform of ehmc_hmc_run_tempered (a new block; no earlier draw changes): block 0xFFFFFFFE with
 *  the counter of the pair's LOWER particle (its global id, the iteration of the swap), float32 (x >> 8) 2^-24,
 *  float64 ((x >> 6) << 27 | y >> 5) 2^-53.  tests/tempering_reference.py::swap_uniform specifies it bit for bit.
 */
#ifndef EHMC_H_
#define EHMC_H_

#include <stdint.h>

#include "ehmc_dlpack.h"

#ifdef __cplusplus
extern "C" {
#endif

#define EHMC_VERSION 110 /* 0.1.1 */
#define EHMC_RNG_STREAM_VERSION 2 /* see "RNG stream" above */

#if defined(__GNUC__)
#define EHMC_API __attribute__((visibility("default")))
#else
#define EHMC_API
#endif

typedef struct ehmc_ctx ehmc_ctx;
typedef struct ehmc_potential ehmc_potential;

typedef enum {
  EHMC_OK = 0,
  EHMC_ERR_INVALID = -1,     /* bad argument: shape, dtype, stride, device, NULL */
  EHMC_ERR_CUDA = -2,        /* CUDA runtime error (no device, launch failure, ...) */
  EHMC_ERR_UNSUPPORTED = -3, /* valid request outside the built kernel set */
  EHMC_ERR_NOMEM = -4
} ehmc_status;

/* Potential families (replace the reference's arbitrary `potential`/`gradient`
 * Python callables, src/HMC.py:52-60, src/integrator.py:73). */
typedef enum {
  /* U = 0.5 * dot(k, q**2)  -- harmonicPotentialND, src/potential.py:18-27.
   * params: k[D].  scalars: none. */
  EHMC_FAMILY_DIAG_GAUSSIAN = 1,
  /* U = 0.5 (q-mu)^T Lambda (q-mu) -- the Gaussian targets of src/tests/test_HMC.py:122-125.
   * params: Lambda[D,D] (row-major), optional mu[D].  scalars: none. */
  EHMC_FAMILY_DENSE_GAUSSIAN = 2,
  /* Neal's funnel, v = q[0]: U = v^2/(2 s^2) + 0.5 e^{-v} sum_{k>=1} q_k^2 + 0.5 (D-1) v.
   * params: none.  scalars: {D, s} or {D, s, scaleV, scaleX}: the same potential of v = scaleV q[0],
   * x_k = scaleX q[k] (rescaled coordinates = diagonal mass matrix, HMC.run(adaptMass=True)). */
  EHMC_FAMILY_FUNNEL = 3,
  /* Each ensemble particle is a B-body system, coordinates d = c*B + b (src/potential.py:83-84):
   * U = -G sum_{i<j} m_i m_j / sqrt(|r_i-r_j|^2 + eps^2); -grad_i U / m_i is getAccelNBody
   * (src/potential.py:30-53) for eps = 0.  params: bodyMass[B].  scalars: {G, eps}. */
  EHMC_FAMILY_NBODY = 4,
  /* Bayesian logistic regression: U = sum_n softplus(x_n.q) - y_n x_n.q + 0.5 |q|^2 / s^2.
   * params: X[N,D] (row-major), y[N].  scalars: {s, precision?}.  precision selects the gradient kernel:
   * 0 (default) CUDA cores, exact fp32 / fp64;  2 tensor cores at float32 accuracy (tcgen05 GEMM chain, every
   * operand a 2-term fp16 split, 3 MMA passes per GEMM; float32 state);  3 auto = 2 when the state is float32 and
   * the split represents X to 2^-20 per column, else 0;  1 tensor cores with bf16-rounded operands (fast, 5e-3
   * gradient accuracy: outside the 1e-5 trajectory tolerance, opt-in only). */
  EHMC_FAMILY_LOGISTIC = 5,
  /* Independent coin biases q_d in (0, 1) with a flat prior -- the reference's own NumPyro sample
   * (samples/NumpyroExamples/CoinToss/CoinToss.py:6-25):
   * U = -sum_d [ k_d ln q_d + (n_d - k_d) ln(1 - q_d) ],  dU/dq_d = -k_d/q_d + (n_d - k_d)/(1 - q_d)
   * (references/NotesOnParticleBasedHMC.pdf eq. 22).  Outside (0, 1) U is NaN, as ln of a negative
   * number is in the reference.  params: successes k[D], trials n[D].  scalars: none.  D <= 32. */
  EHMC_FAMILY_COIN_TOSS = 6,
  /* Normal-normal hierarchical model (eight schools): y_j ~ N(theta_j, sigma_j^2) with sigma_j known,
   * theta_j ~ N(mu, tau^2), mu ~ N(muLoc, muScale^2), tau ~ HalfCauchy(tauScale), j = 0 .. J-1, 1 <= J <= 30,
   * in NumPyro's unconstrained coordinates, D = J + 2:  q[0] = mu, q[1] = eta = ln tau, q[2+j] = theta_j
   * (centered = 1) or thetaTilde_j with theta_j = mu + e^eta thetaTilde_j (centered = 0).  U is minus the log
   * density with the Jacobian of eta, additive constants dropped:
   *   (mu - muLoc)^2 / (2 muScale^2) + softplus(2 eta - 2 ln tauScale) - eta + 0.5 sum_j (y_j - theta_j)^2 / sigma_j^2
   *   centred:      + J eta + 0.5 e^{-2 eta} sum_j (theta_j - mu)^2
   *   non-centred:  + 0.5 sum_j thetaTilde_j^2
   * params: y[J], sigma[J] [, scale[D]]: with scale, the same potential in rescaled coordinates, U'(q) = U(scale q)
   * (diagonal mass matrix, HMC.run(adaptMass=True)).  scalars: {muLoc, muScale, tauScale, centered}. */
  EHMC_FAMILY_HIERARCHICAL_NORMAL = 7,
  /* Mixture of K Gaussians with diagonal covariances, a multimodal target:
   *   U = -log sum_k w_k prod_d N(q_d; mu_kd, sigma_kd^2)
   * with the constants (D/2) log 2 pi and log sum_k w_k dropped; the per-component -sum_d log sigma_kd terms are
   * kept (they weigh the components against each other).  Evaluated as a max-shifted log-sum-exp, so U and grad U
   * stay finite far from every mode.  params: weights[K] (> 0, need not sum to 1), means[K,D], stds[K,D] (> 0).
   * scalars: none.  1 <= K <= 8, D <= 32 (larger: EHMC_ERR_UNSUPPORTED). */
  EHMC_FAMILY_GAUSSIAN_MIXTURE = 8
} ehmc_family;

typedef enum {
  EHMC_LEAPFROG = 0,      /* method="Leapfrog",       src/HMC.py:62-65 */
  EHMC_STORMER_VERLET = 1 /* method="Stormer-Verlet", src/HMC.py:66-69 */
} ehmc_integrator;

/* ehmc_hmc_args.flags */
#define EHMC_FLAG_BUGCOMPAT_MOMENTUM 1u /* p_out of a rejected particle = its OLD POSITION   \
                                           (src/HMC.py:176 writes oldQ, sic); off: old momentum */
#define EHMC_FLAG_REJECT_NONFINITE 2u   /* reject when exp(oldH-newH) is NaN; the reference      \
                                           ACCEPTS those (u > NaN is False, src/HMC.py:168-173) */

#define EHMC_FLAG_REUSE_ENDPOINT 4u     /* the caller guarantees that q and the potential are exactly what the  \
                                           previous ehmc_hmc_iter on this context left behind (nothing else     \
                                           touched them): families that keep an endpoint cache (logistic        \
                                           regression, pairwise gravity) take grad U(q) and U(q) of the start   \
                                           from the kept end of the previous one instead of re-evaluating them  \
                                           -- L instead of L + 1 gradient evaluations per iteration, identical  \
                                           results.  Ignored when no valid cache exists. */

typedef struct {
  uint32_t struct_size;    /* sizeof(ehmc_hmc_args), for ABI growth */
  uint32_t flags;          /* EHMC_FLAG_* */
  int32_t integrator;      /* ehmc_integrator */
  int32_t numSteps;        /* int(simulTime / stepSize), computed by the caller in Python exactly \
                              like src/integrator.py:51 -- never in C */
  double stepSize;         /* h */
  double stepSizeSq;       /* h**2 as Python computes it (src/integrator.py:114) */
  double boltzmann;        /* scipy.constants.Boltzmann */
  double temperature;      /* momentum std = sqrt((mass * boltzmann) * temperature), ensemble.py:88 */
  uint64_t seed;           /* Philox key */
  uint64_t iteration;      /* HMC iteration index (Philox counter word 3) */
  uint64_t particleOffset; /* global index of column 0 (multi-GPU shards) */
  const void* dynamic;     /* optional DEVICE pointer to an ehmc_dynamic: when set, stepSize (and its
                              square) and iteration are read from it by the kernel at run time instead of
                              from this struct (device tensors, small-D and float32 dense families) */
} ehmc_hmc_args;

/* Device-resident control block of an adaptive run: a whole iteration -- trajectory kernel,
 * statistics all-reduce, step-size update (ehmc_adapt_step) -- is enqueued, or replayed from a CUDA
 * graph, without the host reading anything back (build-defined: the reference has no adaptation). */
typedef struct {
  double stepSize;     /* h of the next ehmc_hmc_iter handed this block */
  double logStepSize;
  uint64_t iteration;  /* Philox iteration word of the next ehmc_hmc_iter */
  uint64_t updates;    /* Robbins-Monro updates applied so far (k) */
  uint64_t row;        /* next row of `history` */
} ehmc_dynamic;

/* ---- library / context ---------------------------------------------------- */
EHMC_API int ehmc_version(void);
/* Message of the last failing call on this thread (ctx may be NULL). */
EHMC_API const char* ehmc_last_error(const ehmc_ctx* ctx);
/* device < 0: current device.  Fails with EHMC_ERR_CUDA when no GPU is usable. */
EHMC_API int ehmc_ctx_create(int device, ehmc_ctx** out);
EHMC_API int ehmc_ctx_destroy(ehmc_ctx* ctx);
/* Number of kernels of THIS library launched through ctx since creation. */
EHMC_API int ehmc_ctx_launch_count(const ehmc_ctx* ctx, uint64_t* out);
/* Rows of ehmc_leapfrog / ehmc_stormer_verlet calls on the float32 tensor-core dense kernel whose position left
 * the fp16 operand range of the row's scale (a divergent trajectory: |q| grew more than 256x past
 * max(|q0|, h L |v0|)) since the last reset.  Those rows hold saturated, finite garbage; re-run the call with
 * option "dense_path" = 1 (exact CUDA-core kernel).  ehmc_hmc_iter needs no such check: it rejects those rows.
 * Synchronises the device. */
EHMC_API int ehmc_ctx_overflow_count(ehmc_ctx* ctx, uint64_t* out, int reset);
/* out[0]=SM count, out[1]=SM clock MHz (max), out[2]=total HBM bytes, out[3]=L2 bytes. */
EHMC_API int ehmc_ctx_device_info(const ehmc_ctx* ctx, double out[4]);
/* Tuning / diagnostic knobs:
 *   "dense_path"      0 auto (float32 dense Gaussian on the 3xFP16 tensor-core kernel unless the fp16 split of
 *                     Lambda would lose accuracy: ill-conditioned / wide-range matrices run on CUDA cores),
 *                     1 CUDA cores (exact fp32 FMA), 4 force 3xFP16
 *   "dense_occupancy" 1|2: CTAs/SM variant of the float32 CUDA-core dense kernel
 *   "small_waves"     resident waves of CTAs of the persistent small-D kernel (default 8)
 *   "nbody_ti"        bodies per thread of the N-body kernel (0 auto, 4, 8)
 *   "ens_sshift"      fused ensemble run: log2 of the 32-particle sub-batches a warp takes from the work queue at
 *                     once (-1 auto: 0 below 2^21 particles per GPU, above that 1, or 2 for trajectories of <= 8 steps)
 *   "ens_groups"      fused ensemble run: groups of batches (one float64 statistics row each) per iteration at most
 *                     (0 auto: 4096 for trajectories of more than 8 steps, else 2048)
 *   "host_chunk_mb"   bytes of state per staged chunk on the host path
 *   "tc_debug", "tc_prof", "tc_prof_dump"  profiling aids of the tensor-core dense kernels */
EHMC_API int ehmc_ctx_set_option(ehmc_ctx* ctx, const char* name, double value);
/* Measures the sustained FP32 FMA rate of the device with a register-only FFMA
 * kernel (2 flop per FMA) for about `millis` ms; the FP32 roofline denominator
 * (MEASURED_PEAKS.json records none).  Synchronises the device. */
EHMC_API int ehmc_measure_fp32_peak(ehmc_ctx* ctx, double millis, double* tflops_out);

/* ---- potentials ------------------------------------------------------------ */
/* Builds a device-resident, kernel-ready copy of the family's parameters (params may
 * live on host or device, float32 or float64).  `dtype_bits` (32 or 64) selects the
 * precision the potential will be used with. */
EHMC_API int ehmc_potential_create(ehmc_ctx* ctx, int family, const DLTensor* const* params, int nparams,
                          const double* scalars, int nscalars, int dtype_bits, ehmc_potential** out);
EHMC_API int ehmc_potential_destroy(ehmc_potential* pot);
/* U(q) and/or grad U(q) for every column of q[D,P]: the vectorised form of the
 * reference's potential(q[:, i]) / gradient(q[:, i]) callables (src/HMC.py:102,
 * src/integrator.py:73; harmonicPotentialND on a (D,P) array, tests/test_potential.py:23).
 * energy_out[P] and grad_out[D,P] are each optional (NULL). */
EHMC_API int ehmc_potential_eval(ehmc_ctx* ctx, const ehmc_potential* pot, const DLTensor* q,
                        DLTensor* energy_out, DLTensor* grad_out, void* stream);

/* ---- ensemble initialisation (src/ensemble.py:63-93) ----------------------- */
/* q <- N(0, qStd^2) from the Philox stream with iteration word 0xFFFFFFFFFFFFFFFF. */
EHMC_API int ehmc_set_position(ehmc_ctx* ctx, DLTensor* q, double qStd, uint64_t seed,
                      uint64_t particleOffset, void* stream);
/* p <- z * sqrt((mass * boltzmann) * temperature), z from Philox (seed, iteration). */
EHMC_API int ehmc_set_momentum(ehmc_ctx* ctx, DLTensor* p, const DLTensor* mass, double boltzmann,
                      double temperature, uint64_t seed, uint64_t iteration,
                      uint64_t particleOffset, void* stream);
/* Raw stream: z[D,P] standard normals and/or u[P] uniforms in [0,1) (either may be NULL)
 * exactly as ehmc_hmc_iter would draw them for (seed, iteration) on a D-dimensional state; u without z is the
 * uniform of block 0xFFFFFFFF (a state whose D is a multiple of 4). */
EHMC_API int ehmc_philox_fill(ehmc_ctx* ctx, DLTensor* z, DLTensor* u, uint64_t seed, uint64_t iteration,
                     uint64_t particleOffset, void* stream);

/* ---- integrators ----------------------------------------------------------- */
/* Leapfrog.integrate(), src/integrator.py:105-120: advances q, p IN PLACE by
 * numSteps steps (numSteps + 1 gradient evaluations), one fused kernel. */
EHMC_API int ehmc_leapfrog(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, DLTensor* p,
                  const DLTensor* mass, double stepSize, double stepSizeSq, int numSteps,
                  void* stream);
/* StormerVerlet.integrate(), src/integrator.py:142-163 (numSteps + 1 position updates,
 * backward-difference momentum). */
EHMC_API int ehmc_stormer_verlet(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, DLTensor* p,
                        const DLTensor* mass, double stepSize, double stepSizeSq, int numSteps,
                        void* stream);
/* Reference N-body mode (Integrator(..., gradient=None), src/integrator.py:57-59,75-85):
 * the ensemble's P particles ARE the bodies (D = 3 typically), acceleration from
 * getAccelNBody (src/potential.py:30-53) with G = gravConst; body i finishes all its
 * steps before body i+1 starts (the reference's sequential-in-time order). */
EHMC_API int ehmc_integrate_nbody_mode(ehmc_ctx* ctx, int integrator, DLTensor* q, DLTensor* p,
                              const DLTensor* mass, double gravConst, double stepSize,
                              double stepSizeSq, int numSteps, void* stream);

/* ---- one HMC iteration: the body of getSamples' loop, src/HMC.py:154-179 ---- */
/* momentum refresh (ensemble.py:88-91) -> oldH (HMC.py:108-110) -> integrate (:161) ->
 * newH (:111-114) -> ratio = exp(oldH-newH) (:115) -> reject iff u > min(1, ratio)
 * (:168-173) -> q restored where rejected (:175).
 *   q        [D,P] in/out
 *   p_out    [D,P] optional: the momentum the reference stores in momentum_hmc (:179):
 *            un-flipped integrated p where accepted; where rejected see EHMC_FLAG_BUGCOMPAT_MOMENTUM
 *   mass     [P]
 *   z        [D,P] optional standard normals (the reference's MT19937 draws, parity mode);
 *            NULL -> Philox
 *   u        [P]   optional Metropolis uniforms; NULL -> Philox
 *   accept_out [P] uint8, optional: 1 = accepted
 *   stats_out  [2D+3] float64, optional, OVERWRITTEN with this call's sums over the P
 *            particles: {n_accept, sum min(1,ratio), sum H(kept state), sum_i q[d,i] (D),
 *            sum_i q[d,i]^2 (D)} -- the per-iteration ensemble statistics that cross GPUs.
 */
EHMC_API int ehmc_hmc_iter(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, DLTensor* p_out,
                  const DLTensor* mass, const ehmc_hmc_args* args, const DLTensor* z,
                  const DLTensor* u, DLTensor* accept_out, DLTensor* stats_out, void* stream);

/* ---- the whole loop of getSamples, src/HMC.py:150-179, in ONE launch ---------------------- */
/* numIterations HMC iterations (Philox iterations args.iteration .. + numIterations - 1) with the particle
 * state held on chip in between; iteration k stores the position the reference stores in samples_hmc[:, :, k]
 * (src/HMC.py:178) and the momentum of momentum_hmc[:, :, k] (:179, same conventions as p_out of ehmc_hmc_iter).
 *   q            [D,P] in/out (device)
 *   samples_out  [D*P, S] optional: the reference's (D, P, S) array viewed as 2-D; slots
 *                sampleOffset .. sampleOffset + numIterations - 1 are written
 *   momenta_out  [D*P, S] optional
 *   accepted_out [P] int32 optional: accepted proposals per particle
 * Device tensors and the small-D families only (diagonal / small dense Gaussian, funnel, coin toss, hierarchical
 * normal, Gaussian mixture);
 * EHMC_ERR_UNSUPPORTED otherwise -- call ehmc_hmc_iter per iteration then. */
EHMC_API int ehmc_hmc_run(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, const DLTensor* mass,
                 const ehmc_hmc_args* args, int numIterations, DLTensor* samples_out, DLTensor* momenta_out,
                 int64_t sampleOffset, DLTensor* accepted_out, void* stream);

/* ---- getSamples' loop with parallel tempering (replica exchange), in ONE launch -------------------------------- */
/* Systems of R adjacent particles: particle i is replica r = i mod R of system i / R.  Slot r samples at inverse
 * temperature betas[r]: momentum std sqrt((mass * boltzmann) * temperature) / sqrt(beta_r), Metropolis test on
 * beta_r (oldH - newH) -- with boltzmann * temperature = 1 slot r targets exp(-beta_r U).  After every iteration's
 * Metropolis step the deterministic even-odd schedule proposes swaps: at Philox iteration k the pairs are
 * (r, r + 1) with r = k (mod 2); the lower particle draws u (block 0xFFFFFFFE, see "RNG stream") and the two exchange
 * their states iff u < min(1, exp((beta_r - beta_r+1)(U_r - U_r+1))) (a NaN exponent rejects).  The schedule follows
 * the global iteration, so splitting a run into several calls does not change its results.  At R = 1 (betas = {1})
 * this is ehmc_hmc_run bit for bit. */
typedef struct {
  uint32_t struct_size;   /* sizeof(ehmc_temper_args) */
  int32_t R;              /* replicas per system: 1, 2, 4, 8, 16 or 32 */
  const DLTensor* betas;  /* float64[R] device: 1 = betas[0] > betas[1] > ... > betas[R-1] > 0 (read back once) */
  DLTensor* swaps_out;    /* int32[P] device, optional: accepted swaps of slot r with slot r + 1, per particle */
  DLTensor* roundtrips_out; /* int32[P/R] device, optional: round trips per system -- a state that visited the
                               hottest slot and then reached slot 0 (labels start at the call's first iteration) */
} ehmc_temper_args;

/* numIterations tempered iterations (Philox iterations args.iteration ..), as ehmc_hmc_run:
 *   q            [D,P] in/out (device); P and args.particleOffset multiples of R
 *   samples_out  [D*P, S] optional: slot sampleOffset + k holds the positions after iteration k's swap, so slot r of
 *                a system always holds its beta_r state (slot 0: the target itself)
 *   accepted_out [P] int32 optional: accepted HMC proposals per particle
 * Small-D families, device tensors only, Philox draws only (there is no fed z / u); counts are this call's.
 * EHMC_ERR_INVALID for a bad R, ladder or shard (P or particleOffset not a multiple of R) and for host tensors,
 * EHMC_ERR_UNSUPPORTED for families without a small-D kernel and for args.dynamic. */
EHMC_API int ehmc_hmc_run_tempered(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, const DLTensor* mass,
                                   const ehmc_hmc_args* args, int numIterations, const ehmc_temper_args* temper,
                                   DLTensor* samples_out, int64_t sampleOffset, DLTensor* accepted_out, void* stream);

/* ---- the adaptive ensemble run in ONE launch, with the statistics all-reduce inside the kernel -------------- */
/* Peer-memory mailboxes: one process per GPU creates a communicator, the caller exchanges the opaque handles of
 * all ranks (any transport; the Python binding uses torch.distributed all_gather) and connects.  Needs CUDA IPC /
 * peer access between the GPUs (NVLink / NVSwitch on a B200 box). */
#define EHMC_COMM_MAX_RANKS 16
#define EHMC_COMM_HANDLE_BYTES 64
typedef struct ehmc_comm ehmc_comm;
EHMC_API int ehmc_comm_create(ehmc_ctx* ctx, int rank, int worldSize, ehmc_comm** out);
EHMC_API int ehmc_comm_handle(ehmc_comm* comm, void* out /* EHMC_COMM_HANDLE_BYTES */);
EHMC_API int ehmc_comm_connect(ehmc_comm* comm, const void* handles /* worldSize x EHMC_COMM_HANDLE_BYTES, by rank */);
EHMC_API int ehmc_comm_destroy(ehmc_comm* comm);

typedef struct {
  uint32_t struct_size;      /* sizeof(ehmc_adapt_args) */
  int32_t adaptIterations;   /* Robbins-Monro updates from the first adaptIterations iterations of the call */
  double targetAccept, gain0, kappa, maxMove, minStep, maxStep; /* parallel.StepSizeAdapter */
  double numParticlesTotal;  /* particles of ALL ranks */
  int32_t lag;               /* the statistics of iteration k set the step size of iteration k + 1 + lag: 1 (0 means 1:
                              * the one-iteration-stale pipeline of HMC.run) up to 4.  The lag has to cover the span of an
                              * iteration (hand-out of its batches, the last trajectory, the reductions, the all-reduce)
                              * in units of the time per iteration: 3 for shards of ~2^19 particles on 8 GPUs */
  int32_t reserved;
} ehmc_adapt_args;

/* numIterations iterations of the loop of src/HMC.py:150-179 on the resident ensemble (Philox iterations
 * args.iteration ..), as HMC.run drives it: every iteration's ensemble statistics {n_accept, sum acceptance
 * probability, sum H, sum q_d, sum q_d^2} are summed over the CTAs and over all ranks of `comm` INSIDE the kernel
 * (stores into the peers' mailboxes over NVLink, rank-ordered sum: identical bits on every rank), the step size
 * follows log h += clip(gain0 / k^kappa (mean acceptance probability - target)) with the statistics of iteration
 * k first used by iteration k + 1 + adapt.lag (the all-reduce hides behind the iterations in between), numSteps
 * stays fixed.
 *   state    float64[4] device, in/out: {step size, log step size, updates k, iterations run}
 *   history  float64[S,4] device, optional: {accept rate, mean acceptance probability, mean H, step size used}
 *   moments  float64[2D] device, optional, accumulated: sum q_d, sum q_d^2 over particles and iterations
 *   trace    [D*traceParticles, S] device, optional: kept positions of the first traceParticles local particles,
 *            iteration k in slot traceOffset + k
 * Small-D families (diagonal / small dense Gaussian, funnel, coin toss, hierarchical normal, Gaussian mixture), device
 * tensors,
 * leapfrog; every rank of `comm` (NULL: single GPU) must make the same call. */
EHMC_API int ehmc_hmc_run_ensemble(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, const DLTensor* mass,
                          const ehmc_hmc_args* args, int numIterations, const ehmc_adapt_args* adapt, ehmc_comm* comm,
                          DLTensor* state, DLTensor* history, DLTensor* moments, DLTensor* trace,
                          int64_t traceParticles, int64_t traceOffset, void* stream);

/* ---- per-chain moments for convergence diagnostics (nested R-hat) ------------------------------------------------ */
/* Welford's streaming update of every chain's mean and sum of squared deviations m2 with its n-th draw, in the dtype
 * of q:  n = 1: mean = q, m2 = 0 (nothing is read: the buffers need no initialisation);  n > 1: d = q - mean,
 * mean += d (1/n), m2 += d (q - mean).  The within-chain variance of N draws is m2 / (N - 1).
 *   q        [D,P] device
 *   mean, m2 [D,P] device, same dtype as q, the same row stride as each other; in/out
 * One elementwise kernel on `stream`. */
EHMC_API int ehmc_chain_moments_update(ehmc_ctx* ctx, const DLTensor* q, DLTensor* mean, DLTensor* m2, int64_t n,
                                       void* stream);

/* Optional per-chain moments of ehmc_hmc_run_ensemble_chains: iteration k >= windowStart of the call enters mean / m2
 * as draw n = k - windowStart + 1, with the update of ehmc_chain_moments_update (identical bits). */
typedef struct {
  uint32_t struct_size;  /* sizeof(ehmc_chain_args) */
  DLTensor* mean;        /* [D,P] device, dtype of q */
  DLTensor* m2;          /* [D,P] device, dtype of q, row stride of mean */
  int64_t windowStart;   /* >= 0 */
} ehmc_chain_args;

/* ehmc_hmc_run_ensemble with per-chain moments accumulated inside the same launch (chains = NULL: none; the
 * trajectories, statistics and step sizes do not depend on it). */
EHMC_API int ehmc_hmc_run_ensemble_chains(ehmc_ctx* ctx, const ehmc_potential* pot, DLTensor* q, const DLTensor* mass,
                                          const ehmc_hmc_args* args, int numIterations, const ehmc_adapt_args* adapt,
                                          ehmc_comm* comm, DLTensor* state, DLTensor* history, DLTensor* moments,
                                          DLTensor* trace, int64_t traceParticles, int64_t traceOffset,
                                          const ehmc_chain_args* chains, void* stream);

/* Consumes the (all-reduced) statistics of the iteration that just ran with the block `dynamic`:
 *   history[dynamic.row] = {acceptRate, meanAcceptProb, meanH, stepSize used}  (optional, float64 [S,4])
 *   moments[0:D] += sum q_d, moments[D:2D] += sum q_d^2                        (optional, float64 [2D])
 *   (log h, k) are taken from `state` (NULL: from `dynamic` itself) and, if dynamic.row < adaptRows,
 *       log h += clip(gain0 / k^kappa * (meanAcceptProb - targetAccept), +-maxMove),
 *       clipped to [log minStep, log maxStep]                                   (parallel.StepSizeAdapter)
 *   the result is written to `dynamic`;  dynamic.iteration += stride, dynamic.row += stride.
 * stride = 1, state = NULL: plain sequential adaptation.  stride = 2 with two blocks used alternately
 * (state = the other block) gives the one-iteration-stale pipeline of HMC.run: the update computed from
 * iteration k - 1 is consumed by iteration k + 1 and overlaps iteration k.
 * One tiny kernel on `stream`; every rank computes the same update from the same reduced numbers. */
EHMC_API int ehmc_adapt_step(ehmc_ctx* ctx, const DLTensor* stats, double numParticlesTotal, double targetAccept,
                    double gain0, double kappa, double maxMove, double minStep, double maxStep,
                    uint64_t adaptRows, void* dynamic, const void* state, uint64_t stride, DLTensor* history,
                    DLTensor* moments, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EHMC_H_ */
