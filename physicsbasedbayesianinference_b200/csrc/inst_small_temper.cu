// Instantiations of the tempered multi-iteration kernel (k_small_run_tempered), both dtypes: a translation unit of its
// own, so that it compiles in parallel with the other small-D instances.
#include "inst_small.cuh"
namespace ehmc {
template int run_small_tempered<float>(ehmc_ctx*, const ehmc_potential*, const IterArgs<float>&, int,
                                       const RunArgs<float>&, const TemperRun&, cudaStream_t);
template int run_small_tempered<double>(ehmc_ctx*, const ehmc_potential*, const IterArgs<double>&, int,
                                        const RunArgs<double>&, const TemperRun&, cudaStream_t);
}  // namespace ehmc
