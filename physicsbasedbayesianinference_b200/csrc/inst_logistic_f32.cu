#include "inst_logistic.cuh"
namespace ehmc {
template int launch_logistic<float>(ehmc_ctx*, const ehmc_potential*, const IterArgs<float>&, int, bool, cudaStream_t, int);
template int eval_logistic<float>(ehmc_ctx*, const ehmc_potential*, const float*, long long, long long, float*, float*,
                                long long, cudaStream_t);
template int build_logistic<float>(ehmc_potential*, const std::vector<double>&, const std::vector<double>&, int);
}  // namespace ehmc
