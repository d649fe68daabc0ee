#include "inst_logistic.cuh"
namespace ehmc {
template int launch_logistic<double>(ehmc_ctx*, const ehmc_potential*, const IterArgs<double>&, int, bool, cudaStream_t, int);
template int eval_logistic<double>(ehmc_ctx*, const ehmc_potential*, const double*, long long, long long, double*, double*,
                                long long, cudaStream_t);
template int build_logistic<double>(ehmc_potential*, const std::vector<double>&, const std::vector<double>&, int);
}  // namespace ehmc
