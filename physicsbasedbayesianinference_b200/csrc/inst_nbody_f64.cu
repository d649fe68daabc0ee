#include "inst_nbody.cuh"
namespace ehmc {
template int launch_nbody<double>(ehmc_ctx*, const ehmc_potential*, const IterArgs<double>&, int, bool, cudaStream_t);
template int eval_nbody<double>(ehmc_ctx*, const ehmc_potential*, const double*, long long, long long, double*, double*, long long,
                             cudaStream_t);
template int colstats<double>(ehmc_ctx*, const double*, long long, long long, int, double*, cudaStream_t);
template int build_nbody<double>(ehmc_potential*, const std::vector<double>&);
}  // namespace ehmc
