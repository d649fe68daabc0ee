#include "inst_nbody.cuh"
namespace ehmc {
template int launch_nbody<float>(ehmc_ctx*, const ehmc_potential*, const IterArgs<float>&, int, bool, cudaStream_t);
template int eval_nbody<float>(ehmc_ctx*, const ehmc_potential*, const float*, long long, long long, float*, float*, long long,
                             cudaStream_t);
template int colstats<float>(ehmc_ctx*, const float*, long long, long long, int, double*, cudaStream_t);
template int build_nbody<float>(ehmc_potential*, const std::vector<double>&);
}  // namespace ehmc
