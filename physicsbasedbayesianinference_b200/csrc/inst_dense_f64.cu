#include "inst_dense.cuh"
namespace ehmc {
template int launch_dense<double>(ehmc_ctx*, const ehmc_potential*, const IterArgs<double>&, int, bool, cudaStream_t);
template int dense_particles_per_cta<double>();
template int dense_tnp<double>(int);
template int build_dense<double>(ehmc_potential*, std::vector<double>&, std::vector<double>&);
}  // namespace ehmc
