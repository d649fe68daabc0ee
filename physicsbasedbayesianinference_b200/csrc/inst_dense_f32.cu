#include "inst_dense.cuh"
namespace ehmc {
template int launch_dense<float>(ehmc_ctx*, const ehmc_potential*, const IterArgs<float>&, int, bool, cudaStream_t);
template int dense_particles_per_cta<float>();
template int dense_tnp<float>(int);
template int build_dense<float>(ehmc_potential*, std::vector<double>&, std::vector<double>&);
int dense_tn(int D) { return D <= 32 ? 4 : D <= 64 ? 8 : D <= 104 ? 13 : 16; }
}  // namespace ehmc
