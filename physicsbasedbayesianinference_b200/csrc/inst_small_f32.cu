#include "inst_small.cuh"
namespace ehmc {
template int launch_small<float>(ehmc_ctx*, const ehmc_potential*, const IterArgs<float>&, int, bool, cudaStream_t);
template int eval_small<float>(ehmc_ctx*, const ehmc_potential*, const float*, long long, long long, float*, float*,
                               long long, cudaStream_t);
template int run_small<float>(ehmc_ctx*, const ehmc_potential*, const IterArgs<float>&, int, const RunArgs<float>&, cudaStream_t);

// the dispatcher with nothing to launch (which functors exist does not depend on the dtype)
bool has_small_kernel(const ehmc_potential* p) {
  return with_small_pot<float>(p, nullptr, [](auto, const auto&) { return EHMC_OK; }) == EHMC_OK;
}
}  // namespace ehmc
