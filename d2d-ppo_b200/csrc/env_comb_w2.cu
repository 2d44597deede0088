// CombinatorialEnv step kernels for 8-byte packet-buffer records (max deadline <= 8).
#include "env_comb_step.cuh"
namespace d2d {
template int launch_comb_step<2>(const StepArgs&, int, int, int, cudaStream_t);
template int launch_comb_run<2>(const StepArgs&, const RunArgs&, const CombRunParams&, int, cudaStream_t);
}
