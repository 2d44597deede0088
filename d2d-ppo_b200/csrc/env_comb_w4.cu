// CombinatorialEnv step kernels for 16-byte packet-buffer records (max deadline <= 16).
#include "env_comb_step.cuh"
namespace d2d {
template int launch_comb_step<4>(const StepArgs&, int, int, int, cudaStream_t);
template int launch_comb_run<4>(const StepArgs&, const RunArgs&, int, cudaStream_t);
}
