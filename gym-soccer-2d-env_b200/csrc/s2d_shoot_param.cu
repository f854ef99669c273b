// s2d_shoot_param.cu - SHOOT with the parameterized action space (S2D_ACT_PARAMETERIZED, include/soccer2d.h): the step
// kernels and the fused tcgen05 DDPG actor, one of each for every constants variant.  They live in a translation unit
// of their own for the reason launch_fullgame_scripted (s2d_fullgame.cuh) gives: instantiated next to the other
// kernels, they could change how ptxas compiles the out-of-line functions all of them share.
#include "s2d_rollout_tc5.cuh"

namespace s2d {

cudaError_t launch_shoot_param(int var, int grid, const KernelParams& kp, int k_substeps, cudaStream_t s) {
  constexpr int SCN = S2D_SCENARIO_SHOOT, ACT = S2D_ACT_PARAMETERIZED;
  if (var == kVarNoisy) step_kernel<SCN, ACT, kVarNoisy><<<grid, kBlock, 0, s>>>(kp, k_substeps);
  else if (var == kVarDefault) step_kernel<SCN, ACT, kVarDefault><<<grid, kBlock, 0, s>>>(kp, k_substeps);
  else if (var == kVarRuntime) step_kernel<SCN, ACT, kVarRuntime><<<grid, kBlock, 0, s>>>(kp, k_substeps);
  else return cudaErrorInvalidValue;
  return cudaSuccess;
}

cudaError_t launch_shoot_param_actor(int var, int grid, const KernelParams& kp, int k_substeps, const MlpWeights& w,
                                     float noise, const TrajOut& traj, cudaStream_t s) {
  constexpr int SCN = S2D_SCENARIO_SHOOT, ACT = S2D_ACT_PARAMETERIZED;
  if (var == kVarNoisy)
    rollout_mlp_tc5_kernel<SCN, kVarNoisy, ACT><<<grid, kBlock, 0, s>>>(kp, k_substeps, w, noise, nullptr, nullptr, traj);
  else if (var == kVarDefault)
    rollout_mlp_tc5_kernel<SCN, kVarDefault, ACT><<<grid, kBlock, 0, s>>>(kp, k_substeps, w, noise, nullptr, nullptr, traj);
  else if (var == kVarRuntime)
    rollout_mlp_tc5_kernel<SCN, kVarRuntime, ACT><<<grid, kBlock, 0, s>>>(kp, k_substeps, w, noise, nullptr, nullptr, traj);
  else return cudaErrorInvalidValue;
  return cudaSuccess;
}

}  // namespace s2d
