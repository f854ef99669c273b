// s2d_scripted.cu - the step kernels of FULLGAME with the built-in script compiled in (scripted players:
// include/soccer2d.h, s2d_set_scripted_players): one for every (constants variant, player count, lanes per match) the
// launcher of s2d_api.cu can pick without it.  See launch_fullgame_scripted (s2d_fullgame.cuh) for why they are here.
#include "s2d_fullgame.cuh"

namespace s2d {

cudaError_t launch_fullgame_scripted(int var, int np_template, int lpm, int grid, const KernelParams& kp, int k_substeps,
                                     int np, int half_time, cudaStream_t s) {
#define S2D_GO(VAR, NP, LPM)                                                                                         \
  if (var == VAR && np_template == NP && lpm == LPM) {                                                               \
    fullgame_step_kernel<VAR + kVarScripted, NP, LPM><<<grid, kFgBlock, 0, s>>>(kp, k_substeps, np, half_time);      \
    return cudaSuccess;                                                                                              \
  }
  S2D_GO(kVarHeteroNoisy, 0, 1)
  S2D_GO(kVarHetero, 22, 1)
  S2D_GO(kVarHetero, 0, 1)
  S2D_GO(kVarNoisy, 0, 1)
  S2D_GO(kVarRuntime, 22, 2)
  S2D_GO(kVarRuntime, 22, 1)
  S2D_GO(kVarRuntime, 0, 1)
  S2D_GO(kVarDefault, 22, 2)
  S2D_GO(kVarDefault, 22, 1)
  S2D_GO(kVarDefault, 0, 1)
#undef S2D_GO
  return cudaErrorInvalidValue;  // a variant s2d_api.cu launches without the script that has no scripted twin here
}

}  // namespace s2d
