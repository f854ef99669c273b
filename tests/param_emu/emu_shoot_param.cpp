// emu_shoot_param.cpp - TEST-ONLY: tests/emu (the kernel source compiled for the host, included unchanged) with SHOOT's
// parameterized actions: each 8-float row goes through the kernels' own parameterized_command (s2d_scenarios.cuh), then
// substep<SHOOT, S2D_ACT_COMMAND>, as step_kernel does.
#include "../emu/emu_reachball.cpp"

template <class SP>
static void step_param(Emu* h, const float* actions, int K, float* obs, float* reward, uint8_t* done, uint8_t* result,
                       double* stats) {
  const KernelParams& P = h->kp;
  const SP sp(P.cc);
  const int64_t n = P.num_envs;
  for (int64_t i = 0; i < n; ++i) {
    Episode e;
    LaunchOut out;
    load_episode(P.state, n, i, e);
    const uint64_t gid = (uint64_t)(P.env_id_offset + i);
    for (int k = 0; k < K; ++k) {
      const float* a = actions + (i * K + k) * 8;
      const float4 c = parameterized_command(make_float4(a[0], a[1], a[2], a[3]), make_float4(a[4], a[5], a[6], a[7]));
      substep<S2D_SCENARIO_SHOOT, S2D_ACT_COMMAND>(e, P, sp, gid, i, c.x, c.y, c.z, c.w, out);
    }
    store_episode(P.state, n, i, e);
    scenario_obs<S2D_SCENARIO_SHOOT>(e, obs + i * kObsDim);
    reward[i] = out.reward_sum;
    done[i] = (uint8_t)(out.ended != 0);
    result[i] = (uint8_t)out.last_result();
    stats[0] += out.episodes(); stats[1] += out.goals(); stats[2] += out.outs(); stats[3] += out.timeouts();
    stats[4] += out.ep_steps; stats[5] += out.ret;
  }
}

extern "C" void emu_step_param(void* p, const float* actions, int K, float* obs, float* reward, uint8_t* done,
                               uint8_t* result, float* terminal_obs, double* stats6) {
  Emu* h = (Emu*)p;
  h->kp.terminal_obs = terminal_obs;
  if (h->kp.noise) step_param<NoisySP>(h, actions, K, obs, reward, done, result, stats6);
  else if (h->default_sp) step_param<DefaultSP>(h, actions, K, obs, reward, done, result, stats6);
  else step_param<RuntimeSP>(h, actions, K, obs, reward, done, result, stats6);
}
