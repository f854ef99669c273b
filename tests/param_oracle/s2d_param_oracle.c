/*
 * s2d_param_oracle.c - TEST INFRASTRUCTURE: SHOOT with S2D_ACT_PARAMETERIZED (include/soccer2d.h) on top of the CPU
 * oracle, in the oracle's two builds (f64: the truth, f32: the bit-exact mirror of the CUDA kernels).
 *
 * The spec defines a parameterized row as the S2D_ACT_COMMAND row it stands for, so the cycle is the oracle's,
 * unchanged (this file includes oracle/s2d_oracle.c and adds to it): the simulation is created in command mode and every
 * row is translated into a float command row before the oracle steps it.  The translation is computed in `real` (the f64
 * build rounds its products to float where they enter the float row, as the oracle does for S2D_ACT_TURNING).
 */
#include "../../oracle/s2d_oracle.c"

/* r_clamp turns a NaN into +1, as fminf / fmaxf do in the kernels */
static void param_command(const float* a, float* row) {
  real p[8];
  for (int j = 0; j < 8; ++j) p[j] = r_clamp(RC(-1.0), (real)a[j], RC(1.0));
  row[0] = row[1] = row[2] = row[3] = 0.0f;
  if (p[0] >= p[1] && p[0] >= p[2]) {
    row[0] = (float)S2D_CMD_DASH; row[1] = (float)((p[3] + RC(1.0)) * RC(50.0)); row[2] = (float)(p[4] * RC(180.0));
  } else if (p[1] >= p[2]) {
    row[0] = (float)S2D_CMD_TURN; row[1] = (float)(p[5] * RC(180.0));
  } else {
    row[0] = (float)S2D_CMD_KICK; row[1] = (float)((p[6] + RC(1.0)) * RC(50.0)); row[2] = (float)(p[7] * RC(180.0));
  }
}

/* SHOOT + S2D_ACT_PARAMETERIZED only; the simulation underneath steps command rows */
int s2dop_create(const S2DConfig* cfg, void** out) {
  if (!cfg || cfg->scenario != S2D_SCENARIO_SHOOT || cfg->action_mode != S2D_ACT_PARAMETERIZED) return -1;
  S2DConfig c = *cfg;
  c.action_mode = S2D_ACT_COMMAND;
  return s2do_create(&c, out);
}

/* the command rows [N][K][4] that the parameterized rows [N][K][8] stand for */
void s2dop_translate(const float* actions, int64_t rows, float* commands) {
  for (int64_t r = 0; r < rows; ++r) param_command(actions + r * 8, commands + r * 4);
}

/* s2do_step with parameterized rows [N][K][8] */
void s2dop_step(void* h, const float* actions, int K, real* obs, real* reward, uint8_t* done, uint8_t* result,
                real* term_obs) {
  OSim* s = (OSim*)h;
  const int64_t rows = s->cfg.num_envs * K;
  float* commands = (float*)malloc((size_t)rows * 4 * sizeof(float));
  s2dop_translate(actions, rows, commands);
  s2do_step(h, commands, K, obs, reward, done, result, term_obs);
  free(commands);
}
