/*
 * s2d_script_oracle.c - TEST INFRASTRUCTURE: the built-in script of FULLGAME's scripted players (include/soccer2d.h,
 * s2d_set_scripted_players) on top of the CPU oracle, in the oracle's two builds (f64: the truth, f32: the bit-exact
 * mirror of the CUDA kernel).
 *
 * The script decides from the state at the START of a cycle only, and the kernel puts its command in place of the
 * player's row of the action buffer before anything else reads that row.  So here the cycle itself is the oracle's,
 * unchanged (this file includes oracle/s2d_oracle.c and adds to it): before every cycle the scripted players' rows of a
 * copy of the actions are filled in from the oracle's state, then that one cycle is stepped.  The command crosses into
 * the float action row as any command does (in the f64 build: rounded to float where the proxy's proto message would be).
 */
#include "../../oracle/s2d_oracle.c"

static int script_in_area(const S2DServerParam* sp, real bx, real by, int left) {
  real edge = SP(pitch_half_length) - FG_PENALTY_LENGTH;
  return (left ? bx <= -edge : bx >= edge) && r_fabs(by) <= FG_PENALTY_HALF_WIDTH;
}

/* each side's chaser (-1: none), from the positions the players have now */
static void script_chasers(const OSim* s, const OEnv* e, int* chaser_l, int* chaser_r) {
  const S2DServerParam* sp = &s->cfg.sp;
  const OBall* b = &e->ball;
  int n = e->np, pps = n / 2;
  int area_l = script_in_area(sp, b->x, b->y, 1), area_r = script_in_area(sp, b->x, b->y, 0);
  real best_l = RC(3.0e38), best_r = RC(3.0e38);
  *chaser_l = *chaser_r = -1;
  for (int j = 0; j < n; ++j) {
    int left = j < pps, keeper = j == 0 || j == pps;
    int eligible = !keeper || pps == 1 || (left ? area_l : area_r);
    real dx = e->pl[j].x - b->x, dy = e->pl[j].y - b->y;
    real d2 = dx * dx + dy * dy;
    if (eligible && left && d2 < best_l) { best_l = d2; *chaser_l = j; }
    if (eligible && !left && d2 < best_r) { best_r = d2; *chaser_r = j; }
  }
}

/* the command of scripted player j: the rules of include/soccer2d.h in their order */
static void script_command(const OSim* s, const OEnv* e, uint64_t gid, int j, int chaser, float* out) {
  const S2DServerParam* sp = player_sp(s, gid, j);
  const OPlayer* p = &e->pl[j];
  const OBall* b = &e->ball;
  int pps = e->np / 2, left = j < pps, keeper = j == 0 || j == pps;
  real sg = left ? RC(1.0) : RC(-1.0);
  real hl = SP(pitch_half_length), hw = SP(pitch_half_width);
  real post = SP(goal_width) * RC(0.5) - RC(1.0);
  real obx = sg * b->x, oby = sg * b->y;
  real c = S2D_CMD_NONE, a1 = RC(0.0), a2 = RC(0.0), a3 = RC(0.0);
  int mode = e->play_mode, play_on = mode == S2D_PM_PLAY_ON;
  if (mode == S2D_PM_AFTER_GOAL || mode == S2D_PM_BEFORE_KICK_OFF || mode == S2D_PM_TIME_OVER) {
    /* 1. nobody acts */
  } else if (chaser && (play_on || e->mode_side == p->side)) {
    real dx = b->x - p->x, dy = b->y - p->y;
    real d2 = dx * dx + dy * dy;
    if (play_on && keeper && p->catch_ban == 0 && script_in_area(sp, b->x, b->y, left) && d2 <= FG_CATCH_LENGTH * FG_CATCH_LENGTH) {
      c = S2D_CMD_CATCH;
      a1 = norm_deg(atan2_deg(dy, dx) - p->body);
    } else if (!(r_sqrt(d2) > SP(player_size) + SP(ball_size) + SP(kickable_margin))) {
      real gx = hl - obx, gy = -oby;
      real g2 = gx * gx + gy * gy;
      real tx, ty, speed;
      if (g2 <= RC(625.0)) {
        tx = hl;
        ty = sg * p->y >= RC(0.0) ? -post : post;
        speed = SP(ball_speed_max);
      } else {
        real k = RC(8.0) / r_sqrt(g2);
        tx = obx + gx * k;
        ty = oby + gy * k;
        speed = RC(1.0);
      }
      c = S2D_CMD_SMART_KICK; a1 = sg * tx; a2 = sg * ty; a3 = speed;
    } else if (play_on) {
      c = S2D_CMD_INTERCEPT;
    } else {
      c = S2D_CMD_GOTO; a1 = b->x; a2 = b->y; a3 = RC(100.0);
    }
  } else if (keeper) {
    c = S2D_CMD_GOTO; a1 = sg * (RC(2.5) - hl); a2 = sg * r_clamp(-post, RC(0.3) * oby, post); a3 = RC(100.0);
  } else {
    int k = left ? j : j - pps;
    real fx = r_clamp(RC(2.5) - hl, (real)FG_FORM[k][0] + RC(0.6) * obx, hl - RC(2.5));
    real fy = r_clamp(RC(2.0) - hw, (real)FG_FORM[k][1] + RC(0.3) * oby, hw - RC(2.0));
    c = S2D_CMD_GOTO; a1 = sg * fx; a2 = sg * fy; a3 = RC(60.0);
  }
  out[0] = (float)c; out[1] = (float)a1; out[2] = (float)a2; out[3] = (float)a3;
}

/* one cycle's commands of env i: `row` [np][4] holds the caller's; the scripted players' rows are replaced */
static void script_row(const OSim* s, int64_t i, uint32_t mask, float* row) {
  const OEnv* e = env_at(s, i);
  uint64_t gid = (uint64_t)(s->cfg.env_id_offset + i);
  int chaser_l, chaser_r;
  script_chasers(s, e, &chaser_l, &chaser_r);
  for (int j = 0; j < e->np; ++j)
    if ((mask >> j) & 1u) script_command(s, e, gid, j, j == (j < e->np / 2 ? chaser_l : chaser_r), row + 4 * j);
}

/* the commands the script gives the players of `mask` in every env now: rows [N][np][4] (the others left as they are) */
void s2dos_script_commands(void* h, uint32_t mask, float* rows) {
  OSim* s = (OSim*)h;
  int np = 2 * s->cfg.players_per_side;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < s->cfg.num_envs; ++i) script_row(s, i, mask, rows + (size_t)i * np * 4);
}

/* s2do_step with the players of `mask` played by the script (FULLGAME; mask 0: s2do_step itself).  Outputs as s2do_step:
 * reward summed over the K cycles (in cycle order), done = any, result and term_obs of the last episode that ended. */
void s2dos_step(void* h, uint32_t mask, const float* actions, int K, real* obs, real* reward, uint8_t* done, uint8_t* result,
                real* term_obs) {
  OSim* s = (OSim*)h;
  if (mask == 0 || s->cfg.scenario != S2D_SCENARIO_FULLGAME) {
    s2do_step(h, actions, K, obs, reward, done, result, term_obs);
    return;
  }
  int64_t n = s->cfg.num_envs;
  int np = 2 * s->cfg.players_per_side;
  float* rows = (float*)malloc(sizeof(float) * (size_t)n * np * 4);
  real* rw = (real*)malloc(sizeof(real) * (size_t)n);
  uint8_t* d = (uint8_t*)malloc((size_t)n);
  uint8_t* rs = (uint8_t*)malloc((size_t)n);
  for (int64_t i = 0; i < n; ++i) {
    if (reward) reward[i] = RC(0.0);
    if (done) done[i] = 0;
    if (result) result[i] = 0;
  }
  for (int k = 0; k < K; ++k) {
    for (int64_t i = 0; i < n; ++i)
      memcpy(rows + (size_t)i * np * 4, actions + ((size_t)(i * K + k) * np) * 4, sizeof(float) * np * 4);
    s2dos_script_commands(h, mask, rows);
    s2do_step(h, rows, 1, obs, rw, d, rs, term_obs);
    for (int64_t i = 0; i < n; ++i) {
      if (reward) reward[i] += rw[i];
      if (d[i]) {
        if (done) done[i] = 1;
        if (result) result[i] = rs[i];
      }
    }
  }
  free(rows); free(rw); free(d); free(rs);
}
