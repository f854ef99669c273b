// s2d_scenarios.cuh - the one-player scenarios (ReachBall, Shoot) fused into the lockstep step / reset kernels.
//
// Replaces, per env and per cycle, the whole of Soccer2DEnv.step (soccer_2d_env.py:226-269):
//   decode (in substep)  ReachBallEnv.action_to_rpc_actions      sample_environments/reach_ball_env.py:53-85
//   simulate_cycle       the rcssserver cycle behind the gRPC round trip (server.py:49-103)
//   check_episode        ReachBallEnv.check_trainer_observation  reach_ball_env.py:113-161
//   build_obs            ReachBallEnv.state_to_observation       reach_ball_env.py:87-111
//   place_new_episode    Soccer2DEnv.env_reset + ReachBallEnv.abs_reset / trainer_reset_actions /
//                        get_ball_velocity                       soccer_2d_env.py:179-224, reach_ball_env.py:163-218
#pragma once
#include <math.h>
#include <string.h>

#include <type_traits>

#include "s2d_one_player.cuh"

namespace s2d {

constexpr int kObsDim = 10;        // reach_ball_env.py:48
constexpr int kBallVelTries = 64;  // bound on the rejection loop of reach_ball_env.py:204-212

// Everything a kernel needs, passed by value as a __grid_constant__ (lives in the constant bank).
struct KernelParams {
  CycleConsts cc;
  int64_t num_envs;
  int64_t env_id_offset;
  uint64_t seed;
  int32_t scenario, action_mode, action_space_size, max_steps;
  int32_t auto_reset, change_ball_position, change_ball_velocity, noise;
  float min_distance_to_ball, ball_position_x, ball_position_y, ball_speed, ball_direction;
  float travel_factor;  // (1 - 0.96^max_steps) / (1 - 0.96), reach_ball_env.py:207
  float goto_dist_thr;
  int32_t dash_dirs_whole;  // Discrete(n): every dash of action_table has a whole-degree direction in [-180, 180] and
                            // is not a back dash, so body + direction of a whole-degree body is a memo index
                            // (in the alignment gap before `state`, like scripted_mask below)
  // device buffers (caller-owned, see S2DBuffers)
  void* state;
  const void* actions;
  float* obs;
  float* reward;
  uint8_t* done;
  uint8_t* result;
  float* terminal_obs;
  unsigned long long* stats;  // [kStatSlots][kStatWords]
  int32_t kick_actions;       // SHOOT Discrete(n): the last kick_actions actions are kicks
  uint32_t scripted_mask;     // FULLGAME: bit j = player j is played by the built-in script (s2d_set_scripted_players).
                              // (In the alignment gap before the next pointer: the struct keeps its size and every other
                              // field and kernel argument its offset in the constant bank.)
  const float* player_types;  // FULLGAME, heterogeneous players: [S2D_MAX_PLAYER_TYPES][PT_ROW] (device), else nullptr
  uint8_t type_of[32];        // player -> row of player_types (one assignment for every match of the handle)
  const uint8_t* type_of_match;  // or one assignment per match: [np][Nr] (device, match-minor like the state), else nullptr
  const float4* action_table; // [256] Discrete(n) -> {cmd, power, lowered direction, dash direction rate}, built on the host
  const float2* sincos_memo;  // [kSinCosMemoSize] {sin, cos} of the whole degrees in [-360, 360] (device; s2d_math.cuh)
};

// Fills everything but the buffer pointers from a config.  `table` receives, per Discrete(n) action, the command
// it stands for: Dash(100, dir) with the direction of reach_ball_env.py:84 (evaluated as the reference does: double,
// then the proto float) already lowered by dash_direction (clamp, dash_angle_step snap, direction rate - the part
// of Player::dash that does not depend on the episode); in SHOOT the last kick_actions entries are Kick(100, dir).
inline void make_kernel_params(const S2DConfig& cfg, KernelParams& kp, float4 table[256]) {
  memset(&kp, 0, sizeof(kp));
  kp.cc = make_cycle_consts(cfg.sp);
  kp.cc.collision_model = cfg.collision_model;
  kp.num_envs = cfg.num_envs;
  kp.env_id_offset = cfg.env_id_offset;
  kp.seed = cfg.seed;
  kp.scenario = cfg.scenario;
  kp.action_mode = cfg.action_mode;
  kp.action_space_size = cfg.action_space_size;
  kp.max_steps = cfg.max_steps;
  kp.auto_reset = cfg.auto_reset;
  kp.change_ball_position = cfg.change_ball_position;
  kp.change_ball_velocity = cfg.change_ball_velocity;
  kp.noise = cfg.noise;
  kp.min_distance_to_ball = cfg.min_distance_to_ball;
  kp.ball_position_x = cfg.ball_position_x;
  kp.ball_position_y = cfg.ball_position_y;
  kp.ball_speed = cfg.ball_speed;
  kp.ball_direction = cfg.ball_direction;
  kp.goto_dist_thr = cfg.goto_dist_thr;
  // reach_ball_env.py:207 - the reference uses 0.96 here, not the server's ball_decay
  kp.travel_factor = static_cast<float>((1.0 - pow(0.96, static_cast<double>(cfg.max_steps))) / (1.0 - 0.96));
  kp.kick_actions = cfg.scenario == S2D_SCENARIO_SHOOT ? cfg.kick_actions : 0;
  const int n_dash = cfg.action_space_size - kp.kick_actions;
  const RuntimeSP sp(kp.cc);
  auto direction = [](int a, int n) {
    return n > 0 ? static_cast<float>(fmod(static_cast<double>(a) * 360.0 / static_cast<double>(n), 360.0) - 180.0) : 0.0f;
  };
  // dash_apply turns Dash(100, .) into a back dash when max_dash_power < 0
  kp.dash_dirs_whole = fmaxf(sp.min_dash_power(), fminf(100.0f, sp.max_dash_power())) >= 0.0f;
  for (int a = 0; a < 256; ++a) {
    if (a < n_dash || kp.kick_actions == 0) {
      table[a].x = static_cast<float>(S2D_CMD_DASH);
      table[a].y = 100.0f;
      dash_direction(direction(a, n_dash), sp, table[a].z, table[a].w);
      kp.dash_dirs_whole = kp.dash_dirs_whole && rintf(table[a].z) == table[a].z && fabsf(table[a].z) <= 180.0f;
    } else {
      table[a] = make_float4(static_cast<float>(S2D_CMD_KICK), 100.0f, direction(a - n_dash, kp.kick_actions), 0.0f);
    }
  }
}

// episode statistics: slots spread the atomics over L2 lines; s2d_stats sums them
constexpr int kStatSlots = 256;
constexpr int kStatWords = 8;  // episodes, goals, outs, timeouts, episode_steps, return (double bits), pad, pad
enum { ST_EPISODES = 0, ST_GOALS = 1, ST_OUTS = 2, ST_TIMEOUTS = 3, ST_EP_STEPS = 4, ST_RETURN = 5 };

// what one launch accumulates per env.  `ended` packs three 10-bit counters (episodes that ended as Goal / Out /
// Timeout during the launch: K <= kMaxSubsteps) and, in the top two bits, the result of the last one.
constexpr int kMaxSubsteps = 1023;
struct LaunchOut {
  float reward_sum = 0.0f;
  uint32_t ended = 0;
  uint32_t ep_steps = 0;
  double ret = 0.0;
  __device__ __forceinline__ void count(int result) { ended = ((ended & 0x3fffffffu) + (1u << (10 * (result - 1)))) | (static_cast<uint32_t>(result) << 30); }
  // an episode that had already ended (auto_reset off: S2D_FLAG_DONE) and is stepped on: done / result are reported
  // again, the statistics are not
  __device__ __forceinline__ void report_only(int result) { ended = (ended & 0x3fffffffu) | (static_cast<uint32_t>(result) << 30); }
  // finished episodes to tally: at most one per launch can be a re-report, and then it is the only ending
  __device__ __forceinline__ bool any_ended() const { return ended != 0; }
  __device__ __forceinline__ uint32_t goals() const { return ended & 0x3ffu; }
  __device__ __forceinline__ uint32_t outs() const { return (ended >> 10) & 0x3ffu; }
  __device__ __forceinline__ uint32_t timeouts() const { return (ended >> 20) & 0x3ffu; }
  __device__ __forceinline__ uint32_t episodes() const { return goals() + outs() + timeouts(); }
  __device__ __forceinline__ uint32_t last_result() const { return ended >> 30; }
};

// reach_ball_env.py:113-161.  Rewards accumulate and later endings overwrite `result`, in the reference's
// order Goal -> Out -> Timeout; leaving the pitch ADDS 10 (`reward -= -10.0`, :144).
// body, mem_ang and atan2's result are already in [-180, 180], so AngleDeg's re-normalisations are identities.
// (dx, dy) = ball - player and d2 = dx*dx + dy*dy as left by simulate_cycle.
// Ball and player a few micrometres to a million metres apart (every state an episode reaches, collisions included:
// a resolved overlap leaves them collide_r apart) take the square root and atan2's division without the IEEE range
// guards (s2d_math.cuh, in_range_vector); anything else, such as coincident centres or a component below 2^-100 m,
// takes the IEEE operators out of line.
__device__ __noinline__ inline float2 cold_dist_angle(float dx, float dy, float d2) {
  return make_float2(sqrtf(d2), atan2_deg(dy, dx));
}
__device__ __forceinline__ bool check_episode(Episode& e, const KernelParams& P, float dx, float dy, float d2,
                                              float& reward, int& result) {
  float dist, th;
  if (in_range_vector(dx, dy, d2)) {
    dist = sqrt_in_range(d2);
    th = atan2_deg<true>(dy, dx);
  } else {
    const float2 c = cold_dist_angle(dx, dy, d2);
    dist = c.x;
    th = c.y;
  }
  const float diff = norm_deg_360(th - e.body);
  float rw = e.mem_dist - dist;
  rw += (fabsf(e.mem_ang) - fabsf(diff)) * static_cast<float>(1.0 / 180.0);
  const bool goal = dist < P.min_distance_to_ball;
  const bool out = fabsf(e.px) > 52.5f || fabsf(e.py) > 34.0f;
  const bool timeout = e.step_number > P.max_steps;
  rw = goal ? rw + 10.0f : rw;
  rw = out ? rw - -10.0f : rw;
  rw = timeout ? rw - 5.0f : rw;
  result = timeout ? S2D_RESULT_TIMEOUT : out ? S2D_RESULT_OUT : goal ? S2D_RESULT_GOAL : S2D_RESULT_NONE;
  reward = rw;
  e.mem_dist = dist;
  e.mem_ang = diff;
  return goal || out || timeout;
}

// reach_ball_env.py:87-111.  Must follow a check_episode on the same state: obs[0] is exactly the
// body-to-ball angle that check just stored in mem_ang, so the atan2 is not repeated.
__device__ __forceinline__ void build_obs(const Episode& e, float* o) {
  // A resting ball (the reference's default reset) or one rolling along an axis would send the warp through the slow
  // paths of the IEEE square root (sqrt(0)) and division (zero numerator): those cases are answered without them.
  const bool still = e.bvx == 0.0f && e.bvy == 0.0f;
  const bool axis = e.bvx == 0.0f || e.bvy == 0.0f;
  const float on_axis = e.bvy == 0.0f ? (e.bvx < 0.0f ? 180.0f : 0.0f) : (e.bvy > 0.0f ? 90.0f : -90.0f);
  const float h = hypot2(still ? 1.0f : e.bvx, e.bvy);
  const float t = atan2_deg(axis ? 1.0f : e.bvy, axis ? 2.0f : e.bvx);
  const float speed = still ? 0.0f : h;
  const float bdir = axis ? on_axis : t;
  o[0] = e.mem_ang * static_cast<float>(1.0 / 180.0);
  o[1] = e.body * static_cast<float>(1.0 / 180.0);
  o[2] = e.px * static_cast<float>(1.0 / 52.5);
  o[3] = e.py * static_cast<float>(1.0 / 34.0);
  o[4] = e.bx * static_cast<float>(1.0 / 52.5);
  o[5] = e.by * static_cast<float>(1.0 / 34.0);
  o[6] = speed * static_cast<float>(1.0 / 3.0);
  o[7] = bdir * static_cast<float>(1.0 / 360.0);
  o[8] = e.bvx * static_cast<float>(1.0 / 3.0);
  o[9] = e.bvy * static_cast<float>(1.0 / 3.0);
}

// ---- SHOOT (spec: include/soccer2d.h) ---------------------------------------------------------------
// (pbx, pby) = ball position before this cycle's move.  The reward memory holds the player-ball distance
// (mem_dist) and the ball-goal distance (mem_ang slot).
template <class SP>
__device__ __forceinline__ bool check_shoot(Episode& e, const KernelParams& P, const SP& sp, float d2, float pbx,
                                            float pby, float& reward, int& result) {
  const float d_pb = sqrtf(d2);
  const float d_bg = hypot2(sp.pitch_half_length() - e.bx, 0.0f - e.by);
  float rw = (e.mem_dist - d_pb) * 0.2f + (e.mem_ang - d_bg);
  const float line = sp.pitch_half_length() + sp.ball_size();
  const float post = sp.goal_width() * 0.5f + sp.goal_post_radius();
  bool goal = false;
  if (e.bx > line && !(pbx > line)) {
    const float yc = pby + (e.by - pby) * ((line - pbx) / (e.bx - pbx));
    goal = fabsf(yc) <= post;
  }
  const bool out = !goal && (fabsf(e.bx) > line || fabsf(e.by) > sp.pitch_half_width() + sp.ball_size());
  const bool timeout = !goal && !out && e.step_number > P.max_steps;
  rw = goal ? rw + 10.0f : rw;
  rw = out ? rw - 10.0f : rw;
  rw = timeout ? rw - 5.0f : rw;
  result = goal ? S2D_RESULT_GOAL : out ? S2D_RESULT_OUT : timeout ? S2D_RESULT_TIMEOUT : S2D_RESULT_NONE;
  reward = rw;
  e.mem_dist = d_pb;
  e.mem_ang = d_bg;
  return goal || out || timeout;
}

// same 10 values as ReachBall; the body-to-ball angle is computed here (the memory slot holds a distance)
__device__ __forceinline__ void build_obs_shoot(const Episode& e, float* o) {
  Episode t = e;
  t.mem_ang = norm_deg_360(atan2_deg(e.by - e.py, e.bx - e.px) - e.body);
  build_obs(t, o);
}

template <int SCN>
__device__ __forceinline__ void scenario_obs(const Episode& e, float* o) {
  if (SCN == S2D_SCENARIO_SHOOT) build_obs_shoot(e, o);
  else build_obs(e, o);
}

template <int SCN, class SP>
__device__ __forceinline__ bool scenario_check(Episode& e, const KernelParams& P, const SP& sp, float dx, float dy,
                                               float d2, float pbx, float pby, float& reward, int& result) {
  if (SCN == S2D_SCENARIO_SHOOT) return check_shoot(e, P, sp, d2, pbx, pby, reward, result);
  return check_episode(e, P, dx, dy, d2, reward, result);
}

// trainer_reset_actions' draws (integers: x in [-50,50], y in [-30,30], body in [0,360]; ball velocity by
// bounded rejection: the ball must stay on the pitch for max_steps cycles): what DoMoveBall / DoMovePlayer carry.
struct Placement {
  float px, py, body, bx, by, bvx, bvy;
};

__device__ __forceinline__ bool ball_stays_inside(const KernelParams& P, float bx, float by, float s_try, float sn, float cs) {
  const float travel = s_try * P.travel_factor;
  return fabsf(bx + travel * cs) <= 52.5f && fabsf(by + travel * sn) <= 34.0f;
}

// one thread draws everything (reset kernel; many lanes of a warp resetting at once)
__device__ __forceinline__ Placement draw_placement(const KernelParams& P, uint64_t gid, uint32_t episode, int first_try = 0,
                                                    float bx_known = 0.0f, float by_known = 0.0f) {
  Placement pl;
  if (first_try == 0) {
    const uint4 w = philox4x32_10(P.seed, gid, episode, RNG_RESET, 0);
    pl.px = static_cast<float>(u32_to_int(w.x, -50, 50));
    pl.py = static_cast<float>(u32_to_int(w.y, -30, 30));
    pl.body = static_cast<float>(u32_to_int(w.z, 0, 360));
    pl.bx = P.ball_position_x;
    pl.by = P.ball_position_y;
    if (P.change_ball_position) {
      const uint4 w2 = philox4x32_10(P.seed, gid, episode, RNG_RESET, 1);
      pl.bx = static_cast<float>(u32_to_int(w.w, -50, 50));
      pl.by = static_cast<float>(u32_to_int(w2.x, -30, 30));
    }
  } else {  // continuing a search the warp started (tries first_try .. kBallVelTries-1): only the velocity is used
    pl.px = pl.py = pl.body = 0.0f;
    pl.bx = bx_known;
    pl.by = by_known;
  }
  float speed = P.ball_speed, d = P.ball_direction;
  if (P.change_ball_velocity) {
    speed = 0.0f;
    d = 0.0f;
    uint4 wv = make_uint4(0, 0, 0, 0);
#pragma unroll 1
    for (int t = first_try; t < kBallVelTries; ++t) {
      if ((t & 1) == 0 || t == first_try)
        wv = philox4x32_10(P.seed, gid, episode, RNG_BALLVEL, static_cast<uint32_t>(t >> 1));
      const float s_try = u32_to_unit((t & 1) ? wv.z : wv.x) * 3.0f;
      const float d_try = static_cast<float>(u32_to_int((t & 1) ? wv.w : wv.y, 0, 360));
      float sn, cs;
      sincos_deg(d_try, sn, cs);
      if (ball_stays_inside(P, pl.bx, pl.by, s_try, sn, cs)) {
        speed = s_try;
        d = d_try;
        break;
      }
    }
  }
  float sn, cs;
  sincos_deg(d, sn, cs);
  pl.bvx = speed * cs;
  pl.bvy = speed * sn;
  return pl;
}

#ifndef S2D_HOST_EMU
// The same draws for ONE episode, made by the whole warp (a lane whose episode ended while its 31 neighbours wait):
// lanes 0-1 compute the two placement blocks, lanes 2-31 thirty ball-velocity blocks (tries 0..59), every lane
// evaluates one try per round, and a ballot picks the first accepted one - exactly the try the sequential loop of
// draw_placement stops at.  Returns the placement in every lane.
template <bool MEMO = true>
__device__ __forceinline__ Placement draw_placement_warp(const KernelParams& P, uint64_t gid, uint32_t episode, int lane) {
  const unsigned full = 0xffffffffu;
  const bool placement_lane = lane < 2;
  const uint4 w = philox4x32_10(P.seed, gid, episode, placement_lane ? RNG_RESET : RNG_BALLVEL,
                                static_cast<uint32_t>(placement_lane ? lane : lane - 2));
  Placement pl;
  pl.px = static_cast<float>(u32_to_int(__shfl_sync(full, w.x, 0), -50, 50));
  pl.py = static_cast<float>(u32_to_int(__shfl_sync(full, w.y, 0), -30, 30));
  pl.body = static_cast<float>(u32_to_int(__shfl_sync(full, w.z, 0), 0, 360));
  const uint32_t ubx = __shfl_sync(full, w.w, 0), uby = __shfl_sync(full, w.x, 1);
  pl.bx = P.change_ball_position ? static_cast<float>(u32_to_int(ubx, -50, 50)) : P.ball_position_x;
  pl.by = P.change_ball_position ? static_cast<float>(u32_to_int(uby, -30, 30)) : P.ball_position_y;
  float speed = P.ball_speed, sn, cs;
  if (P.change_ball_velocity) {
    speed = 0.0f;
    bool found = false;
#pragma unroll 1
    for (int round = 0; round < 2 && !found; ++round) {
      const int t = 32 * round + lane, block = t >> 1;
      const bool have = block < 30;
      const int src = have ? 2 + block : 2;
      const uint32_t qx = __shfl_sync(full, w.x, src), qy = __shfl_sync(full, w.y, src), qz = __shfl_sync(full, w.z, src),
                     qw = __shfl_sync(full, w.w, src);
      const float s_try = u32_to_unit((t & 1) ? qz : qx) * 3.0f;
      const float d_try = static_cast<float>(u32_to_int((t & 1) ? qw : qy, 0, 360));
      float tsn, tcs;
      if (MEMO && P.sincos_memo) sincos_deg_memo(d_try, P.sincos_memo, tsn, tcs);  // whole degrees in [0, 360]: always a hit
      else sincos_deg(d_try, tsn, tcs);
      const unsigned ok = __ballot_sync(full, have && ball_stays_inside(P, pl.bx, pl.by, s_try, tsn, tcs));
      if (ok) {
        const int first = __ffs(ok) - 1;
        speed = __shfl_sync(full, s_try, first);
        sn = __shfl_sync(full, tsn, first);
        cs = __shfl_sync(full, tcs, first);
        found = true;
      }
    }
    if (!found) {  // tries 60..63: practically never; every lane walks them alone (same result in all lanes)
      const Placement rest = draw_placement(P, gid, episode, 60, pl.bx, pl.by);
      pl.bvx = rest.bvx;
      pl.bvy = rest.bvy;
      return pl;
    }
  } else {
    sincos_deg(P.ball_direction, sn, cs);
  }
  pl.bvx = speed * cs;
  pl.bvy = speed * sn;
  return pl;
}
#endif

// DoMoveBall / DoMovePlayer (vel = 0) / DoRecover.  The caller still owes the episode ONE idle server cycle and the
// priming check (the reference's reset observes the state one cycle after placement, reach_ball_env.py:163-168).
template <class SP>
__device__ __forceinline__ void apply_placement(Episode& e, const Placement& pl, const SP& sp) {
  e.episode += 1u;
  e.step_number = 0;
  e.ep_return = 0.0f;
  e.bx = pl.bx; e.by = pl.by; e.bvx = pl.bvx; e.bvy = pl.bvy;
  e.px = pl.px; e.py = pl.py; e.vx = 0.0f; e.vy = 0.0f;
  e.body = norm_deg(pl.body);
  e.flags = 0u;
  recover(e, sp);
}

template <class SP>
__device__ __forceinline__ void place_new_episode(Episode& e, const KernelParams& P, const SP& sp, uint64_t gid) {
  apply_placement(e, draw_placement(P, gid, e.episode), sp);
}

// per-lane row store (terminal observations, reset kernel): 40-byte rows are 8-byte aligned
__device__ __forceinline__ void lane_store_row(float* __restrict__ dst, int64_t env, const float* row) {
  float2* o = reinterpret_cast<float2*>(dst + env * kObsDim);
#pragma unroll
  for (int j = 0; j < kObsDim / 2; ++j) o[j] = make_float2(row[2 * j], row[2 * j + 1]);
}

// the second half of Soccer2DEnv.reset: the idle cycle after the placement and the priming check
template <int SCN, class SP>
__device__ __forceinline__ void finish_reset(Episode& e, const KernelParams& P, const SP& sp, uint64_t gid) {
  float dx, dy, d2, rw;
  int rs;
  const float pbx = e.bx, pby = e.by;
  simulate_cycle<false, false>(e, S2D_CMD_NONE, 0.0f, 0.0f, 0.0f, sp, dx, dy, d2, P.seed, gid);
  scenario_check<SCN>(e, P, sp, dx, dy, d2, pbx, pby, rw, rs);  // reach_ball_env.py:166: primes the memory, reward discarded
}

// Soccer2DEnv.reset for one env: placement, the idle cycle, the priming check.
template <int SCN, class SP>
__device__ __forceinline__ void reset_episode(Episode& e, const KernelParams& P, const SP& sp, uint64_t gid) {
  place_new_episode(e, P, sp, gid);
  finish_reset<SCN>(e, P, sp, gid);
}

// ONE env-step = what Soccer2DEnv.step does: decode the action, run the server cycle, score it; when the
// episode ends, record it and (auto_reset) start the next one (placement, idle cycle, priming check).
//   discrete:   (a0..a3) = the action's table entry {cmd, power, lowered direction, dash rate}
//   continuous: a0 in [-1, 1]                                                    (ReachBall)
//   turning:    [turn_prob, turn_angle, dash_prob, dash_angle], :65-68           (ReachBall)
//   command:    {cmd, a, b, c} = proto PlayerAction dash / turn / kick / body_go_to_point
// DEFER_END: leave the end of the episode (tally, terminal observation, auto-reset) to the caller and return the
// episode's result, S2D_RESULT_NONE while it goes on (step_kernel: the warp handles endings together, end_of_episode).
template <int SCN, int ACT, class SP, bool DEFER_END = false>
__device__ __forceinline__ int substep(Episode& e, const KernelParams& P, const SP& sp, uint64_t gid, int64_t i, float a0,
                                        float a1, float a2, float a3, LaunchOut& out,
                                        const float2* sincos_memo = nullptr, bool memo_direct = false) {
  constexpr bool kTurns = ACT == S2D_ACT_TURNING || ACT == S2D_ACT_COMMAND;
  constexpr bool kKicks = ACT == S2D_ACT_COMMAND || SCN == S2D_SCENARIO_SHOOT;
  e.step_number += 1;  // reach_ball_env.py:55
  int cmd = S2D_CMD_DASH;
  float power = 100.0f, dir, rate;
  if (ACT == S2D_ACT_DISCRETE) {
    if (SCN == S2D_SCENARIO_SHOOT) {
      cmd = static_cast<int>(a0);
      power = a1;
    }
    dir = a2;
    rate = a3;
  } else if (ACT == S2D_ACT_CONTINUOUS) {
    dash_direction(a0 * 180.0f, sp, dir, rate);
  } else if (ACT == S2D_ACT_TURNING) {
    const float tp = clampf(-1.0f, a0, 1.0f), ta = clampf(-1.0f, a1, 1.0f);
    const float dp = clampf(-1.0f, a2, 1.0f), da = clampf(-1.0f, a3, 1.0f);
    const float u = u32_to_unit(philox4x32_10(P.seed, gid, e.cycle, RNG_ACTION, 0).x);
    const bool turn_selected = u < softmax_first(dp, tp);  // :69-72: tested against the DASH logit's weight
    cmd = turn_selected ? S2D_CMD_TURN : S2D_CMD_DASH;
    power = turn_selected ? 0.0f : 100.0f;
    dash_direction(da * 180.0f, sp, dir, rate);
    dir = turn_selected ? ta * 180.0f : dir;
  } else {
    decode_command(e, make_float4(a0, a1, a2, a3), P.goto_dist_thr, sp, cmd, power, dir, rate);
  }
  float dx, dy, d2, rw;
  int rs;
  const float pbx = e.bx, pby = e.by;
  simulate_cycle<kTurns, kKicks>(e, cmd, power, dir, rate, sp, dx, dy, d2, P.seed, gid, sincos_memo, memo_direct);
  const bool done = scenario_check<SCN>(e, P, sp, dx, dy, d2, pbx, pby, rw, rs);
  out.reward_sum += rw;
  e.ep_return += rw;
  if (DEFER_END) return rs;
  if (done) {
    if (e.flags & S2D_FLAG_DONE) {
      out.report_only(rs);
    } else {
      out.count(rs);
      out.ep_steps += static_cast<uint32_t>(e.step_number);
      out.ret += static_cast<double>(e.ep_return);
    }
    if (P.terminal_obs) {
      float row[kObsDim];
      scenario_obs<SCN>(e, row);
      lane_store_row(P.terminal_obs, i, row);
    }
    if (P.auto_reset) {
      reset_episode<SCN>(e, P, sp, gid);
    } else {
      e.flags |= S2D_FLAG_DONE;
    }
  }
  return S2D_RESULT_NONE;
}

#ifndef S2D_HOST_EMU
// Coalesced write of one warp's observations: each lane parks its row in shared memory, then the warp
// streams the 32 x 10 floats out as 80 float4 (512 contiguous bytes per store instruction).
__device__ __forceinline__ void warp_store_obs(float* __restrict__ dst, int64_t warp_first_env, int64_t n,
                                               const float* row, bool lane_valid, float* stage /* [320] */) {
  const int lane = threadIdx.x & 31;
  if (lane_valid) {
#pragma unroll
    for (int j = 0; j < kObsDim; ++j) stage[lane * kObsDim + j] = row[j];
  }
  __syncwarp();
  const int64_t rows = (n - warp_first_env) < 32 ? (n - warp_first_env) : 32;
  const int nvec = static_cast<int>(rows) * kObsDim / 4;  // full float4s
  float4* out4 = reinterpret_cast<float4*>(dst + warp_first_env * kObsDim);  // 32*10*4 B = 1280 B: 16-B aligned
  const float4* st4 = reinterpret_cast<const float4*>(stage);
  for (int v = lane; v < nvec; v += 32) st_stream(out4 + v, st4[v]);
  const int tail = static_cast<int>(rows) * kObsDim - nvec * 4;  // only in the last, ragged warp
  if (lane < tail) dst[warp_first_env * kObsDim + nvec * 4 + lane] = stage[nvec * 4 + lane];
  __syncwarp();
}

// warp-level sum of the launch's episode statistics, then one lane adds them to a stats slot
__device__ __forceinline__ void flush_tally(const LaunchOut& t, unsigned long long* stats) {
  const unsigned full = 0xffffffffu;
  if (!__any_sync(full, (t.ended & 0x3fffffffu) != 0)) return;
  const uint32_t g = __reduce_add_sync(full, t.goals()), o = __reduce_add_sync(full, t.outs()),
                 to = __reduce_add_sync(full, t.timeouts()), st = __reduce_add_sync(full, t.ep_steps);
  double r = t.ret;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) r += __shfl_xor_sync(full, r, s);
  if ((threadIdx.x & 31) == 0) {
    const unsigned warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    unsigned long long* slot = stats + static_cast<size_t>(warp_global % kStatSlots) * kStatWords;
    atomicAdd(slot + ST_EPISODES, static_cast<unsigned long long>(g + o + to));
    if (g) atomicAdd(slot + ST_GOALS, static_cast<unsigned long long>(g));
    if (o) atomicAdd(slot + ST_OUTS, static_cast<unsigned long long>(o));
    if (to) atomicAdd(slot + ST_TIMEOUTS, static_cast<unsigned long long>(to));
    atomicAdd(slot + ST_EP_STEPS, static_cast<unsigned long long>(st));
    atomicAdd(reinterpret_cast<double*>(slot + ST_RETURN), r);
  }
}

// ---- kernels --------------------------------------------------------------------------------------

#ifndef S2D_BLOCK
#define S2D_BLOCK 128
#endif
constexpr int kBlock = S2D_BLOCK;
#ifndef S2D_MIN_BLOCKS
#define S2D_MIN_BLOCKS 8  // resident blocks per SM the step kernel is compiled for (register budget)
#endif

// K lockstep cycles of every env in one launch; state stays in registers in between.
// actions[N][K] (uint8 / float) or [N][K][4] (float): a lane's K actions are contiguous in memory; the first
// access pulls the lane's sector(s) into L1 and the following cycles hit there (ld.global.nc).
// SCN: scenario; ACT: action encoding; VAR: how the constants come in (kVarRuntime: constant bank, kVarDefault: the
// default ServerParam folded at compile time, kVarNoisy: constant bank + rcssserver noise).
// kVarHetero / kVarHeteroNoisy (FULLGAME): per-player PlayerType values from the handle's type table.
constexpr int kVarRuntime = 0, kVarDefault = 1, kVarNoisy = 2, kVarHetero = 3, kVarHeteroNoisy = 4;
template <int VAR>
struct VariantSP {
  using type = typename std::conditional<
      VAR == kVarDefault, DefaultSP,
      typename std::conditional<
          VAR == kVarNoisy, NoisySP,
          typename std::conditional<VAR == kVarHetero, HeteroSP<false>,
                                    typename std::conditional<VAR == kVarHeteroNoisy, HeteroSP<true>, RuntimeSP>::type>::type>::type>::type;
};

// The end of an episode inside the K loop, handled by the warp as a whole: one vote per step replaces a divergent
// branch.  Episodes end in few lanes at a time (about one step in 60 per lane), and a lane that drew its next placement
// alone would hold its 31 neighbours for ~560 instructions; so with up to kWarpDrawMax lanes due the warp makes each
// lane's draws together (draw_placement_warp), with more (synchronised time-outs) every due lane draws for itself in
// parallel.  Both orders consume the same Philox words: the results are identical.
#ifndef S2D_SINCOS_MEMO_MIN_K
#define S2D_SINCOS_MEMO_MIN_K 4  // launches of fewer cycles are bound by HBM: they leave the L1 to the streams
#endif
constexpr int kSinCosMemoMinK = S2D_SINCOS_MEMO_MIN_K;
#ifndef S2D_WARP_DRAW_MAX
#define S2D_WARP_DRAW_MAX 3
#endif
constexpr int kWarpDrawMax = S2D_WARP_DRAW_MAX;

// ONE_PIECE / MEMO: the step kernels' refinements (one lane due: placement and idle cycle in one piece; the draws'
// sin / cos from the whole-degree memo); the fused-policy kernels, at their register limit, are faster without them.
template <int SCN, class SP, bool ONE_PIECE = true, bool MEMO = true>
__device__ __forceinline__ void end_of_episode(Episode& e, const KernelParams& P, const SP& sp, uint64_t gid, int64_t i,
                                               bool valid, int rs, LaunchOut& out) {
  const unsigned full = 0xffffffffu;
  const bool done = rs != S2D_RESULT_NONE;
  unsigned pending = __ballot_sync(full, done);
  if (pending == 0u) return;
  if (done) {
    if (e.flags & S2D_FLAG_DONE) {
      out.report_only(rs);
    } else {
      out.count(rs);
      out.ep_steps += static_cast<uint32_t>(e.step_number);
      out.ret += static_cast<double>(e.ep_return);
    }
    if (P.terminal_obs && valid) {
      float row[kObsDim];
      scenario_obs<SCN>(e, row);
      lane_store_row(P.terminal_obs, i, row);
    }
    if (!P.auto_reset) e.flags |= S2D_FLAG_DONE;
  }
  if (!P.auto_reset) return;
  if (ONE_PIECE && (pending & (pending - 1u)) == 0u) {
    // the usual case, ONE lane due: it places its new episode and runs the idle cycle in one piece, so that the
    // compiler sees a player at rest with full stamina there (most of that cycle folds away)
    const int lane = threadIdx.x & 31, src = __ffs(pending) - 1;
    const uint32_t g_lo = __shfl_sync(full, static_cast<uint32_t>(gid), src);
    const uint32_t g_hi = __shfl_sync(full, static_cast<uint32_t>(gid >> 32), src);
    const uint32_t episode = __shfl_sync(full, e.episode, src);
    const Placement pl = draw_placement_warp<MEMO>(P, (static_cast<uint64_t>(g_hi) << 32) | g_lo, episode, lane);
    if (done) {
      apply_placement(e, pl, sp);
      finish_reset<SCN>(e, P, sp, gid);
    }
  } else if (__popc(pending) <= kWarpDrawMax) {
    const int lane = threadIdx.x & 31;
    do {
      const int src = __ffs(pending) - 1;
      pending &= pending - 1u;
      const uint32_t g_lo = __shfl_sync(full, static_cast<uint32_t>(gid), src);
      const uint32_t g_hi = __shfl_sync(full, static_cast<uint32_t>(gid >> 32), src);
      const uint32_t episode = __shfl_sync(full, e.episode, src);
      const Placement pl = draw_placement_warp<MEMO>(P, (static_cast<uint64_t>(g_hi) << 32) | g_lo, episode, lane);
      if (lane == src) apply_placement(e, pl, sp);
    } while (pending);
    if (done) finish_reset<SCN>(e, P, sp, gid);
  } else if (done) {
    reset_episode<SCN>(e, P, sp, gid);
  }
}

template <int SCN, int ACT, int VAR>
__global__ void __launch_bounds__(kBlock, S2D_MIN_BLOCKS) step_kernel(const __grid_constant__ KernelParams P, const int K) {
  using SP = typename VariantSP<VAR>::type;
  const SP sp(P.cc);
  __shared__ __align__(16) float s_stage[kBlock / 32][32 * kObsDim];
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  const int64_t n = P.num_envs;
  const bool valid = i < n;
  const uint64_t gid = static_cast<uint64_t>(P.env_id_offset + i);
  float* stage = s_stage[threadIdx.x >> 5];
  const int64_t warp_first = i - (threadIdx.x & 31);

  Episode e;
  LaunchOut out;
  float obs_row[kObsDim];

  // Every lane of the warp runs the K loop (the lanes past the end of a ragged last warp replay env n-1 and store
  // nothing), so that the warp can handle the end of an episode together, see end_of_episode.
  const int64_t il = valid ? i : n - 1;
  load_episode(P.state, n, il, e);
  if (ACT == S2D_ACT_DISCRETE) {
    // ReachBall: bodies are whole degrees (placement) and never turn, dash directions are snapped to whole degrees:
    // the dash's sin / cos come from the memo (s2d_math.cuh; 5.8 KB, it stays in L1 next to the action table) when
    // the launch is long enough for that to matter.
    const float2* memo = (SCN != S2D_SCENARIO_SHOOT && K >= kSinCosMemoMinK) ? P.sincos_memo : nullptr;
    // When the table's directions and every body of the warp are whole degrees in [-180, 180], body + direction is the
    // memo index itself, for the whole launch: a new episode's body is a whole degree too (draw_placement).  A body
    // imported off that grid keeps its warp on sincos_deg_memo's per-cycle test until the next launch.
    // The K loop is compiled twice, so that the choice costs nothing per cycle.
    const bool memo_direct = memo && P.dash_dirs_whole &&
                             __all_sync(0xffffffffu, rintf(e.body) == e.body && fabsf(e.body) <= 180.0f);
    auto k_loop = [&](auto direct) {
      // the 4 KB action table stays in L1 (read-only path); `act` walks the lane's K action bytes
      const uint8_t* act = static_cast<const uint8_t*>(P.actions) + il * K;
#pragma unroll 1
      for (int k = K; k > 0; --k, ++act) {
        int rs;
        if (SCN == S2D_SCENARIO_SHOOT) {
          const float4 t = __ldg(P.action_table + __ldg(act));
          rs = substep<SCN, ACT, SP, true>(e, P, sp, gid, i, t.x, t.y, t.z, t.w, out);
        } else {  // ReachBall: always Dash(100, .): only the lowered direction and its rate are needed
          const float2 t = __ldg(reinterpret_cast<const float2*>(P.action_table + __ldg(act)) + 1);
          rs = substep<SCN, ACT, SP, true>(e, P, sp, gid, i, 0.f, 0.f, t.x, t.y, out, memo, decltype(direct)::value);
        }
        end_of_episode<SCN>(e, P, sp, gid, i, valid, rs, out);
      }
    };
    if (SCN != S2D_SCENARIO_SHOOT && memo_direct) k_loop(std::true_type());
    else k_loop(std::false_type());
  } else if (ACT == S2D_ACT_CONTINUOUS) {
    // Box(1): the direction a * 180 is snapped to dash_angle_step = 1 as well and nobody turns - whole degrees again
    const float2* memo = K >= kSinCosMemoMinK ? P.sincos_memo : nullptr;
    const float* act = static_cast<const float*>(P.actions) + il * K;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
      const int rs = substep<SCN, ACT, SP, true>(e, P, sp, gid, i, __ldg(act + k), 0.f, 0.f, 0.f, out, memo);
      end_of_episode<SCN>(e, P, sp, gid, i, valid, rs, out);
    }
  } else {
    const float4* act = static_cast<const float4*>(P.actions) + il * K;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
      const float4 a = __ldg(act + k);
      const int rs = substep<SCN, ACT, SP, true>(e, P, sp, gid, i, a.x, a.y, a.z, a.w, out);
      end_of_episode<SCN>(e, P, sp, gid, i, valid, rs, out);
    }
  }
  if (valid) {
    store_episode(P.state, n, i, e);
    scenario_obs<SCN>(e, obs_row);
    P.reward[i] = out.reward_sum;
    P.done[i] = static_cast<uint8_t>(out.ended != 0);
    P.result[i] = static_cast<uint8_t>(out.last_result());
  } else {
    out = LaunchOut();  // a replayed lane tallies nothing
  }
  warp_store_obs(P.obs, warp_first, n, obs_row, valid, stage);
  flush_tally(out, P.stats);
}

// Soccer2DEnv.reset for every env (mask == nullptr) or the envs with a non-zero mask byte.
template <int SCN, bool NOISY>
__global__ void __launch_bounds__(kBlock) reset_kernel(const __grid_constant__ KernelParams P,
                                                       const uint8_t* __restrict__ mask) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  if (i >= P.num_envs) return;
  if (mask && !mask[i]) return;
  const typename std::conditional<NOISY, NoisySP, RuntimeSP>::type sp(P.cc);
  Episode e;
  load_episode(P.state, P.num_envs, i, e);
  reset_episode<SCN>(e, P, sp, static_cast<uint64_t>(P.env_id_offset + i));
  store_episode(P.state, P.num_envs, i, e);
  float row[kObsDim];
  scenario_obs<SCN>(e, row);
  lane_store_row(P.obs, i, row);
  P.reward[i] = 0.0f;
  P.done[i] = 0;
  P.result[i] = 0;
}
#endif  // !S2D_HOST_EMU

}  // namespace s2d
