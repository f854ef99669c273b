// s2d_one_player.cuh - per-episode state and the rcssserver-style cycle for the one-player scenarios
// (ReachBall: sample_environments/reach_ball_env.py; Shoot: 1v0 with the kick model).
//
// One thread owns one episode; everything below lives in registers between the state load and the state
// store of a launch.  The arithmetic follows the fp32 SPEC of s2d_math.cuh (no implicit fma).  Every function
// takes the constants through an accessor type SP (RuntimeSP or DefaultSP, s2d_params.h).
//
// What each function stands in for (the reference only *launches* these; soccer_2d_env.py:356-398):
//   dash / turn / kick        rcssserver Player::dash, Player::turn, Player::kick
//   move_object               rcssserver MPObject::_inc (accel clamp, speed clamp, move, decay)
//   collide_ball_player       rcssserver Stadium::collisions specialised to one player and the ball
//   update_stamina            rcssserver Player::updateStamina
//   recover                   trainer (recover) = proto DoRecover (idl/service.proto:1407)
#pragma once
#include "s2d_math.cuh"
#include "s2d_params.h"

namespace s2d {

// HBM layout: five 16-byte planes, plane-major (plane p of env i at state + (p * N + i) * 16), so that a
// warp reads / writes 512 contiguous bytes per plane with one 128-bit access per lane.
//   plane 0  float4 {player x, y, vx, vy}
//   plane 1  float4 {body_direction (deg), stamina, effort, recovery}
//   plane 2  float4 {ball x, y, vx, vy}
//   plane 3  float4 {distance_to_ball memory, body_ball_angle_diff memory, stamina_capacity, episode return}
//   plane 4  uint4  {step_number, cycle, episode, flags | play_mode << 8 | scores << 16}
constexpr int kStatePlanes = 5;
constexpr int kStateBytesPerEnv = kStatePlanes * 16;

struct Episode {
  float px, py, vx, vy;
  float body, stamina, effort, recovery;
  float bx, by, bvx, bvy;
  float mem_dist, mem_ang, capacity, ep_return;
  int step_number;
  uint32_t cycle, episode, flags;
};

__device__ __forceinline__ void load_episode(const void* state, int64_t n, int64_t i, Episode& e) {
  const float4* f = reinterpret_cast<const float4*>(state);
  const float4 a = ld_stream(f + i), b = ld_stream(f + n + i), c = ld_stream(f + 2 * n + i),
               d = ld_stream(f + 3 * n + i);
  const uint4 u = ld_stream(reinterpret_cast<const uint4*>(state) + 4 * n + i);
  e.px = a.x; e.py = a.y; e.vx = a.z; e.vy = a.w;
  e.body = b.x; e.stamina = b.y; e.effort = b.z; e.recovery = b.w;
  e.bx = c.x; e.by = c.y; e.bvx = c.z; e.bvy = c.w;
  e.mem_dist = d.x; e.mem_ang = d.y; e.capacity = d.z; e.ep_return = d.w;
  e.step_number = static_cast<int>(u.x); e.cycle = u.y; e.episode = u.z; e.flags = u.w;
}

__device__ __forceinline__ void store_episode(void* state, int64_t n, int64_t i, const Episode& e) {
  float4* f = reinterpret_cast<float4*>(state);
  st_stream(f + i, make_float4(e.px, e.py, e.vx, e.vy));
  st_stream(f + n + i, make_float4(e.body, e.stamina, e.effort, e.recovery));
  st_stream(f + 2 * n + i, make_float4(e.bx, e.by, e.bvx, e.bvy));
  st_stream(f + 3 * n + i, make_float4(e.mem_dist, e.mem_ang, e.capacity, e.ep_return));
  st_stream(reinterpret_cast<uint4*>(state) + 4 * n + i,
            make_uint4(static_cast<uint32_t>(e.step_number), e.cycle, e.episode, e.flags));
}

// ---- noise ------------------------------------------------------------------------------------------
// rcssserver's player_rand / ball_rand / kick_rand, drawn from the counter-based RNG: one Philox block per
// (env, server cycle, agent) - agent = player index, kBallAgent = the ball - and a second block (32 + agent) for a
// kicker's kick-noise direction.  Streams do not depend on sharding or on K; with noise off (SP::kNoise == false,
// the comparison mode of the north star) none of this is compiled in.
struct NoiseCtx {
  uint64_t seed, gid;
  uint32_t cycle;
};
constexpr uint32_t kBallAgent = 31;
__device__ __forceinline__ float u11(uint32_t w) { return u32_to_unit(w) * 2.0f - 1.0f; }  // uniform in [-1, 1)
__device__ __forceinline__ uint4 noise_block(const NoiseCtx& nz, uint32_t sub) {
  return philox4x32_10(nz.seed, nz.gid, nz.cycle, RNG_NOISE, sub);
}

// ---- commands -------------------------------------------------------------------------------------

template <class SP>
__device__ __forceinline__ void recover(Episode& e, const SP& sp) {
  e.stamina = sp.stamina_max();
  e.recovery = sp.recover_init();
  e.effort = sp.effort_max();
  e.capacity = sp.stamina_capacity();
}

// The direction half of (dash power dir): clamp, snap to dash_angle_step, and the direction-dependent rate
// (forward 1, sideways side_dash_rate, backwards back_dash_rate).  It depends on the command only, not on
// the episode, so Discrete(n) actions get it from a table built with this very function on the host.
template <class SP>
S2D_HD void dash_direction(float dir, const SP& sp, float& snapped, float& rate) {
  dir = fmaxf(sp.min_dash_angle(), fminf(dir, sp.max_dash_angle()));
  if (sp.dash_angle_step() > 1.0e-10f) dir = sp.dash_angle_step() * rintf(dir * sp.inv_dash_angle_step());
  const float ad = fabsf(dir);
  const float over = (ad - 90.0f) * static_cast<float>(1.0 / 90.0);
  const float under = ad * static_cast<float>(1.0 / 90.0);
  const float rate_back = sp.back_dash_rate() - ((sp.back_dash_rate() - sp.side_dash_rate()) * (1.0f - over));
  const float rate_fwd = sp.side_dash_rate() + ((1.0f - sp.side_dash_rate()) * (1.0f - under));
  rate = fmaxf(0.0f, fminf(ad > 90.0f ? rate_back : rate_fwd, 1.0f));
  snapped = dir;
}

// The episode half: stamina is charged first, then the effective power is scaled by effort, the rate and
// dash_power_rate.  Gives the player's acceleration (it is the only contribution in a cycle).
template <class SP>
__device__ __forceinline__ void dash_apply(Episode& e, float power, float dir, float rate, const SP& sp, float& ax,
                                           float& ay, bool left_team = true, const float2* sincos_memo = nullptr) {
  power = clampf(sp.min_dash_power(), power, sp.max_dash_power());
  const bool back = power < 0.0f;
  float need = back ? power * -2.0f : power;
  need = fmin_(need, e.stamina + sp.extra_stamina());
  e.stamina = fmax_(0.0f, e.stamina - need);
  power = back ? need * -0.5f : need;
  float eff = fabsf(e.effort * power * rate * sp.dash_power_rate());
  const float slow = left_team ? sp.slowness_on_top_for_left_team() : sp.slowness_on_top_for_right_team();
  if (slow != 1.0f && e.py < 0.0f) eff = cold_div(eff, slow);
  dir = back ? dir + 180.0f : dir;
  float s, c;
  if (sincos_memo) sincos_deg_memo(e.body + dir, sincos_memo, s, c);  // the same bits, see s2d_math.cuh
  else sincos_deg(e.body + dir, s, c);
  ax = eff * c;
  ay = eff * s;
}

// (turn moment): the faster the player moves, the less it turns (inertia_moment)
template <class SP>
__device__ __forceinline__ void turn(Episode& e, float moment, const SP& sp, const NoiseCtx& nz, uint32_t agent = 0) {
  moment = clampf(sp.min_moment(), moment, sp.max_moment());
  if (SP::kNoise) moment = moment * (1.0f + sp.player_rand() * u11(noise_block(nz, agent).z));
  const float speed = hypot2_or_zero(e.vx, e.vy);
  e.body = norm_deg(e.body + moment / (1.0f + sp.inertia_moment() * speed));
}

// (kick power dir): only inside the kickable area; power falls off by up to 25 % with the angle between
// body and ball and by up to 25 % with the distance.  Adds to the ball's acceleration.
template <class SP>
__device__ __forceinline__ bool kick(Episode& e, float power, float dir, const SP& sp, float& bax, float& bay,
                                     const NoiseCtx& nz, uint32_t agent = 0) {
  power = clampf(0.0f, power, sp.max_power());
  dir = clampf(sp.min_moment(), dir, sp.max_moment());
  const float dx = e.bx - e.px, dy = e.by - e.py;
  const float dist = hypot2(dx, dy);
  if (dist > sp.kickable_area()) return false;
  const float dir_diff = fabsf(norm_deg_360(atan2_deg(dy, dx) - e.body));
  const float dist_ball = dist - sp.player_size() - sp.ball_size();
  const float eff = power * sp.kick_power_rate() *
                    (1.0f - 0.25f * dir_diff * static_cast<float>(1.0 / 180.0) - 0.25f * dist_ball / sp.kickable_margin());
  float s, c;
  sincos_deg(e.body + dir, s, c);
  bax += eff * c;
  bay += eff * s;
  if (SP::kNoise) {  // a random push whose size grows with power, with the awkwardness of the kick and with ball speed
    const uint4 w = noise_block(nz, agent), w2 = noise_block(nz, 32u + agent);
    const float pos_rate = 0.5f + 0.25f * (dir_diff * static_cast<float>(1.0 / 180.0) + dist_ball / sp.kickable_margin());
    const float speed_rate = 0.5f + 0.5f * (hypot2(e.bvx, e.bvy) / (sp.ball_speed_max() * sp.ball_decay()));
    const float max_rand = sp.kick_rand() * (power / sp.max_power()) * (pos_rate + speed_rate);
    const float mag = u32_to_unit(w.w) * max_rand;
    float ns, nc;
    sincos_deg(u11(w2.x) * 180.0f, ns, nc);
    bax += mag * nc;
    bay += mag * ns;
  }
  return true;
}

// Body_GoToPoint (idl/service.proto:684-688) as the proxy lowers it to ONE server command (simplified librcsc
// rule): inside dist_thr -> nothing; facing error above max(15 deg, asin(dist_thr / dist)) -> turn towards the
// target, compensating inertia; else dash straight with the power that reaches the target this cycle.
template <class SP>
__device__ __forceinline__ void lower_goto(const Episode& e, float tx, float ty, float dist_thr, float max_power,
                                           const SP& sp, int& cmd, float& power, float& dir) {
  const float dx = tx - e.px, dy = ty - e.py;
  const float dist = hypot2(dx, dy);
  cmd = S2D_CMD_NONE;
  power = 0.0f;
  dir = 0.0f;
  if (dist < dist_thr) return;
  const float ang = norm_deg_360(atan2_deg(dy, dx) - e.body);
  const float ratio = dist_thr / dist;
  // asin(ratio) exceeds 15 degrees only for ratio > sin(15 deg) = 0.2588: below 0.25 the threshold is exactly 15
  const float athr = ratio > 0.25f ? fmax_(15.0f, atan2_deg(ratio, sqrtf(fmax_(0.0f, 1.0f - ratio * ratio)))) : 15.0f;
  if (fabsf(ang) > athr) {
    const float speed = hypot2_or_zero(e.vx, e.vy);
    cmd = S2D_CMD_TURN;
    dir = clampf(sp.min_moment(), ang * (1.0f + sp.inertia_moment() * speed), sp.max_moment());
    return;
  }
  float sn, cs;
  sincos_deg(e.body, sn, cs);
  const float v_along = e.vx * cs + e.vy * sn;
  const float need = (dist - v_along) / (e.effort * sp.dash_power_rate());
  cmd = S2D_CMD_DASH;
  power = clampf(0.0f, need, max_power);
}

// d^n for 0 <= n <= 63 by binary powering (the order of the multiplications is part of the fp32 spec)
__device__ __forceinline__ float pow_int(float d, int n) {
  float r = 1.0f;
#pragma unroll
  for (int bit = 0; bit < 6; ++bit) {
    r = ((n >> bit) & 1) ? r * d : r;
    d = d * d;
  }
  return r;
}
// how far an object drifts in n cycles per unit of velocity: (1 - d^n) / (1 - d)
__device__ __forceinline__ float inertia_factor(float decay, int n) { return (1.0f - pow_int(decay, n)) / (1.0f - decay); }

// Body_TurnToPoint / Body_TurnToBall / Body_TurnToAngle / Body_KickOneStep / Body_StopBall (include/soccer2d.h,
// S2D_CMD_TURN_TO_POINT ..): rewrites the command in place as the ONE turn or kick the proxy would send.
// Out of line and fed by value (player, ball, constants accessor): taking the address of the episode for a cold call
// would put it on the stack in the hot loop.
struct Kinematics {
  float px, py, vx, vy, body, bx, by, bvx, bvy;
};
template <class SP>
__device__ __noinline__ float4 lower_body_action_cold(const Kinematics e, float4 a, const SP sp) {
  const int c = static_cast<int>(a.x);
  if (c == S2D_CMD_TURN_TO_POINT || c == S2D_CMD_TURN_TO_BALL || c == S2D_CMD_TURN_TO_ANGLE) {
    float ang;
    if (c == S2D_CMD_TURN_TO_ANGLE) {
      ang = norm_deg(norm_deg(a.y) - e.body);
    } else {
      const float nf = rintf(c == S2D_CMD_TURN_TO_BALL ? a.y : a.w);
      const int n = static_cast<int>(clampf(0.0f, nf, 63.0f));
      float tx = a.y, ty = a.z;
      if (c == S2D_CMD_TURN_TO_BALL) {
        const float fb = inertia_factor(sp.ball_decay(), n);
        tx = e.bx + e.bvx * fb;
        ty = e.by + e.bvy * fb;
      }
      const float fp = inertia_factor(sp.player_decay(), n);
      const float mx = e.px + e.vx * fp, my = e.py + e.vy * fp;
      ang = norm_deg_360(atan2_deg(ty - my, tx - mx) - e.body);
    }
    const float speed = hypot2(e.vx, e.vy);
    a = make_float4(static_cast<float>(S2D_CMD_TURN),
                    clampf(sp.min_moment(), ang * (1.0f + sp.inertia_moment() * speed), sp.max_moment()), 0.0f, 0.0f);
  } else if (c == S2D_CMD_KICK_ONE_STEP || c == S2D_CMD_STOP_BALL) {
    const float dx = e.bx - e.px, dy = e.by - e.py;
    const float dist = hypot2(dx, dy);
    if (dist > sp.kickable_area()) return make_float4(static_cast<float>(S2D_CMD_NONE), 0.0f, 0.0f, 0.0f);
    float wx = 0.0f, wy = 0.0f;  // the velocity the ball should leave with
    if (c == S2D_CMD_KICK_ONE_STEP) {
      const float first_speed = clampf(0.0f, a.w, sp.ball_speed_max());
      float s, cs;
      sincos_deg(atan2_deg(a.z - e.by, a.y - e.bx), s, cs);
      wx = first_speed * cs;
      wy = first_speed * s;
    }
    const float ax = wx - e.bvx, ay = wy - e.bvy;
    const float acc = hypot2(ax, ay);
    const float dir_diff = fabsf(norm_deg_360(atan2_deg(dy, dx) - e.body));
    const float dist_ball = dist - sp.player_size() - sp.ball_size();
    const float rate = sp.kick_power_rate() *
                       (1.0f - 0.25f * dir_diff * static_cast<float>(1.0 / 180.0) - 0.25f * dist_ball / sp.kickable_margin());
    a = make_float4(static_cast<float>(S2D_CMD_KICK), clampf(0.0f, acc / rate, sp.max_power()),
                    norm_deg_360(atan2_deg(ay, ax) - e.body), 0.0f);
  } else if (c == S2D_CMD_SMART_KICK) {  // release if one kick can do it, else stage (include/soccer2d.h)
    const float dx = e.bx - e.px, dy = e.by - e.py;
    const float dist = hypot2(dx, dy);
    if (dist > sp.kickable_area()) return make_float4(static_cast<float>(S2D_CMD_NONE), 0.0f, 0.0f, 0.0f);
    const float first_speed = clampf(0.0f, a.w, sp.ball_speed_max());
    float s, cs;
    sincos_deg(atan2_deg(a.z - e.by, a.y - e.bx), s, cs);
    float ax = first_speed * cs - e.bvx, ay = first_speed * s - e.bvy;
    float acc = hypot2(ax, ay);
    const float dir_diff = fabsf(norm_deg_360(atan2_deg(dy, dx) - e.body));
    const float dist_ball = dist - sp.player_size() - sp.ball_size();
    const float rate = sp.kick_power_rate() *
                       (1.0f - 0.25f * dir_diff * static_cast<float>(1.0 / 180.0) - 0.25f * dist_ball / sp.kickable_margin());
    if (!(acc <= sp.max_power() * rate)) {
      const float nx = e.px + e.vx, ny = e.py + e.vy;
      sincos_deg(atan2_deg(a.z - ny, a.y - nx), s, cs);
      const float d = sp.player_size() + sp.ball_size() + 0.3f * sp.kickable_margin();
      const float sax = ((nx + d * cs) - e.bx) - e.bvx, say = ((ny + d * s) - e.by) - e.bvy;
      const float sacc = hypot2(sax, say);
      if (sacc >= 0.05f) {  // (else it is staged already: release with what max_power gives)
        ax = sax;
        ay = say;
        acc = sacc;
      }
    }
    a = make_float4(static_cast<float>(S2D_CMD_KICK), clampf(0.0f, acc / rate, sp.max_power()),
                    norm_deg_360(atan2_deg(ay, ax) - e.body), 0.0f);
  } else if (c == S2D_CMD_INTERCEPT) {
    // drift sums 1 + d + d^2 + ...: where ball and player are after t cycles if nobody touches them
    const float reach0 = 0.8f * sp.kickable_area();
    float fb = 0.0f, fp = 0.0f, pwb = 1.0f, pwp = 1.0f, tx = e.bx, ty = e.by;
#pragma unroll 1
    for (int t = 1; t <= 30; ++t) {
      fb += pwb;
      fp += pwp;
      pwb *= sp.ball_decay();
      pwp *= sp.player_decay();
      tx = e.bx + e.bvx * fb;
      ty = e.by + e.bvy * fb;
      const float mx = e.px + e.vx * fp, my = e.py + e.vy * fp;
      const float ddx = tx - mx, ddy = ty - my;
      const float reach = reach0 + static_cast<float>(t - 1) * sp.player_speed_max();
      if (ddx * ddx + ddy * ddy <= reach * reach) break;
    }
    a = make_float4(static_cast<float>(S2D_CMD_GOTO), tx, ty, 100.0f);
  }
  return a;
}
template <class SP>
__device__ __forceinline__ void lower_body_action(const Episode& e, float4& a, const SP& sp) {
  a = lower_body_action_cold(Kinematics{e.px, e.py, e.vx, e.vy, e.body, e.bx, e.by, e.bvx, e.bvy}, a, sp);
}

// S2D_ACT_COMMAND: {cmd, a, b, c} = proto PlayerAction dash / turn / kick / body_go_to_point (S2D_CMD_*).
// Dashes come out with the direction already lowered by dash_direction.
template <class SP>
__device__ __forceinline__ void decode_command(const Episode& e, float4 a, float goto_dist_thr, const SP& sp, int& cmd,
                                               float& power, float& dir, float& rate) {
  if (a.x >= static_cast<float>(S2D_CMD_TURN_TO_POINT)) lower_body_action(e, a, sp);
  const int c = static_cast<int>(a.x);
  cmd = S2D_CMD_NONE;
  power = 0.0f;
  dir = 0.0f;
  rate = 0.0f;
  if (c == S2D_CMD_DASH || c == S2D_CMD_KICK) {
    cmd = c;
    power = a.y;
    dir = a.z;
  } else if (c == S2D_CMD_TURN) {
    cmd = c;
    dir = a.y;
  } else if (c == S2D_CMD_GOTO) {
    lower_goto(e, a.y, a.z, goto_dist_thr, a.w, sp, cmd, power, dir);
  }
  if (cmd == S2D_CMD_DASH) dash_direction(dir, sp, dir, rate);
}

// ---- one cycle ------------------------------------------------------------------------------------

// MPObject::_inc.  The two clamps compare SQUARED lengths (no square root unless a clamp applies).
// NOISE: vel += (U(-m, m), U(-m, m)) with m = rnd * |vel|, drawn for `agent`.
template <bool NOISE = false>
__device__ __forceinline__ void move_object(float& x, float& y, float& vx, float& vy, float ax, float ay,
                                            float accel_max, float accel_max2, float speed_max, float speed_max2,
                                            float decay, float rnd = 0.0f, const NoiseCtx* nz = nullptr,
                                            uint32_t agent = 0) {
  if (ax != 0.0f || ay != 0.0f) {
    const float a2 = ax * ax + ay * ay;
    if (a2 > accel_max2) {
      const float k = cold_div(accel_max, sqrtf(a2));
      ax *= k;
      ay *= k;
    }
    vx += ax;
    vy += ay;
    const float v2 = vx * vx + vy * vy;
    if (v2 > speed_max2) {
      const float k = cold_div(speed_max, sqrtf(v2));
      vx *= k;
      vy *= k;
    }
  }
  if (NOISE) {
    const uint4 w = noise_block(*nz, agent);
    const float m = rnd * hypot2(vx, vy);
    vx += m * u11(w.x);
    vy += m * u11(w.y);
  }
  x += vx;
  y += vy;
  vx *= decay;
  vy *= decay;
}

constexpr float kCollideEps = 1.0e-6f;

// Where an object at (bx, by) moving with (bvx, bvy) goes when it overlaps an object at (px, py): back along its own
// velocity until the two are `rr` apart; if it is not moving (or that line misses), straight out along the line of
// centres; coincident centres separate along x (`side` = +1 or -1).  The ball of a ball-player contact in both collision
// models, and every colliding object in the BACKTRACE model (include/soccer2d.h).
__device__ __forceinline__ float2 ball_back_trace(float px, float py, float bx, float by, float bvx, float bvy, float rr,
                                                  float side = 1.0f) {
  const float dx = bx - px, dy = by - py;
  const float v = hypot2(bvx, bvy);
  if (v > 1.0e-10f) {
    const float ux = bvx / v, uy = bvy / v;
    const float du = dx * ux + dy * uy;
    const float disc = du * du - (dx * dx + dy * dy - rr * rr);
    if (disc >= 0.0f) {
      const float t = du + sqrtf(disc);
      if (t >= 0.0f) return make_float2(bx - t * ux, by - t * uy);
    }
  }
  const float d = hypot2(dx, dy);
  if (d < 1.0e-10f) return make_float2(px + side * rr, py);
  return make_float2(px + dx / d * rr, py + dy / d * rr);
}

// Ball overlapping the single player (rare): up to ten relaxation rounds as in the server.  MIDPOINT model: the player
// keeps its place (the average of its proposals is its own position).  The caller applies vel *= -0.1 to both.
__device__ __noinline__ inline float2 resolve_ball_player_overlap(float px, float py, float bx, float by, float bvx, float bvy,
                                                           float r) {
  const float r2 = r * r;
  const float rr = r + kCollideEps;
#pragma unroll 1
  for (int round = 0; round < 10; ++round) {
    const float dx = bx - px, dy = by - py;
    if (!(dx * dx + dy * dy < r2)) break;
    const float2 b = ball_back_trace(px, py, bx, by, bvx, bvy, rr);
    bx = b.x;
    by = b.y;
  }
  return make_float2(bx, by);
}
// BACKTRACE model: the player backs up along its own velocity as well.  Returns {ball x, y, player x, y}.
__device__ __noinline__ inline float4 resolve_ball_player_overlap_backtrace(float px, float py, float vx, float vy, float bx, float by,
                                                                     float bvx, float bvy, float r) {
  const float r2 = r * r;
  const float rr = r + kCollideEps;
#pragma unroll 1
  for (int round = 0; round < 10; ++round) {
    const float dx = bx - px, dy = by - py;
    if (!(dx * dx + dy * dy < r2)) break;
    const float2 b = ball_back_trace(px, py, bx, by, bvx, bvy, rr);
    const float2 q = ball_back_trace(bx, by, px, py, vx, vy, rr, -1.0f);
    px = q.x;
    py = q.y;
    bx = b.x;
    by = b.y;
  }
  return make_float4(bx, by, px, py);
}

template <class SP>
// (dx, dy) = ball - player and d2 = dx*dx + dy*dy come from the caller, which re-uses them for the reward when
// nothing collided (the common case).  Returns true when something was moved.
__device__ __forceinline__ bool collide_ball_player(Episode& e, float d2, const SP& sp) {
  uint32_t hit = 0;
  if (d2 < sp.collide_r2()) {
    hit = S2D_FLAG_BALL_COLLIDED | S2D_FLAG_PLAYER_COLLIDED;
    if (sp.collision_model() == S2D_COLLISION_BACKTRACE) {
      const float4 b = resolve_ball_player_overlap_backtrace(e.px, e.py, e.vx, e.vy, e.bx, e.by, e.bvx, e.bvy, sp.collide_r());
      e.bx = b.x;
      e.by = b.y;
      e.px = b.z;
      e.py = b.w;
    } else {
      const float2 b = resolve_ball_player_overlap(e.px, e.py, e.bx, e.by, e.bvx, e.bvy, sp.collide_r());
      e.bx = b.x;
      e.by = b.y;
    }
    e.bvx *= -0.1f;
    e.bvy *= -0.1f;
    e.vx *= -0.1f;
    e.vy *= -0.1f;
  }
  e.flags = (e.flags & ~(S2D_FLAG_BALL_COLLIDED | S2D_FLAG_PLAYER_COLLIDED)) | hit;
  return hit != 0;
}

// Player::updateStamina, written with selects instead of nested branches.
template <class SP>
__device__ __forceinline__ void update_stamina(Episode& e, const SP& sp) {
  {  // recovery decays below recover_dec_thr * stamina_max
    float r = e.recovery > sp.recover_min() ? e.recovery - sp.recover_dec() : e.recovery;
    r = r < sp.recover_min() ? sp.recover_min() : r;
    e.recovery = e.stamina <= sp.recover_dec_stamina() ? r : e.recovery;
  }
  {  // effort decays below effort_dec_thr * stamina_max ...
    float f = e.effort > sp.effort_min() ? e.effort - sp.effort_dec() : e.effort;
    f = f < sp.effort_min() ? sp.effort_min() : f;
    e.effort = e.stamina <= sp.effort_dec_stamina() ? f : e.effort;
  }
  {  // ... and comes back above effort_inc_thr * stamina_max
    float f = e.effort + sp.effort_inc();
    f = f > sp.effort_max() ? sp.effort_max() : f;
    e.effort = (e.stamina >= sp.effort_inc_stamina() && e.effort < sp.effort_max()) ? f : e.effort;
  }
  float inc = fmin_(e.recovery * sp.stamina_inc_max(), sp.stamina_max() - e.stamina);
  const bool capped = sp.stamina_capacity() >= 0.0f;
  inc = (capped && inc > e.capacity) ? e.capacity : inc;
  e.stamina += inc;
  e.capacity = capped ? fmax_(0.0f, e.capacity - inc) : e.capacity;
}

// One server cycle with at most one body command.  Order as in rcssserver's Stadium::step: commands were
// applied on receipt, then every object moves, then collisions, then stamina, then the clock.
// For S2D_CMD_DASH, (dir, rate) come from dash_direction.  TURNS / KICKS say whether the caller can issue those
// commands at all (compile-time pruning).
// Outputs (dx, dy) = ball - player after the cycle and d2 = dx*dx + dy*dy, which the scenario's scoring re-uses.
template <bool TURNS, bool KICKS, class SP>
__device__ __forceinline__ void simulate_cycle(Episode& e, int cmd, float power, float dir, float rate, const SP& sp,
                                               float& dx, float& dy, float& d2, uint64_t seed, uint64_t gid,
                                               const float2* sincos_memo = nullptr) {
  float ax = 0.0f, ay = 0.0f, bax = 0.0f, bay = 0.0f;
  const NoiseCtx nz{seed, gid, e.cycle};
  if (KICKS) e.flags &= ~S2D_FLAG_KICKED;
  if (cmd == S2D_CMD_DASH) {
    dash_apply(e, power, dir, rate, sp, ax, ay, true, sincos_memo);
  } else if (TURNS && cmd == S2D_CMD_TURN) {
    turn(e, dir, sp, nz);
  } else if (KICKS && cmd == S2D_CMD_KICK) {
    if (kick(e, power, dir, sp, bax, bay, nz)) e.flags |= S2D_FLAG_KICKED;
  }
  move_object<SP::kNoise>(e.px, e.py, e.vx, e.vy, ax, ay, sp.player_accel_max(), sp.player_accel_max2(),
                          sp.player_speed_max(), sp.player_speed_max2(), sp.player_decay(), sp.player_rand(), &nz, 0u);
  move_object<SP::kNoise>(e.bx, e.by, e.bvx, e.bvy, bax, bay, sp.ball_accel_max(), sp.ball_accel_max2(),
                          sp.ball_speed_max(), sp.ball_speed_max2(), sp.ball_decay(), sp.ball_rand(), &nz, kBallAgent);
  dx = e.bx - e.px;
  dy = e.by - e.py;
  d2 = dx * dx + dy * dy;
  if (collide_ball_player(e, d2, sp)) {
    dx = e.bx - e.px;
    dy = e.by - e.py;
    d2 = dx * dx + dy * dy;
  }
  update_stamina(e, sp);
  e.cycle += 1u;
}

}  // namespace s2d
