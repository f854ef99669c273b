// s2d_fullgame.cuh - the FULLGAME scenario (BASELINE configs[3]): up to 11 v 11, one THREAD per match.
//
// Thread t of the grid owns match t and walks its players in a loop; the 32 lanes of a warp are 32 different matches.
// Nothing is exchanged between lanes, every lane carries work (a warp-per-match mapping leaves 10 of 32 lanes idle and
// repeats the ball / referee arithmetic in all of them: 956 warp-instructions per match and cycle, round 1), and the
// state is laid out match-minor in HBM, so that the lanes of a warp read and write 512 contiguous bytes per access.
// A player streams through registers, one at a time (its three plane entries and its command are fetched while the
// previous player computes); a copy of the positions sits in shared memory for the n-body parts of the cycle (nearest
// pair, collisions, offside line, dead-ball clearance).
//
// Physics per player = the one-player functions of s2d_one_player.cuh (dash / turn / kick / Body_GoToPoint lowering,
// MPObject::_inc, stamina) plus rcssserver's Stadium::collisions for n players; referee subset: goals, ball out ->
// kick-in / corner kick / goal kick, kick-off after a goal, offside, time over.  NOT in the reference (which only ever
// runs one player with the referee off, soccer_2d_env.py:363-369): the spec is include/soccer2d.h.
//
// Sums over the players of a match (kick accelerations on the ball, collision proposals for the ball) are part of the
// fp32 spec: they are added as a 32-leaf xor-butterfly (leaf = player index, absent players and non-contributors 0.0),
// see tree_sum32 - the order include/soccer2d.h fixes for those sums.
#pragma once
#include "s2d_scenarios.cuh"

namespace s2d {

constexpr int kFgObsDim = 120;        // 4 ball + 22 x 5 player + 6 referee values (rows are 16-byte multiples)
constexpr int kFgDropBallTime = 100;  // cycles a dead ball waits for the awarded side before play resumes
constexpr int kFgMaxPlayers = 22;
constexpr float kFgFreeKickDist = 9.15f;  // the distance opponents keep from a dead ball
constexpr float kFgOffsideArea = 2.5f;    // offside_active_area_size: a marked player this close to the ball takes part
constexpr int kFgAfterGoalWait = 50;      // stopped cycles between a goal and the kick-off
constexpr int kFgTackleCycles = 10;       // tackle_cycles: how long a player lies on the ground after a tackle
constexpr int kFgCatchBan = 5;            // catch_ban_cycle
constexpr float kFgCatchLength = 1.2f, kFgCatchWidth = 1.0f;             // catch_area_l, catch_area_w
constexpr float kFgPenaltyLength = 16.5f, kFgPenaltyHalfWidth = 20.16f;  // the penalty area

// HBM layout of N matches with np players each: plane-major, MATCH-MINOR (consecutive matches are consecutive in
// memory, so a warp = 32 matches touches 512 contiguous bytes per float4 access).  Rows hold Nr = N rounded up to the
// block size (64) entries: every thread of the grid owns a column, so warps are always whole (the columns past N are
// scratch matches that are simulated and never reported):
//   PA float4 [np][Nr] {x, y, vx, vy}           PB float4 [np][Nr] {body, stamina, effort, recovery}
//   PC float  [np][Nr] stamina_capacity
//   EB float4 [Nr] ball {x, y, vx, vy}          EF float4 [Nr] {episode return, player separation bound, offside marks (bits), -}
//   EI uint4  [Nr] {step_number, cycle, episode, mode | side<<8 | last_touch<<10 | timer<<12 | ball_collided<<20 | done<<21}
//   EJ uint4  [Nr] {score_l, score_r, collided mask (bit = player), kicked mask}
//   EK uint4  [Nr] {tackle counters of players 0-7, 8-15, 16-21 (a nibble each), catch bans (left keeper | right << 4)}
constexpr int kFgBlock = 64;  // matches (= threads) per block
struct FgLayout {
  int64_t n;
  int np;
  __host__ __device__ size_t nr() const { return (static_cast<size_t>(n) + kFgBlock - 1) / kFgBlock * kFgBlock; }
  __host__ __device__ size_t pa() const { return 0; }
  __host__ __device__ size_t pb() const { return nr() * np * 16; }
  __host__ __device__ size_t pc() const { return nr() * np * 32; }
  __host__ __device__ size_t eb() const { return pc() + nr() * np * 4; }
  __host__ __device__ size_t ef() const { return eb() + nr() * 16; }
  __host__ __device__ size_t ei() const { return ef() + nr() * 16; }
  __host__ __device__ size_t ej() const { return ei() + nr() * 16; }
  __host__ __device__ size_t ek() const { return ej() + nr() * 16; }
  __host__ __device__ size_t bytes() const { return ek() + nr() * 16; }
};

#ifndef S2D_HOST_EMU

struct Match {
  int step_number;
  uint32_t cycle, episode;
  int mode, side, last_touch, timer;
  int score_l, score_r;
  float ep_return;
  float sep;  // lower bound on the smallest player-player distance (see fg_collisions); 0 = unknown
  uint32_t offside;  // bit = player marked offside at the last pass of its team (all bits from one team)
  bool done_flag;
  float bx, by, bvx, bvy;  // the ball
  uint32_t tk0, tk1, tk2;  // cycles each player still lies on the ground after a tackle: a nibble per player
  uint32_t ban;            // cycles until the goalkeepers may catch again (left | right << 4)
};

#ifndef S2D_FG_AHEAD
#define S2D_FG_AHEAD 2  // player rows the L2 is asked for ahead of the register prefetch (measured: 0 -> 201 us, 1..3 -> 190 us)
#endif
#ifndef S2D_FG_MIN_BLOCKS
// Register budget of the step kernel.  Measured after the store pattern stopped being the bound (profiles/README.md):
// 10 blocks (96 registers, spills and rebuilt pointers in the player loop) 172 us per 2^18-match cycle, 7 or 8 blocks
// (124 registers, nothing spilled, 8 blocks = 16 warps resident) 160-164 us, 6 blocks (144 registers, 12 warps) 176 us;
// a 32 K-match shard 39 -> 34 us.
#define S2D_FG_MIN_BLOCKS 7
#endif

// The block's shared memory: per player a row of kFgBlock entries (lane-minor: conflict-free).
struct FgShared {
  float2 xy[kFgMaxPlayers][kFgBlock];  // position (the same values as plane PA holds)
  float oldx[kFgMaxPlayers][kFgBlock]; // x before this cycle's move (the offside line is drawn at the moment of the pass)
  float obs[20][kFgBlock];             // four players' worth of the observation row on its way out (five float4); after the
                                       // player loop rows 0-4 of a column bring the collision resolver's outcome back
#ifdef S2D_FG_PAD
  char pad[S2D_FG_PAD];                // (tuning aid: lowers the number of resident blocks)
#endif
  uint32_t kicked[kFgBlock];           // per thread: the players (bits) that kicked this cycle.  Kicks are rare; as a register
                                       // variable the mask was spilled, and its reload (an L2 round trip: the SM's L1 is
                                       // given to shared memory) sat in front of every player: 10 % of the kernel's time
};

// Plane pointers of one match (column t of every row), advanced by a row to go from player j to player j + 1.
struct FgPlanes {
  float4* pa;
  float4* pb;
  float* pc;
  const uint8_t* types;  // this match's column of the per-match player types ([np][Nr], s2d_set_player_types_per_match), else nullptr
  size_t row, rowc;  // elements per row
  __device__ __forceinline__ FgPlanes(const KernelParams& P, const FgLayout& L, int64_t env) {
    char* base = static_cast<char*>(P.state);
    pa = reinterpret_cast<float4*>(base + L.pa()) + env;
    pb = reinterpret_cast<float4*>(base + L.pb()) + env;
    pc = reinterpret_cast<float*>(base + L.pc()) + env;
    types = P.type_of_match ? P.type_of_match + env : nullptr;
    row = L.nr();
    rowc = L.nr();
  }
};

// heterogeneous players: points sp at the constants of player j of this match (its own assignment if the handle has
// one per match, else the handle's)
template <class SP>
__device__ __forceinline__ void fg_point_at_type(SP& sp, const KernelParams& P, const FgPlanes& g, const int j) {
  if constexpr (SP::kHetero)
    sp.row = sp.table + PT_ROW * (g.types ? static_cast<int>(__ldg(g.types + static_cast<size_t>(j) * g.row)) : static_cast<int>(P.type_of[j]));
}

// 4-4-2 kick-off formation of the left team (own half); the right team is the mirror image
__device__ __constant__ float kFgFormX[11] = {-50, -36, -36, -36, -36, -20, -20, -20, -20, -9, -9};
__device__ __constant__ float kFgFormY[11] = {0, -20, -7, 7, 20, -24, -8, 8, 24, -10, 10};

// Sum of 32 leaves in xor-butterfly order ((i, i^16), then (i, i^8), ...): leaf i = v[i] where bit i of `mask` is set,
// else 0.0.  Cold (only cycles with a kick or a ball collision get here), so the leaves live in local memory.
__device__ __noinline__ inline float tree_sum32(const float* v, uint32_t mask) {
  float leaf[32];
#pragma unroll 1
  for (int i = 0; i < 32; ++i) leaf[i] = ((mask >> i) & 1u) ? v[i] : 0.0f;
#pragma unroll 1
  for (int s = 16; s > 0; s >>= 1) {
#pragma unroll 1
    for (int i = 0; i < s; ++i) leaf[i] = leaf[i] + leaf[i + s];
  }
  return leaf[0];
}

// kick-off placement of one player: formation spot plus a +-2 m jitter drawn per (episode, kick-off, player)
__device__ __forceinline__ void fg_place_player(float2& xy, float& body, const KernelParams& P, uint64_t gid, uint32_t episode,
                                                int j, int pps, int kick_offs) {
  const bool left = j < pps;
  const int k = left ? j : j - pps;
  const uint4 w = philox4x32_10(P.seed, gid, episode, RNG_RESET,
                                static_cast<uint32_t>(2 + j) + 32u * (static_cast<uint32_t>(kick_offs) & 0xFFFFu));
  const float jx = u32_to_unit(w.x) * 4.0f - 2.0f, jy = u32_to_unit(w.y) * 4.0f - 2.0f;
  const float fx = kFgFormX[k], fy = kFgFormY[k];
  xy.x = (left ? fx : -fx) + jx;
  xy.y = (left ? fy : -fy) + jy;
  body = left ? 0.0f : 180.0f;
}

// every player to its kick-off spot, at rest, facing the opponents (after a goal; cold)
__device__ __noinline__ inline void fg_kick_off_formation(FgShared& S, int t, FgPlanes g, const KernelParams& P, uint64_t gid,
                                                   uint32_t episode, int np, int kick_offs) {
#pragma unroll 1
  for (int j = 0; j < np; ++j) {
    float2 xy;
    float body;
    fg_place_player(xy, body, P, gid, episode, j, np >> 1, kick_offs);
    S.xy[j][t] = xy;
    *g.pa = make_float4(xy.x, xy.y, 0.0f, 0.0f);
    float4 b = *g.pb;
    b.x = body;
    *g.pb = b;
    g.pa += g.row;
    g.pb += g.row;
  }
}

// new match: scores 0, kick-off formation, everybody recovered, kick-off for the left team
template <class SP>
__device__ __noinline__ void fg_reset(FgShared& S, int t, FgPlanes g, Match& m, const KernelParams& P, SP sp, uint64_t gid, int np) {
  m.score_l = 0;
  m.score_r = 0;
#pragma unroll 1
  for (int j = 0; j < np; ++j) {
    fg_point_at_type(sp, P, g, j);
    float2 xy;
    Episode p;
    fg_place_player(xy, p.body, P, gid, m.episode, j, np >> 1, 0);
    recover(p, sp);
    S.xy[j][t] = xy;
    *g.pa = make_float4(xy.x, xy.y, 0.0f, 0.0f);
    *g.pb = make_float4(p.body, p.stamina, p.effort, p.recovery);
    *g.pc = p.capacity;
    g.pa += g.row;
    g.pb += g.row;
    g.pc += g.rowc;
  }
  m.bx = m.by = m.bvx = m.bvy = 0.0f;
  m.tk0 = m.tk1 = m.tk2 = m.ban = 0u;
  m.episode += 1u;
  m.step_number = 0;
  m.ep_return = 0.0f;
  m.sep = 0.0f;
  m.offside = 0u;
  m.done_flag = false;
  m.mode = S2D_PM_KICK_OFF;
  m.side = S2D_SIDE_LEFT;
  m.timer = 0;
  m.last_touch = S2D_SIDE_UNKNOWN;
}

// The command of player `agent` in the 32 matches of a warp.  Every lane may carry a different command, so a switch over
// the command would make the warp walk dash, turn, kick and go-to-point one after the other, each with its own sincos /
// atan2 / sqrt.  Here the commands are decomposed into the pieces they share, each evaluated ONCE per warp under a vote
// (`full` = the lanes of the warp that hold a match) and with per-lane operands:
//   geometry to a reference point  (go-to-point: the target, kick: the ball)  -> distance, relative angle
//   speed                          (turn and go-to-point's turn: inertia)
//   sincos(body + direction)       (dash, go-to-point's dash (direction 0), kick)
// Per lane the arithmetic is the sequence of decode_command + dash_apply / turn / kick (s2d_one_player.cuh), so the
// results are the same bit for bit.  Returns whether the player kicked (kax, kay = its push on the ball).
template <class SP>
__device__ __forceinline__ bool fg_commands(Episode& p, float4 a, float goto_dist_thr, const SP& sp, const NoiseCtx& nz,
                                            const unsigned full, int agent, bool left, bool may_kick, bool may_dash, float& ax,
                                            float& ay, float& kax, float& kay) {
  // the proxy's other body actions become a plain turn or kick first (rare: one vote when nobody uses them)
  if (__any_sync(full, a.x >= static_cast<float>(S2D_CMD_TURN_TO_POINT))) {
    if (a.x >= static_cast<float>(S2D_CMD_TURN_TO_POINT)) lower_body_action(p, a, sp);
  }
  const int c = static_cast<int>(a.x);
  const bool is_goto = c == S2D_CMD_GOTO;
  const bool is_kick = c == S2D_CMD_KICK && may_kick;
  const bool user_dash = c == S2D_CMD_DASH, user_turn = c == S2D_CMD_TURN;

  // The operands of the three long chains of a command - geometry to the reference point (square root, atan2), the
  // player's speed (square root; a turn's inertia), sin / cos of body + direction (dash, kick) - are all known once
  // the command is decoded, before go-to-point has decided anything.  They are evaluated up front in ONE block, side by
  // side, for every lane whose command MAY need them: this kernel is bound by the length of the thread's dependency
  // chain, not by issue slots, and three independent chains overlap where three voted blocks in a row did not.
  const bool may_turn = user_turn || is_goto;                  // superset of do_turn
  const bool may_dsh = (user_dash || is_goto) && may_dash;     // superset of do_dash
  float dist = 0.0f, rel = 0.0f, speed = 0.0f;
  float dir = 0.0f, rate = 1.0f, sn = 0.0f, cs = 1.0f;
  const float user_power = clampf(sp.min_dash_power(), a.y, sp.max_dash_power());
  const bool back = user_dash && user_power < 0.0f;
  auto dash_kick_direction = [&]() {  // dash direction (go-to-point dashes straight: direction 0) and the one sincos
    dash_direction(user_dash ? a.z : 0.0f, sp, dir, rate);
    const float kick_dir = clampf(sp.min_moment(), a.z, sp.max_moment());
    const float d = is_kick ? kick_dir : back ? dir + 180.0f : dir;
    sincos_deg(p.body + d, sn, cs);  // (of the body angle before this cycle's turn: who turns neither dashes nor kicks)
  };
  if (__any_sync(full, is_goto || is_kick || user_turn)) {
    // (lanes that are not concerned get harmless operands: a zero numerator or denominator, or sqrt(0), would send
    // the whole warp through the slow paths of the IEEE division and square root)
    const float dx = is_goto ? a.y - p.px : is_kick ? p.bx - p.px : 1.0f;
    const float dy = is_goto ? a.z - p.py : is_kick ? p.by - p.py : 0.5f;
    dist = hypot2(dx, dy);
    rel = norm_deg_360(atan2_deg(dy, dx) - p.body);
    speed = hypot2_or_zero(may_turn ? p.vx : 1.0f, may_turn ? p.vy : 0.0f);  // (a standing player: often)
    dash_kick_direction();
  } else if (__any_sync(full, may_dsh)) {  // nobody but dashers in the warp
    dash_kick_direction();
  }

  // go-to-point decides: nothing (arrived) | turn towards the target | dash straight at it
  bool goto_turn = false, goto_dash = false;
  if (__any_sync(full, is_goto)) {
    const bool on_the_way = is_goto && !(dist < goto_dist_thr);
    const float ratio = goto_dist_thr / (is_goto ? dist : 1.0f);
    float athr = 15.0f;  // asin(ratio) exceeds 15 degrees only for ratio > sin(15 deg) = 0.2588
    if (__any_sync(full, on_the_way && ratio > 0.25f)) {
      const float wide = fmax_(15.0f, atan2_deg(ratio, sqrtf(fmax_(0.0f, 1.0f - ratio * ratio))));
      athr = ratio > 0.25f ? wide : 15.0f;
    }
    goto_turn = on_the_way && fabsf(rel) > athr;
    goto_dash = on_the_way && !goto_turn;
  }

  // turn
  const bool do_turn = user_turn || goto_turn;
  if (__any_sync(full, do_turn)) {
    const float inertia = 1.0f + sp.inertia_moment() * (do_turn ? speed : 0.2f);
    float moment = goto_turn ? clampf(sp.min_moment(), rel * inertia, sp.max_moment()) : user_turn ? a.y : 1.0f;
    moment = clampf(sp.min_moment(), moment, sp.max_moment());
    if (SP::kNoise) moment = moment * (1.0f + sp.player_rand() * u11(noise_block(nz, static_cast<uint32_t>(agent)).z));
    const float body = norm_deg(p.body + moment / inertia);
    p.body = do_turn ? body : p.body;
  }

  const bool do_dash = (user_dash || goto_dash) && may_dash;  // (AfterGoal: the clock stands still, only turns work)

  // dash
  if (__any_sync(full, do_dash)) {
    float power = user_power;
    if (__any_sync(full, goto_dash)) {
      const float v_along = p.vx * cs + p.vy * sn;
      const float need = (dist - v_along) / (goto_dash ? p.effort * sp.dash_power_rate() : 1.0f);
      const float reach = clampf(sp.min_dash_power(), clampf(0.0f, need, a.w), sp.max_dash_power());
      power = goto_dash ? reach : power;
    }
    float need = back ? power * -2.0f : power;
    need = fmin_(need, p.stamina + sp.extra_stamina());
    const float stamina = fmax_(0.0f, p.stamina - need);
    power = back ? need * -0.5f : need;
    float eff = fabsf(p.effort * power * rate * sp.dash_power_rate());
    const float slow = left ? sp.slowness_on_top_for_left_team() : sp.slowness_on_top_for_right_team();
    if (slow != 1.0f && p.py < 0.0f) eff = cold_div(eff, slow);
    p.stamina = do_dash ? stamina : p.stamina;
    ax = do_dash ? eff * cs : 0.0f;
    ay = do_dash ? eff * sn : 0.0f;
  }

  // kick
  bool kicked = false;
  if (__any_sync(full, is_kick)) {
    kicked = is_kick && !(dist > sp.kickable_area());
    const float power = clampf(0.0f, a.y, sp.max_power());
    const float dir_diff = fabsf(rel);
    const float dist_ball = dist - sp.player_size() - sp.ball_size();
    const float eff = power * sp.kick_power_rate() *
                      (1.0f - 0.25f * dir_diff * static_cast<float>(1.0 / 180.0) - 0.25f * dist_ball / sp.kickable_margin());
    float bax = 0.0f, bay = 0.0f;
    bax += eff * cs;
    bay += eff * sn;
    if (SP::kNoise) {
      if (__any_sync(full, kicked)) {
        const uint4 w = noise_block(nz, static_cast<uint32_t>(agent)), w2 = noise_block(nz, 32u + static_cast<uint32_t>(agent));
        const float pos_rate = 0.5f + 0.25f * (dir_diff * static_cast<float>(1.0 / 180.0) + dist_ball / sp.kickable_margin());
        const float speed_rate = 0.5f + 0.5f * (hypot2(p.bvx, p.bvy) / (sp.ball_speed_max() * sp.ball_decay()));
        const float max_rand = sp.kick_rand() * (power / sp.max_power()) * (pos_rate + speed_rate);
        const float mag = u32_to_unit(w.w) * max_rand;
        float ns, nc;
        sincos_deg(u11(w2.x) * 180.0f, ns, nc);
        bax += mag * nc;
        bay += mag * ns;
      }
    }
    kax = kicked ? bax : 0.0f;
    kay = kicked ? bay : 0.0f;
  }
  return kicked;
}


__device__ __forceinline__ float butterfly_sum(float v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

// Stadium::collisions for the matches of a warp that have an overlap (`need`: one bit per lane = match).  Overlaps are
// rare (a few per cent of the matches per cycle), and resolving one is an O(np^2) affair that would hold the other 31
// matches of the warp: so the WARP resolves each such match together, lane l = player l of that match - positions come
// from shared memory, partner positions are shuffle broadcasts, the ball's proposals are summed with an xor butterfly.
// In a round every object collects the positions proposed for it and moves to their average; afterwards whatever
// collided gets vel *= -0.1 once.  The lane that owns the match finds the masks (players that collided, players that touched the
// ball) and the ball in rows 0-4 of its observation staging column (nothing is passed by reference: a variable whose
// address a non-inlined function has seen lives in local memory for good); the player lanes write positions and velocities back (shared memory, plane PA and,
// when `obs_rows` (the observation tensor) is set - last cycle of a launch -, the row the player loop has already written).
__device__ __noinline__ inline void fg_resolve_collisions(FgShared& S, const int t, const int tid, const int lane, const int lpm, const FgPlanes g,
                                                   const float mbx, const float mby, const float mbvx, const float mbvy,
                                                   const int np, unsigned need,
                                                   const bool dead, const float r, const float r2, const int model, float* obs_rows,
                                                   const int64_t env, const bool valid) {
  // (t = this thread's match column in shared memory; with lpm lanes per match, lane l holds column t - l / lpm + ..)
  const unsigned full = 0xffffffffu;
  const bool active = lane < np;
  const float h = r2 / 2.0f + kCollideEps;
#pragma unroll 1
  while (need) {
    const int src = __ffs(need) - 1;
    need &= need - 1u;
    const int dcol = src / lpm - lane / lpm;  // from this thread's match to the match being resolved
    const int ts = t + dcol;                  // its column in shared memory
    float bx = __shfl_sync(full, mbx, src), by = __shfl_sync(full, mby, src);
    const float bvx = __shfl_sync(full, mbvx, src), bvy = __shfl_sync(full, mbvy, src);
    const bool ball_fixed = __shfl_sync(full, static_cast<int>(dead), src) != 0;
    const bool report = __shfl_sync(full, static_cast<int>(valid), src) != 0;
    float2 pos = active ? S.xy[lane][ts] : make_float2(0.0f, 0.0f);
    float4* const my_pa = g.pa + dcol + static_cast<size_t>(active ? lane : 0) * g.row;  // (player lane, match src)
    float2 vel = make_float2(0.0f, 0.0f);  // BACKTRACE: every object backs up along its own velocity
    if (model == S2D_COLLISION_BACKTRACE && active) {
      const float4 a = *my_pa;
      vel = make_float2(a.z, a.w);
    }
    bool collided = false, ballhit = false, ball_any = false;
#pragma unroll 1
    for (int round = 0; round < 10; ++round) {
      // Pass 1, without a branch: which players overlap this lane's player (bit j), and does the ball.  The tests are the
      // specification's own (ex * ex + ey * ey < r2 * r2, ...).  Almost every pair says no, so finding the few that say
      // yes first keeps the expensive part below out of the 22-iteration loop.
      uint32_t hits = 0;
#pragma unroll 2
      for (int j = 0; j < np; ++j) {
        const float xj = __shfl_sync(full, pos.x, j), yj = __shfl_sync(full, pos.y, j);
        const float ex = pos.x - xj, ey = pos.y - yj;
        hits |= (ex * ex + ey * ey < r2 * r2) ? 1u << j : 0u;
      }
      hits &= active ? ~(1u << lane) : 0u;
      const float dx = bx - pos.x, dy = by - pos.y;
      const bool bc = active && !ball_fixed && dx * dx + dy * dy < r * r;
      hits |= bc ? 1u << lane : 0u;
      const bool col = hits != 0u;
      collided |= col;
      ballhit |= bc;
      // Pass 2: the proposals, partner by partner in increasing player index (the order of these sums is part of the
      // fp32 spec); bit `lane` stands for the ball.  Lanes take as many turns as the busiest of them has partners.
      int cnt = 0;
      float sx = 0.0f, sy = 0.0f, bpx = 0.0f, bpy = 0.0f;
#pragma unroll 1
      for (uint32_t rest = hits; __any_sync(full, rest != 0u); rest &= rest - 1u) {
        const int j = rest ? __ffs(rest) - 1 : lane;
        const float xj = __shfl_sync(full, pos.x, j), yj = __shfl_sync(full, pos.y, j);
        if (rest == 0u) continue;
        if (j == lane) {
          const float2 b = ball_back_trace(pos.x, pos.y, bx, by, bvx, bvy, r + kCollideEps);
          bpx = b.x;
          bpy = b.y;
          float2 own = pos;
          if (model == S2D_COLLISION_BACKTRACE) own = ball_back_trace(bx, by, pos.x, pos.y, vel.x, vel.y, r + kCollideEps, -1.0f);
          sx += own.x;
          sy += own.y;
        } else if (model == S2D_COLLISION_BACKTRACE) {
          const float2 own = ball_back_trace(xj, yj, pos.x, pos.y, vel.x, vel.y, r2 + kCollideEps, lane < j ? 1.0f : -1.0f);
          sx += own.x;
          sy += own.y;
        } else {
          const float ex = pos.x - xj, ey = pos.y - yj;
          const float mx = (pos.x + xj) / 2.0f, my = (pos.y + yj) / 2.0f;
          const float d = hypot2(ex, ey);
          float ux, uy;
          if (d < 1.0e-10f) {
            ux = lane < j ? 1.0f : -1.0f;
            uy = 0.0f;
          } else {
            ux = ex / d;
            uy = ey / d;
          }
          sx += mx + ux * h;
          sy += my + uy * h;
        }
        cnt += 1;
      }
      const int bcnt = __popc(__ballot_sync(full, bc));
      const float bsx = butterfly_sum(bpx), bsy = butterfly_sum(bpy);
      if (bcnt) {
        bx = bsx / static_cast<float>(bcnt);
        by = bsy / static_cast<float>(bcnt);
        ball_any = true;
      }
      if (cnt) {
        pos.x = sx / static_cast<float>(cnt);
        pos.y = sy / static_cast<float>(cnt);
      }
      if (!__any_sync(full, col)) break;
    }
    const unsigned cm = __ballot_sync(full, collided), tm = __ballot_sync(full, ballhit);
    if (collided) {  // (active lanes only)
      S.xy[lane][ts] = pos;
      const float4 a = *my_pa;
      const float vx = a.z * -0.1f, vy = a.w * -0.1f;
      *my_pa = make_float4(pos.x, pos.y, vx, vy);
      if (obs_rows && report) {
        float* o = obs_rows + (env + dcol) * kFgObsDim + 4 + 5 * lane;
        o[0] = pos.x * static_cast<float>(1.0 / 52.5);
        o[1] = pos.y * static_cast<float>(1.0 / 34.0);
        o[2] = vx;
        o[3] = vy;
      }
    }
    if (lane == src) {  // the outcome, left in the owner's (free by now) observation staging column
      S.obs[0][tid] = bx;
      S.obs[1][tid] = by;
      S.obs[2][tid] = __uint_as_float(ball_any ? 1u : 0u);
      S.obs[3][tid] = __uint_as_float(cm);
      S.obs[4][tid] = __uint_as_float(tm);
    }
  }
  __syncwarp();  // what the player lanes wrote (shared memory, plane PA) is read by the matches' own threads next
}

// Offside marks (OffsideRef), taken at the moment of a pass by ONE team in PlayOn: the passer's team-mates that are, in
// their direction of attack, beyond the ball, the half-way line and the second-last opponent.  Positions are those
// before the cycle's move (S.oldx, the ball before its move).  Cold: only cycles with a kick.
__device__ __noinline__ inline uint32_t fg_offside_marks(const FgShared& S, int t, int np, bool att_left, uint32_t kick_mask, float ball_x) {
  const int pps = np >> 1;
  const float sgn = att_left ? 1.0f : -1.0f;
  const int d0 = att_left ? pps : 0, a0 = att_left ? 0 : pps;
  float last = -3.0e38f, second = -3.0e38f;  // the two largest of the defenders (equal values count twice)
#pragma unroll 1
  for (int j = d0; j < d0 + pps; ++j) {
    const float v = sgn * S.oldx[j][t];
    if (v > last) {
      second = last;
      last = v;
    } else if (v > second) {
      second = v;
    }
  }
  const float line_x = fmaxf(fmaxf(second, sgn * ball_x), 0.0f);
  uint32_t marks = 0;
#pragma unroll 1
  for (int j = a0; j < a0 + pps; ++j)
    if (((kick_mask >> j) & 1u) == 0u && sgn * S.oldx[j][t] > line_x) marks |= 1u << j;
  return marks;
}

// The 120-float observation row of a match: ball, 22 x {x, y, vx, vy, body}, referee state (absent players zero).
// Written by the match's own thread as 15 full 32-byte sectors; the plane entries of the next four players are in
// flight while the current four are converted and stored.
struct FgObsGroup {
  float4 a[4];
  float body[4];
};
__device__ __forceinline__ void fg_obs_load(FgObsGroup& q, const float4* pa, const float4* pb, size_t row, int first, int np) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    q.a[k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    q.body[k] = 0.0f;
    if (first + k < np) {
      q.a[k] = pa[static_cast<size_t>(first + k) * row];
      q.body[k] = reinterpret_cast<const float*>(pb + static_cast<size_t>(first + k) * row)[0];
    }
  }
}
__device__ __forceinline__ void fg_write_obs(float* __restrict__ dst, int64_t env, const FgPlanes& g, const Match& m, int np,
                                             int half_time) {
  float4* row = reinterpret_cast<float4*>(dst + env * kFgObsDim);
  FgObsGroup nxt;
  fg_obs_load(nxt, g.pa, g.pb, g.row, 0, np);
  // carry: the float4 that completes a 32-byte sector with the first float4 of the next group (row[0] = the ball)
  float4 carry = make_float4(m.bx * static_cast<float>(1.0 / 52.5), m.by * static_cast<float>(1.0 / 34.0),
                             m.bvx * static_cast<float>(1.0 / 3.0), m.bvy * static_cast<float>(1.0 / 3.0));
#pragma unroll 1
  for (int grp = 0; grp < 6; ++grp) {  // four players = 20 floats = 5 float4; the last group: 2 players + the 6 referee values
    const FgObsGroup cur = nxt;
    if (grp < 5) fg_obs_load(nxt, g.pa, g.pb, g.row, 4 * grp + 4, np);
    float f[20];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      f[5 * q + 0] = cur.a[q].x * static_cast<float>(1.0 / 52.5);
      f[5 * q + 1] = cur.a[q].y * static_cast<float>(1.0 / 34.0);
      f[5 * q + 2] = cur.a[q].z;
      f[5 * q + 3] = cur.a[q].w;
      f[5 * q + 4] = cur.body[q] * static_cast<float>(1.0 / 180.0);
    }
    if (grp == 5) {
      f[10] = static_cast<float>(m.mode);
      f[11] = static_cast<float>(m.side);
      f[12] = static_cast<float>(m.score_l);
      f[13] = static_cast<float>(m.score_r);
      f[14] = static_cast<float>(m.step_number) / static_cast<float>(2 * half_time);
      f[15] = 0.0f;
    }
    // float4 index of this group's first value: 1 + 5 grp.  Even groups start on the odd half of a sector (completed
    // by `carry`), odd groups on the even half and leave their fifth float4 as the next carry.
    float4* o = row + 5 * grp;
    const float4 v0 = make_float4(f[0], f[1], f[2], f[3]), v1 = make_float4(f[4], f[5], f[6], f[7]);
    const float4 v2 = make_float4(f[8], f[9], f[10], f[11]), v3 = make_float4(f[12], f[13], f[14], f[15]);
    const float4 v4 = make_float4(f[16], f[17], f[18], f[19]);
    if ((grp & 1) == 0) {  // row + 5 grp is sector aligned: {carry, v0} {v1, v2} {v3, v4}
      st_stream_256(o, carry, v0);
      st_stream_256(o + 2, v1, v2);
      st_stream_256(o + 4, v3, v4);
    } else {               // row + 5 grp + 1 is sector aligned: {v0, v1} {v2, v3}, v4 carried
      st_stream_256(o + 1, v0, v1);
      st_stream_256(o + 3, v2, v3);
      carry = v4;
    }
  }
}

// ---- the built-in script (scripted players; spec: include/soccer2d.h, s2d_set_scripted_players) ----
// A kernel variant: VAR + kVarScripted is the same kernel with the script compiled in; the launcher picks it only when
// the handle's mask is non-zero, so the kernels without it are the ones that ran before the script existed.
constexpr int kVarScripted = 8;

// the ball inside the penalty area of the left (right) team
template <class SP>
__device__ __forceinline__ bool fg_in_penalty_area(const SP& sp, float bx, float by, bool left) {
  const float edge = sp.pitch_half_length() - kFgPenaltyLength;
  return (left ? bx <= -edge : bx >= edge) && fabsf(by) <= kFgPenaltyHalfWidth;
}

// Chaser of each side: its player nearest to the ball (positions at the start of the cycle, S.xy; ties go to the lower
// index).  The goalkeeper takes part only while the ball is in its own penalty area, or when it is its side's only player.
template <class SP>
__device__ __forceinline__ void fg_script_chasers(const FgShared& S, int t, const SP& sp, const Match& m, int np, int& chaser_l,
                                                  int& chaser_r) {
  const int pps = np >> 1;
  const bool area_l = fg_in_penalty_area(sp, m.bx, m.by, true), area_r = fg_in_penalty_area(sp, m.bx, m.by, false);
  float best_l = 3.0e38f, best_r = 3.0e38f;
  chaser_l = chaser_r = -1;
#pragma unroll 1
  for (int j = 0; j < np; ++j) {
    const bool left = j < pps;
    const bool keeper = j == 0 || j == pps;
    const bool eligible = !keeper || pps == 1 || (left ? area_l : area_r);
    const float2 xy = S.xy[j][t];
    const float dx = xy.x - m.bx, dy = xy.y - m.by;
    const float d2 = dx * dx + dy * dy;
    if (eligible && left && d2 < best_l) {
      best_l = d2;
      chaser_l = j;
    }
    if (eligible && !left && d2 < best_r) {
      best_r = d2;
      chaser_r = j;
    }
  }
}

// The command of scripted player j (start-of-cycle position / body in `pa` / `body`, catch bans `ban`), in the rules'
// order of the spec.  fp32, no contraction, IEEE division and square root (DESIGN.md section 4).
template <class SP>
__device__ __forceinline__ float4 fg_script_command(const SP& sp, const Match& m, const float4 pa, const float body, const int j,
                                                    const int pps, const bool chaser, const uint32_t ban) {
  const bool left = j < pps;
  const float sg = left ? 1.0f : -1.0f;  // own frame: (sg x, sg y)
  const bool keeper = j == 0 || j == pps;
  const float hl = sp.pitch_half_length(), hw = sp.pitch_half_width();
  const float post = sp.goal_width() * 0.5f - 1.0f;
  const float obx = sg * m.bx, oby = sg * m.by;  // the ball in the own frame
  if (m.mode == S2D_PM_AFTER_GOAL || m.mode == S2D_PM_BEFORE_KICK_OFF || m.mode == S2D_PM_TIME_OVER)
    return make_float4(static_cast<float>(S2D_CMD_NONE), 0.0f, 0.0f, 0.0f);
  const bool play_on = m.mode == S2D_PM_PLAY_ON;
  if (chaser && (play_on || m.side == (left ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT))) {
    const float dx = m.bx - pa.x, dy = m.by - pa.y;
    const float d2 = dx * dx + dy * dy;
    const uint32_t my_ban = j == 0 ? ban & 15u : (ban >> 4) & 15u;
    if (play_on && keeper && my_ban == 0u && fg_in_penalty_area(sp, m.bx, m.by, left) && d2 <= kFgCatchLength * kFgCatchLength)
      return make_float4(static_cast<float>(S2D_CMD_CATCH), norm_deg(atan2_deg(dy, dx) - body), 0.0f, 0.0f);
    if (!(sqrtf(d2) > sp.kickable_area())) {
      // kick target: within 25 m of the goal centre the far post (seen from the kicker: the ball's side flips while it
      // is staged around the kicker's feet) at ball_speed_max, else 8 m further towards the goal at 1
      const float gx = hl - obx, gy = -oby;
      const float g2 = gx * gx + gy * gy;
      float tx, ty, speed;
      if (g2 <= 625.0f) {
        tx = hl;
        ty = sg * pa.y >= 0.0f ? -post : post;
        speed = sp.ball_speed_max();
      } else {
        const float k = 8.0f / sqrtf(g2);
        tx = obx + gx * k;
        ty = oby + gy * k;
        speed = 1.0f;
      }
      return make_float4(static_cast<float>(S2D_CMD_SMART_KICK), sg * tx, sg * ty, speed);
    }
    if (play_on) return make_float4(static_cast<float>(S2D_CMD_INTERCEPT), 0.0f, 0.0f, 0.0f);
    return make_float4(static_cast<float>(S2D_CMD_GOTO), m.bx, m.by, 100.0f);
  }
  if (keeper) return make_float4(static_cast<float>(S2D_CMD_GOTO), sg * (2.5f - hl), sg * clampf(-post, 0.3f * oby, post), 100.0f);
  const int k = left ? j : j - pps;
  const float fx = clampf(2.5f - hl, kFgFormX[k] + 0.6f * obx, hl - 2.5f);
  const float fy = clampf(2.0f - hw, kFgFormY[k] + 0.3f * oby, hw - 2.0f);
  return make_float4(static_cast<float>(S2D_CMD_GOTO), sg * fx, sg * fy, 60.0f);
}

// One cycle of the match.  Commands: float4 {cmd, a, b, c} of player j at act[j].  Returns done.
// `obs_row` != nullptr (last cycle of a launch, 11 v 11): the player loop writes the players' part of the observation
// row as it goes (the values are in registers then), and whatever moves a player afterwards patches its entry;
// obs_dirty is raised where the whole row has to be written again (kick-off).
//
// LPM = lanes per match (1, 2 or 4 adjacent lanes).  With more than one, the lanes of a match share its players in the
// two player loops (sub-lane h takes the groups of four players h, h + LPM, ...) and in the pair scan, merge what they
// found with shuffles, and repeat the cheap per-match arithmetic (ball, referee) redundantly - bit-identical by
// construction.  It shortens the dependent chain of a cycle: for shards too small to fill the GPU with one thread per match.
template <int LPM, bool SCRIPT, class SP>
__device__ __forceinline__ bool fg_cycle(FgShared& S, const int t, const int tid, const FgPlanes& g, Match& m, const KernelParams& P,
                                         SP& sp, uint64_t gid, int np, int half_time, const float4* __restrict__ act,
                                         float* obs_row, const bool valid, bool& obs_dirty, float& reward, int& result,
                                         uint32_t& collided_mask, uint32_t& kicked_mask, bool& ball_collided) {
  const unsigned full = 0xffffffffu;
  const int pps = np >> 1;
  const int h = tid & (LPM - 1);  // sub-lane within the match
  const int lane = tid & 31;
  // the players of this sub-lane, in the order it walks them; LPM = 1: simply 0 .. np - 1
  auto player_at = [&](int it) { return LPM == 1 ? it : 4 * ((it >> 2) * LPM + h) + (it & 3); };
  const int iters = LPM == 1 ? np : 4 * ((((np + 3) >> 2) + LPM - 1) / LPM);
  const unsigned left_set = (1u << pps) - 1u;
  bool dead = m.mode != S2D_PM_PLAY_ON;
  const bool dead_at_start = dead;
  const bool stopped = m.mode == S2D_PM_AFTER_GOAL;  // the server's clock stands still: nothing moves, only turns work
  int caught = -1;                                   // the goalkeeper (player index) that caught the ball this cycle
  m.step_number += 1;
  const NoiseCtx nz{P.seed, gid, m.cycle};
  {  // the match's command row (np x 16 bytes, 32-byte aligned): ask the L2 for its lines now, the loop loads them later
    const char* row = reinterpret_cast<const char*>(act);
    const int bytes = np * 16;
#pragma unroll 1
    for (int o = 0; o < bytes; o += 128) prefetch_l2(row + o);
    prefetch_l2(row + bytes - 32);
  }

  // ---- every player: command, move, stamina (the private part of the player streams through registers) ----
  S.kicked[tid] = 0u;
  float kx[32], ky[32];  // the kickers' pushes on the ball (local memory; written only when somebody kicks)
  float moved2 = 0.0f;
  const uint32_t tk0_in = m.tk0, tk1_in = m.tk1, tk2_in = m.tk2, ban_in = m.ban;
  int chaser_l = -1, chaser_r = -1;  // scripted players: each side's chaser, from the positions before anybody moves
  if constexpr (SCRIPT) {
    fg_script_chasers(S, t, sp, m, np, chaser_l, chaser_r);
    if (LPM > 1) __syncwarp();  // (the other sub-lanes overwrite S.xy in the player loop)
  }
  {
    // software pipeline: the plane entries of this sub-lane's next player are in flight while the current one
    // computes; the commands come two players (one 32-byte sector) at a time, so the loop walks the players in pairs
    // (np is even, and pairs do not straddle the groups of four the sub-lanes take turns with)
    const int j_first = player_at(0);
    float4 n_a = make_float4(0.f, 0.f, 0.f, 0.f), n_b = make_float4(0.f, 0.f, 0.f, 1.f), n_cmd0 = n_a, n_cmd1 = n_a;
    float n_c = 0.0f;
    if (j_first < np) {
      n_a = ld_stream(g.pa + static_cast<size_t>(j_first) * g.row);
      n_b = ld_stream(g.pb + static_cast<size_t>(j_first) * g.row);
      n_c = ld_stream(g.pc + static_cast<size_t>(j_first) * g.rowc);
      ld_nc_256(act + j_first, n_cmd0, n_cmd1);
    }
    constexpr int kAhead = LPM == 1 ? S2D_FG_AHEAD : 0;  // rows the L2 is asked for ahead of the register prefetch
#pragma unroll
    for (int a = 1; a <= kAhead; ++a) {
      if (a < np) {
        prefetch_l2(g.pa + a * g.row);
        prefetch_l2(g.pb + a * g.row);
        prefetch_l2(g.pc + a * g.rowc);
      }
    }

    // `on`: the sub-lane has a player in this slot (with LPM > 1 the sub-lanes own 8 / 6 / 4 / 4 or 12 / 10 players and all
    // walk the longest list, so that the warp votes of fg_commands stay whole); j_next: the player it handles after this one
    auto one_player = [&](const int j, float4 a, const bool on, const int j_next) {
      if (LPM == 2 && obs_row) __syncwarp();  // (the observation staging columns are read across the two sub-lanes)
      fg_point_at_type(sp, P, g, on ? j : 0);
      const float4 pa = n_a, b = n_b;
      const float cap = n_c;
      float4* const wpa = g.pa + static_cast<size_t>(j) * g.row;
      float4* const wpb = g.pb + static_cast<size_t>(j) * g.row;
      float* const wpc = g.pc + static_cast<size_t>(j) * g.rowc;
      if (j_next < np) {
        n_a = ld_stream(g.pa + static_cast<size_t>(j_next) * g.row);
        n_b = ld_stream(g.pb + static_cast<size_t>(j_next) * g.row);
        n_c = ld_stream(g.pc + static_cast<size_t>(j_next) * g.rowc);
      }
      if (kAhead > 0 && j + 1 + kAhead < np) {
        prefetch_l2(wpa + (1 + kAhead) * g.row);
        prefetch_l2(wpb + (1 + kAhead) * g.row);
        prefetch_l2(wpc + (1 + kAhead) * g.rowc);
      }
      if constexpr (SCRIPT) {  // a scripted player's row of the action buffer is replaced by the script's command
        if (on && ((P.scripted_mask >> j) & 1u))
          a = fg_script_command(sp, m, pa, b.x, j, pps, j == (j < pps ? chaser_l : chaser_r), ban_in);
      }
      if (!on) a.x = static_cast<float>(S2D_CMD_NONE);
      const bool left = j < pps;
      const int my_side = left ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
      Episode p;
      p.px = pa.x; p.py = pa.y; p.vx = pa.z; p.vy = pa.w;
      p.body = b.x; p.stamina = b.y; p.effort = b.z; p.recovery = b.w;
      p.capacity = cap;
      p.bx = m.bx; p.by = m.by; p.bvx = m.bvx; p.bvy = m.bvy;
      if (on) S.oldx[j][t] = p.px;
      float ax = 0.0f, ay = 0.0f, kax = 0.0f, kay = 0.0f;
      // tackle / catch and their after-effects (Player::tackle, Player::goalieCatch; spec: include/soccer2d.h).  One
      // vote skips all of it while nobody in the warp tackles, catches, lies on the ground or waits for its next catch.
      float4 cmd = a;
      bool tackled = false;
      float tkx = 0.0f, tky = 0.0f;  // a tackle's push on the ball
      const int raw = static_cast<int>(a.x);
      if (__any_sync(full, on && ((m.tk0 | m.tk1 | m.tk2 | m.ban) != 0u || raw == S2D_CMD_TACKLE || raw == S2D_CMD_CATCH)) && on) {
        const int word = j >> 3, shift = (j & 7) * 4;
        const uint32_t w = word == 0 ? m.tk0 : word == 1 ? m.tk1 : m.tk2;
        uint32_t count = (w >> shift) & 15u;
        const bool keeper = j == 0 || j == pps;
        const int ban_shift = j == 0 ? 0 : 4;
        uint32_t ban = keeper ? (m.ban >> ban_shift) & 15u : 0u;
        if (!stopped && ban > 0u) ban -= 1u;
        if (!stopped && count > 0u) {  // on the ground after a tackle: whatever it was told, it does nothing
          count -= 1u;
          cmd.x = static_cast<float>(S2D_CMD_NONE);
        } else if (raw == S2D_CMD_TACKLE) {
          cmd.x = static_cast<float>(S2D_CMD_NONE);
          if (!stopped) {
            float sn, cs;
            sincos_deg(p.body, sn, cs);
            const float dx = p.bx - p.px, dy = p.by - p.py;
            const float rx = dx * cs + dy * sn, ry = dy * cs - dx * sn;  // the ball in the body frame, x ahead
            count = kFgTackleCycles;
            bool ok = false;
            if (rx > 0.0f) {
              const float fx = rx * static_cast<float>(1.0 / 2.0), fy = fabsf(ry) * static_cast<float>(1.0 / 1.25);
              const float fx2 = fx * fx, fy2 = fy * fy;
              const float fail = (fx2 * fx2) * fx2 + (fy2 * fy2) * fy2;
              if (fail < 1.0f)
                ok = u32_to_unit(philox4x32_10(P.seed, gid, m.cycle, RNG_TACKLE, static_cast<uint32_t>(j)).x) < 1.0f - fail;
            }
            if (ok && !dead_at_start) {
              const float d = clampf(-180.0f, a.y, 180.0f);
              float eff = 100.0f * (1.0f - fabsf(d) * static_cast<float>(1.0 / 180.0)) * 0.027f;
              eff = eff * (1.0f - 0.5f * fabsf(atan2_deg(ry, rx)) * static_cast<float>(1.0 / 180.0));
              sincos_deg(p.body + d, sn, cs);
              tkx = eff * cs;
              tky = eff * sn;
              tackled = true;
            }
          }
        } else if (raw == S2D_CMD_CATCH) {
          cmd.x = static_cast<float>(S2D_CMD_NONE);
          if (!stopped && !dead_at_start && keeper && ban == 0u) {
            const float d = clampf(-180.0f, a.y, 180.0f);
            float sn, cs;
            sincos_deg(p.body + d, sn, cs);
            const float dx = p.bx - p.px, dy = p.by - p.py;
            const float rx = dx * cs + dy * sn, ry = dy * cs - dx * sn;
            const bool in_rect = rx >= 0.0f && rx <= kFgCatchLength && fabsf(ry) <= kFgCatchWidth * static_cast<float>(1.0 / 2.0);
            const float edge = sp.pitch_half_length() - kFgPenaltyLength;
            const bool in_area = (j == 0 ? p.bx <= -edge : p.bx >= edge) && fabsf(p.by) <= kFgPenaltyHalfWidth;
            if (in_rect && in_area) {
              caught = j;
              ban = kFgCatchBan;
            }
          }
        }
        const uint32_t nw = (w & ~(15u << shift)) | (count << shift);
        m.tk0 = word == 0 ? nw : m.tk0;
        m.tk1 = word == 1 ? nw : m.tk1;
        m.tk2 = word == 2 ? nw : m.tk2;
        if (keeper) m.ban = (m.ban & ~(15u << ban_shift)) | (ban << ban_shift);
      }
      bool kicked = fg_commands(p, cmd, P.goto_dist_thr, sp, nz, full, j, left, (!dead_at_start || my_side == m.side) && !stopped,
                                !stopped, ax, ay, kax, kay);
      if (tackled) {  // counts as a kick: last touch, kicked flag, offside
        kicked = true;
        kax = tkx;
        kay = tky;
      }
      if (stopped) {
        p.vx = 0.0f;
        p.vy = 0.0f;
      }
      if (kicked && on) {
        S.kicked[tid] |= 1u << j;
        kx[j] = kax;
        ky[j] = kay;
      }
      move_object<SP::kNoise>(p.px, p.py, p.vx, p.vy, ax, ay, sp.player_accel_max(), sp.player_accel_max2(),
                              sp.player_speed_max(), sp.player_speed_max2(), sp.player_decay(), sp.player_rand(), &nz,
                              static_cast<uint32_t>(j));
      if (!on) return;
      const float stepx = p.px - pa.x, stepy = p.py - pa.y;
      moved2 = fmaxf(moved2, stepx * stepx + stepy * stepy);
      if (!stopped) update_stamina(p, sp);
      S.xy[j][t] = make_float2(p.px, p.py);
      st_stream(wpa, make_float4(p.px, p.py, p.vx, p.vy));
      st_stream(wpb, make_float4(p.body, p.stamina, p.effort, p.recovery));
      st_stream(wpc, p.capacity);
      if (obs_row) {  // (uniform) four players = 20 floats = five float4 of the row, starting at float4 1 + 5 (j / 4)
        const int q = j & 3, grp = j >> 2;
        float(*stg)[kFgBlock] = S.obs + 5 * q;
        stg[0][tid] = p.px * static_cast<float>(1.0 / 52.5);
        stg[1][tid] = p.py * static_cast<float>(1.0 / 34.0);
        stg[2][tid] = p.vx;
        stg[3][tid] = p.vy;
        stg[4][tid] = p.body * static_cast<float>(1.0 / 180.0);
        auto f4 = [&](int r) { return make_float4(S.obs[r][tid], S.obs[r + 1][tid], S.obs[r + 2][tid], S.obs[r + 3][tid]); };
        if (LPM <= 2) {
          // Whole 32-byte sectors only (a half-written sector costs the L2 about as much as two whole ones: measured,
          // profiles/micro/fg_layout.cu).  A group's five float4 start at an odd float4 of the row in the even groups and
          // at an even one in the odd groups, so an odd group leaves its last float4 (rows 16-19) behind for the first
          // float4 of the next one.  The first float4 of group 0 shares its sector with the ball and the last two floats
          // of player 21 share theirs with the referee's values: those two sectors are written at the end of the launch.
          // With two lanes per match the even groups are the first sub-lane's and the odd ones the second's: the float4
          // left behind sits in the neighbour's column (written a whole group of players ago; the __syncwarp at the top
          // of every player slot orders it).
          const int left_behind = LPM == 1 ? tid : tid | 1;
          if (valid) {
            float4* o = reinterpret_cast<float4*>(obs_row) + 5 * grp;  // the group's values are o[1] .. o[5]
            if ((grp & 1) == 0) {
              if (q == 0 && grp > 0)
                st_stream_256(o, make_float4(S.obs[16][left_behind], S.obs[17][left_behind], S.obs[18][left_behind], S.obs[19][left_behind]), f4(0));
              if (q == 3) {
                st_stream_256(o + 2, f4(4), f4(8));
                st_stream_256(o + 4, f4(12), f4(16));
              }
            } else if (q == 3) {
              st_stream_256(o + 1, f4(0), f4(4));
              st_stream_256(o + 3, f4(8), f4(12));
            } else if (j == np - 1) {  // players 20 and 21: floats 104..111
              st_stream_256(o + 1, f4(0), f4(4));
            }
          }
        } else if (valid && (q == 3 || j == np - 1)) {
          float4* o = reinterpret_cast<float4*>(obs_row) + 1 + 5 * grp;
          st_stream(o, f4(0));
          st_stream(o + 1, f4(4));
          if (q == 3) {
            st_stream(o + 2, f4(8));
            st_stream(o + 3, f4(12));
            st_stream(o + 4, f4(16));
          }
        }
      }
    };
#pragma unroll 1
    for (int it = 0; it < iters; it += 2) {
      const int j = player_at(it), j_after = it + 2 < iters ? player_at(it + 2) : np;  // (j is even)
      const bool on = j < np;
      const float4 c0 = n_cmd0, c1 = n_cmd1;
      if (j_after < np) ld_nc_256(act + j_after, n_cmd0, n_cmd1);
      one_player(j, c0, on, on ? j + 1 : np);
      one_player(j + 1, c1, on, j_after);
    }
  }
  uint32_t kick_mask = S.kicked[tid];
  if (LPM > 1) {  // what the sub-lanes of a match found, merged: every one of them goes on with the whole picture
    __syncwarp();
    uint32_t d0 = m.tk0 ^ tk0_in, d1 = m.tk1 ^ tk1_in, d2 = m.tk2 ^ tk2_in, db = m.ban ^ ban_in;  // (disjoint nibbles)
#pragma unroll
    for (int sft = 1; sft < LPM; sft <<= 1) {
      kick_mask |= __shfl_xor_sync(full, kick_mask, sft);
      moved2 = fmaxf(moved2, __shfl_xor_sync(full, moved2, sft));
      caught = max(caught, __shfl_xor_sync(full, caught, sft));
      d0 |= __shfl_xor_sync(full, d0, sft);
      d1 |= __shfl_xor_sync(full, d1, sft);
      d2 |= __shfl_xor_sync(full, d2, sft);
      db |= __shfl_xor_sync(full, db, sft);
    }
    m.tk0 = tk0_in ^ d0;
    m.tk1 = tk1_in ^ d1;
    m.tk2 = tk2_in ^ d2;
    m.ban = ban_in ^ db;
    if (kick_mask) {  // the pushes of the kickers the other sub-lanes handled (cold; the lanes of a match are converged)
      const unsigned group = ((1u << LPM) - 1u) << (lane & ~(LPM - 1));
#pragma unroll 1
      for (uint32_t rest = kick_mask; rest; rest &= rest - 1u) {
        const int j = __ffs(rest) - 1, owner = (j >> 2) & (LPM - 1);
        const float vx = h == owner ? kx[j] : 0.0f, vy = h == owner ? ky[j] : 0.0f;
        kx[j] = __shfl_sync(group, vx, owner, LPM);
        ky[j] = __shfl_sync(group, vy, owner, LPM);
      }
    }
  }

  // ---- the kicks: acceleration of the ball, last touch, a dead ball comes alive, offside marks ----
  float bax = 0.0f, bay = 0.0f;
  if (kick_mask) {  // without a kicker both sums are exactly zero
    bax = tree_sum32(kx, kick_mask);
    bay = tree_sum32(ky, kick_mask);
  }
  const bool kick_l = (kick_mask & left_set) != 0, kick_r = (kick_mask & ~left_set) != 0;
  if (kick_l != kick_r) m.last_touch = kick_l ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
  const int mode_at_kick = m.mode;
  if (dead && ((m.side == S2D_SIDE_LEFT && kick_l) || (m.side == S2D_SIDE_RIGHT && kick_r))) {
    m.mode = S2D_PM_PLAY_ON;
    dead = false;
  }
  kicked_mask = kick_mask;
  if (caught >= 0) {  // the goalkeeper holds the ball: free kick for its side; what the others did to the ball is void
    m.mode = S2D_PM_FREE_KICK;
    m.side = caught < pps ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
    m.timer = 0;
    m.last_touch = m.side;
    dead = true;
  }
  if (kick_mask && !dead) {
    m.offside = 0u;  // whoever kicks: the old marks are void
    const bool exempt = mode_at_kick == S2D_PM_KICK_IN || mode_at_kick == S2D_PM_CORNER_KICK || mode_at_kick == S2D_PM_GOAL_KICK;
    if (kick_l != kick_r && !exempt) m.offside = fg_offside_marks(S, t, np, kick_l, kick_mask, m.bx);
  }

  // ---- the ball moves ----
  const float pbx = m.bx, pby = m.by;
  if (!dead) {
    move_object<SP::kNoise>(m.bx, m.by, m.bvx, m.bvy, bax, bay, sp.ball_accel_max(), sp.ball_accel_max2(),
                            sp.ball_speed_max(), sp.ball_speed_max2(), sp.ball_decay(), sp.ball_rand(), &nz, kBallAgent);
  } else {
    m.bvx = 0.0f;
    m.bvy = 0.0f;
  }
  if (caught >= 0) {  // in the keeper's hands
    const float2 k = S.xy[caught][t];
    m.bx = k.x;
    m.by = k.y;
  }

  // ---- second walk over the players, now that ball and play mode are settled: a dead ball keeps the side that does
  // ---- not take the kick 9.15 m away; a live ball is tested against every player ----
  const float r = sp.player_size() + sp.ball_size();
  const float r2 = sp.player_size() + sp.player_size();
  const bool clearing = dead && m.mode != S2D_PM_TIME_OVER && m.mode != S2D_PM_AFTER_GOAL;
  const bool own_half = m.mode == S2D_PM_KICK_OFF;  // Referee::placePlayersInTheirField
  uint32_t ball_mask = 0;  // players the live ball overlaps
  float cleared2 = 0.0f;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
    const int j = player_at(it);
    if (j >= np) continue;
    float2 xy = S.xy[j][t];
    const bool left = j < pps;
    const int my_side = left ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
    bool placed = false;
    float sx = 0.0f, sy = 0.0f;  // how far the referee moved the player
    if (own_half && (left ? xy.x > 0.0f : xy.x < 0.0f)) {
      const float nx = left ? -sp.player_size() : sp.player_size();
      sx = nx - xy.x;
      xy.x = nx;
      placed = true;
    }
    const float cx = xy.x - m.bx, cy = xy.y - m.by;
    const float c2 = cx * cx + cy * cy;
    if (clearing && my_side != m.side && c2 < kFgFreeKickDist * kFgFreeKickDist) {
      const float c = sqrtf(c2);
      float ux = left ? -1.0f : 1.0f, uy = 0.0f;
      if (c >= 1.0e-6f) {
        ux = cx / c;
        uy = cy / c;
      }
      const float nx = m.bx + ux * kFgFreeKickDist, ny = m.by + uy * kFgFreeKickDist;
      sx += nx - xy.x;
      sy += ny - xy.y;
      xy = make_float2(nx, ny);
      placed = true;
    }
    if (placed) {
      cleared2 = fmaxf(cleared2, sx * sx + sy * sy);
      S.xy[j][t] = xy;
      g.pa[static_cast<size_t>(j) * g.row] = make_float4(xy.x, xy.y, 0.0f, 0.0f);
      if (obs_row && valid) {
        float* o = obs_row + 4 + 5 * j;
        o[0] = xy.x * static_cast<float>(1.0 / 52.5);
        o[1] = xy.y * static_cast<float>(1.0 / 34.0);
        o[2] = 0.0f;
        o[3] = 0.0f;
      }
    }
    if (!dead && c2 < r * r) ball_mask |= 1u << j;
  }
  if (LPM > 1) {
#pragma unroll
    for (int sft = 1; sft < LPM; sft <<= 1) {
      ball_mask |= __shfl_xor_sync(full, ball_mask, sft);
      cleared2 = fmaxf(cleared2, __shfl_xor_sync(full, cleared2, sft));
    }
    __syncwarp();  // the referee's placements are in shared memory for the other sub-lanes
  }

  // ---- collisions ----
  // `sep` (kept in the match state) is a LOWER BOUND on the smallest distance between two players.  Every cycle it
  // shrinks by twice the farthest any player moved; only when it drops below the collision distance is the exact
  // minimum measured (all pairs, from shared memory) - and then for every match of the warp, since the lanes walk the
  // pairs together anyway.  Without a close pair and without a ball overlap the relaxation rounds - which would change
  // nothing - are skipped, so the results do not depend on this shortcut.
  {
    float moved, cleared;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(moved) : "f"(moved2));
    asm("sqrt.approx.f32 %0, %1;" : "=f"(cleared) : "f"(cleared2));
    m.sep -= 2.002f * (moved + cleared) + 1.0e-6f;
  }
  bool pairs_close = false;
  if (__any_sync(full, m.sep < r2)) {
    // (the smallest squared distance, with sm_100's packed fp32 instructions: {dx, dy} and their squares take one issue
    // slot each.  The value only feeds the bound and the conservative test below - the resolver makes the exact tests in
    // the fp32 spec's own arithmetic - so it does not matter that the assembler may fuse packed operations.)
    float m2 = 3.0e38f;
#pragma unroll 1
    for (int i = h; i + 1 < np; i += LPM) {
      const unsigned long long pi = *reinterpret_cast<const unsigned long long*>(&S.xy[i][t]);
#pragma unroll 4
      for (int j = i + 1; j < np; ++j) {
        const unsigned long long pj = *reinterpret_cast<const unsigned long long*>(&S.xy[j][t]);
        unsigned long long d;
        float sx, sy;
        asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pi), "l"(pj));
        asm("mul.rn.f32x2 %0, %0, %0;" : "+l"(d));
        asm("mov.b64 {%0, %1}, %2;" : "=f"(sx), "=f"(sy) : "l"(d));
        m2 = fminf(m2, sx + sy);
      }
    }
#pragma unroll
    for (int sft = 1; sft < LPM; sft <<= 1) m2 = fminf(m2, __shfl_xor_sync(full, m2, sft));
    pairs_close = m2 < r2 * r2 * 1.000001f;  // (a last-bit difference from the resolver's own sums must not hide a pair)
    m.sep = sqrtf(m2) * 0.999f;
  }
  collided_mask = 0;
  ball_collided = false;
  uint32_t touch = 0;
  {
    constexpr unsigned kFirstSubLanes = LPM == 1 ? 0xffffffffu : LPM == 2 ? 0x55555555u : 0x11111111u;
    const unsigned need = __ballot_sync(full, (pairs_close || ball_mask != 0u) && !stopped) & kFirstSubLanes;  // (AfterGoal: nothing moves)
    if (need) {
      fg_resolve_collisions(S, t, tid, lane, LPM, g, m.bx, m.by, m.bvx, m.bvy, np, need, dead, r, r2, sp.collision_model(),
                            obs_row ? P.obs : nullptr, static_cast<int64_t>(blockIdx.x) * (kFgBlock / LPM) + t, valid);
      const int first = lane & ~(LPM - 1);  // the sub-lane that stood for the match
      if ((need >> first) & 1u) {
        const int col = tid & ~(LPM - 1);
        m.bx = S.obs[0][col];
        m.by = S.obs[1][col];
        ball_collided = __float_as_uint(S.obs[2][col]) != 0u;
        collided_mask = __float_as_uint(S.obs[3][col]);
        touch = __float_as_uint(S.obs[4][col]);
        if (ball_collided) {
          m.bvx *= -0.1f;
          m.bvy *= -0.1f;
        }
        m.sep = 0.0f;  // players were pushed around: measure again next cycle
      }
    }
  }
  {
    const bool hit_l = (touch & left_set) != 0, hit_r = (touch & ~left_set) != 0;
    if (hit_l != hit_r) m.last_touch = hit_l ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
    if (m.offside && (touch & ((m.offside & left_set) ? ~left_set : left_set))) m.offside = 0u;  // the defenders got the ball
  }

  // ---- referee ----
  int goal_l = 0, goal_r = 0;
  const float bx_phys = m.bx;
  bool kick_off = false;
  const float line = sp.pitch_half_length() + sp.ball_size();
  const float side_line = sp.pitch_half_width() + sp.ball_size();
  bool offside_called = false;
  if (!dead && m.offside) {  // a marked player within 2.5 m of the ball takes part in play: free kick where it stands
    uint32_t part = 0;
#pragma unroll 1
    for (uint32_t rest = m.offside; rest; rest &= rest - 1u) {
      const int j = __ffs(rest) - 1;
      const float2 xy = S.xy[j][t];
      const float ox = xy.x - m.bx, oy = xy.y - m.by;
      if (ox * ox + oy * oy < kFgOffsideArea * kFgOffsideArea) part |= 1u << j;
    }
    if (part) {
      const int who = __ffs(part) - 1;
      const float2 f = S.xy[who][t];
      m.mode = S2D_PM_FREE_KICK;
      m.side = who < pps ? S2D_SIDE_RIGHT : S2D_SIDE_LEFT;
      m.timer = 0;
      m.bx = clampf(-sp.pitch_half_length(), f.x, sp.pitch_half_length());
      m.by = clampf(-sp.pitch_half_width(), f.y, sp.pitch_half_width());
      m.bvx = 0.0f;
      m.bvy = 0.0f;
      offside_called = true;
    }
  }
  if (offside_called) {
    // (the ball was re-placed inside the pitch: nothing else to rule on this cycle)
  } else if (!dead && !(fabsf(m.bx) > line || fabsf(m.by) > side_line)) {
    // ball inside the field: every ruling below needs it beyond a line, so there is nothing to decide (the common case)
  } else if (!dead) {
    const float bx = m.bx, by = m.by;
    const float post = sp.goal_width() * 0.5f + sp.goal_post_radius();
    if (bx > line && !(pbx > line)) {
      const float yc = pby + (by - pby) * ((line - pbx) / (bx - pbx));
      goal_l = fabsf(yc) <= post;
    } else if (bx < -line && !(pbx < -line)) {
      const float yc = pby + (by - pby) * ((-line - pbx) / (bx - pbx));
      goal_r = fabsf(yc) <= post;
    }
    if (goal_l || goal_r) {
      if (goal_l) m.score_l += 1;
      else m.score_r += 1;
      m.mode = S2D_PM_AFTER_GOAL;  // AfterGoal_ + the scoring side: the clock stops for kFgAfterGoalWait cycles
      m.side = goal_l ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
      m.timer = 0;
      m.last_touch = S2D_SIDE_UNKNOWN;
      m.bvx = 0.0f;
      m.bvy = 0.0f;
    } else if (fabsf(bx) > line) {  // over a goal line outside the goal: corner kick or goal kick
      const int defending = bx > 0.0f ? S2D_SIDE_RIGHT : S2D_SIDE_LEFT;
      const float sx = bx > 0.0f ? 1.0f : -1.0f, sy = by > 0.0f ? 1.0f : -1.0f;
      if (m.last_touch == defending) {
        m.mode = S2D_PM_CORNER_KICK;
        m.side = defending == S2D_SIDE_LEFT ? S2D_SIDE_RIGHT : S2D_SIDE_LEFT;
        m.bx = sx * (sp.pitch_half_length() - 1.0f);
        m.by = sy * (sp.pitch_half_width() - 1.0f);
      } else {
        m.mode = S2D_PM_GOAL_KICK;
        m.side = defending;
        m.bx = sx * (sp.pitch_half_length() - 5.5f);
        m.by = sy * 9.16f;
      }
      m.bvx = 0.0f;
      m.bvy = 0.0f;
      m.timer = 0;
    } else if (fabsf(by) > side_line) {
      m.mode = S2D_PM_KICK_IN;
      m.side = m.last_touch == S2D_SIDE_LEFT ? S2D_SIDE_RIGHT : S2D_SIDE_LEFT;
      m.bx = clampf(-sp.pitch_half_length(), bx, sp.pitch_half_length());
      m.by = by > 0.0f ? sp.pitch_half_width() : -sp.pitch_half_width();
      m.bvx = 0.0f;
      m.bvy = 0.0f;
      m.timer = 0;
    }
  } else {
    m.timer += 1;
    if (m.mode == S2D_PM_AFTER_GOAL) {
      if (m.timer >= kFgAfterGoalWait) {  // kick-off for the side that conceded
        kick_off = true;
        m.mode = S2D_PM_KICK_OFF;
        m.side = m.side == S2D_SIDE_LEFT ? S2D_SIDE_RIGHT : S2D_SIDE_LEFT;
        m.timer = 0;
      }
    } else if (m.timer >= kFgDropBallTime) {
      m.mode = S2D_PM_PLAY_ON;
      m.timer = 0;
    }
  }
  if (kick_off) {
    m.sep = 0.0f;
    obs_dirty = true;
    fg_kick_off_formation(S, t, g, P, gid, m.episode, np, m.score_l + m.score_r);
    m.bx = m.by = m.bvx = m.bvy = 0.0f;
  }
  if (m.mode != S2D_PM_PLAY_ON) m.offside = 0u;  // marks live only while play goes on
  m.cycle += stopped ? 0u : 1u;
  reward = static_cast<float>(goal_l - goal_r) * 10.0f + (bx_phys - pbx) * 0.01f;
  const bool done = m.step_number >= 2 * half_time;
  result = !done ? S2D_RESULT_NONE : m.score_l > m.score_r ? 1 : m.score_r > m.score_l ? 2 : 3;
  if (done) m.mode = S2D_PM_TIME_OVER;
  if (LPM > 1) __syncwarp();  // (kick-off placements: shared memory and planes, for the other sub-lanes' next cycle)
  return done;
}

// match-level state: four coalesced 16-byte loads / stores per lane
__device__ __forceinline__ void fg_load(const KernelParams& P, const FgLayout& L, int64_t env, Match& m) {
  const char* base = static_cast<const char*>(P.state);
  const float4 ball = ld_stream(reinterpret_cast<const float4*>(base + L.eb()) + env);
  const float4 ef = ld_stream(reinterpret_cast<const float4*>(base + L.ef()) + env);
  const uint4 ei = ld_stream(reinterpret_cast<const uint4*>(base + L.ei()) + env);
  const uint4 ej = ld_stream(reinterpret_cast<const uint4*>(base + L.ej()) + env);
  m.bx = ball.x; m.by = ball.y; m.bvx = ball.z; m.bvy = ball.w;
  m.ep_return = ef.x;
  m.sep = ef.y;
  m.offside = __float_as_uint(ef.z);
  m.step_number = static_cast<int>(ei.x); m.cycle = ei.y; m.episode = ei.z;
  m.mode = ei.w & 0xff; m.side = (ei.w >> 8) & 3; m.last_touch = (ei.w >> 10) & 3; m.timer = (ei.w >> 12) & 0xff;
  m.done_flag = (ei.w >> 21) & 1;
  m.score_l = static_cast<int>(ej.x); m.score_r = static_cast<int>(ej.y);
  const uint4 ek = ld_stream(reinterpret_cast<const uint4*>(base + L.ek()) + env);
  m.tk0 = ek.x; m.tk1 = ek.y; m.tk2 = ek.z; m.ban = ek.w;
}

__device__ __forceinline__ void fg_store(const KernelParams& P, const FgLayout& L, int64_t env, const Match& m,
                                         uint32_t collided_mask, uint32_t kicked_mask, bool ball_collided) {
  char* base = static_cast<char*>(P.state);
  st_stream(reinterpret_cast<float4*>(base + L.eb()) + env, make_float4(m.bx, m.by, m.bvx, m.bvy));
  st_stream(reinterpret_cast<float4*>(base + L.ef()) + env, make_float4(m.ep_return, m.sep, __uint_as_float(m.offside), 0.0f));
  const uint32_t packed = static_cast<uint32_t>(m.mode) | (static_cast<uint32_t>(m.side) << 8) |
                          (static_cast<uint32_t>(m.last_touch) << 10) | (static_cast<uint32_t>(m.timer) << 12) |
                          (ball_collided ? 1u << 20 : 0u) | (m.done_flag ? 1u << 21 : 0u);
  st_stream(reinterpret_cast<uint4*>(base + L.ei()) + env, make_uint4(static_cast<uint32_t>(m.step_number), m.cycle, m.episode, packed));
  st_stream(reinterpret_cast<uint4*>(base + L.ej()) + env,
            make_uint4(static_cast<uint32_t>(m.score_l), static_cast<uint32_t>(m.score_r), collided_mask, kicked_mask));
  st_stream(reinterpret_cast<uint4*>(base + L.ek()) + env, make_uint4(m.tk0, m.tk1, m.tk2, m.ban));
}

// heterogeneous players: the block copies the type table to shared memory; the player loops point sp.row at the row of
// the player they are at
template <class SP>
__device__ __forceinline__ void fg_bind_player_types(SP& sp, const KernelParams& P) {
  if constexpr (SP::kHetero) {
    __shared__ float s_types[S2D_MAX_PLAYER_TYPES * PT_ROW];
    for (int k = threadIdx.x; k < S2D_MAX_PLAYER_TYPES * PT_ROW; k += blockDim.x) s_types[k] = __ldg(P.player_types + k);
    __syncthreads();
    sp.table = s_types;
    sp.row = s_types;
  }
}

// K lockstep cycles of every match; actions float4 [N][K][np].  NP = 22 is the 11 v 11 instantiation (player count and
// team masks become immediates); NP = 0 takes the player count at run time.
template <int VAR, int NP, int LPM>
__global__ void __launch_bounds__(kFgBlock, S2D_FG_MIN_BLOCKS) fullgame_step_kernel(const __grid_constant__ KernelParams P, const int K,
                                                                 const int np_runtime, const int half_time) {
  static_assert(LPM == 1 || LPM == 2 || LPM == 4, "lanes per match");
  const int np = NP ? NP : np_runtime;
  constexpr bool SCRIPT = (VAR & kVarScripted) != 0;
  using SP = typename VariantSP<VAR & ~kVarScripted>::type;
  SP sp(P.cc);
  __shared__ FgShared S;
  fg_bind_player_types(sp, P);
  const int tid = threadIdx.x;
  const int t = tid / LPM;  // the match's column in the block's shared memory; the block holds kFgBlock / LPM matches
  // Every thread owns (with LPM > 1: shares) a column of the state (rows are padded to 64), so warps are whole: the
  // columns past num_envs are scratch matches - they run the commands of the last real match and report nothing.
  const int64_t env = static_cast<int64_t>(blockIdx.x) * (kFgBlock / LPM) + t;
  const bool valid = env < P.num_envs;
  const bool writer = valid && (tid & (LPM - 1)) == 0;  // the sub-lane that reports the match
  const int64_t env_in = valid ? env : P.num_envs - 1;
  const FgLayout L{P.num_envs, np};
  if (env >= static_cast<int64_t>(L.nr())) return;  // (whole warps: nr is a multiple of 64)
  const FgPlanes g(P, L, env);
  const uint64_t gid = static_cast<uint64_t>(P.env_id_offset + env);

  Match m;
  fg_load(P, L, env, m);
  if constexpr (SCRIPT) {  // the script's chaser pre-pass reads every player's position from shared memory
#pragma unroll 1
    for (int j = tid & (LPM - 1); j < np; j += LPM) {
      const float4 a = ld_stream(g.pa + static_cast<size_t>(j) * g.row);
      S.xy[j][t] = make_float2(a.x, a.y);
    }
    if (LPM > 1) __syncwarp();
  }
  uint32_t collided_mask = 0, kicked_mask = 0;
  bool ball_collided = false, obs_dirty = false;
  float reward_sum = 0.0f;
  uint32_t any_done = 0, last_result = 0;
  const float4* act = static_cast<const float4*>(P.actions) + (env_in * K) * np;
  float* const my_obs = P.obs + env_in * kFgObsDim;
#pragma unroll 1
  for (int k = K; k > 0; --k, act += np) {
    float rw;
    int rs;
    // in the last cycle of an 11 v 11 launch the player loop writes the observation row itself
    float* const obs_row = (NP == kFgMaxPlayers && k == 1) ? my_obs : nullptr;
    const bool done = fg_cycle<LPM, SCRIPT>(S, t, tid, g, m, P, sp, gid, np, half_time, act, obs_row, valid, obs_dirty, rw, rs, collided_mask,
                                    kicked_mask, ball_collided);
    reward_sum += rw;
    m.ep_return += rw;
    if (done) {
      any_done = 1;
      last_result = static_cast<uint32_t>(rs);
      if (!m.done_flag && writer) {  // (a finished match stepped on with auto_reset off is tallied once)
        unsigned long long* slot = P.stats + static_cast<size_t>(env % kStatSlots) * kStatWords;
        atomicAdd(slot + ST_EPISODES, 1ull);
        atomicAdd(slot + (rs == 1 ? ST_GOALS : rs == 2 ? ST_OUTS : ST_TIMEOUTS), 1ull);
        atomicAdd(slot + ST_EP_STEPS, static_cast<unsigned long long>(m.step_number));
        atomicAdd(reinterpret_cast<double*>(slot + ST_RETURN), static_cast<double>(m.ep_return));
      }
      if (P.terminal_obs && writer) fg_write_obs(P.terminal_obs, env, g, m, np, half_time);
      if (P.auto_reset) {
        if (LPM > 1) __syncwarp();  // (the terminal observation reads the planes the reset rewrites)
        Match mc = m;  // (see fg_resolve_collisions' call)
        fg_reset(S, t, g, mc, P, sp, gid, np);
        m = mc;
        collided_mask = kicked_mask = 0;
        ball_collided = false;
        obs_dirty = true;
        if (LPM > 1) __syncwarp();
      } else {
        m.done_flag = true;
      }
    }
  }
  if (!writer) return;
  fg_store(P, L, env, m, collided_mask, kicked_mask, ball_collided);
  if (NP != kFgMaxPlayers || obs_dirty) {
    fg_write_obs(P.obs, env, g, m, np, half_time);  // the whole row from the planes
  } else {
    // the players' part is written, up to the two sectors they share with the ball (floats 0..7) and with the referee's
    // six values (floats 112..119): both are written whole, the players' halves from the planes (as the player loop
    // wrote them, or as the referee / the collisions left them since)
    float4* row = reinterpret_cast<float4*>(my_obs);
    const float4 a0 = ld_stream(g.pa), a21 = ld_stream(g.pa + static_cast<size_t>(kFgMaxPlayers - 1) * g.row);
    const float body21 = ld_stream(reinterpret_cast<const float*>(g.pb + static_cast<size_t>(kFgMaxPlayers - 1) * g.row));
    st_stream_256(row,
                  make_float4(m.bx * static_cast<float>(1.0 / 52.5), m.by * static_cast<float>(1.0 / 34.0),
                              m.bvx * static_cast<float>(1.0 / 3.0), m.bvy * static_cast<float>(1.0 / 3.0)),
                  make_float4(a0.x * static_cast<float>(1.0 / 52.5), a0.y * static_cast<float>(1.0 / 34.0), a0.z, a0.w));
    st_stream_256(row + 28,
                  make_float4(a21.w, body21 * static_cast<float>(1.0 / 180.0), static_cast<float>(m.mode), static_cast<float>(m.side)),
                  make_float4(static_cast<float>(m.score_l), static_cast<float>(m.score_r),
                              static_cast<float>(m.step_number) / static_cast<float>(2 * half_time), 0.0f));
  }
  P.reward[env] = reward_sum;
  P.done[env] = static_cast<uint8_t>(any_done);
  P.result[env] = static_cast<uint8_t>(last_result);
}

// Launches fullgame_step_kernel<var + kVarScripted, np_template, lpm> (s2d_scripted.cu); cudaErrorInvalidValue, and no
// launch, for a combination it does not instantiate.  The scripted variants live in a
// translation unit of their own: sharing one with the kernels without the script changed how ptxas compiled the
// out-of-line functions they have in common, and with them the code of kernels that had not changed.
cudaError_t launch_fullgame_scripted(int var, int np_template, int lpm, int grid, const KernelParams& kp, int k_substeps,
                                     int np, int half_time, cudaStream_t s);

template <bool HETERO>
__global__ void __launch_bounds__(kFgBlock) fullgame_reset_kernel(const __grid_constant__ KernelParams P,
                                                                  const uint8_t* __restrict__ mask, const int np,
                                                                  const int half_time) {
  using SP = typename std::conditional<HETERO, HeteroSP<false>, RuntimeSP>::type;
  SP sp(P.cc);
  __shared__ FgShared S;
  fg_bind_player_types(sp, P);
  const int t = threadIdx.x;
  const int64_t env = static_cast<int64_t>(blockIdx.x) * kFgBlock + t;
  const bool valid = env < P.num_envs;
  if (valid && mask && !mask[env]) return;  // (the scratch columns past num_envs are reset with every call)
  const FgLayout L{P.num_envs, np};
  const FgPlanes g(P, L, env);
  Match m;
  fg_load(P, L, env, m);
  fg_reset(S, t, g, m, P, sp, static_cast<uint64_t>(P.env_id_offset + env), np);
  fg_store(P, L, env, m, 0u, 0u, false);
  if (!valid) return;
  fg_write_obs(P.obs, env, g, m, np, half_time);
  P.reward[env] = 0.0f;
  P.done[env] = 0;
  P.result[env] = 0;
}

#endif  // !S2D_HOST_EMU

}  // namespace s2d
