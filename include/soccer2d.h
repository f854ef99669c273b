/*
 * soccer2d.h - C ABI of libsoccer2d.so: the batched lockstep 2D-soccer simulator (sm_100a).
 *
 * This is the drop-in boundary for ONE path of CLSFramework/gym-soccer-2d-env: Soccer2DEnv.step/reset.
 * The reference has no FFI for this path - it crosses three process boundaries instead
 * (multiprocessing.Queue x4, gRPC, rcssserver UDP).  Each entry point below names the reference
 * interface it replaces (paths relative to the reference root):
 *
 *   s2d_create / s2d_destroy   Soccer2DEnv.__init__ / close        soccer_2d_env.py:30-95, :280-299
 *                              (spawn gRPC server + rcssserver + proxy, _wait_for_agents)
 *   s2d_reset                  Soccer2DEnv.reset -> env_reset      soccer_2d_env.py:179-224
 *                              + ReachBallEnv.abs_reset /          sample_environments/reach_ball_env.py:163-197
 *                                trainer_reset_actions (DoMoveBall, DoMovePlayer, DoRecover)
 *   s2d_step / s2d_step_host   Soccer2DEnv.step                    soccer_2d_env.py:226-269
 *                              = action_to_rpc_actions             reach_ball_env.py:53-85
 *                              + GrpcAgent.GetPlayerActions /      server.py:49-67, :85-103
 *                                GetTrainerActions round trip
 *                              + one rcssserver cycle (external)   soccer_2d_env.py:356-383
 *                              + state_to_observation              reach_ball_env.py:87-111
 *                              + check_trainer_observation         reach_ball_env.py:113-161
 *   s2d_bind_pipeline /        the same step, submitted asynchronously from host buffers (copies overlap compute)
 *   s2d_submit_host / s2d_wait_host
 *   s2d_stats                  InfoCollectorCallback tallies       utils/info_collector_callback.py:17-53
 *   s2d_export_env             proto State/WorldModel of one env   idl/service.proto:306-359
 *   S2DServerParam             proto ServerParam / PlayerType      idl/service.proto:1435-1732
 *   S2D_PM_*, S2D_SIDE_*       proto GameModeType / Side           idl/service.proto:267-301, :88-92
 *   S2D_CMD_*                  proto PlayerAction oneof            idl/service.proto:1291-1308
 *
 * Conventions: plain pointers and sizes only; every function returns 0 or a negative S2D_ERR_* code and
 * never throws; s2d_last_error() gives the message.  All device buffers are owned by the caller (PyTorch
 * tensors in the Python host); a handle owns only parameters and launch configuration.  A handle is bound
 * to one CUDA device and is not thread-safe.  All work is enqueued on the caller's stream
 * (`stream` = cudaStream_t as void*); nothing synchronises except s2d_stats and s2d_export_env.
 */
#ifndef SOCCER2D_H_
#define SOCCER2D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S2D_ABI_VERSION 14

/* error codes */
#define S2D_OK 0
#define S2D_ERR_INVALID (-1)   /* bad argument / config */
#define S2D_ERR_UNBOUND (-2)   /* s2d_bind has not been called or a required buffer is NULL */
#define S2D_ERR_CUDA (-3)      /* CUDA runtime error (message in s2d_last_error) */
#define S2D_ERR_NO_DEVICE (-4) /* no usable CUDA device: there is NO CPU fallback */

/* scenarios */
#define S2D_SCENARIO_REACHBALL 0 /* sample_environments/reach_ball_env.py: 1 player + ball */
#define S2D_SCENARIO_SHOOT 1     /* 1v0 shoot-on-goal: kick model + goal / ball-out detection (spec below) */
#define S2D_SCENARIO_FULLGAME 2  /* 11 v 11: dash/turn/kick, stamina, collisions, play modes */

/* SHOOT scenario (BASELINE configs[2]; not in the reference, which has ReachBall only - this is the spec):
 *   one player (left team) + ball, reset distribution and observation as ReachBall;
 *   goal   = the ball is beyond x = +(pitch_half_length + ball_size) this cycle, was not the cycle before, and the
 *            segment between the two positions meets that line at |y| <= goal_width/2 + goal_post_radius
 *            (rcssserver's referee rule)                                   -> done, result GOAL,    reward +10
 *   out    = otherwise |x| > pitch_half_length + ball_size or |y| > pitch_half_width + ball_size (own goal
 *            included)                                                     -> done, result OUT,     reward -10
 *   else step_number > max_steps                                           -> done, result TIMEOUT, reward -5
 *   shaping every step: 0.2 * (d_player_ball[t-1] - d_player_ball[t]) + (d_ball_goal[t-1] - d_ball_goal[t]),
 *            d_ball_goal measured to the centre of the right goal (pitch_half_length, 0).
 *   Discrete(n): the first n - kick_actions actions are Dash(100, (a*360/n_dash)%360-180) as in ReachBall, the last
 *            kick_actions are Kick(100, (j*360/kick_actions)%360-180). */

/* FULLGAME scenario (BASELINE configs[3]; not in the reference - this is the spec):
 *   players_per_side v players_per_side (1..11); player index p < pps = left team, uniform number p+1; p >= pps = right
 *   team.  Actions: S2D_ACT_COMMAND, one {cmd, a, b, c} per player and cycle.  Every player: dash / turn / kick /
 *   Body_GoToPoint, stamina, player-player and ball-player collisions as in the one-player scenarios.
 *   A match lasts 2 * half_time_cycles cycles, then done with result 1 = left wins, 2 = right wins, 3 = draw.
 *   Reset / kick-off: 4-4-2 formation in the own half, each player jittered by +-2 m (Philox), left faces 0 deg, right
 *   180 deg, ball at the centre, play mode KickOff for the left team (after a goal: for the conceding side, next cycle).
 *   Referee subset (play modes = proto GameModeType, idl/service.proto:267-301):
 *     goal       ball beyond x = +-(pitch_half_length + ball_size) having crossed the line between the posts
 *                (|y| <= goal_width/2 + goal_post_radius at the crossing)      -> score, AfterGoal for the scoring side
 *     after goal (AfterGoal_, proto GameModeType 8) the server's clock stands still for 50 cycles (rcssserver: only
 *                `stoped_cycle` advances, S2DEnvSnapshot.stoped_cycle here): nothing moves or collides, velocities are zero, dash / kick
 *                / tackle / catch have no effect and cost no stamina, turn works, stamina is not updated, `cycle` does not
 *                advance (step_number does: an env step is an env step).  Then: kick-off formation, KickOff for the
 *                conceding side.
 *     kick-off   while the mode is KickOff every player stays in its own half: after the players have moved, one beyond the
 *                half-way line is put back at x = -+player_size on its side, at rest (Referee::placePlayersInTheirField);
 *                the 9.15 m clearance then applies to the side that does not kick off
 *     goal line  crossed elsewhere: last touched by the defending side -> CornerKick for the attackers at
 *                (+-(half_length - 1), +-(half_width - 1)); else GoalKick for the defenders at (+-(half_length - 5.5), +-9.16)
 *     side line  |y| > pitch_half_width + ball_size -> KickIn for the side that did not touch it last, ball on the line
 *     dead ball  (KickOff, KickIn, CornerKick, GoalKick, FreeKick): the ball rests and takes no part in collisions; only the awarded
 *                side's kicks count, the first one resumes PlayOn; after 100 cycles without it play resumes anyway.
 *     last touch = side of the last kicker(s) / of the player(s) the ball collided with (unchanged if both sides did).
 *     clearance  while the ball is dead, after the players have moved, every player of the side that does NOT take the
 *                kick and stands closer than 9.15 m to the ball is placed on that circle (on the line ball -> player; a
 *                player exactly on the ball goes towards its own goal) with velocity zero (Referee::clearPlayersFromBall).
 *     offside    (OffsideRef) when ONE team kicks the ball in PlayOn - not the kick that takes a kick-in, corner kick or
 *                goal kick - its players other than the kickers who are, in their direction of attack, beyond the ball,
 *                the half-way line and the second-last opponent (positions before that cycle's move) are marked; any
 *                kick replaces the marks, the other team touching the ball or a dead ball clears them.  A marked player
 *                closer than 2.5 m (offside_active_area_size) to the ball after the collisions -> FreeKick for the other
 *                team with the ball where that player stands (lowest player index if several), nothing else is ruled
 *                on in that cycle.
 *     tackle     S2D_CMD_TACKLE (Player::tackle, rcssserver defaults as constants: tackle_dist 2.0, tackle_back_dist 0,
 *                tackle_width 1.25, tackle_exponent 6, tackle_cycles 10, tackle_power_rate 0.027, max_tackle_power 100,
 *                max_back_tackle_power 0).  Ball relative to the player in its body frame (x ahead): behind (x <= 0) the
 *                tackle fails; else fail = (x / 2.0)^6 + (|y| / 1.25)^6; with fail < 1 it succeeds when a uniform draw
 *                (counter RNG: seed, global env id, cycle, player) is below 1 - fail.  Success, in PlayOn only: the ball is
 *                pushed like a kick by 100 (1 - |dir| / 180) 0.027 (1 - 0.5 |angle of the ball in the body frame| / 180)
 *                towards body + dir (dir clamped to +-180); it counts as a kick for last touch, kicked flags and offside.
 *                Either way the player can do nothing for the next 10 cycles (its commands are ignored).  The foul flag of
 *                the proto message is ignored (no cards).
 *     catch      S2D_CMD_CATCH, goalkeepers only (player 0 of each team), PlayOn, not within 5 cycles (catch_ban_cycle) of
 *                its last catch: succeeds (catch_probability 1) when the ball is inside the keeper's own penalty area
 *                (|x| >= pitch_half_length - 16.5 on its side, |y| <= 20.16) and inside the catch rectangle - 1.2 long
 *                (catch_area_l), 1.0 wide (catch_area_w), starting at the keeper and pointing to body + dir.  Then: FreeKick
 *                for the keeper's side with the ball in the keeper's hands (at its position, at rest), last touch = its side.
 *     Not modelled: fouls and cards, back tackles, the keeper carrying the ball with `move`, the stretched catch area.
 *     Heterogeneous player types: s2d_set_player_types.
 *   Reward (left team's view) per cycle: 10 * (goals by left - goals by right) + 0.01 * (ball x after physics - before).
 *   Observation: 120 floats = ball {x/52.5, y/34, vx/3, vy/3}, then per player {x/52.5, y/34, vx, vy, body/180}
 *   (absent players zero), then [114] play mode, [115] side awarded, [116] left score, [117] right score,
 *   [118] step_number / (2 * half_time_cycles), [119] 0.
 *   Sums over the players of a match (kick pushes on the ball, collision proposals for the ball) are added as a 32-leaf
 *   xor butterfly ((i, i^16), (i, i^8), ... ; leaf = player index, the others 0.0): part of the fp32 result.
 *   State buffer: s2d_state_bytes(cfg) = Nr * (np * 36 + 80) bytes, Nr = N rounded up to 64; plane-major, match-minor
 *   (layout: DESIGN.md). */

/* FULLGAME scripted players (s2d_set_scripted_players; not in the reference - this is the spec).  One fixed baseline team
 * that runs inside the step kernel, so that a team, or one player, can be trained against it without writing the others.
 * Bit j of the handle's mask set: player j (left team first) plays by the rules below and its row of the action buffer
 * is ignored.  Mask 0 (the default): nothing changes.  The script's command then goes through the cycle exactly as a
 * command from the action buffer would (catch ban, tackle counters, kick-off confinement, dead-ball clearance).
 *   Inputs: the state at the START of the cycle - the ball, the player's own position, velocity, body and catch ban, the
 *   play mode and its side, and the other players' positions only.  No randomness.  fp32 arithmetic as the rest of the cycle.
 *   Notation: sg = +1 for the left team, -1 for the right; own frame (sg x, sg y) (the point reflection of the kick-off
 *   formation); L = pitch_half_length, W = pitch_half_width, P = goal_width / 2 - 1; F_k = the kick-off spot of team slot k
 *   (left-team coordinates, 4-4-2: (-50, 0) (-36, -20) (-36, -7) (-36, 7) (-36, 20) (-20, -24) (-20, -8) (-20, 8)
 *   (-20, 24) (-9, -10) (-9, 10)); b' = (bx', by') = the ball in the own frame; clamp(v, a) = max(-a, min(v, a));
 *   d2 = dx * dx + dy * dy with (dx, dy) = ball - player; "in the penalty area" as for catch (|x| >= L - 16.5 on the own
 *   side, |y| <= 20.16).
 *   Chaser of each side (decided once per cycle, before anybody moves): the side's player with the smallest d2, ties to
 *   the lower index.  The goalkeeper (player 0 / players_per_side) takes part only while the ball is in its own penalty
 *   area, or when it is its side's only player.
 *   Kick target T (own frame): gx = L - bx', gy = -by', g2 = gx * gx + gy * gy.
 *     g2 <= 625 (within 25 m of the goal centre): shoot at the far post as seen from the kicker, T = (L, py' >= 0 ? -P : P)
 *       (py' = the kicker's own-frame y: the ball's own side of the goal flips back and forth while a kick is staged
 *       around the kicker's feet), first speed ball_speed_max;
 *     else dribble: k = 8 / sqrt(g2), T = (bx' + gx * k, by' + gy * k), first speed 1.
 *   Rules for scripted player j of side s, the first that applies:
 *     1. play mode AfterGoal, BeforeKickOff or TimeOver: NONE.
 *     2. j is s's chaser and the mode is PlayOn or a dead ball for s:
 *        a. PlayOn, j is the goalkeeper, its catch ban is 0, the ball is in its penalty area and d2 <= 1.2 * 1.2:
 *           CATCH(norm_deg(atan2(dy, dx) - body)) (degrees, -180..180);
 *        b. else sqrt(d2) <= kickable_area (of j's player type): SMART_KICK(sg T, first speed);
 *        c. else PlayOn: INTERCEPT;
 *        d. else (dead ball for s): GOTO(ball, max_dash_power 100).
 *     3. j is the goalkeeper: GOTO(sg (2.5 - L, clamp(0.3 by', P)), 100).
 *     4. everybody else: GOTO(sg (clamp(F_k.x + 0.6 bx', L - 2.5), clamp(F_k.y + 0.3 by', W - 2)), 60).
 *   It does not pass, tackle, mark, or use stamina wisely; it is a baseline, not helios-base.  Two scripted teams against
 *   each other score little (the two chasers kick the ball into each other: profiles/README.md). */

/* action encodings (reach_ball_env.py:39-47, :53-85) */
#define S2D_ACT_DISCRETE 0   /* uint8  [N][K]      Discrete(n): Dash(100, (a*360/n)%360-180) (+ kicks in SHOOT)  */
#define S2D_ACT_CONTINUOUS 1 /* float  [N][K][1]   Box(-1,1,(1,)): Dash(100, a*180)               (REACHBALL)   */
#define S2D_ACT_TURNING 2    /* float  [N][K][4]   [turn_prob, turn_angle, dash_prob, dash_angle] (REACHBALL)   */
#define S2D_ACT_COMMAND 3    /* float4 [N][K][P]   {cmd, a, b, c} per player: see S2D_CMD_* (proto PlayerAction) */
#define S2D_ACT_PARAMETERIZED 4 /* float [N][K][8] dash / turn / kick with continuous arguments (SHOOT; spec below)  */

/* SHOOT + S2D_ACT_PARAMETERIZED (the HFO parameterized action space without tackle; not in the reference - this is the spec).
 * Row a[0..7]; every component is first clamped: c(x) = max(-1, min(x, 1)) (fminf / fmaxf order: a NaN becomes +1).
 *   a[0], a[1], a[2]  weights of dash, turn, kick: the largest c() selects the command, ties to the lower index.
 *   The row then IS the S2D_ACT_COMMAND row (fp32, one rounding per operation as written):
 *     dash  {DASH, (c(a[3]) + 1) * 50, c(a[4]) * 180, 0}   power 0..100, direction lowered by dash_direction as every dash
 *     turn  {TURN, c(a[5]) * 180, 0, 0}
 *     kick  {KICK, (c(a[6]) + 1) * 50, c(a[7]) * 180, 0}   no effect unless the ball is kickable, as every kick
 *   No randomness: unlike S2D_ACT_TURNING's sampled choice, the same row in the same state gives the same command.
 *   Reset, reward, done, results and the 10-float observation are SHOOT's, unchanged.  32 bytes per env and cycle. */

/* S2D_ACT_COMMAND: cmd stored as a float; arguments as in the proto messages */
#define S2D_CMD_NONE 0 /* no body command this cycle                                  */
#define S2D_CMD_DASH 1 /* a = power, b = relative_direction   (service.proto:380-383) */
#define S2D_CMD_TURN 2 /* a = relative_direction              (service.proto:390-392) */
#define S2D_CMD_KICK 3 /* a = power, b = relative_direction   (service.proto:394-397) */
#define S2D_CMD_GOTO 4 /* a,b = target x,y, c = max_dash_power; distance_threshold = S2DConfig.goto_dist_thr (:684-688) */
/* More of the proxy's body actions, each lowered to ONE turn or kick (librcsc's rules; n = cycles of inertia to look
 * ahead, rounded and clamped to 0..63: an object with velocity v and decay d drifts v (1 - d^n) / (1 - d) in n cycles):
 *   TURN_TO_POINT  face the point as seen from where the player will be after n cycles; the moment is the angle
 *                  times (1 + inertia_moment * speed), clamped - what librcsc sends to cancel the server's inertia
 *   TURN_TO_BALL   the same towards where the ball will be after n cycles
 *   TURN_TO_ANGLE  the same towards an absolute body direction
 *   KICK_ONE_STEP  if the ball is kickable: the kick that gives the ball `first_speed` (<= ball_speed_max) towards the
 *                  target in one cycle - acceleration = wanted velocity - ball velocity, power = |acceleration| / kick
 *                  rate (force mode: clamped to max_power), direction = its angle relative to the body; else nothing
 *   STOP_BALL      KICK_ONE_STEP with a wanted velocity of zero
 *   INTERCEPT      go to where the ball can first be met (simplified librcsc intercept table): for t = 1..30 cycles the
 *                  ball's drift position b_t and the player's own drift position m_t are compared; the first t with
 *                  |b_t - m_t| <= 0.8 kickable_area + (t - 1) player_speed_max (one cycle is kept for turning) gives the
 *                  target b_t, else b_30; then Body_GoToPoint(target, max_dash_power 100) decides turn or dash */
#define S2D_CMD_TURN_TO_POINT 5 /* a,b = target x,y, c = n           Body_TurnToPoint  (:777-780) */
#define S2D_CMD_TURN_TO_BALL 6  /* a = n                              Body_TurnToBall   (:773-775) */
#define S2D_CMD_TURN_TO_ANGLE 7 /* a = angle                          Body_TurnToAngle  (:769-771) */
#define S2D_CMD_KICK_ONE_STEP 8 /* a,b = target x,y, c = first_speed  Body_KickOneStep  (:747-751, force_mode) */
#define S2D_CMD_STOP_BALL 9     /*                                    Body_StopBall     (:753-754) */
#define S2D_CMD_INTERCEPT 10    /*                                    Body_Intercept    (:742-745; save_recovery and face_point ignored) */
/* FULLGAME only (ignored = no command elsewhere): */
#define S2D_CMD_TACKLE 11       /* a = power_or_dir (a direction, deg)  Tackle            (:399-402; foul ignored) */
#define S2D_CMD_CATCH 12        /* a = direction relative to the body   Catch             (:404-406; the proxy aims at the ball) */
/* Body_SmartKick (:690-695): the kick that gives the ball `first_speed` towards the target, planned over more than one
 * cycle when one kick cannot do it.  Stateless, decided anew every cycle:
 *   release  if the acceleration it needs is within what max_power yields at the ball's current place: as KICK_ONE_STEP;
 *   stage    else the ball is kicked to the staging point - on the line from where the player will be next cycle
 *            (position + velocity) to the target, player_size + ball_size + 0.3 kickable_margin in front of it: the
 *            acceleration asked for is staging point - (ball position + ball velocity), the power is clamped to
 *            max_power.  If that acceleration is below 0.05 the ball IS staged: release with whatever max_power gives.
 *            From the staging point (close, in front when the player faces the target) the kick rate is near its best
 *            and the ball is slow: 2-3 cycles in all. */
#define S2D_CMD_SMART_KICK 13   /* a,b = target x,y, c = first_speed    Body_SmartKick    (:690-695; first_speed_threshold, max_steps ignored) */

/* Collision models (S2DConfig.collision_model).  rcssserver's Stadium::collisions repeats up to ten rounds in which every
 * overlapping pair proposes new positions, every object moves to the average of its proposals, and what collided gets
 * vel *= -0.1 at the end.  The binary is not available offline (SURVEY.md Appendix A.5 marks the pair rule with a
 * warning sign), so both readings of the pair rule are implemented, bit-exact against the oracle:
 *   MIDPOINT   (default; our reading of Stadium::calcCollPos / calcBallCollPos) player-player: both are placed
 *              symmetrically about their midpoint, (size_i + size_j) / 2 + eps each (coincident centres separate along x,
 *              lower index towards +x); ball-player: the ball is moved back along its own velocity until the two touch
 *              (straight out along the line of centres if it is at rest or its line of motion misses), the player keeps
 *              its place.
 *   BACKTRACE  (the other reading, MPObject::collide backing each object up) EVERY colliding object is moved back along
 *              its OWN velocity until it touches the other one, taken at its current place: both players of a pair, and
 *              in a ball-player contact the player as well as the ball.  An object at rest, or whose line of motion
 *              misses, is pushed straight out along the line of centres (coincident centres: along x, the lower index /
 *              the ball towards +x).  eps = 1e-6 in both. */
#define S2D_COLLISION_MIDPOINT 0
#define S2D_COLLISION_BACKTRACE 1

/* episode results: info['result'] of reach_ball_env.py:126,140,145,150 */
#define S2D_RESULT_NONE 0
#define S2D_RESULT_GOAL 1
#define S2D_RESULT_OUT 2
#define S2D_RESULT_TIMEOUT 3

/* play modes / sides (values = proto enums) */
#define S2D_PM_BEFORE_KICK_OFF 0
#define S2D_PM_TIME_OVER 1
#define S2D_PM_PLAY_ON 2
#define S2D_PM_KICK_OFF 3
#define S2D_PM_KICK_IN 4
#define S2D_PM_FREE_KICK 5
#define S2D_PM_CORNER_KICK 6
#define S2D_PM_GOAL_KICK 7
#define S2D_PM_AFTER_GOAL 8
#define S2D_SIDE_UNKNOWN 0
#define S2D_SIDE_LEFT 1
#define S2D_SIDE_RIGHT 2

/* flag bits of the per-env `flags` word (state plane 4, .z) */
#define S2D_FLAG_BALL_COLLIDED 0x1u   /* ball collided in the last simulated cycle   */
#define S2D_FLAG_PLAYER_COLLIDED 0x2u /* player collided in the last simulated cycle */
#define S2D_FLAG_KICKED 0x4u          /* a kick was applied in the last cycle        */
#define S2D_FLAG_DONE 0x8u            /* episode ended and auto_reset is off         */

/* Physics constants.  Field names = proto ServerParam / PlayerType; defaults = rcssserver's
 * (s2d_default_server_param).  All float: the kernels compute in fp32. */
typedef struct S2DServerParam {
  float pitch_half_length, pitch_half_width, goal_width, goal_post_radius;
  float ball_size, ball_decay, ball_rand, ball_speed_max, ball_accel_max;
  float player_size, player_decay, player_rand, player_speed_max, player_accel_max;
  float dash_power_rate, inertia_moment;
  float min_dash_power, max_dash_power, min_dash_angle, max_dash_angle, dash_angle_step;
  float side_dash_rate, back_dash_rate;
  float min_power, max_power, min_moment, max_moment;
  float kick_power_rate, kickable_margin, kick_rand;
  float stamina_max, stamina_inc_max, extra_stamina, stamina_capacity;
  float recover_init, recover_min, recover_dec, recover_dec_thr;
  float effort_init, effort_max, effort_min, effort_dec, effort_dec_thr, effort_inc, effort_inc_thr;
  float slowness_on_top_for_left_team, slowness_on_top_for_right_team;
  float reserved[5];
} S2DServerParam;

typedef struct S2DConfig {
  int32_t struct_size; /* sizeof(S2DConfig): checked by s2d_create */
  int32_t scenario;    /* S2D_SCENARIO_* */
  int64_t num_envs;    /* envs held by THIS handle (this rank's shard) */
  int64_t env_id_offset; /* global id of local env 0: RNG is keyed on the global id, so shards reproduce */
  uint64_t seed;
  int32_t device;      /* CUDA device ordinal */
  int32_t action_mode; /* S2D_ACT_* */
  int32_t action_space_size; /* Discrete(n), n <= 256 */
  int32_t max_steps;   /* reach_ball_env.py:33 */
  int32_t auto_reset;  /* 1: a finished episode is re-drawn inside the step kernel (VecEnv convention) */
  int32_t change_ball_position, change_ball_velocity; /* reach_ball_env.py:26-27 */
  int32_t noise;       /* 0 = noise off (player_rand = ball_rand = kick_rand = 0) */
  int32_t players_per_side; /* FULLGAME: 1..11 */
  int32_t half_time_cycles; /* FULLGAME: cycles per half (rcssserver: 3000) */
  int32_t kick_actions;     /* SHOOT + S2D_ACT_DISCRETE: how many of the action_space_size actions are kicks */
  int32_t collision_model;  /* S2D_COLLISION_* (below); 0 = default */
  int32_t reserved_i[2];
  float min_distance_to_ball; /* reach_ball_env.py:32 */
  float ball_position_x, ball_position_y, ball_speed, ball_direction; /* reach_ball_env.py:28-31 */
  float goto_dist_thr; /* Body_GoToPoint.distance_threshold for S2D_CMD_GOTO */
  float reserved_f[3];
  S2DServerParam sp;
} S2DConfig;

/* Device buffers, owned by the caller.  Sizes come from the s2d_*_bytes helpers. */
typedef struct S2DBuffers {
  void* state;         /* s2d_state_bytes(cfg), 256-B aligned; plane-major SoA (layout in DESIGN.md) */
  void* actions;       /* k_max * s2d_action_bytes(cfg); 16-byte aligned (FULLGAME: actions, obs, terminal_obs 32-byte) */
  float* obs;          /* [num_envs][s2d_obs_dim(cfg)] row-major fp32 */
  float* reward;       /* [num_envs] (sum over the K substeps of one launch) */
  uint8_t* done;       /* [num_envs] 1 if an episode ended during the launch */
  uint8_t* result;     /* [num_envs] S2D_RESULT_* of the episode that ended (else 0) */
  float* terminal_obs; /* optional [num_envs][obs_dim]: last observation of an episode that ended; may be NULL */
  void* stats;         /* s2d_stats_bytes(cfg): per-warp partial accumulators */
} S2DBuffers;

/* Totals since create (or the last s2d_stats_reset): what InfoCollectorCallback tallies. */
typedef struct S2DStats {
  uint64_t episodes, goals, outs, timeouts;
  uint64_t episode_steps; /* sum of episode lengths */
  uint64_t env_steps;     /* env-steps simulated (incl. the extra reset cycles NOT counted) */
  double return_sum;      /* sum of episode returns */
  double reserved;
} S2DStats;

/* One env on the host: the fields of proto WorldModel the path consumes (idl/service.proto:306-349). */
typedef struct S2DPlayerSnapshot {
  float x, y, vx, vy, body_direction, stamina, effort, recovery, stamina_capacity;
  int32_t side, uniform_number, collided, kicked;
} S2DPlayerSnapshot;
typedef struct S2DEnvSnapshot {
  int32_t cycle, stoped_cycle, game_mode_type, game_mode_side;
  int32_t step_number, episode, left_score, right_score;
  float ball_x, ball_y, ball_vx, ball_vy;
  float mem_distance_to_ball, mem_body_ball_angle_diff, episode_return;
  int32_t ball_collided, num_players, flags;
  S2DPlayerSnapshot players[22];
} S2DEnvSnapshot;

typedef struct S2DSim* S2DHandle;

int s2d_abi_version(void);
const char* s2d_error_string(int code);
const char* s2d_last_error(S2DHandle h); /* h may be NULL: last create error */

int s2d_default_server_param(S2DServerParam* out);
int s2d_default_config(S2DConfig* out, int scenario);

size_t s2d_state_bytes(const S2DConfig* cfg);
size_t s2d_action_bytes(const S2DConfig* cfg); /* bytes of ONE substep's actions for all envs */
size_t s2d_stats_bytes(const S2DConfig* cfg);
int s2d_obs_dim(const S2DConfig* cfg);
int s2d_num_players(const S2DConfig* cfg);

int s2d_create(const S2DConfig* cfg, S2DHandle* out);
int s2d_destroy(S2DHandle h);
int s2d_bind(S2DHandle h, const S2DBuffers* buffers);

/* Start a new episode in every env (mask == NULL) or in the envs whose device mask byte is non-zero;
 * writes obs.  Equivalent of Soccer2DEnv.reset (placement, recover, one idle cycle, reward priming). */
int s2d_reset(S2DHandle h, const uint8_t* device_mask_or_null, void* stream);

/* Advance every env by k_substeps cycles in ONE kernel launch, reading actions[N][k] from buffers.actions. */
int s2d_step(S2DHandle h, int k_substeps, void* stream);

/* Same, with HOST buffers: copies actions host->device, steps, copies obs/reward/done/result back, all
 * asynchronously on `stream` (use pinned memory).  Any of the h_* outputs may be NULL to skip that copy. */
int s2d_step_host(S2DHandle h, int k_substeps, const void* h_actions, float* h_obs, float* h_reward,
                  uint8_t* h_done, uint8_t* h_result, void* stream);

/* Pipelined host-buffer stepping: the copies of one step overlap the kernel and the copies of the next ones.
 * s2d_bind_pipeline_slot gives the handle another set of device actions / obs / reward / done / result (/ terminal_obs)
 * buffers (slot 1 .. S2D_MAX_PIPELINE_SLOTS - 1; slot 0 = the buffers of s2d_bind; state and stats are shared);
 * s2d_bind_pipeline(h, b) = s2d_bind_pipeline_slot(h, 1, b).  s2d_submit_host enqueues H2D(actions) -> step kernel ->
 * D2H(outputs) for one slot on three internal streams and returns at once; rotate the slots between consecutive
 * submissions and call s2d_wait_host(slot) before reading that slot's host outputs (or re-using its host action
 * buffer).  Host buffers should be pinned.
 * ONE device-to-host copy per step: when a slot's device outputs and its host outputs are both laid out as
 * s2d_output_layout says (obs | reward | done | result inside one block), s2d_submit_host and s2d_step_host move the
 * whole block with a single cudaMemcpyAsync instead of four.
 * Ordering: s2d_reset / s2d_step / s2d_step_host / s2d_rollout_* / s2d_stats / s2d_export_env issued on the caller's
 * stream while slots are in flight first wait (on the device) for every submitted kernel and for slot 0's copies,
 * and the next s2d_submit_host waits for that caller-stream work: the shared state is never raced.
 * What the library cannot see is work the CALLER enqueues on its own stream that touches slot 0's buffers (a copy into
 * the bound action tensor before s2d_step, a kernel reading obs after it).  s2d_fence(h, stream) orders both ways: work
 * enqueued on `stream` after the call waits for everything the pipeline has submitted, and the next s2d_submit_host
 * waits for everything enqueued on `stream` before the call.  Device-side only; the host does not block. */
#define S2D_MAX_PIPELINE_SLOTS 4
int s2d_fence(S2DHandle h, void* stream);
int s2d_bind_pipeline(S2DHandle h, const S2DBuffers* second_slot);
int s2d_bind_pipeline_slot(S2DHandle h, int slot, const S2DBuffers* slot_buffers);
int s2d_submit_host(S2DHandle h, int k_substeps, int slot, const void* h_actions, float* h_obs, float* h_reward,
                    uint8_t* h_done, uint8_t* h_result);
int s2d_wait_host(S2DHandle h, int slot); /* blocks the calling thread until the slot's outputs are on the host */

/* Offsets (256-byte aligned) of the per-step outputs inside ONE block of `bytes` bytes, for callers that want the single
 * copy described above: allocate the block once on the device and once in pinned host memory and hand the carved
 * pointers to s2d_bind / s2d_bind_pipeline_slot / s2d_submit_host.  terminal_obs (optional) sits after the others and
 * is not part of the per-step copy (only the rows of finished episodes are ever read). */
typedef struct S2DOutputLayout {
  size_t obs, reward, done, result; /* byte offsets */
  size_t step_bytes;                /* obs .. end of result: what one step copies to the host */
  size_t terminal_obs;              /* byte offset; the block then has `bytes_with_terminal_obs` bytes */
  size_t bytes, bytes_with_terminal_obs;
} S2DOutputLayout;
int s2d_output_layout(const S2DConfig* cfg, S2DOutputLayout* out);

/* Zero-fills the bound state and statistics buffers (asynchronously on `stream`).  The reset kernels READ the episode
 * and cycle counters from the state (the RNG is keyed on them), so a caller that binds freshly allocated device memory
 * must call this (or memset the buffers itself) before the first s2d_reset - otherwise episodes differ from run to run.
 * Not needed when the buffers come zero-initialised (torch.zeros in the Python host) or from a checkpoint. */
int s2d_clear(S2DHandle h, void* stream);

int s2d_stats(S2DHandle h, S2DStats* host_out, void* stream);   /* reduces the partials; synchronises */
int s2d_stats_reset(S2DHandle h, void* stream);
/* env-steps simulated so far (S2DStats.env_steps) without touching the device: for callers that reduce the statistics
 * buffer on the device themselves (Soccer2DVecEnv.allreduce_stats_async) */
int s2d_env_steps(S2DHandle h, uint64_t* out);
int s2d_export_env(S2DHandle h, int64_t local_env, S2DEnvSnapshot* host_out, void* stream); /* synchronises */

/* Heterogeneous players (FULLGAME; proto PlayerType, idl/service.proto:1697-1732).  rcssserver draws 18 player types
 * when it starts (HeteroPlayer: each type trades one quality against another) and every player is of one of them;
 * type 0 is the default player = the ServerParam values.  The fields below are the ones the cycle reads; the others of
 * the proto message either do not vary with rcssserver's default player.conf (player_size, player_speed_max,
 * kick_power_rate delta ranges are [0, 0]; kick_power_rate is kept because the proto carries it) or belong to
 * commands this library does not simulate (catch, tackle, foul). */
#define S2D_MAX_PLAYER_TYPES 18
typedef struct S2DPlayerType {
  float player_decay;    /* :1701 */
  float inertia_moment;  /* :1702 */
  float dash_power_rate; /* :1703 */
  float stamina_inc_max; /* :1700 */
  float kickable_margin; /* :1705 */
  float kick_rand;       /* :1706 */
  float extra_stamina;   /* :1707 */
  float effort_max;      /* :1708; also the effort a player starts an episode with */
  float effort_min;      /* :1709 */
  float kick_power_rate; /* :1710 */
  float reserved[6];
} S2DPlayerType;

/* types[0] = the default player of `sp`; types[1..n-1] drawn like rcssserver's HeteroPlayer from (seed, type id) with
 * the default player.conf ranges (SURVEY.md Appendix A.1 lineage: player_decay +-0.1 <-> inertia_moment x25,
 * dash_power_rate -0.0012..+0.0008 <-> stamina_inc_max x-6000, kickable_margin +-0.1 <-> kick_rand x1,
 * extra_stamina 0..50 <-> effort_max / effort_min x-0.004).  Host only, deterministic. */
int s2d_generate_player_types(uint64_t seed, const S2DServerParam* sp, S2DPlayerType* out, int n);

/* Gives the handle its player types: type_of_player[j] in [0, n) for player j (left team first, s2d_num_players
 * entries), the same assignment in every match of the handle.  Call before the first s2d_reset (effort starts at the
 * type's effort_max).  From then on the step / reset kernels read the per-player values; n = 0 returns the handle to
 * homogeneous players.  FULLGAME only. */
int s2d_set_player_types(S2DHandle h, const S2DPlayerType* types, int n, const uint8_t* type_of_player);
/* The same with an assignment of its own for every match, as rcssserver hands out its types match by match:
 * type_of_player is a HOST array [num_envs][s2d_num_players] (row e = the players of local match e).  The handle keeps a
 * device copy (num_players bytes per match, read once per player and cycle).  The type TABLE stays one per handle: the
 * matches differ in who plays with which of the n types, not in the types themselves. */
int s2d_set_player_types_per_match(S2DHandle h, const S2DPlayerType* types, int n, const uint8_t* type_of_player);

/* FULLGAME: the players played by the built-in script (spec above): bit j = player j, left team first; bits >= s2d_num_players
 * are rejected (S2D_ERR_INVALID), as is any other scenario.  0 = none (the default).  Takes effect from the next launch
 * enqueued (s2d_step, s2d_step_host, s2d_submit_host); with a non-zero mask the step runs a variant of the kernel with
 * the script compiled in. */
int s2d_set_scripted_players(S2DHandle h, uint32_t mask);

/* Closed-loop rollout with the policy inside the kernel (S2D_ACT_DISCRETE; REACHBALL with at most 16 actions, SHOOT
 * with at most 24).
 * The reference's caller is SB3 DQN (dqn_stable_baselines3.py:33-55): MlpPolicy = obs -> 64 -> 64 -> n_actions with
 * ReLU, `action = argmax Q(obs)`, `env.step(action)`.  s2d_rollout_mlp runs k_substeps cycles of
 *     observe -> Q-network (tensor cores: tcgen05.mma, TF32 operands, fp32 accumulate in tensor memory) -> action -> step
 * per launch without the observation or the action leaving the SM; with probability `epsilon` the action is uniform
 * random instead (counter RNG keyed on (seed, global env id, cycle)).  Outputs as s2d_step (obs after the last cycle,
 * reward summed, done / result, statistics); `actions_out` (device, uint8 [num_envs][k_substeps]) and `q_out` (device,
 * float [num_envs][16] for REACHBALL, [num_envs][24] for SHOOT: the Q-values seen before the LAST cycle, absent actions
 * -3e38) are optional.
 * Weights: device pointers in torch nn.Linear layout (weight [out][in] row-major, bias [out]); hidden must be 64.
 * TF32 has 10 mantissa bits: Q agrees with an fp32 evaluation to about 1e-3 of its scale, so the greedy action can
 * differ from an fp32 policy's on near-ties. */
typedef struct S2DMlpPolicy {
  const float* w1; const float* b1; /* [64][obs_dim], [64] */
  const float* w2; const float* b2; /* [64][64], [64] */
  const float* w3; const float* b3; /* [n_actions][64], [n_actions] */
  int32_t hidden;                   /* 64 */
  int32_t precision;                /* 0 (default): TF32 operands on tcgen05.mma with the accumulators in tensor memory
                                       (Q-networks and actors); 1: bf16 operands, mma.sync (Q-networks only; ~1e-2 of
                                       Q's scale); 2: TF32 operands on warp-level mma.sync (the round-1 kernels, kept
                                       for comparison) */
} S2DMlpPolicy;
int s2d_rollout_mlp(S2DHandle h, const S2DMlpPolicy* policy, int k_substeps, float epsilon, void* actions_out,
                    void* q_out, void* stream);

/* The same rollout as a collector for a replay buffer: every cycle's transition is written out, time-major (device
 * buffers, each optional).  obs[k] is what the policy saw in cycle k and obs[k + 1] the observation after it; when
 * done[k] is set that next observation already belongs to the next episode (auto-reset), which is all a TD target
 * masked by (1 - done) needs. */
typedef struct S2DTrajectory {
  float* obs;       /* [k_substeps + 1][num_envs][obs_dim] */
  uint8_t* actions; /* [k_substeps][num_envs] */
  float* reward;    /* [k_substeps][num_envs] */
  uint8_t* done;    /* [k_substeps][num_envs] */
  float* actions_f; /* [k_substeps][num_envs][action_dim]: the Box actions of s2d_rollout_actor_collect */
} S2DTrajectory;
int s2d_rollout_mlp_collect(S2DHandle h, const S2DMlpPolicy* policy, int k_substeps, float epsilon,
                            const S2DTrajectory* trajectory, void* stream);

/* The same for a deterministic actor (DDPG, ddpg_stable_baselines3.py / dqn_ddpg_stable_baselines3.py): REACHBALL with
 * S2D_ACT_CONTINUOUS (Box(1)) or S2D_ACT_TURNING (Box(4)), or SHOOT with S2D_ACT_PARAMETERIZED (Box(8); precision 0
 * only, and `actions_f` 16-byte aligned).  `actor` = obs -> 64 -> 64 -> action_dim with ReLU and a
 * final tanh (w3: [action_dim][64]); `noise` = half-width of a uniform exploration noise added to every component
 * before the clip to [-1, 1] (0: the deterministic policy).  `trajectory` may be NULL; its `actions` is not used. */
int s2d_rollout_actor_collect(S2DHandle h, const S2DMlpPolicy* actor, int k_substeps, float noise,
                              const S2DTrajectory* trajectory, void* stream);

/* Host-buffer path, for measurement: how many pipeline slots are bound (0 = no pipeline) and how many device-to-host
 * copies the last s2d_step_host / s2d_submit_host issued (1 when the packed output block went out in one piece). */
int s2d_pipeline_info(S2DHandle h, int* slots_bound, int* d2h_copies_last_step);

/* Launch geometry actually used (for bench.py's gpu_launches / DESIGN.md): blocks, threads, kernels per step call */
int s2d_launch_info(S2DHandle h, int* grid, int* block, int* kernels_per_step);

#ifdef __cplusplus
}
#endif
#endif /* SOCCER2D_H_ */
