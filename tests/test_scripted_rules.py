"""CPU-only: FULLGAME's scripted players (include/soccer2d.h "FULLGAME scripted players"), rule by rule on the C oracle
with the script's rules (tests/script_oracle), in its f64 and f32 builds.  The GPU is held to the f32 build bit for bit in
tests/test_gpu_scripted.py."""
import numpy as np
import pytest

import oracle_lib as OL
import script_oracle_lib as SL

P, PPS = 22, 11
K = P * 12
ALL = (1 << P) - 1
NONE, GOTO, INTERCEPT, CATCH, SMART_KICK = 0, 4, 10, 12, 13


def make(kind, n=4, mask=ALL, seed=1, half_time=10 ** 6):
    cfg = OL.default_config(n, 2, kind, action_mode=OL.ACT_COMMAND, players_per_side=PPS, half_time_cycles=half_time,
                            auto_reset=0, seed=seed)
    sim = SL.ScriptedOracleSim(cfg, kind, mask)
    sim.reset()
    return sim


def scene(sim, ball, players, mode=2, side=0, ban=(0, 0)):
    """every env: the kick-off formation, except `players` {index: (x, y, vx, vy, body)}; ball (x, y, vx, vy); play mode"""
    st = sim.get_state_fg()
    for j, v in players.items():
        st[:, j * 12:j * 12 + 5] = v
    st[:, K:K + 4] = ball
    st[:, K + 8], st[:, K + 9], st[:, K + 10] = mode, side, 0
    sim.set_state_fg(st)
    extra = np.zeros((sim.n, P + 2))
    extra[:, P:] = ban
    sim.set_extra_fg(extra)


def idle(n):
    return np.zeros((n, P * 4), np.float32)


def formation_spot(j, bx, by, hl=52.5, hw=34.0):
    left = j < PPS
    sg = 1.0 if left else -1.0
    fx, fy = OL_FORM[j if left else j - PPS]
    return (sg * np.clip(fx + 0.6 * sg * bx, -(hl - 2.5), hl - 2.5), sg * np.clip(fy + 0.3 * sg * by, -(hw - 2), hw - 2))


OL_FORM = [(-50, 0), (-36, -20), (-36, -7), (-36, 7), (-36, 20), (-20, -24), (-20, -8), (-20, 8), (-20, 24), (-9, -10), (-9, 10)]
KINDS = pytest.mark.parametrize("kind", ["f64", "f32"])


@KINDS
def test_chaser_intercepts_and_the_others_go_to_their_formation_spots(kind):
    sim = make(kind)
    scene(sim, (10.0, 5.0, 0.3, 0.0), {9: (8.0, 5.0, 0, 0, 0), 15: (13.0, 6.0, 0, 0, 180)})
    c = sim.script_commands()[0]
    assert c[9, 0] == INTERCEPT and c[15, 0] == INTERCEPT  # the nearest of each side
    for j in range(P):
        if j in (9, 15):
            continue
        tx, ty = (2.5 - 52.5, np.clip(0.3 * 5.0, -6.01, 6.01)) if j == 0 else (52.5 - 2.5, -np.clip(-0.3 * 5.0, -6.01, 6.01)) \
            if j == PPS else formation_spot(j, 10.0, 5.0)
        assert c[j, 0] == GOTO and c[j, 1:3] == pytest.approx((tx, ty), abs=1e-4), j
        assert c[j, 3] == (100.0 if j in (0, PPS) else 60.0)
    before = sim.get_state_fg()[0]
    for _ in range(5):
        sim.step(idle(sim.n))
    after = sim.get_state_fg()[0]
    for j in (2, 5, 13, 20):  # non-chasers close in on their spots
        tx, ty = formation_spot(j, 10.0, 5.0)
        assert np.hypot(after[j * 12] - tx, after[j * 12 + 1] - ty) < np.hypot(before[j * 12] - tx, before[j * 12 + 1] - ty) - 1.0
    assert np.hypot(after[9 * 12] - after[K], after[9 * 12 + 1] - after[K + 1]) < 2.5


@KINDS
def test_kickable_chaser_shoots_at_the_far_post_near_the_goal_and_dribbles_farther_out(kind):
    sim = make(kind)
    scene(sim, (35.5, 5.0, 0, 0), {10: (35.0, 5.0, 0, 0, 0)})  # left player 10, 17.8 m from the goal centre
    c = sim.script_commands()[0]
    assert c[10, 0] == SMART_KICK and tuple(c[10, 1:]) == pytest.approx((52.5, -6.01, 3.0))
    for _ in range(4):
        sim.step(idle(sim.n))
    s = sim.get_state_fg()[0]
    ang = np.degrees(np.arctan2(s[K + 3], s[K + 2]))
    want = np.degrees(np.arctan2(-6.01 - s[K + 1], 52.5 - s[K]))
    assert np.hypot(s[K + 2], s[K + 3]) > 1.5 and abs(ang - want) < 10
    # the same for the right team, mirrored: player 20 at (-35, -5) shoots at (-52.5, +6.01)
    scene(sim, (-35.5, -5.0, 0, 0), {20: (-35.0, -5.0, 0, 0, 180)})
    c = sim.script_commands()[0]
    assert c[20, 0] == SMART_KICK and tuple(c[20, 1:]) == pytest.approx((-52.5, 6.01, 3.0))
    # 50 m out: a dribble, 8 m towards the goal centre at first speed 1
    scene(sim, (0.5, 0.0, 0, 0), {10: (0.0, 0.0, 0, 0, 0), 9: (-20, -20, 0, 0, 0)})
    c = sim.script_commands()[0]
    assert c[10, 0] == SMART_KICK and tuple(c[10, 1:]) == pytest.approx((8.5, 0.0, 1.0))
    for _ in range(3):
        sim.step(idle(sim.n))
    s = sim.get_state_fg()[0]
    assert 0.3 < s[K + 2] <= 1.0 + 1e-6 and abs(s[K + 3]) < 0.05


@KINDS
def test_keeper_catches_in_its_area_but_not_outside_it_or_while_banned(kind):
    sim = make(kind)
    scene(sim, (-47.2, 0.2, -0.3, 0.0), {0: (-48.0, 0.0, 0, 0, 0)})
    assert sim.script_commands()[0, 0, 0] == CATCH
    sim.step(idle(sim.n))
    s = sim.get_state_fg()[0]
    assert (s[K + 8], s[K + 9]) == (5, 1) and s[K:K + 2] == pytest.approx(s[0:2])  # free kick left, the ball in its hands
    # outside its penalty area the keeper is no chaser: it keeps its goal, somebody else goes for the ball
    scene(sim, (-30.0, 0.2, 0, 0), {0: (-30.8, 0.0, 0, 0, 0)})
    c = sim.script_commands()[0]
    assert c[0, 0] == GOTO and c[0, 1] == pytest.approx(-50.0)
    sim.step(idle(sim.n))
    assert sim.get_state_fg()[0, K + 8] == 2
    # banned: it kicks the ball away instead
    scene(sim, (-47.2, 0.2, 0, 0), {0: (-48.0, 0.0, 0, 0, 0)}, ban=(3, 0))
    assert sim.script_commands()[0, 0, 0] == SMART_KICK
    sim.step(idle(sim.n))
    assert sim.get_state_fg()[0, K + 8] == 2


@KINDS
def test_kick_in_only_the_awarded_chaser_goes_to_the_ball_and_its_kick_resumes_play(kind):
    sim = make(kind)
    scene(sim, (10.0, 34.0, 0, 0), {}, mode=4, side=2)  # kick-in for the right team
    c = sim.script_commands()[0]
    right_chaser = [j for j in range(PPS, P) if c[j, 0] == GOTO and tuple(c[j, 1:3]) == pytest.approx((10.0, 34.0))]
    assert len(right_chaser) == 1 and c[right_chaser[0], 3] == 100.0
    assert all(c[j, 3] == 60.0 or j == 0 for j in range(PPS))  # the left team keeps its shape
    for t in range(99):
        sim.step(idle(sim.n))
        s = sim.get_state_fg()[0]
        if s[K + 8] == 2:
            break
    assert s[K + 8] == 2 and s[K + 13] == 2 and t < 60  # play resumed by the right team's kick, not by the referee's clock
    assert s[right_chaser[0] * 12 + 10] == 1


@KINDS
def test_after_a_catch_the_keeper_takes_the_free_kick(kind):
    sim = make(kind)
    scene(sim, (-47.2, 0.2, -0.3, 0.0), {0: (-48.0, 0.0, 0, 0, 0)})
    sim.step(idle(sim.n))
    assert sim.get_state_fg()[0, K + 8] == 5
    for t in range(60):
        sim.step(idle(sim.n))
        s = sim.get_state_fg()[0]
        if s[K + 8] == 2:
            break
    assert s[K + 8] == 2 and s[0 * 12 + 10] == 1 and s[K + 13] == 1 and t < 10


@KINDS
def test_nobody_acts_after_a_goal(kind):
    sim = make(kind)
    scene(sim, (53.0, 0.0, 0, 0), {}, mode=8, side=1)
    assert (sim.script_commands()[:, :, 0] == NONE).all()


@KINDS
def test_a_scripted_players_action_row_is_ignored(kind):
    """garbage in the scripted players' rows gives the same match as NONE there"""
    n, mask = 16, SL.team_mask(P, "right") | 1 << 3
    a, b = make(kind, n, mask), make(kind, n, mask)
    rng = np.random.default_rng(0)
    for _ in range(200):
        act = (rng.uniform(-1, 1, (n, P, 4)) * [0, 100, 100, 100]).astype(np.float32)
        act[:, :, 0] = rng.integers(0, 14, (n, P))
        garbage = act.copy()
        for j in range(P):
            if (mask >> j) & 1:
                act[:, j] = 0
                garbage[:, j, 0] = rng.choice([1, 3, 11, 12, 13, 14, 99], n)
        a.step(act.reshape(n, -1))
        b.step(garbage.reshape(n, -1))
        assert np.array_equal(a.obs, b.obs) and np.array_equal(a.reward, b.reward)
    assert np.array_equal(a.get_state_fg(), b.get_state_fg()) and np.array_equal(a.get_extra_fg(), b.get_extra_fg())


@KINDS
def test_mask_zero_is_the_oracle_itself(kind):
    n = 16
    cfg = OL.default_config(n, 2, kind, action_mode=OL.ACT_COMMAND, players_per_side=PPS, half_time_cycles=100, seed=4)
    a, b = SL.ScriptedOracleSim(cfg, kind, 0), OL.OracleSim(cfg, kind)
    assert np.array_equal(a.reset(), b.reset())
    rng = np.random.default_rng(1)
    for _ in range(250):
        act = np.zeros((n, P, 4), np.float32)
        act[:, :, 0] = rng.integers(0, 14, (n, P))
        act[:, :, 1:] = rng.uniform(-60, 60, (n, P, 3))
        a.step(act.reshape(n, -1), 1)
        b.step(act.reshape(n, -1), 1)
        assert np.array_equal(a.obs, b.obs) and np.array_equal(a.reward, b.reward) and np.array_equal(a.done, b.done)
    assert np.array_equal(a.get_state_fg(), b.get_state_fg())


def test_scripted_left_beats_an_idle_right_team():
    """64 matches of 2 x 300 cycles, the right team standing still (NONE).  First run (f64): the left team won all 64,
    192 goals to 0."""
    n = 64
    sim = make("f64", n, SL.team_mask(P, "left"), seed=3, half_time=300)
    for _ in range(600):
        sim.step(idle(n))
    s = sim.get_state_fg()
    assert (s[:, K + 11] > s[:, K + 12]).mean() >= 0.95 and s[:, K + 12].sum() == 0


def test_scripted_against_scripted():
    """256 matches of 2 x 300 cycles, both teams scripted.  First run (f64): 39 goals to 31; of the play modes only
    PlayOn, KickOff, AfterGoal, FreeKick (keeper catches) and the final TimeOver occurred - the script dribbles at the goal
    centre and shoots inside the posts, so the ball hardly ever leaves the pitch (the other dead-ball modes are exercised
    from hand-made states: the kick-in scene above and tests/test_gpu_scripted.py)."""
    n = 256
    sim = make("f64", n, ALL, seed=3, half_time=300)
    modes = set()
    for _ in range(600):
        sim.step(idle(n))
        modes |= set(sim.obs[:, 114].astype(int).tolist())
    s = sim.get_state_fg()
    assert s[:, K + 11].sum() >= 20 and s[:, K + 12].sum() >= 20
    assert {2, 3, 5, 8} <= modes


def dead_ball_states(sim, rng):
    """every match from its kick-off formation into a dead ball - kick-in, free kick, corner kick or goal kick, for
    either side, the ball where the referee puts it - with a random timer below 20"""
    st = sim.get_state_fg()
    n = sim.n
    modes = np.arange(n) % 4 + 4  # 4 kick-in, 5 free kick, 6 corner kick, 7 goal kick
    sides = (np.arange(n) // 4) % 2 + 1
    for i in range(n):
        sy = rng.choice([-1.0, 1.0])
        att = 1.0 if sides[i] == 1 else -1.0  # the awarded side attacks towards +x (left) or -x (right)
        bx, by = {4: (rng.uniform(-45, 45), sy * 34.0), 5: (rng.uniform(-40, 40), rng.uniform(-25, 25)),
                  6: (att * 51.5, sy * 33.0), 7: (-att * 47.0, sy * 9.16)}[int(modes[i])]
        st[i, K:K + 4] = [np.float32(bx), np.float32(by), 0.0, 0.0]
        st[i, K + 8:K + 11] = [modes[i], sides[i], int(rng.integers(0, 10))]
    sim.set_state_fg(st)
    return modes, sides


def test_scripted_teams_take_every_dead_ball():
    """Scripted against scripted from kick-ins, free kicks, corner kicks and goal kicks for either side: in (nearly)
    every match the awarded side's chaser walks to the ball and kicks it, which resumes play before the referee's
    100-cycle limit.  First run (f64, 256 matches, 64 of each mode): all 256 resumed by the awarded side's kick - kick-ins
    after 9-61 cycles, free kicks 0-50, corner kicks 64-68 (the chaser walks there from its formation spot), goal kicks
    9-12."""
    n = 256
    sim = make("f64", n, ALL, seed=5)
    modes, sides = dead_ball_states(sim, np.random.default_rng(2))
    resumed = np.full(n, -1)
    for c in range(90):
        sim.step(idle(n))
        s = sim.get_state_fg()
        newly = (resumed < 0) & (s[:, K + 8] == 2)
        assert (s[newly, K + 13] == sides[newly]).all()  # the first kick was the awarded side's
        resumed[newly] = c
    for m in (4, 5, 6, 7):
        assert (resumed[modes == m] >= 0).mean() >= 0.95, m
