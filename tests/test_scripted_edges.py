"""CPU-only: the scripted players' rules at their edges - the chaser's tie order, the goalkeeper's eligibility, the catch
direction - stated as hand-computed expectations and checked on the C oracle (f64 and f32 builds, tests/script_oracle)
and on the Python restatement of the header (tests/scripted_twin.py)."""
import math

import numpy as np
import pytest

import fullgame_twin as T
import oracle_lib as OL
import script_oracle_lib as SL
import scripted_twin as ST
from oracle import soccer2d_oracle as O

KINDS = pytest.mark.parametrize("kind", ["f64", "f32"])


def make(kind, pps=11):
    cfg = OL.default_config(2, 2, kind, action_mode=OL.ACT_COMMAND, players_per_side=pps, half_time_cycles=10 ** 6,
                            auto_reset=0, seed=1)
    sim = SL.ScriptedOracleSim(cfg, kind, (1 << (2 * pps)) - 1)
    sim.reset()
    return sim, cfg


def scene(sim, ball, players, mode=2, side=0, ban=(0, 0)):
    p = 2 * int(sim.cfg.players_per_side)
    k = 12 * p
    st = sim.get_state_fg()
    for j, v in players.items():
        st[:, j * 12:j * 12 + 5] = v
    st[:, k:k + 4] = ball
    st[:, k + 8], st[:, k + 9], st[:, k + 10] = mode, side, 0
    sim.set_state_fg(st)
    extra = np.zeros((sim.n, p + 2))
    extra[:, p:] = ban
    sim.set_extra_fg(extra)


def both(sim, cfg):
    """the script's commands of env 0: from the C oracle and from the twin"""
    p = 2 * int(cfg.players_per_side)
    c = sim.script_commands()[0]
    m = T.Match(sim.get_state_fg()[0].tolist(), p)
    m.set_extra(sim.get_extra_fg()[0])
    sp = O.ServerParam(**{k: getattr(cfg.sp, k) for k in OL.SP_FIELDS if hasattr(O.ServerParam(), k)})
    t = ST.script_rows(m, np.zeros((p, 4), np.float32), (1 << p) - 1, sp, [sp] * p)
    return c, t


@KINDS
def test_equidistant_players_the_lower_index_chases(kind):
    sim, cfg = make(kind)
    # left players 3 and 7 exactly 2 m from the ball (binary fractions: the squared distances are equal in any precision)
    scene(sim, (10.0, 0.0, 0, 0), {3: (10.0, 2.0, 0, 0, 0), 7: (10.0, -2.0, 0, 0, 0), 14: (12.0, 1.5, 0, 0, 180),
                                   18: (12.0, -1.5, 0, 0, 180)})
    for c in both(sim, cfg):
        assert c[3, 0] == ST.INTERCEPT and c[7, 0] == ST.GOTO
        assert c[14, 0] == ST.INTERCEPT and c[18, 0] == ST.GOTO


@KINDS
def test_keeper_chases_only_in_its_own_area_or_alone(kind):
    sim, cfg = make(kind)
    # the ball just inside the left penalty area (x = -36): the keeper is nearest and chases
    scene(sim, (-36.0, 0.0, 0, 0), {0: (-37.5, 0.0, 0, 0, 0), 1: (-33.0, 0.0, 0, 0, 0)})
    for c in both(sim, cfg):
        assert c[0, 0] == ST.INTERCEPT and c[1, 0] == ST.GOTO
    # 0.25 m further out: the keeper keeps its goal, the nearest field player chases
    scene(sim, (-35.75, 0.0, 0, 0), {0: (-37.25, 0.0, 0, 0, 0), 1: (-33.0, 0.0, 0, 0, 0)})
    for c in both(sim, cfg):
        assert c[0, 0] == ST.GOTO and c[0, 1] == pytest.approx(-50.0) and c[1, 0] == ST.INTERCEPT
    # the ball in the RIGHT team's area does not make the left keeper eligible
    scene(sim, (40.0, 0.0, 0, 0), {0: (39.0, 0.0, 0, 0, 0), 1: (30.0, 0.0, 0, 0, 0)})
    for c in both(sim, cfg):
        assert c[0, 0] == ST.GOTO and c[1, 0] == ST.INTERCEPT
    # one player a side: the keeper is its side's only player and chases anywhere
    sim1, cfg1 = make(kind, pps=1)
    scene(sim1, (0.0, 5.0, 0, 0), {0: (-10.0, 0.0, 0, 0, 0), 1: (10.0, 0.0, 0, 0, 180)})
    for c in both(sim1, cfg1):
        assert c[0, 0] == ST.INTERCEPT and c[1, 0] == ST.INTERCEPT


@KINDS
def test_catch_is_aimed_at_the_ball_relative_to_the_body(kind):
    sim, cfg = make(kind)
    # keeper at (-48, 0) facing 30 deg; the ball 1 m away at 75 deg: CATCH(45)
    bx, by = -48.0 + math.cos(math.radians(75)), math.sin(math.radians(75))
    scene(sim, (bx, by, 0, 0), {0: (-48.0, 0.0, 0, 0, 30.0)})
    for c in both(sim, cfg):
        assert c[0, 0] == ST.CATCH and c[0, 1] == pytest.approx(45.0, abs=1e-3)
    # the right keeper, body -170, the ball at +150 (world): relative -40 after wrapping
    bx, by = 48.0 + math.cos(math.radians(150)), math.sin(math.radians(150))
    scene(sim, (bx, by, 0, 0), {11: (48.0, 0.0, 0, 0, -170.0)})
    for c in both(sim, cfg):
        assert c[11, 0] == ST.CATCH and c[11, 1] == pytest.approx(-40.0, abs=1e-3)
    sim.step(np.zeros((sim.n, 22 * 4), np.float32))
    s = sim.get_state_fg()[0]
    assert (s[22 * 12 + 8], s[22 * 12 + 9]) == (5, 2)  # caught: free kick for the right team
