"""CPU-only: the C oracle with the scripted players' rules (tests/script_oracle, f64 build) against an independent
Python restatement of the script written from include/soccer2d.h (tests/scripted_twin.py) driving the FULLGAME twin
(tests/fullgame_twin.py), one cycle ahead from random states - the pattern of the twin tests in tests/test_oracle_c.py."""
import numpy as np
import pytest

import fullgame_twin as T
import helpers as H
import script_oracle_lib as SL
import scripted_twin as ST
from oracle import soccer2d_oracle as O
from soccer2d_b200 import _abi

P, PPS = 22, 11
K = P * 12
SCALE = np.concatenate([np.tile([52.5, 34.0, 1.05, 1.05, 180.0, 8000.0, 1.0, 1.0, 130600.0, 1, 1, 1], P),
                        [52.5, 34.0, 3.0, 3.0, 1], np.ones(12)])
MASKS = {"all": (1 << P) - 1, "right": SL.team_mask(P, "right"), "all_but_one": ((1 << P) - 1) & ~(1 << 9)}


def random_states(sim, rng, rnd):
    """players scattered or crowding the ball, the ball anywhere incl. at a keeper's feet and inside the penalty areas,
    every play mode with either side; some players on the ground, some keepers banned"""
    n = sim.n
    st = sim.get_state_fg()
    for i in range(n):
        P_ = st[i, :K].reshape(P, 12)
        bx = rng.choice([rng.uniform(-50, 50), rng.uniform(-52, -36), rng.uniform(36, 52), 52.4, -40.0])
        by = rng.choice([rng.uniform(-30, 30), rng.uniform(-20, 20), 33.95, 0.0])
        P_[:, 0] = rng.uniform(-52, 52, P)
        P_[:, 1] = rng.uniform(-33, 33, P)
        crowd = rng.integers(0, 6)
        P_[:crowd, 0] = bx + rng.uniform(-1.0, 1.0, crowd)
        P_[:crowd, 1] = by + rng.uniform(-1.0, 1.0, crowd)
        P_[:, 2:4] = rng.uniform(-0.4, 0.4, (P, 2))
        P_[:, 4] = rng.uniform(-180, 180, P)
        P_[:, 5] = rng.uniform(0, 8000, P)
        P_[:, 6] = rng.uniform(0.6, 1.0, P)
        P_[:, 7] = rng.uniform(0.5, 1.0, P)
        if rng.uniform() < 0.3:  # the ball within reach of a goalkeeper (catch or kick), inside or just outside its area
            side = int(rng.integers(0, 2))
            P_[PPS * side, 0:2] = [(-1) ** (side + 1) * rng.uniform(33, 51), rng.uniform(-22, 22)]
            th, d = rng.uniform(-np.pi, np.pi), rng.uniform(0.0, 1.6)
            bx, by = P_[PPS * side, 0] + d * np.cos(th), P_[PPS * side, 1] + d * np.sin(th)
        elif rng.uniform() < 0.3:  # the ball at a field player's feet (shoot or dribble)
            j = int(rng.integers(1, P))
            th, d = rng.uniform(-np.pi, np.pi), rng.uniform(0.0, 1.2)
            bx, by = P_[j, 0] + d * np.cos(th), P_[j, 1] + d * np.sin(th)
        st[i, K:K + 4] = [bx, by, rng.uniform(-2, 2), rng.uniform(-2, 2)]
        mode = int(rng.choice([2, 2, 2, 3, 4, 5, 6, 7, 8, 1]))
        st[i, K + 5] = rnd
        st[i, K + 8:K + 11] = [mode, int(rng.integers(1, 3)) if mode != 2 else 0, int(rng.choice([0, 5, 99]))]
        st[i, K + 13] = int(rng.integers(0, 3))
        st[i, K + 15] = st[i, K + 16] = 0
    sim.set_state_fg(st)
    extra = np.zeros((n, P + 2))
    extra[:, :P] = np.where(rng.uniform(size=(n, P)) < 0.1, rng.integers(1, 11, (n, P)), 0)
    extra[:, P:] = np.where(rng.uniform(size=(n, 2)) < 0.3, rng.integers(1, 6, (n, 2)), 0)
    sim.set_extra_fg(extra)
    return extra


@pytest.mark.parametrize("who", sorted(MASKS))
def test_script_c_oracle_equals_the_python_twin_on_random_states(who):
    mask = MASKS[who]
    n, half = 96, 10 ** 6
    cfg = H.make_config(n, "command", scenario=_abi.SCENARIO_FULLGAME, seed=2, half_time_cycles=half, goto_dist_thr=0.5,
                        auto_reset=0)
    sim = SL.ScriptedOracleSim(cfg, "f64", mask)
    sim.reset()
    base = O.ServerParam(**{k: getattr(cfg.sp, k) for k in _abi._SP_FIELDS if hasattr(O.ServerParam(), k)})
    sps = [base] * P
    rng = np.random.default_rng({"all": 1, "right": 2, "all_but_one": 3}[who])
    seen = set()
    for rnd in range(10):
        extra = random_states(sim, rng, rnd)
        before = sim.get_state_fg()
        c_cmds = sim.script_commands()
        act = H.random_commands(rng, n * P).reshape(n, P, 4)  # (what the scripted rows hold must not matter)
        act[:, :, 0] = np.where(rng.uniform(size=(n, P)) < 0.1, 12, act[:, :, 0])
        sim.step(act.reshape(n, -1))
        after, extra_after = sim.get_state_fg(), sim.get_extra_fg()
        for i in range(n):
            m = T.Match(before[i].tolist(), P)
            m.set_extra(extra[i])
            rows = ST.script_rows(m, act[i], mask, base, sps)
            for j in range(P):
                if (mask >> j) & 1:
                    assert np.array_equal(rows[j], c_cmds[i, j]), (rnd, i, j, rows[j], c_cmds[i, j])
                    seen.add(int(rows[j, 0]))
            rw, done, _ = T.cycle(m, rows, sps, base, int(cfg.seed), i, 0.5, half)
            assert m.extra() == extra_after[i].tolist(), (rnd, i)
            assert rw == pytest.approx(float(sim.reward[i]), abs=1e-9), (rnd, i)
            m.ep_return += rw
            err = np.abs(np.array(m.vector()) - after[i]) / SCALE
            err[4:K:12] = np.minimum(err[4:K:12], np.abs(2.0 - err[4:K:12]))
            assert err.max() < 1e-9, (rnd, i, int(err.argmax()))
    assert {ST.NONE, ST.GOTO, ST.INTERCEPT, ST.CATCH, ST.SMART_KICK} <= seen, sorted(seen)
