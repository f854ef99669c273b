"""GPU: FULLGAME's scripted players (include/soccer2d.h "FULLGAME scripted players", s2d_set_scripted_players) against
the CPU oracle with the same rules (tests/script_oracle): bit for bit against its fp32 build, on whole trajectories and
on one cycle from hand-made states; and the host API around it."""
import numpy as np
import pytest
import torch

import helpers as H
import script_oracle_lib as SL
from test_gpu_fullgame import gpu_extra_fg, gpu_state_fg, same_state, same_step, set_gpu_extra_fg, set_gpu_state_fg
from soccer2d_b200 import Soccer2DVecEnv, _abi

pytestmark = pytest.mark.gpu


def masks(p):
    """all players, the right team, all but one (player 9 of 22, player 3 of 8)"""
    full = (1 << p) - 1
    return {"all": full, "right": SL.team_mask(p, "right"), "all_but_one": full & ~(1 << (9 if p == 22 else 3))}


@pytest.mark.parametrize("pps,k,lanes,variant", [(11, 1, "1", "default"), (11, 3, "1", "default"), (11, 1, "2", "default"),
                                                 (11, 3, "2", "default"), (4, 1, "1", "default"), (4, 3, "1", "default"),
                                                 (11, 1, "1", "noise"), (11, 3, "1", "types_per_match"),
                                                 (4, 1, "1", "types_per_match")])
@pytest.mark.parametrize("who", ["all", "right", "all_but_one"])
def test_scripted_trajectories_bit_exact_against_fp32_oracle(pps, k, lanes, variant, who, monkeypatch):
    """Whole matches (auto-reset on, 2 x 150 cycles, no masked resets: the matches stay in phase) with the players of
    the mask scripted and the others on random commands; the GPU equals the fp32 oracle after every launch."""
    monkeypatch.setenv("S2D_FG_LANES", lanes)  # (read when the handle is created; the two-lane mapping is 11 v 11 only)
    n, p = 320, 2 * pps
    mask = masks(p)[who]
    kw = dict(noise=True) if variant == "noise" else dict(hetero_seed=7, hetero_per_match=True) if variant == "types_per_match" else {}
    env = Soccer2DVecEnv(n, scenario="fullgame", device="cuda:0", seed=11, substeps=k, terminal_obs=True,
                         players_per_side=pps, half_time_cycles=150, scripted_players=[j for j in range(p) if (mask >> j) & 1], **kw)
    assert env.scripted_players == tuple(j for j in range(p) if (mask >> j) & 1)
    sim = SL.ScriptedOracleSim(env.cfg, "f32", mask)
    if env.type_of_player is not None:
        types = (_abi.PlayerType * len(env.player_types))()
        for j, t in enumerate(env.player_types):
            for name, v in t.items():
                setattr(types[j], name, v)
        sim.set_player_types(types, len(env.player_types), env.type_of_player)
    assert np.array_equal(env.reset(), sim.reset())
    rng = np.random.default_rng(3)
    modes = set()
    for t in range(660 // k):
        act = H.random_commands(rng, n * k * p).reshape(n, k, p, 4)
        env.step_torch(torch.from_numpy(act))
        sim.step(act.reshape(n, -1), k)
        same_step(env, sim)
        modes |= set(sim.obs[:, 114].astype(int).tolist())
        if t % 50 == 49:
            same_state(env, sim)
    same_state(env, sim)
    st, so = env.stats(), sim.stats(_abi.Stats())
    for key in ("episodes", "goals", "outs", "timeouts", "episode_steps", "env_steps"):
        assert st[key] == getattr(so, key), key
    assert st["episodes"] >= 2 * n
    assert {2, 3, 8} <= modes  # PlayOn, KickOff, and goals (AfterGoal)


@pytest.mark.parametrize("lanes", ["1", "2"])
@pytest.mark.parametrize("who", ["all", "right", "all_but_one"])
def test_scripted_random_states_bit_exact(who, lanes, monkeypatch):
    """One cycle from hand-made states (every play mode, the ball near the lines and at the keepers' feet, players lying
    on the ground, banned keepers), the scripted players' rows full of random commands that must be ignored."""
    monkeypatch.setenv("S2D_FG_LANES", lanes)
    n, p = 512, 22
    mask = masks(p)[who]
    env = Soccer2DVecEnv(n, scenario="fullgame", device="cuda:0", seed=2, half_time_cycles=10 ** 6, auto_reset=False)
    env.set_scripted_players([j for j in range(p) if (mask >> j) & 1])
    sim = SL.ScriptedOracleSim(env.cfg, "f32", mask)
    env.reset_torch()
    sim.reset()
    rng = np.random.default_rng(9)
    k = p * 12
    cmds = set()
    for rnd in range(8):
        st = sim.get_state_fg()
        for i in range(n):
            P = st[i, :k].reshape(p, 12)
            bx, by = rng.choice([rng.uniform(-50, 50), 52.4, -52.4, 40.0, -40.0]), rng.choice([rng.uniform(-30, 30), 33.95, -33.95, 0.0])
            P[:, 0] = rng.uniform(-52, 52, p)
            P[:, 1] = rng.uniform(-33, 33, p)
            crowd = rng.integers(0, 5)
            P[:crowd, 0] = bx + rng.uniform(-1.0, 1.0, crowd)
            P[:crowd, 1] = by + rng.uniform(-1.0, 1.0, crowd)
            P[:, 2:4] = rng.uniform(-0.4, 0.4, (p, 2))
            P[:, 4] = rng.uniform(-180, 180, p)
            P[:, 5] = rng.uniform(0, 8000, p)
            P[:, 0:9] = P[:, 0:9].astype(np.float32)
            P[:, 9:11] = 0
            if rng.uniform() < 0.3:  # the ball at a goalkeeper's feet, inside its penalty area
                side = int(rng.integers(0, 2))
                P[11 * side, 0:2] = np.float32([(-1) ** (side + 1) * rng.uniform(40, 51), rng.uniform(-15, 15)])
                th = rng.uniform(-np.pi, np.pi)
                d = rng.uniform(0.0, 1.5)
                bx, by = P[11 * side, 0] + d * np.cos(th), P[11 * side, 1] + d * np.sin(th)
            st[i, k:k + 4] = np.float32([bx, by, rng.uniform(-2, 2), rng.uniform(-2, 2)])
            mode = int(rng.choice([2, 2, 2, 3, 4, 5, 6, 7, 8]))
            st[i, k + 4] = 0
            st[i, k + 5] = rnd
            st[i, k + 8:k + 11] = [mode, int(rng.integers(1, 3)) if mode != 2 else 0, int(rng.choice([0, 5, 99]))]
            st[i, k + 13] = int(rng.integers(0, 3))
            st[i, k + 14] = st[i, k + 15] = st[i, k + 16] = 0
        sim.set_state_fg(st)
        set_gpu_state_fg(env, st)
        extra = np.zeros((n, p + 2))
        extra[:, :p] = np.where(rng.uniform(size=(n, p)) < 0.1, rng.integers(1, 11, (n, p)), 0)
        extra[:, p:] = np.where(rng.uniform(size=(n, 2)) < 0.2, rng.integers(1, 6, (n, 2)), 0)
        sim.set_extra_fg(extra)
        set_gpu_extra_fg(env, extra)
        same_state(env, sim)
        cmds |= set(sim.script_commands(mask)[:, :, 0].astype(int).ravel().tolist())
        act = H.random_commands(rng, n * p).reshape(n, 1, p, 4)
        env.step_torch(torch.from_numpy(act))
        sim.step(act.reshape(n, -1))
        same_step(env, sim)
        same_state(env, sim)
    assert {0, 4, 10, 12, 13} <= cmds  # every command the script gives: NONE, GOTO, INTERCEPT, CATCH, SMART_KICK
    env.close()


def test_scripted_players_api():
    env = Soccer2DVecEnv(64, scenario="fullgame", device="cuda:0", seed=1, players_per_side=4, half_time_cycles=50)
    assert env.scripted_players == ()
    env.set_scripted_players("left")
    assert env.scripted_players == (0, 1, 2, 3)
    env.set_scripted_players("right")
    assert env.scripted_players == (4, 5, 6, 7)
    env.set_scripted_players([7, 1])
    assert env.scripted_players == (1, 7)
    for bad in ([8], [-1], "both"):
        with pytest.raises(ValueError):
            env.set_scripted_players(bad)
    with pytest.raises(_abi.Soccer2DError):  # the library itself refuses players beyond the match
        _abi.check(env.lib.s2d_set_scripted_players(env.handle, 1 << 8), env.handle)
    env.set_scripted_players(None)
    assert env.scripted_players == ()
    env.close()
    rb = Soccer2DVecEnv(8, device="cuda:0")
    with pytest.raises(ValueError):
        rb.set_scripted_players("left")
    with pytest.raises(_abi.Soccer2DError):
        _abi.check(rb.lib.s2d_set_scripted_players(rb.handle, 1), rb.handle)
    rb.close()


def test_scripted_mask_changes_between_launches():
    """the mask reaches the next launch: a run that switches masks between launches equals the oracle doing the same"""
    n, p = 192, 22
    env = Soccer2DVecEnv(n, scenario="fullgame", device="cuda:0", seed=4, half_time_cycles=200)
    sim = SL.ScriptedOracleSim(env.cfg, "f32", 0)
    assert np.array_equal(env.reset(), sim.reset())
    rng = np.random.default_rng(1)
    for who in ["left", None, "right", range(p), [0, 11], None] * 20:
        env.set_scripted_players(who)
        sim.set_scripted(env.scripted_mask(who))
        act = H.random_commands(rng, n * p).reshape(n, 1, p, 4)
        env.step_torch(torch.from_numpy(act))
        sim.step(act.reshape(n, -1))
        same_step(env, sim)
    same_state(env, sim)
    env.close()


def test_full_game_env_with_scripted_players():
    from sample_environments.full_game_env import FullGameEnv
    env = FullGameEnv(device="cuda:0", seed=3, players_per_side=11, half_time_cycles=100, scripted_players="right")
    assert env.scripted_players == tuple(range(11, 22)) and env.controlled_players == tuple(range(11))
    assert env.action_space.shape == (11, 4)
    obs = env.reset()
    assert obs.shape == (120,)
    goto_ball = np.zeros((11, 4), np.float32)
    total, done, steps = 0.0, False, 0
    while not done:
        goto_ball[:, 0], goto_ball[:, 1], goto_ball[:, 2], goto_ball[:, 3] = 10, 0, 0, 0  # everybody intercepts
        obs, r, done, info = env.step(goto_ball)
        total += r
        steps += 1
    assert steps == 200 and info["result"] in ("Goal", "Out", "Timeout")
    with pytest.raises(ValueError):
        env.step(np.zeros((22, 4), np.float32))
    env.set_scripted_players([0, 5])
    assert env.action_space.shape == (20, 4)
    env.set_scripted_players(None)
    assert env.action_space.shape == (22, 4)
    env.close()


@pytest.mark.parametrize("who,lanes,k", [("all", "1", 1), ("all", "2", 3), ("right", "1", 3), ("right", "2", 1)])
def test_scripted_dead_balls_bit_exact(who, lanes, k, monkeypatch):
    """Trajectories that start in kick-ins, free kicks, corner kicks and goal kicks for either side (the modes a
    scripted match seldom reaches by itself): the scripted chasers walk to the ball and take the kick over many cycles,
    bit for bit as the fp32 oracle; every dead ball awarded to a scripted side is resumed by that side's kick."""
    from test_scripted_rules import dead_ball_states
    monkeypatch.setenv("S2D_FG_LANES", lanes)
    n, p = 256, 22
    mask = masks(p)[who]
    env = Soccer2DVecEnv(n, scenario="fullgame", device="cuda:0", seed=5, substeps=k, half_time_cycles=10 ** 6,
                         auto_reset=False, scripted_players=[j for j in range(p) if (mask >> j) & 1])
    sim = SL.ScriptedOracleSim(env.cfg, "f32", mask)
    env.reset_torch()
    sim.reset()
    modes, sides = dead_ball_states(sim, np.random.default_rng(7))
    set_gpu_state_fg(env, sim.get_state_fg())
    same_state(env, sim)
    rng = np.random.default_rng(8)
    resumed = np.zeros(n, bool)
    kk = p * 12
    for t in range(96 // k):
        act = H.random_commands(rng, n * k * p).reshape(n, k, p, 4)
        env.step_torch(torch.from_numpy(act))
        sim.step(act.reshape(n, -1), k)
        same_step(env, sim)
        g = gpu_state_fg(env)
        resumed |= (g[:, kk + 8] == 2) & (g[:, kk + 13] == sides)
    same_state(env, sim)
    scripted_side = sides == 2 if who == "right" else np.ones(n, bool)
    for m in (4, 5, 6, 7):
        sel = (modes == m) & scripted_side
        assert sel.any() and resumed[sel].mean() >= 0.9, (m, resumed[sel].mean())
    env.close()
