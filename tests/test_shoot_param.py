"""CPU-only: Shoot with the parameterized action space (S2D_ACT_PARAMETERIZED, include/soccer2d.h).  The two oracles
(C, Python) agree, the fp32 build tracks the f64 truth, the kernel source compiled for the host equals the fp32 build bit
for bit, and a parameterized row steps exactly as the S2D_ACT_COMMAND row it stands for."""
import ctypes as C

import numpy as np
import pytest

import emu_lib as EL
import helpers as H
import oracle_lib as OL
import param_lib as PL
from oracle import soccer2d_oracle as O
from soccer2d_b200 import _abi

SHOOT = _abi.SCENARIO_SHOOT


def _cfg(n, mode="parameterized", **kw):
    return PL.config(n, **kw) if mode == "parameterized" else PL.command_config(n, **kw)


@pytest.mark.parametrize("scenario", [_abi.SCENARIO_REACHBALL, _abi.SCENARIO_FULLGAME])
def test_parameterized_actions_are_shoot_only(scenario):
    """config_ok runs before the device check: these answers need no GPU"""
    lib = _abi.load()
    cfg = H.make_config(4, _abi.ACT_PARAMETERIZED, scenario=scenario)
    h = C.c_void_p()
    assert lib.s2d_create(C.byref(cfg), C.byref(h)) == _abi.S2D_ERR_INVALID
    assert b"action_mode 4 is not valid" in lib.s2d_last_error(None)
    ok = _cfg(4)
    assert lib.s2d_action_bytes(C.byref(ok)) == 4 * 32
    rc = lib.s2d_create(C.byref(ok), C.byref(h))
    assert rc in (_abi.S2D_OK, _abi.S2D_ERR_NO_DEVICE)
    if rc == _abi.S2D_OK:
        lib.s2d_destroy(h)


def test_translation_matches_the_spec_on_edge_values():
    """the host translation (numpy float32), the Python restatement and the C oracle's against hand-computed rows"""
    nan = float("nan")
    rows = np.array([
        [0.5, 0.5, 0.5, 1, 0.25, 0, 0, 0],        # three-way tie -> dash, power (1 + 1) * 50
        [0.2, 0.7, 0.7, 0, 0, -0.5, 0, 0],        # turn / kick tie -> turn
        [-3, -2, -1.5, 0, 0, 0, -1, 2],           # all clamp to -1 -> dash; kick args unused
        [0, 0.1, nan, 0, 0, 0, 0.5, nan],         # NaN weight -> +1 -> kick; NaN direction -> +1 -> 180
        [nan, nan, 1, nan, -7, 0, 0, 0],          # dash (tie at +1, lower index), power 100, direction -180
        [-1, 1, -1, 0, 0, 1.5, 0, 0],             # turn 180
    ], np.float32)
    want = [[1, 100, 45, 0], [2, -90, 0, 0], [1, 50, 0, 0], [3, 75, 180, 0], [1, 100, -180, 0], [2, 180, 0, 0]]
    assert np.array_equal(PL.to_command(rows), np.array(want, np.float32))
    assert [list(PL.to_command_f64(r)) for r in rows] == want
    for kind in ("f32", "f64"):  # the C oracle's translation, both builds
        assert np.array_equal(PL.ParamOracleSim(_cfg(1), kind).translate(rows), np.array(want, np.float32))
    with pytest.raises(ValueError):  # the oracle takes SHOOT's parameterized configs only
        PL.ParamOracleSim(_cfg(1, "command"), "f32")


def test_c_f64_equals_python_oracle():
    """the C and Python restatements of Shoot + parameterized rows agree (chase-and-shoot rows plus random ones)"""
    n, steps = 6, 500
    cfg = _cfg(n, seed=4, env_id_offset=50, max_steps=120)
    sim = PL.ParamOracleSim(cfg, "f64")
    pc = O.ShootConfig(seed=4, max_steps=120, sp=O.ServerParam().as_f32())
    py = [PL.ParamShootOracle(pc, env_id=50 + i) for i in range(n)]
    obs = sim.reset().copy()
    for i, o in enumerate(py):
        assert np.allclose(o.reset(), obs[i], rtol=0, atol=1e-12)
    rng = np.random.default_rng(6)
    results, kicks = set(), 0
    for _ in range(steps):
        act = PL.chase_and_shoot(sim.obs, rng)
        obs, rew, done, res = sim.step(act)
        for i, o in enumerate(py):
            po, pr, pd, pres, _ = o.step(act[i, 0])
            assert pd == bool(done[i]) and pres == int(res[i])
            assert pr == pytest.approx(float(rew[i]), rel=1e-10, abs=1e-10)
            assert H.obs_close(po, obs[i], 0) < 1e-10
            results.add(pres)
            kicks += o.player.kicked
    assert {0, 1} <= results and kicks > 20


def test_fp32_spec_tracks_f64_truth():
    """the C f32 build (the kernels' arithmetic) against the f64 truth one cycle ahead: flags exact, floats within 1e-5
    of their scale.  Dribbling is chaotic (each kick multiplies a position error), so the f64 run is re-synchronised to
    the f32 state before every cycle, as tests/test_gpu_parity.py does for the command rows."""
    n = 128
    cfg = _cfg(n, seed=2024, change_ball_velocity=1, max_steps=150)
    t, s = PL.ParamOracleSim(cfg, "f64"), PL.ParamOracleSim(cfg, "f32")
    assert H.obs_close(t.reset(), s.reset()) < H.TOL
    rng = np.random.default_rng(5)
    goals = kicks = 0
    for _ in range(400):
        g = s.get_state()
        for i in range(n):
            t.set_state(i, g[i])
        act = PL.chase_and_shoot(s.obs, rng)
        ot, rt, dt, rest = t.step(act)
        os_, rs, ds, ress = s.step(act)
        assert np.array_equal(dt, ds) and np.array_equal(rest, ress)
        # next to the ball the direction to it is ill-conditioned (position error / distance): scale those columns
        assert H.obs_close(ot, os_, angle_scale=0.02) < H.TOL
        assert np.abs(rt - rs).max() < H.TOL * 100.0
        goals += int((rest == _abi.RESULT_GOAL).sum())
        st, ss = t.get_state(), s.get_state()
        kicks += int(((ss[:, 19].astype(int) & _abi.FLAG_KICKED) != 0).sum())
        assert np.array_equal(st[:, 16:], ss[:, 16:])  # step_number, cycle, episode, collision / kick flags
        assert H.state_err(st, ss) < H.TOL
    assert goals > 20 and kicks > 200


@pytest.mark.parametrize("k", [1, 3, 16])
@pytest.mark.parametrize("sp", [{}, dict(kickable_margin=0.9, kick_power_rate=0.03, player_decay=0.5, inertia_moment=3.0)])
def test_kernel_source_bit_exact(k, sp):
    """csrc's translation + substep compiled for the host == the C f32 build, bit for bit (default ServerParam: the
    constant-folded path; the other: runtime constants)"""
    n = 257
    cfg = _cfg(n, seed=7, change_ball_velocity=1, max_steps=60 if k == 1 else 150, sp=sp)
    emu, sim = PL.ParamEmuSim(cfg), PL.ParamOracleSim(cfg, "f32")
    assert EL.lib().emu_uses_default_sp(emu.h) == (0 if sp else 1)
    assert np.array_equal(emu.reset(), sim.reset())
    rng = np.random.default_rng(0)
    episodes = 0
    for t in range(600 // k):
        act = PL.chase_and_shoot(sim.obs, rng, k, random_share=0.3)
        emu.step(act, k)
        sim.step(act, k)
        assert np.array_equal(emu.done, sim.done) and np.array_equal(emu.result, sim.result)
        assert np.array_equal(emu.obs, sim.obs) and np.array_equal(emu.reward, sim.reward)
        d = emu.done.astype(bool)
        assert np.array_equal(emu.term_obs[d], sim.term_obs[d])
        episodes += int(d.sum())
    assert np.array_equal(emu.get_state(), sim.get_state())
    assert episodes > n
    st = sim.stats(_abi.Stats())
    assert [st.episodes, st.goals, st.outs, st.timeouts, st.episode_steps] == [int(x) for x in emu.stats6[:5]]
    assert st.return_sum == pytest.approx(emu.stats6[5], rel=1e-12)


@pytest.mark.parametrize("kind", ["f64", "f32", "emu"])
def test_parameterized_equals_command_rows(kind):
    """a parameterized run equals a S2D_ACT_COMMAND run fed the rows translated on the host: in numpy float32 (one
    rounding per operation) for the fp32 arithmetic, by the Python oracle (double, then rounded to float) for f64"""
    n, k = 129, 2
    kw = dict(seed=9, change_ball_velocity=1, max_steps=100)
    if kind == "emu":
        par, cmd = PL.ParamEmuSim(_cfg(n, **kw)), EL.EmuSim(_cfg(n, "command", **kw))
    else:
        par, cmd = PL.ParamOracleSim(_cfg(n, **kw), kind), OL.OracleSim(_cfg(n, "command", **kw), kind)
    translate = PL.to_command
    if kind == "f64":
        translate = lambda a: np.array([[PL.to_command_f64(r) for r in row] for row in a], np.float32)  # noqa: E731
    assert np.array_equal(par.reset(), cmd.reset())
    rng = np.random.default_rng(3)
    kicked = 0
    for _ in range(200):
        act = PL.chase_and_shoot(par.obs, rng, k, random_share=0.4)
        par.step(act, k)
        cmd.step(translate(act), k)
        for a, b in ((par.obs, cmd.obs), (par.reward, cmd.reward), (par.done, cmd.done), (par.result, cmd.result)):
            assert np.array_equal(a, b)
        kicked += int((par.get_state()[:, 19].astype(int) & _abi.FLAG_KICKED != 0).sum())
    assert np.array_equal(par.get_state(), cmd.get_state())
    assert kicked > 50


def test_python_env_surface_without_a_device():
    """the Shoot kwargs carry the new switch, off by default (every existing configuration unchanged)"""
    from soccer2d_b200.vec_env import SHOOT_DEFAULTS
    assert SHOOT_DEFAULTS["use_parameterized_action"] is False
    assert _abi.ACT_PARAMETERIZED == 4
