"""GPU: Shoot with the parameterized action space (S2D_ACT_PARAMETERIZED: dash / turn / kick with continuous arguments,
include/soccer2d.h) - the step kernels and the fused tcgen05 DDPG actor of csrc/s2d_shoot_param.cu - against the C
fp32 oracle, against command rows translated on the host, and against a torch actor followed by the step kernel."""
import ctypes as C

import numpy as np
import pytest
import torch

import param_lib as PL
from soccer2d_b200 import Soccer2DVecEnv, _abi
from test_gpu_parity import assert_same_step, gpu_state, set_gpu_state

pytestmark = pytest.mark.gpu

PARAM = dict(scenario="shoot", device="cuda:0", use_parameterized_action=True)
# a ServerParam away from the defaults: the runtime-constant kernel, with the kick model's constants changed too
OTHER_SP = dict(kickable_margin=0.9, kick_power_rate=0.03, player_decay=0.5, inertia_moment=3.0, ball_decay=0.9)


@pytest.mark.parametrize("n,k,variant,auto_reset", [
    (1, 1, "default", True), (33, 4, "noise", True), (1001, 16, "runtime", True), (1001, 1, "noise", False),
    (33, 16, "default", False), (1, 4, "runtime", False), (1001, 4, "default", True), (33, 1, "runtime", True),
    (1001, 16, "noise", True)])
def test_bit_exact_against_fp32_oracle(n, k, variant, auto_reset):
    """obs, reward, done, result, terminal obs, the full state and the statistics equal the C f32 build bit for bit,
    for every constants variant (noise / default ServerParam / another ServerParam), with and without auto-reset"""
    env = Soccer2DVecEnv(n, seed=21, substeps=k, terminal_obs=True, max_steps=60, change_ball_velocity=True,
                         auto_reset=auto_reset, noise=variant == "noise", server_param=OTHER_SP if variant == "runtime" else None,
                         **PARAM)
    assert env.action_space.shape == (8,) and tuple(env.actions.shape) == (n, k, 8) and env.actions.dtype == torch.float32
    sim = PL.ParamOracleSim(env.cfg, "f32")
    assert np.array_equal(env.reset(), sim.reset())
    rng = np.random.default_rng(1)
    episodes = 0
    for t in range(max(24, 480 // k)):
        act = PL.chase_and_shoot(sim.obs, rng, k, random_share=0.3)
        env.step_torch(torch.from_numpy(act))
        sim.step(act, k)
        episodes += assert_same_step(env, sim)
        if not auto_reset and t % 16 == 15:  # start the finished episodes again
            mask = sim.done.copy()
            env.reset_torch(torch.from_numpy(mask).cuda())
            sim.reset(mask)
            assert np.array_equal(env.obs.cpu().numpy(), sim.obs)
    assert np.array_equal(gpu_state(env), sim.get_state())
    st, so = env.stats(), sim.stats(_abi.Stats())
    assert (st["episodes"], st["goals"], st["outs"], st["timeouts"], st["episode_steps"]) == \
        (so.episodes, so.goals, so.outs, so.timeouts, so.episode_steps)
    assert st["return_sum"] == pytest.approx(so.return_sum, rel=1e-9)
    assert episodes > 0
    env.close()


def test_rows_with_ties_bounds_out_of_range_values_and_nan():
    """every choice, exact ties between weights, +-1, values beyond [-1, 1] and NaN: bit-exact against the oracle and the
    same as the command rows they stand for"""
    n = 4096 + 3
    par = Soccer2DVecEnv(n, seed=5, substeps=2, max_steps=80, **PARAM)
    cmd = Soccer2DVecEnv(n, scenario="shoot", device="cuda:0", seed=5, substeps=2, max_steps=80, use_command_action=True)
    sim = PL.ParamOracleSim(par.cfg, "f32")
    assert np.array_equal(par.reset(), sim.reset()) and np.array_equal(cmd.reset(), sim.obs)
    rng = np.random.default_rng(2)
    chosen = np.zeros(4, np.int64)
    for _ in range(60):
        act = PL.random_rows(rng, n, 2)
        rows = PL.to_command(act)
        chosen += np.bincount(rows[..., 0].astype(int).ravel(), minlength=4)
        par.step_torch(torch.from_numpy(act))
        cmd.step_torch(torch.from_numpy(rows))
        sim.step(act, 2)
        assert_same_step(par, sim)
        for name in ("obs", "reward", "done_u8", "result", "state"):
            assert torch.equal(getattr(par, name), getattr(cmd, name)), name
    assert chosen[1:].min() > 10000  # dash, turn and kick all taken
    par.close()
    cmd.close()


def test_kicks_happen_from_hand_placed_states():
    """the ball at the player's feet (written through state_planes): parameterized kicks of every power and direction
    set S2D_FLAG_KICKED and move the ball, bit-exact against the oracle, and equal to the command rows"""
    n = 512
    par = Soccer2DVecEnv(n, seed=3, max_steps=200, auto_reset=False, **PARAM)
    cmd = Soccer2DVecEnv(n, scenario="shoot", device="cuda:0", seed=3, max_steps=200, auto_reset=False, use_command_action=True)
    sim = PL.ParamOracleSim(par.cfg, "f32")
    par.reset_torch()
    cmd.reset_torch()
    sim.reset()
    rng = np.random.default_rng(4)
    kicked = 0
    for rnd in range(8):
        for i in range(n):
            px, py, body = rng.uniform(-40, 40), rng.uniform(-25, 25), float(rng.integers(-180, 180))
            d, a = rng.uniform(0.3, 1.0), np.radians(body + rng.uniform(-90, 90))
            st = [px, py, 0, 0, body, 8000, 1, 1, 130600, px + d * np.cos(a), py + d * np.sin(a), 0, 0, d, 30, 0, 0,
                  3 + rnd, 1, 0]
            st = list(np.float32(st).astype(np.float64))
            set_gpu_state(par, i, st)
            set_gpu_state(cmd, i, st)
            sim.set_state(i, np.array(st))
        for e in (par, cmd):
            e.state_planes()[1][:, 3] = 0  # flags: a fresh episode (set_gpu_state leaves them)
        for t in range(3):
            act = PL.random_rows(rng, n)
            act[:, 0, :3] = [-1, -1, 1]  # kick ...
            act[: n // 8, 0, 2] = act[: n // 8, 0, 0]  # ... or, in an eighth of the rows, a dash / kick tie (dash)
            par.step_torch(torch.from_numpy(act))
            cmd.step_torch(torch.from_numpy(PL.to_command(act)))
            sim.step(act)
            assert_same_step(par, sim)
            g = gpu_state(par)
            assert np.array_equal(g, sim.get_state()) and torch.equal(par.state, cmd.state)
            kicked += int(((g[:, 19].astype(int) & _abi.FLAG_KICKED) != 0).sum())
    assert kicked > 5 * n  # most of the 7 / 8 * n first-cycle kicks of each round, and some later ones
    par.close()
    cmd.close()


def test_host_mapped_single_env_and_factory():
    """the gym single-env path (host-mapped I/O) and the factory pick the switch up from SHOOT_DEFAULTS"""
    from sample_environments.environment_factory import EnvironmentFactory
    env = EnvironmentFactory().create("shoot", None, None, None, device="cuda:0", seed=1, use_parameterized_action=True)
    assert env.action_space.shape == (8,) and env.use_parameterized_action
    vec = Soccer2DVecEnv(1, seed=1, auto_reset=False, host_mapped_io=True, **PARAM)
    assert vec.actions.device.type == "cpu"
    env.reset()
    vec.reset()
    rng = np.random.default_rng(0)
    for _ in range(50):
        a = PL.random_rows(rng, 1)[0, 0]
        o1, r1, d1, _ = env.step(a)
        o2, r2, d2, _ = vec.step_host(a)
        assert np.array_equal(o1, o2[0]) and r1 == r2[0] and d1 == bool(d2[0])
        if d1:
            env.reset()
            vec.reset()
    with pytest.raises(ValueError):
        env.step(np.zeros(4, np.float32))
    v = EnvironmentFactory().create_vec("shoot", 64, device="cuda:0", use_parameterized_action=True)
    assert v.action_mode == _abi.ACT_PARAMETERIZED
    v.close()
    vec.close()
    env.close()


# ---- the DDPG actor inside the step kernel (s2d_rollout_actor_collect) -------------------------------------------------

@pytest.mark.parametrize("n", [2048, 2048 + 9])
def test_fused_actor_rollout_matches_actor_then_step(n):
    """Even and odd N (the two trajectory store paths).  The recorded actions equal torch's fp32 actor on the recorded
    observations to TF32 accuracy; replaying them through the step kernel reproduces every observation, reward, done
    flag and the state bit for bit; the exploration noise on all 8 components is uniform of the given half-width."""
    from soccer2d_b200.rollout import Actor, mlp_layers
    torch.manual_seed(2)
    k = 5
    kw = dict(seed=6, change_ball_velocity=True, max_steps=50, **PARAM)
    fused = Soccer2DVecEnv(n, substeps=k, **kw)
    plain = Soccer2DVecEnv(n, substeps=1, **kw)
    actor = Actor(10, 8).cuda()
    with torch.no_grad():
        for p in actor.parameters():
            p.mul_(2.0)
    fused.reset_torch()
    plain.reset_torch()
    traj = {"obs": torch.zeros((k + 1, n, 10), device="cuda"), "actions": torch.zeros((k, n, 8), device="cuda"),
            "reward": torch.zeros((k, n), device="cuda"), "done": torch.zeros((k, n), dtype=torch.uint8, device="cuda")}
    worst = 0.0
    for launch in range(20):
        fused.rollout_actor(mlp_layers(actor), k, 0.0, traj=traj)
        assert torch.equal(traj["obs"][0], plain.obs)
        for j in range(k):
            with torch.no_grad():
                want = actor(plain.obs)
            worst = max(worst, float((traj["actions"][j] - want).abs().max()))
            plain.step_torch(traj["actions"][j].reshape(plain.actions.shape).contiguous())
            assert torch.equal(traj["obs"][j + 1], plain.obs)
            assert torch.equal(traj["reward"][j], plain.reward) and torch.equal(traj["done"][j], plain.done_u8)
        assert torch.equal(fused.state, plain.state)
    assert worst < 5e-3, worst
    assert fused.stats()["episodes"] == plain.stats()["episodes"] > 0
    det = torch.zeros((k, n, 8), device="cuda")
    noisy = torch.zeros((k, n, 8), device="cuda")
    state = fused.state.clone()
    fused.rollout_actor(mlp_layers(actor), k, 0.0, traj={"actions": det})
    fused.state.copy_(state)
    fused.rollout_actor(mlp_layers(actor), k, 0.25, traj={"actions": noisy})
    d = noisy[0] - det[0]  # first cycle: the same state, so the same deterministic action
    for c in range(8):
        inside = det[0, :, c].abs() < 0.7
        assert int(inside.sum()) > 200, c
        dc = d[:, c][inside]
        assert float(dc.abs().max()) <= 0.25 + 1e-6 and float(dc.std()) == pytest.approx(0.25 / 3 ** 0.5, rel=0.1), c
    assert float(noisy.abs().max()) <= 1.0
    # components 4..7 draw their own counter: not a copy of 0..3
    assert not torch.equal(d[:, 4:], d[:, :4])
    fused.close()
    plain.close()


def test_fused_actor_precisions_and_alignment_are_checked():
    """precision 1 (bf16) and 2 (mma.sync) are refused for this space, as is a misaligned actions_f"""
    from soccer2d_b200.rollout import Actor, mlp_layers
    env = Soccer2DVecEnv(64, seed=1, **PARAM)
    env.reset_torch()
    layers = mlp_layers(Actor(10, 8).cuda())
    with pytest.raises(_abi.Soccer2DError):
        env.rollout_actor(layers, 2, precision="tf32_mma_sync")
    lib = _abi.load()
    ptrs = [t.data_ptr() for wb in layers for t in wb]
    stream = torch.cuda.current_stream().cuda_stream
    for precision in (1, 2):
        pol = _abi.MlpPolicy(*ptrs, 64, precision)
        assert lib.s2d_rollout_actor_collect(env.handle, C.byref(pol), 2, 0.0, None, stream) == _abi.S2D_ERR_INVALID
    buf = torch.zeros(2 * 64 * 8 + 1, device="cuda")
    t = _abi.Trajectory()
    t.actions_f = buf[1:].data_ptr()
    pol = _abi.MlpPolicy(*ptrs, 64, 0)
    assert lib.s2d_rollout_actor_collect(env.handle, C.byref(pol), 2, 0.0, C.byref(t), stream) == _abi.S2D_ERR_INVALID
    with pytest.raises(ValueError):
        env.rollout_actor(mlp_layers(Actor(10, 4).cuda()), 2)  # an actor with the wrong number of outputs
    env.rollout_actor(layers, 2)
    torch.cuda.synchronize()
    env.close()


@pytest.mark.parametrize("n", [33, 1000 + 7])
def test_kernels_stay_inside_their_buffers(n):
    """every buffer of the step and actor kernels is the middle of a larger tensor filled with a sentinel"""
    from soccer2d_b200.rollout import Actor, mlp_layers
    lib = _abi.load()
    guard, k = 4096, 3
    env = Soccer2DVecEnv(n, seed=1, substeps=k, terminal_obs=True, max_steps=4, **PARAM)
    big = []

    def guarded(nbytes):
        buf = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
        buf[guard:guard + nbytes] = 0
        big.append((buf, nbytes))
        return buf[guard:guard + nbytes]

    views = {name: guarded(getattr(env, name).numel() * getattr(env, name).element_size())
             for name in ("state", "obs", "reward", "done_u8", "result", "terminal_obs", "stats_buf")}
    actions = guarded(env.actions.numel() * 4)
    actions.view(torch.float32).copy_((torch.rand(env.actions.numel(), device="cuda") * 3 - 1.5))
    b = _abi.Buffers(state=views["state"].data_ptr(), actions=actions.data_ptr(), obs=views["obs"].data_ptr(),
                     reward=views["reward"].data_ptr(), done=views["done_u8"].data_ptr(), result=views["result"].data_ptr(),
                     terminal_obs=views["terminal_obs"].data_ptr(), stats=views["stats_buf"].data_ptr())
    torch.cuda.synchronize()
    _abi.check(lib.s2d_bind(env.handle, C.byref(b)), env.handle)
    stream = torch.cuda.current_stream().cuda_stream
    _abi.check(lib.s2d_reset(env.handle, None, stream), env.handle)
    for _ in range(6):
        _abi.check(lib.s2d_step(env.handle, k, stream), env.handle)
    t = _abi.Trajectory()
    traj = {"obs": guarded((k + 1) * n * 40), "actions_f": guarded(k * n * 32), "reward": guarded(k * n * 4),
            "done": guarded(k * n)}
    for name, v in traj.items():
        setattr(t, name, v.data_ptr())
    layers = mlp_layers(Actor(10, 8).cuda())
    pol = _abi.MlpPolicy(*[x.data_ptr() for wb in layers for x in wb], 64, 0)
    for _ in range(4):
        _abi.check(lib.s2d_rollout_actor_collect(env.handle, C.byref(pol), k, 0.1, C.byref(t), stream), env.handle)
    torch.cuda.synchronize()
    for buf, nbytes in big:
        assert bool((buf[:guard] == 0xA5).all()) and bool((buf[guard + nbytes:] == 0xA5).all())
    assert float(views["obs"].view(torch.float32).abs().sum()) > 0 and float(traj["actions_f"].view(torch.float32).abs().sum()) > 0
    assert int(traj["done"].sum()) > 0
    env.close()


# ---- learning ------------------------------------------------------------------------------------------------------

def _random_goal_rate(env, agent, steps=300):
    before = env.stats()
    for _ in range(steps):
        agent.rollout_step(0.0, store=False, random=True)
    after = env.stats()
    return (after["goals"] - before["goals"]) / max(1, after["episodes"] - before["episodes"])


@pytest.mark.parametrize("fused,steps", [(False, 1600), (True, 3000)])
def test_ddpg_learns_to_shoot(fused, steps):
    """DDPG (ddpg_b200.py --scenario shoot) on the parameterized space beats the random actor's goal rate, measured in
    the same run.  Observed on a B200 (seed 0, 4096 envs): the random actor scored no goal in about 6 000 episodes; the
    noise-free trained actor reached a 2.4 % goal rate (torch collection, 1 600 steps) and 2.6 % (fused collection,
    3 000 steps).  The margin, 0.5 percentage points, is about a fifth of that."""
    from soccer2d_b200.rollout import DDPGConfig, DeviceDDPG
    from soccer2d_b200.vec_env import SHOOT_DEFAULTS
    env = Soccer2DVecEnv(4096, scenario="shoot", device="cuda:0", seed=0, terminal_obs=True,
                         **dict(SHOOT_DEFAULTS, use_parameterized_action=True))
    agent = DeviceDDPG(env, DDPGConfig(seed=0, learning_starts=1 << 15))
    random_rate = _random_goal_rate(env, agent)
    if fused:
        agent.learn_fused(steps, k=8)
    else:
        agent.learn(steps)
    trained = agent.evaluate(400, fused=fused)
    print("random goal rate", random_rate, "trained", trained)
    assert trained["episodes"] > 4096
    assert trained["goal_rate"] > random_rate + 0.005, (trained, random_rate)
    env.close()
