"""Soccer2DVecEnv - N lockstep episodes held in GPU memory, stepped by libsoccer2d.so.

Vectorised face of the reference's `Soccer2DEnv.step/reset` (soccer_2d_env.py:179-269) for the scenario
classes of sample_environments/: instead of one env whose every step is a gRPC + UDP round trip to an
external rcssserver, `num_envs` independent episodes advance together in one CUDA kernel launch.  The obs,
reward, done and result tensors are persistent CUDA tensors that the kernel writes directly (zero copy).

Duck-types stable_baselines3.common.vec_env.VecEnv (num_envs, observation_space, action_space, reset,
step_async, step_wait, step, close, get_attr, set_attr, env_method, env_is_wrapped, seed) with auto-reset,
`infos[i]['terminal_observation']` and `infos[i]['result']` (what utils/info_collector_callback.py:17-53
tallies).  The torch-native calls (`reset_torch`, `step_torch`) return device tensors and build no infos.
"""
from __future__ import annotations

import ctypes as C
import operator
from collections.abc import Sequence

import numpy as np
import torch

from . import _abi
from .spaces import Box, Discrete

# kwargs of ReachBallEnv.__init__ (sample_environments/reach_ball_env.py:26-36) with the reference defaults
REACHBALL_DEFAULTS = dict(
    change_ball_position=True, change_ball_velocity=False, ball_position_x=0, ball_position_y=0, ball_speed=0,
    ball_direction=0, min_distance_to_ball=5.0, max_steps=200, use_continuous_action=True, action_space_size=16,
    use_turning=False)

# 1v0 shoot-on-goal (BASELINE configs[2]; spec in include/soccer2d.h): Discrete(24) = 16 dashes + 8 kicks by default;
# use_parameterized_action=True: Box(-1, 1, (8,)) = HFO's dash / turn / kick with continuous arguments
SHOOT_DEFAULTS = dict(
    change_ball_position=True, change_ball_velocity=False, ball_position_x=0, ball_position_y=0, ball_speed=0,
    ball_direction=0, max_steps=200, action_space_size=24, kick_actions=8, use_parameterized_action=False)

# full match, up to 11 v 11 (BASELINE configs[3]; spec in include/soccer2d.h): command actions for every player
FULLGAME_DEFAULTS = dict(players_per_side=11, half_time_cycles=3000)

_SCENARIOS = {"reachball": _abi.SCENARIO_REACHBALL, "shoot": _abi.SCENARIO_SHOOT, "fullgame": _abi.SCENARIO_FULLGAME}
_DEFAULTS = {"reachball": REACHBALL_DEFAULTS, "shoot": SHOOT_DEFAULTS, "fullgame": FULLGAME_DEFAULTS}


try:  # when Stable-Baselines3 is installed, be a real VecEnv so that SB3 does not wrap us in a DummyVecEnv
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase  # type: ignore
except Exception:  # noqa: BLE001 - SB3 is not part of this image
    _VecEnvBase = object


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _carve(block: torch.Tensor, offset: int, shape, dtype) -> torch.Tensor:
    """typed view of `shape` at byte `offset` of a uint8 block (offsets of s2d_output_layout are 256-byte aligned)"""
    shape = (shape,) if isinstance(shape, int) else tuple(shape)
    nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    return block[offset:offset + nbytes].view(dtype).view(shape)


class _SharedInfo(dict):
    """The info dict of every env whose episode goes on: ONE object shared by all of them (step_wait must not build
    num_envs dicts per step).  Read-only; `.copy()` gives a plain dict, which is what SB3's VecMonitor mutates."""

    def _ro(self, *a, **k):
        raise TypeError("the info dict of a running episode is shared between envs; copy() it before writing")

    __setitem__ = __delitem__ = update = pop = popitem = clear = setdefault = _ro


_RUNNING = _SharedInfo(result=None)


def per_match_type_assignment(seed: int, first_match: int, num_matches: int, players_per_side: int, num_types: int):
    """uint8 [num_matches][2 * players_per_side]: the goalkeepers keep type 0, the field players of a team get different
    non-default types (rcssserver's pt_max = 1) in an order that depends on (seed, GLOBAL match id, team) only."""
    with np.errstate(over="ignore"):
        gid = np.arange(first_match, first_match + num_matches, dtype=np.uint64)
        x = (gid[:, None, None] * np.uint64(2) + np.arange(2, dtype=np.uint64)[None, :, None]) * np.uint64(64) \
            + np.arange(num_types - 1, dtype=np.uint64)[None, None, :] + np.uint64(seed & 0xFFFFFFFF) * np.uint64(0x9E3779B97F4A7C15)
        x = x + np.uint64(0x9E3779B97F4A7C15)  # splitmix64
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    order = np.argsort(x, axis=2, kind="stable").astype(np.uint8) + 1  # a permutation of the non-default types per team
    field = players_per_side - 1
    reps = -(-field // (num_types - 1))  # (more field players than non-default types: go round again)
    order = np.tile(order, (1, 1, reps))[:, :, :field]
    out = np.zeros((num_matches, 2, players_per_side), dtype=np.uint8)
    out[:, :, 1:] = order
    return out.reshape(num_matches, 2 * players_per_side)


class LazyInfos(Sequence):
    """`infos` of Soccer2DVecEnv.step_wait: behaves like the list of per-env info dicts SB3 expects, but nothing is built
    until somebody looks.  Every running env answers with one shared read-only {'result': None}; an env whose episode
    ended gets its own dict {'result': 'Goal' | 'Out' | 'Timeout'[, 'terminal_observation': row]} on first access.
    `infos[:]` and iteration give plain lists (what VecMonitor copies).  It reads the step's host arrays, which the env
    recycles after `host_ring` further steps: an access later than that raises instead of returning another step's data."""
    __slots__ = ("_env", "_n", "_done", "_result", "_term", "_serial", "_cache")

    def __init__(self, env, done, result, term):
        self._env, self._n, self._done, self._result, self._term = env, env.num_envs, done, result, term
        self._serial, self._cache = env._step_serial, None

    def __len__(self):
        return self._n

    def _finished(self) -> dict:
        if self._cache is None:
            if self._env._step_serial - self._serial >= self._env.host_ring:
                raise RuntimeError("these infos belong to a step whose host buffers have been recycled; read infos within "
                                   f"{self._env.host_ring - 1} steps or construct the env with a larger host_ring")
            idx = np.flatnonzero(self._done).tolist()
            names, result, term = _abi.RESULT_NAMES, self._result, self._term
            if term is None:
                self._cache = {i: {"result": names[int(result[i])]} for i in idx}
            else:
                self._cache = {i: {"result": names[int(result[i])], "terminal_observation": term[i].copy()} for i in idx}
            self._done = self._result = self._term = None
        return self._cache

    def __getitem__(self, i):
        if isinstance(i, slice):
            out = [_RUNNING] * self._n
            for j, info in self._finished().items():
                out[j] = info
            return out[i]
        i = operator.index(i)
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError("info index out of range")
        return self._finished().get(i, _RUNNING)

    def __iter__(self):
        return iter(self[:])

    def __eq__(self, other):
        return self[:] == (other[:] if isinstance(other, LazyInfos) else other)

    def __repr__(self):
        return f"LazyInfos({self._n} envs, {len(self._finished())} finished)"


class Soccer2DVecEnv(_VecEnvBase):
    """`num_envs` ReachBall episodes on one GPU.

    num_envs       episodes held by THIS process (its shard)
    scenario       "reachball" (case-insensitive, as environment_factory.py:25)
    device         CUDA device; there is no CPU mode
    seed           Philox key; with `env_id_offset` (global id of local env 0) it fixes every episode,
                   independent of how envs are sharded over GPUs
    substeps       K cycles fused per launch; actions then carry a K axis: [N, K(, A)]
    auto_reset     finished episodes restart inside the kernel (VecEnv convention)
    terminal_obs   also keep the last observation of finished episodes (needed for SB3 infos)
    server_param   dict of overrides for the physics constants (proto ServerParam names)
    use_command_action   actions are proto-style commands {cmd, a, b, c} (S2D_CMD_*: dash / turn / kick /
                   body_go_to_point) instead of the scenario's own action space; shape [N, K, 4] float32
    goto_dist_thr  Body_GoToPoint.distance_threshold for CMD_GOTO
    hetero_seed    fullgame: draw rcssserver's 18 heterogeneous player types from this seed and give every player but
                   the two goalkeepers a random one of them (see `set_player_types` for an explicit assignment)
    hetero_per_match   with hetero_seed: every match gets an assignment of its own (rcssserver hands its types out match
                   by match): per team ten different non-default types (pt_max = 1), drawn from a hash of (hetero_seed,
                   global match id, team), so shards reproduce the global run
    noise          rcssserver's player_rand / ball_rand / kick_rand noise from the counter-based RNG, keyed on
                   (seed, global env id, server cycle, agent): reproducible, independent of sharding and of
                   `substeps`.  Off by default (the mode in which runs are compared with the double-precision CPU truth)
    scripted_players   fullgame: players played by the built-in script inside the step kernel (include/soccer2d.h,
                   s2d_set_scripted_players): None (nobody), "left", "right", or an iterable of player indices (left team
                   first).  Their rows of the action tensor keep their place in its [N, K, players, 4] layout and are
                   ignored.  The reward stays the left team's view.  See `set_scripted_players`
    collision_model  "midpoint" (default) or "backtrace": which reading of rcssserver's pair rule Stadium::collisions uses
                   (include/soccer2d.h "Collision models"; the binary is not available offline, both are implemented)
    host_numa_node NUMA node for the pinned host staging blocks of step_host / submit_host (soccer2d_b200.numa: the node of
                   this rank's GPU keeps the copies off the inter-socket link); None = wherever the driver allocates
    host_ring      step_wait() hands out views of pinned host blocks, `host_ring` of them in rotation: the arrays (and the
                   lazily built infos) of one step stay valid for the next host_ring - 1 steps - long enough for SB3's
                   collect_rollouts / VecMonitor / VecNormalize, which copy what they keep - and no num_envs-sized copy is
                   made per step.  step_wait(copy=True) returns private copies instead
    host_mapped_io actions / obs / reward / done / result live in PINNED HOST memory that the kernel reads and writes
                   directly over PCIe (unified addressing): no memcpy calls at all - the lowest-latency path for a
                   handful of envs (the single-env gym API uses it); the state stays in HBM
    **kwargs       the scenario kwargs: ReachBallEnv's (same names and defaults as the reference) or SHOOT_DEFAULTS
    """

    metadata = {"render.modes": ["human"]}  # soccer_2d_env.py:28

    def __init__(self, num_envs: int, scenario: str = "reachball", device="cuda", seed: int = 0, substeps: int = 1,
                 env_id_offset: int = 0, auto_reset: bool = True, terminal_obs: bool = False,
                 server_param: dict | None = None, use_command_action: bool = False, goto_dist_thr: float = 0.5,
                 noise: bool = False, host_mapped_io: bool = False, hetero_seed: int | None = None, hetero_per_match: bool = False,
                 host_numa_node: int | None = None, host_ring: int = 4, collision_model: str = "midpoint", scripted_players=None, **kwargs):
        if scenario.lower() not in _SCENARIOS:
            raise ValueError(f"Environment {scenario} not found.")  # environment_factory.py:28
        self.scenario = scenario.lower()
        defaults = _DEFAULTS[self.scenario]
        unknown = set(kwargs) - set(defaults)
        if unknown:
            raise TypeError(f"unknown {self.scenario} kwargs: {sorted(unknown)}")
        self.lib = _abi.load()
        if not torch.cuda.is_available():
            raise _abi.Soccer2DError(_abi.S2D_ERR_NO_DEVICE, "no CUDA device: soccer2d_b200 has no CPU fallback")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("Soccer2DVecEnv runs on CUDA devices only")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs = int(num_envs)
        self.host_numa_node = host_numa_node
        self.host_ring = max(2, int(host_ring))
        self._ring, self._ring_pos, self._step_serial = None, 0, 0
        self.substeps = int(substeps)
        self.kw = dict(defaults, **kwargs)
        for k, v in self.kw.items():
            setattr(self, k, v)
        self.seed_value = int(seed)
        self.env_id_offset = int(env_id_offset)
        self.auto_reset = bool(auto_reset)

        cfg = _abi.Config()
        _abi.check(self.lib.s2d_default_config(C.byref(cfg), _SCENARIOS[scenario.lower()]))
        cfg.num_envs = self.num_envs
        cfg.env_id_offset = self.env_id_offset
        cfg.seed = self.seed_value & 0xFFFFFFFFFFFFFFFF
        cfg.device = self.device.index
        self.num_players = 1
        if self.scenario == "fullgame":
            use_command_action = True
            cfg.players_per_side = int(self.kw["players_per_side"])
            cfg.half_time_cycles = int(self.kw["half_time_cycles"])
            self.num_players = 2 * cfg.players_per_side
        if use_command_action:
            cfg.action_mode = _abi.ACT_COMMAND
        elif self.kw.get("use_parameterized_action", False):
            cfg.action_mode = _abi.ACT_PARAMETERIZED
        elif self.kw.get("use_continuous_action", False):
            cfg.action_mode = _abi.ACT_TURNING if self.kw["use_turning"] else _abi.ACT_CONTINUOUS
        else:
            cfg.action_mode = _abi.ACT_DISCRETE
        cfg.action_space_size = int(self.kw.get("action_space_size", 16))
        cfg.kick_actions = int(self.kw.get("kick_actions", 0))
        cfg.goto_dist_thr = float(goto_dist_thr)
        cfg.noise = int(bool(noise))
        if collision_model not in _abi.COLLISION_MODELS:
            raise ValueError(f"collision_model must be one of {sorted(_abi.COLLISION_MODELS)}")
        cfg.collision_model = _abi.COLLISION_MODELS[collision_model]
        cfg.max_steps = int(self.kw.get("max_steps", 200))
        cfg.auto_reset = int(self.auto_reset)
        cfg.change_ball_position = int(bool(self.kw.get("change_ball_position", True)))
        cfg.change_ball_velocity = int(bool(self.kw.get("change_ball_velocity", False)))
        cfg.min_distance_to_ball = float(self.kw.get("min_distance_to_ball", 5.0))
        cfg.ball_position_x = float(self.kw.get("ball_position_x", 0))
        cfg.ball_position_y = float(self.kw.get("ball_position_y", 0))
        cfg.ball_speed = float(self.kw.get("ball_speed", 0))
        cfg.ball_direction = float(self.kw.get("ball_direction", 0))
        for k, v in (server_param or {}).items():
            if k not in _abi._SP_FIELDS:
                raise KeyError(f"unknown ServerParam field {k!r}")
            setattr(cfg.sp, k, float(v))
        self.cfg = cfg
        self.action_mode = cfg.action_mode

        # spaces exactly as reach_ball_env.py:39-48
        if self.scenario == "fullgame":  # one command per player
            lo = np.tile(np.array([0, -180, -180, -180], dtype=np.float32), (self.num_players, 1))
            hi = np.tile(np.array([4, 180, 180, 180], dtype=np.float32), (self.num_players, 1))
            self.action_space = Box(low=lo, high=hi, dtype=np.float32)
        elif cfg.action_mode == _abi.ACT_COMMAND:  # {cmd, a, b, c}: cmd in 0..4, arguments in metres / degrees / power
            self.action_space = Box(low=np.array([0, -180, -180, -180], dtype=np.float32),
                                    high=np.array([4, 180, 180, 180], dtype=np.float32), dtype=np.float32)
        elif cfg.action_mode == _abi.ACT_TURNING:
            self.action_space = Box(low=np.array([-1, -1, -1, -1], dtype=np.float32),
                                    high=np.array([1, 1, 1, 1], dtype=np.float32), dtype=np.float32)
        elif cfg.action_mode == _abi.ACT_PARAMETERIZED:  # [w_dash, w_turn, w_kick, dash power, dash dir, turn dir, kick power, kick dir]
            self.action_space = Box(low=-1, high=1, shape=(8,), dtype=np.float32)
        elif cfg.action_mode == _abi.ACT_CONTINUOUS:
            self.action_space = Box(low=-1, high=1, shape=(1,), dtype=np.float32)
        else:
            self.action_space = Discrete(cfg.action_space_size)
        self.observation_space = Box(low=-1, high=1, shape=(self.lib.s2d_obs_dim(C.byref(cfg)),), dtype=np.float32)

        self.handle = C.c_void_p()
        _abi.check(self.lib.s2d_create(C.byref(cfg), C.byref(self.handle)))

        # ---- device buffers: owned here (PyTorch), bound into the handle ---------------------------
        n, k, dev = self.num_envs, self.substeps, self.device
        self.host_mapped_io = bool(host_mapped_io)
        self.obs_dim = self.lib.s2d_obs_dim(C.byref(cfg))
        self.state = torch.zeros(self.lib.s2d_state_bytes(C.byref(cfg)), dtype=torch.uint8, device=dev)
        if self.host_mapped_io:
            torch.cuda.init()
            io = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory()  # noqa: E731  device-visible host memory
        else:
            io = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        if cfg.action_mode == _abi.ACT_DISCRETE:
            self.actions = io((n, k), torch.uint8)
        elif cfg.action_mode == _abi.ACT_CONTINUOUS:
            self.actions = io((n, k), torch.float32)
        elif self.scenario == "fullgame":
            self.actions = io((n, k, self.num_players, 4), torch.float32)
        elif cfg.action_mode == _abi.ACT_PARAMETERIZED:
            self.actions = io((n, k, 8), torch.float32)
        else:
            self.actions = io((n, k, 4), torch.float32)
        assert self.actions.numel() * self.actions.element_size() == self.lib.s2d_action_bytes(C.byref(cfg)) * k
        # obs | reward | done | result (| terminal_obs) are carved out of ONE block (s2d_output_layout), so that the
        # host-buffer calls can bring a step's outputs back with a single device-to-host copy
        self.layout = lay = _abi.OutputLayout()
        _abi.check(self.lib.s2d_output_layout(C.byref(cfg), C.byref(lay)))
        self._with_term = bool(terminal_obs)
        self.out_block = io(lay.bytes_with_terminal_obs if terminal_obs else lay.bytes, torch.uint8)
        self.obs, self.reward, self.done_u8, self.result, self.terminal_obs = self._carve_outputs(self.out_block)
        self.done = self.done_u8.view(torch.bool)
        self.stats_buf = torch.zeros(self.lib.s2d_stats_bytes(C.byref(cfg)), dtype=torch.uint8, device=dev)
        self._bufs = bufs = _abi.Buffers(
            state=self.state.data_ptr(), actions=self.actions.data_ptr(), obs=self.obs.data_ptr(),
            reward=self.reward.data_ptr(), done=self.done_u8.data_ptr(), result=self.result.data_ptr(),
            terminal_obs=self.terminal_obs.data_ptr() if terminal_obs else None, stats=self.stats_buf.data_ptr())
        _abi.check(self.lib.s2d_bind(self.handle, C.byref(bufs)), self.handle)
        self._pinned = None
        self._pipe = None
        self._pending = None
        self._numa_blocks = []
        self._user_dirty = False
        self.player_types = None
        self.type_of_player = None
        if hetero_seed is not None:
            types = self.generate_player_types(int(hetero_seed))
            pps = self.num_players // 2
            if hetero_per_match:
                pick = per_match_type_assignment(int(hetero_seed), self.env_id_offset, self.num_envs, pps, len(types))
            else:
                pick = np.random.default_rng(int(hetero_seed)).integers(1, len(types), size=self.num_players)
                pick[0] = pick[pps] = 0  # goalkeepers keep the default type, as rcssserver requires
            self.set_player_types(types, pick)
        self.scripted_players = ()
        if scripted_players is not None:
            self.set_scripted_players(scripted_players)
        if _VecEnvBase is not object:
            _VecEnvBase.__init__(self, self.num_envs, self.observation_space, self.action_space)
        self.render_mode = None  # soccer_2d_env.py:36; SB3 reads it with get_attr("render_mode")
        self._closed = False

    def _carve_outputs(self, block: torch.Tensor):
        lay, n = self.layout, self.num_envs
        return (_carve(block, lay.obs, (n, self.obs_dim), torch.float32), _carve(block, lay.reward, n, torch.float32),
                _carve(block, lay.done, n, torch.uint8), _carve(block, lay.result, n, torch.uint8),
                _carve(block, lay.terminal_obs, (n, self.obs_dim), torch.float32) if self._with_term else None)

    def pinned_bytes(self, nbytes: int) -> torch.Tensor:
        """page-locked uint8 host tensor, on `host_numa_node` when one was given"""
        if self.host_numa_node is None:
            return torch.empty(int(nbytes), dtype=torch.uint8, pin_memory=True)
        from .numa import PinnedBlock
        pb = PinnedBlock(nbytes, self.host_numa_node)
        self._numa_blocks.append(pb)  # keeps the registration alive as long as the env
        return pb.tensor

    def pinned_like(self, t: torch.Tensor) -> torch.Tensor:
        """page-locked host tensor of t's shape / dtype (see pinned_bytes), e.g. for the actions of submit_host"""
        return self.pinned_bytes(t.numel() * t.element_size()).view(t.dtype).view(t.shape)

    def _pinned_outputs(self) -> dict:
        """one pinned host block with the device block's layout: a step's outputs arrive in ONE copy"""
        block = self.pinned_bytes(self.layout.bytes)
        self._with_term, keep = False, self._with_term
        obs, reward, done, result, _ = self._carve_outputs(block)
        self._with_term = keep
        return dict(block=block, obs=obs, reward=reward, done=done, result=result)

    # ---- torch-native API: device tensors in, device tensors out, no host sync ------------------------
    def reset_torch(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        """New episode in every env, or in the envs where `mask` (bool/uint8 [N], on the device) is set."""
        ptr = None
        if mask is not None:
            mask = mask.to(device=self.device).view(-1)
            mask = mask.view(torch.uint8) if mask.dtype == torch.bool else mask.to(torch.uint8)
            mask = mask.contiguous()
            assert mask.numel() == self.num_envs
            ptr = mask.data_ptr()
        _abi.check(self.lib.s2d_reset(self.handle, ptr, _stream_ptr(self.device)), self.handle)
        self._user_dirty = True
        return self.obs

    def _fence(self) -> None:
        """order this stream against the host-buffer pipeline in both directions (s2d_fence); no-op without one"""
        if self._pipe is not None:
            _abi.check(self.lib.s2d_fence(self.handle, _stream_ptr(self.device)), self.handle)

    def step_torch(self, actions: torch.Tensor | None = None):
        """One launch = `substeps` cycles of every env.  `actions=None` uses what is already in
        `self.actions` (a policy may write there directly).  Returns (obs, reward, done, result): views of
        the persistent tensors, valid until the next step."""
        if actions is not None:
            self._fence()  # slot 0's kernel may still be reading the tensor this copy overwrites
            self.actions.copy_(actions.to(self.device).reshape(self.actions.shape), non_blocking=True)
        _abi.check(self.lib.s2d_step(self.handle, self.substeps, _stream_ptr(self.device)), self.handle)
        self._user_dirty = True
        return self.obs, self.reward, self.done, self.result

    def bind_actions(self, actions: torch.Tensor) -> None:
        """Point the kernels at another device tensor of the same shape/dtype (no copy): lets a policy, or a
        pool of pre-generated action blocks, feed the step without a device-to-device copy."""
        assert actions.is_cuda and actions.device == self.device and actions.is_contiguous()
        assert actions.shape == self.actions.shape and actions.dtype == self.actions.dtype
        self.actions = actions
        self._bufs.actions = actions.data_ptr()
        _abi.check(self.lib.s2d_bind(self.handle, C.byref(self._bufs)), self.handle)

    # ---- host API: host buffers in / host buffers out (the reference-facing call) --------------------
    def host_buffers(self) -> dict:
        """Pinned host staging tensors: 'actions' (fill it in place for zero-copy submission) and the
        outputs 'obs', 'reward', 'done', 'result' that step_host fills."""
        if self._pinned is None:
            self._pinned = dict(self._pinned_outputs(), actions=self.pinned_like(self.actions))
        return self._pinned

    def step_host(self, actions=None, out: dict | None = None, sync: bool = True):
        """Host actions in, host results out: H2D of the actions, the step launch and D2H of
        obs/reward/done/result are enqueued by ONE C-ABI call (s2d_step_host), then the stream is drained.
        `actions`: numpy array / CPU tensor of the action shape (pinned memory makes the copy asynchronous),
        or None to submit host_buffers()['actions'].  Returns numpy views of the pinned output buffers (`out`: another
        block of _pinned_outputs() to receive them; sync=False leaves the stream un-drained)."""
        if self.host_mapped_io:  # the kernel reads the actions from / writes the results to host memory itself
            if actions is not None:
                self.actions.numpy()[...] = np.asarray(actions).reshape(tuple(self.actions.shape))
            _abi.check(self.lib.s2d_step(self.handle, self.substeps, _stream_ptr(self.device)), self.handle)
            torch.cuda.current_stream(self.device).synchronize()
            return self.obs.numpy(), self.reward.numpy(), self.done_u8.numpy().view(np.bool_), self.result.numpy()
        p = self.host_buffers()
        if actions is None:
            src = p["actions"]
        elif isinstance(actions, torch.Tensor):
            src = actions.to(dtype=self.actions.dtype).reshape(self.actions.shape).contiguous()
            assert not src.is_cuda
        else:
            src = torch.from_numpy(np.ascontiguousarray(
                np.asarray(actions).reshape(tuple(self.actions.shape)), dtype=p["actions"].numpy().dtype))
        self._host_src = src  # keep the host source alive until the copy has happened
        o = out if out is not None else p
        _abi.check(self.lib.s2d_step_host(self.handle, self.substeps, src.data_ptr(), o["obs"].data_ptr(),
                                          o["reward"].data_ptr(), o["done"].data_ptr(), o["result"].data_ptr(),
                                          _stream_ptr(self.device)), self.handle)
        if sync:
            torch.cuda.current_stream(self.device).synchronize()
        return o["obs"].numpy(), o["reward"].numpy(), o["done"].numpy().view(np.bool_), o["result"].numpy()

    # ---- pipelined host API: submit step i+1 while the results of step i are still coming back ---------
    def enable_pipeline(self, slots: int = 3) -> None:
        """Allocate `slots` - 1 further slots (device actions + output block, pinned host output block) and bind them;
        slot 0 = this env's own buffers.  With three slots the device-to-host copy of step i, the kernel of step i + 1
        and the host-to-device copy of step i + 2 run at the same time."""
        if getattr(self, "_pipe", None) is not None:
            return
        if not 2 <= slots <= _abi.MAX_PIPELINE_SLOTS:
            raise ValueError(f"slots must be in 2..{_abi.MAX_PIPELINE_SLOTS}")
        dev = self.device
        torch.cuda.current_stream(dev).synchronize()
        device = [None]
        for k in range(1, slots):
            block = torch.zeros_like(self.out_block, device=dev)
            obs, reward, done, result, term = self._carve_outputs(block)
            actions = torch.zeros_like(self.actions, device=dev)
            b = _abi.Buffers(state=self.state.data_ptr(), actions=actions.data_ptr(), obs=obs.data_ptr(),
                             reward=reward.data_ptr(), done=done.data_ptr(), result=result.data_ptr(),
                             terminal_obs=term.data_ptr() if term is not None else None, stats=self.stats_buf.data_ptr())
            _abi.check(self.lib.s2d_bind_pipeline_slot(self.handle, k, C.byref(b)), self.handle)
            device.append(dict(block=block, actions=actions, obs=obs, reward=reward, done=done, result=result,
                               terminal_obs=term))
        host = [self._pinned_outputs() for _ in range(slots)]
        self._pipe = dict(device=device, host=host, next_slot=0, keep=[None] * slots, slots=slots)

    def submit_host(self, actions) -> int:
        """Enqueue one step from host `actions` (pinned CPU tensor / numpy array of the action shape) and return
        its ticket (the slot).  At most `slots` steps can be in flight: wait_host() the oldest one before re-using
        its slot."""
        self.enable_pipeline()
        pipe = self._pipe
        slot = pipe["next_slot"]
        pipe["next_slot"] = (slot + 1) % pipe["slots"]
        if isinstance(actions, torch.Tensor):
            src = actions.to(dtype=self.actions.dtype).reshape(self.actions.shape).contiguous()
        else:
            src = torch.from_numpy(np.ascontiguousarray(np.asarray(actions).reshape(tuple(self.actions.shape))))
            src = src.to(dtype=self.actions.dtype)
        pipe["keep"][slot] = src  # keep the host source alive until the copy has happened
        ho = pipe["host"][slot]
        if self._user_dirty:  # what this stream still does with the state / slot 0's tensors comes first
            self._fence()
            self._user_dirty = False
        _abi.check(self.lib.s2d_submit_host(self.handle, self.substeps, slot, src.data_ptr(), ho["obs"].data_ptr(),
                                            ho["reward"].data_ptr(), ho["done"].data_ptr(), ho["result"].data_ptr()),
                   self.handle)
        return slot

    def pipeline_info(self) -> dict:
        """slots bound and the number of device-to-host copies the last host-buffer step needed (1 = packed block)"""
        slots, copies = C.c_int(0), C.c_int(0)
        _abi.check(self.lib.s2d_pipeline_info(self.handle, C.byref(slots), C.byref(copies)), self.handle)
        return {"slots": slots.value, "d2h_copies_last_step": copies.value}

    def wait_host(self, ticket: int):
        """Block until the step submitted with `ticket` is on the host; returns numpy views of that slot's pinned
        outputs (valid until the slot is submitted again)."""
        _abi.check(self.lib.s2d_wait_host(self.handle, int(ticket)), self.handle)
        ho = self._pipe["host"][ticket]
        return ho["obs"].numpy(), ho["reward"].numpy(), ho["done"].numpy().view(np.bool_), ho["result"].numpy()

    # ---- SB3 VecEnv surface ---------------------------------------------------------------------------
    def reset(self) -> np.ndarray:
        obs = self.reset_torch()
        if self.host_mapped_io:
            torch.cuda.current_stream(self.device).synchronize()
            return obs.numpy().copy()
        return obs.cpu().numpy()

    def step_async(self, actions) -> None:
        self._pending = actions

    def step_wait(self, copy: bool = False):
        """SB3's VecEnv.step_wait.  Python work per step is O(1): the arrays are views of a pinned host block out of a
        ring of `host_ring` (see the class docstring; copy=True for private copies) and `infos` is a LazyInfos that builds
        dicts only for the envs whose episode ended, and only when read ('result' is what
        utils/info_collector_callback.py:23-27 looks at; 'terminal_observation' with terminal_obs=True)."""
        actions, self._pending = self._pending, None
        if self.host_mapped_io:
            obs, reward, done, result = self.step_host(actions)
            obs, reward, done, result = obs.copy(), reward.copy(), done.copy(), result.copy()
            term = self.terminal_obs.numpy() if self.terminal_obs is not None else None
            self._step_serial += 1
            return obs, reward, done, LazyInfos(self, done, result, term)
        if self._ring is None:
            self._ring = []
            for _ in range(self.host_ring):
                blk = self._pinned_outputs()
                if self.terminal_obs is not None:
                    blk["term"] = self.pinned_like(self.terminal_obs)
                self._ring.append(blk)
        self._ring_pos = (self._ring_pos + 1) % self.host_ring
        blk = self._ring[self._ring_pos]
        term = blk.get("term")
        obs, reward, done, result = self.step_host(actions, out=blk, sync=term is None)
        if term is not None:  # the whole block in one more async copy: no second synchronisation, no gather kernel
            term.copy_(self.terminal_obs, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            term = term.numpy()
        self._step_serial += 1
        if copy:
            obs, reward, done, result = obs.copy(), reward.copy(), done.copy(), result.copy()
            term = term.copy() if term is not None else None
        return obs, reward, done, LazyInfos(self, done, result, term)

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        if not self._closed:
            self._closed = True
            if self.handle:
                self.lib.s2d_destroy(self.handle)
                self.handle = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def seed(self, seed=None):
        return [None] * self.num_envs  # the Philox key is fixed at construction

    # kernel constants: fixed when the handle is created
    _FROZEN = frozenset(REACHBALL_DEFAULTS) | frozenset(SHOOT_DEFAULTS) | frozenset(FULLGAME_DEFAULTS) | {
        "num_envs", "substeps", "scenario", "device", "seed_value", "env_id_offset", "auto_reset", "observation_space",
        "action_space"}

    def get_attr(self, attr_name, indices=None):
        return [getattr(self, attr_name)] * len(self._indices(indices))

    def set_attr(self, attr_name, value, indices=None):
        """All envs are one object: an attribute set for some of them is set for all (SB3 wrappers use this for
        bookkeeping attributes such as render_mode); episode parameters are kernel constants and cannot change."""
        if attr_name in self._FROZEN:
            raise AttributeError(f"{attr_name} is fixed at construction (it is a kernel constant)")
        setattr(self, attr_name, value)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        """Calls the method ONCE on this object and repeats its result per requested env."""
        if method_name.startswith("_") or not callable(getattr(self, method_name, None)):
            raise AttributeError(f"{method_name}: per-env Python methods do not exist on the GPU path")
        return [getattr(self, method_name)(*args, **kwargs)] * len(self._indices(indices))

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * len(self._indices(indices))

    def render(self, mode="human"):
        return None

    def _indices(self, indices):
        if indices is None:
            return range(self.num_envs)
        return [indices] if isinstance(indices, int) else indices

    # ---- statistics, export, checkpoint ---------------------------------------------------------------
    def stats(self) -> dict:
        """Totals since construction / reset_stats(): what InfoCollectorCallback counts per 100 episodes
        (utils/info_collector_callback.py:37-53), plus episode length and return sums."""
        st = _abi.Stats()
        _abi.check(self.lib.s2d_stats(self.handle, C.byref(st), _stream_ptr(self.device)), self.handle)
        return {k: getattr(st, k) for k in
                ("episodes", "goals", "outs", "timeouts", "episode_steps", "env_steps", "return_sum")}

    def reset_stats(self) -> None:
        _abi.check(self.lib.s2d_stats_reset(self.handle, _stream_ptr(self.device)), self.handle)

    def allreduce_stats(self, group=None) -> dict:
        """Sum of stats() over all ranks (one small all-reduce; NCCL when the process group is NCCL)."""
        from .sharding import allreduce_stats
        return allreduce_stats(self.stats(), device=self.device, group=group)

    def allreduce_stats_async(self, group=None):
        """The same sum without a host synchronisation and without touching the stepping stream: the 256 partial
        accumulators are reduced on the device on a SIDE stream (ordered after the launches enqueued so far), the
        NCCL all-reduce follows on that stream, and a StatsFuture is returned at once - call `.result()` when the
        numbers are needed (a training loop that reports every M launches: SURVEY.md section 8e)."""
        from .sharding import allreduce_stats_async
        dev = self.device
        if getattr(self, "_stats_stream", None) is None:
            self._stats_stream = torch.cuda.Stream(dev)
        side = self._stats_stream
        self._fence()  # (launches of the host-buffer pipeline count too)
        side.wait_stream(torch.cuda.current_stream(dev))
        steps = C.c_uint64(0)
        _abi.check(self.lib.s2d_env_steps(self.handle, C.byref(steps)), self.handle)
        with torch.cuda.stream(side):
            slots = self.stats_buf.view(torch.int64).view(-1, 8)
            counts = torch.cat([slots[:, :5].sum(0), torch.tensor([steps.value], dtype=torch.int64, device=dev)])
            ret = self.stats_buf.view(torch.float64).view(-1, 8)[:, 5].sum().reshape(1)
            snapshot = torch.cuda.Event()
            snapshot.record(side)
        # later launches wait for this snapshot (two tiny reductions), not for the collective that follows it
        torch.cuda.current_stream(dev).wait_event(snapshot)
        counts.record_stream(side)
        ret.record_stream(side)
        return allreduce_stats_async(counts, ret, group=group, stream=side)

    def export_env(self, i: int) -> _abi.EnvSnapshot:
        """Host snapshot of env `i`: the WorldModel fields the reference path reads (idl/service.proto:306-349)."""
        snap = _abi.EnvSnapshot()
        _abi.check(self.lib.s2d_export_env(self.handle, int(i), C.byref(snap), _stream_ptr(self.device)), self.handle)
        return snap

    def export_state(self, i: int, unum: int = 1, side: int = 1) -> dict:
        """proto `State` of env `i` as seen by player `unum` of `side`, as nested dicts keyed by the proto field names
        (idl/service.proto:306-359); `json_format.ParseDict(d, service_pb2.State())` turns it into the message."""
        from .proto_state import state_dict
        return state_dict(self.export_env(i), unum=unum, side=side,
                          kickable_area=self.cfg.sp.player_size + self.cfg.sp.ball_size + self.cfg.sp.kickable_margin,
                          type_of_player=self.type_of_player)

    def state_planes(self):
        """One-player scenarios: views of the SoA planes (float32 [4, N, 4], int32 [N, 4]) - layout in DESIGN.md."""
        assert self.scenario != "fullgame", "use export_env / fullgame_planes for the match layout"
        n = self.num_envs
        f = self.state[: 4 * n * 16].view(torch.float32).view(4, n, 4)
        u = self.state[4 * n * 16:].view(torch.int32).view(n, 4)
        return f, u

    def fullgame_planes(self) -> dict:
        """FULLGAME: views of the planes, indexed [match, player(, field)] (in memory they are match-minor - player rows
        of N consecutive matches - see csrc/s2d_fullgame.cuh FgLayout)."""
        assert self.scenario == "fullgame"
        n, p = self.num_envs, self.num_players
        nr = (n + 63) // 64 * 64  # rows are padded to the kernel's block size (scratch matches past num_envs)
        off = 0
        out = {}
        for name in ("pa", "pb"):
            out[name] = self.state[off:off + nr * p * 16].view(torch.float32).view(p, nr, 4)[:, :n].permute(1, 0, 2)
            off += nr * p * 16
        out["pc"] = self.state[off:off + nr * p * 4].view(torch.float32).view(p, nr)[:, :n].t()
        off += nr * p * 4
        for name, dt in (("ball", torch.float32), ("ef", torch.float32), ("ei", torch.int32), ("ej", torch.int32),
                         ("ek", torch.int32)):
            out[name] = self.state[off:off + nr * 16].view(dt).view(nr, 4)[:n]
            off += nr * 16
        assert off == self.state.numel()
        return out

    # ---- closed-loop rollout with the Q-network inside the kernel (s2d_rollout_mlp) ------------------------------
    def rollout_mlp(self, layers, k: int | None = None, epsilon: float = 0.0, actions_out: torch.Tensor | None = None,
                    q_out: torch.Tensor | None = None, traj: dict | None = None, precision: str = "tf32") -> None:
        """`k` cycles of observe -> Q(obs) -> (epsilon-)greedy action -> step in ONE launch (Discrete actions: ReachBall
        with n <= 16, Shoot with n <= 24).
        `layers` = [(weight, bias)] * 3 of a 64-64 ReLU MLP as torch nn.Linear stores them (float32 CUDA tensors:
        [64, 10], [64], [64, 64], [64], [n, 64], [n]), e.g. `[(l.weight, l.bias) for l in qnet.linears]`.
        Outputs land in the env's obs / reward / done_u8 / result tensors as after `step_torch`; optional
        `actions_out` uint8 [N, k] receives the actions taken and `q_out` float32 [N, 16] (Shoot: [N, 24]) the Q-values of the last cycle.
        `precision`: "tf32" (default: TF32 operands on tcgen05.mma, accumulators in tensor memory), "tf32_mma_sync" (the
        same operands on warp-level mma.sync: the round-1 kernel) or "bf16" (mma.sync; Q-values agree with fp32 only to ~1e-2).
        `traj` (s2d_rollout_mlp_collect): time-major tensors for every cycle's transition, any of obs float32
        [k + 1, N, 10], actions uint8 [k, N], reward float32 [k, N], done uint8 [k, N] - what a replay buffer takes."""
        k = self.substeps if k is None else int(k)
        self._user_dirty = True
        ptrs = []
        for (w, b), shape in zip(layers, ((64, self.obs_dim), (64, 64), (self.cfg.action_space_size, 64))):
            if tuple(w.shape) != shape or tuple(b.shape) != shape[:1]:
                raise ValueError(f"rollout_mlp: expected weight {shape} and bias {shape[:1]}, got {tuple(w.shape)} / {tuple(b.shape)}")
            for t in (w, b):
                if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous() or t.device != self.device:
                    raise ValueError("rollout_mlp: weights must be contiguous float32 tensors on the env's device")
            ptrs += [w.data_ptr(), b.data_ptr()]
        if actions_out is not None:
            assert actions_out.dtype == torch.uint8 and tuple(actions_out.shape) == (self.num_envs, k) and actions_out.is_contiguous()
        if q_out is not None:
            width = 24 if self.scenario == "shoot" else 16
            assert q_out.dtype == torch.float32 and tuple(q_out.shape) == (self.num_envs, width) and q_out.is_contiguous()
        pol = _abi.MlpPolicy(*ptrs, 64, {"tf32": 0, "tf32_tcgen05": 0, "bf16": 1, "tf32_mma_sync": 2}[precision])
        if traj is not None:
            assert actions_out is None and q_out is None, "traj replaces actions_out / q_out"
            want = {"obs": ((k + 1, self.num_envs, self.obs_dim), torch.float32), "actions": ((k, self.num_envs), torch.uint8),
                    "reward": ((k, self.num_envs), torch.float32), "done": ((k, self.num_envs), torch.uint8)}
            t = _abi.Trajectory()
            for name, ten in traj.items():
                shape, dt = want[name]
                assert tuple(ten.shape) == shape and ten.dtype == dt and ten.is_contiguous() and ten.device == self.device, name
                setattr(t, name, ten.data_ptr())
            _abi.check(self.lib.s2d_rollout_mlp_collect(self.handle, C.byref(pol), k, float(epsilon), C.byref(t),
                                                        _stream_ptr(self.device)), self.handle)
            return
        _abi.check(self.lib.s2d_rollout_mlp(self.handle, C.byref(pol), k, float(epsilon),
                                            actions_out.data_ptr() if actions_out is not None else None,
                                            q_out.data_ptr() if q_out is not None else None, _stream_ptr(self.device)),
                   self.handle)

    def rollout_actor(self, layers, k: int | None = None, noise: float = 0.0, traj: dict | None = None,
                      precision: str = "tf32") -> None:
        """`k` cycles of observe -> actor(obs) -> Box action -> step in ONE launch (ReachBall with the Box(1) or the Box(4)
        turning action space, Shoot with the Box(8) parameterized one): the DDPG counterpart of `rollout_mlp`
        (s2d_rollout_actor_collect).  `layers` = [(weight, bias)] * 3 of a 64-64 ReLU MLP whose last layer has
        action_dim rows; tanh is applied in the kernel.  `noise`: the half-width of a uniform exploration noise on every
        component.  `traj`: time-major tensors, any of obs float32 [k + 1, N, 10], actions float32 [k, N, action_dim],
        reward float32 [k, N], done uint8 [k, N].  `precision`: "tf32" (default: tcgen05.mma, accumulators in tensor
        memory) or "tf32_mma_sync" (the warp-level kernel of round 1; not for Shoot's parameterized actions)."""
        k = self.substeps if k is None else int(k)
        self._user_dirty = True
        ad = {_abi.ACT_TURNING: 4, _abi.ACT_PARAMETERIZED: 8}.get(self.action_mode, 1)
        ptrs = []
        for (w, b), shape in zip(layers, ((64, self.obs_dim), (64, 64), (ad, 64))):
            if tuple(w.shape) != shape or tuple(b.shape) != shape[:1]:
                raise ValueError(f"rollout_actor: expected weight {shape} and bias {shape[:1]}, got {tuple(w.shape)} / {tuple(b.shape)}")
            for t in (w, b):
                if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous() or t.device != self.device:
                    raise ValueError("rollout_actor: weights must be contiguous float32 tensors on the env's device")
            ptrs += [w.data_ptr(), b.data_ptr()]
        pol = _abi.MlpPolicy(*ptrs, 64, {"tf32": 0, "tf32_tcgen05": 0, "tf32_mma_sync": 2}[precision])
        t = _abi.Trajectory()
        want = {"obs": ((k + 1, self.num_envs, self.obs_dim), torch.float32, "obs"),
                "actions": ((k, self.num_envs, ad), torch.float32, "actions_f"),
                "reward": ((k, self.num_envs), torch.float32, "reward"), "done": ((k, self.num_envs), torch.uint8, "done")}
        for name, ten in (traj or {}).items():
            shape, dt, field = want[name]
            assert tuple(ten.shape) == shape and ten.dtype == dt and ten.is_contiguous() and ten.device == self.device, name
            setattr(t, field, ten.data_ptr())
        _abi.check(self.lib.s2d_rollout_actor_collect(self.handle, C.byref(pol), k, float(noise),
                                                      C.byref(t) if traj is not None else None, _stream_ptr(self.device)),
                   self.handle)

    # ---- heterogeneous players (fullgame; proto PlayerType, idl/service.proto:1697-1732) ------------------------
    def generate_player_types(self, seed: int, n: int = _abi.MAX_PLAYER_TYPES) -> list:
        """rcssserver's HeteroPlayer draws for this env's ServerParam: [type 0 = default player, n - 1 drawn types]"""
        out = (_abi.PlayerType * n)()
        _abi.check(self.lib.s2d_generate_player_types(int(seed) & 0xFFFFFFFFFFFFFFFF, C.byref(self.cfg.sp), out, n))
        return list(out)

    def set_player_types(self, types, type_of_player) -> None:
        """`types`: list of _abi.PlayerType (or dicts of its fields); `type_of_player[j]`: the type of player j (left
        team first), the same in every match - or `type_of_player[e][j]` ([num_envs][num_players]): an assignment of its
        own for every match, as rcssserver hands out its types match by match.  Call before reset(): effort starts at
        the type's effort_max."""
        arr = (_abi.PlayerType * len(types))()
        for k, t in enumerate(types):
            d = t if isinstance(t, dict) else t.as_dict()
            for name, v in d.items():
                setattr(arr[k], name, float(v))
        tof = np.ascontiguousarray(np.asarray(type_of_player, dtype=np.uint8))
        if tof.shape == (self.num_envs, self.num_players):
            setter = self.lib.s2d_set_player_types_per_match
        elif tof.shape == (self.num_players,):
            setter = self.lib.s2d_set_player_types
        else:
            raise ValueError(f"type_of_player needs {self.num_players} entries, or [{self.num_envs}][{self.num_players}]")
        _abi.check(setter(self.handle, arr, len(types), tof.ctypes.data_as(C.POINTER(C.c_uint8))), self.handle)
        self.player_types = [arr[k].as_dict() for k in range(len(types))]
        self.type_of_player = tof.copy()

    # ---- scripted players (fullgame; include/soccer2d.h "FULLGAME scripted players") ------------------------------
    def scripted_mask(self, players) -> int:
        """None / "left" / "right" / an iterable of player indices -> the bit mask of s2d_set_scripted_players"""
        pps = self.num_players // 2
        if players is None:
            return 0
        if isinstance(players, str):
            if players == "left":
                return (1 << pps) - 1
            if players == "right":
                return ((1 << self.num_players) - 1) & ~((1 << pps) - 1)
            raise ValueError(f"scripted_players: {players!r} is not 'left', 'right', None or a list of player indices")
        mask = 0
        for j in players:
            j = int(j)
            if not 0 <= j < self.num_players:
                raise ValueError(f"scripted_players: player {j} does not exist (0..{self.num_players - 1})")
            mask |= 1 << j
        return mask

    def set_scripted_players(self, players) -> None:
        """Players played by the built-in script from the next step on: None (nobody), "left", "right" or an iterable of
        player indices (left team first).  Their rows of the action tensor are ignored.  fullgame only (ValueError)."""
        if self.scenario != "fullgame":
            raise ValueError("scripted players exist in the fullgame scenario only")
        mask = self.scripted_mask(players)
        _abi.check(self.lib.s2d_set_scripted_players(self.handle, mask), self.handle)
        self.scripted_players = tuple(j for j in range(self.num_players) if (mask >> j) & 1)

    def state_dict(self) -> dict:
        return {"state": self.state.clone(), "stats": self.stats_buf.clone(), "seed": self.seed_value,
                "env_id_offset": self.env_id_offset, "num_envs": self.num_envs}

    def load_state_dict(self, sd: dict) -> None:
        assert sd["num_envs"] == self.num_envs and sd["seed"] == self.seed_value and sd["env_id_offset"] == self.env_id_offset
        self.state.copy_(sd["state"])
        self.stats_buf.copy_(sd["stats"])
