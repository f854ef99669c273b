"""Soccer2DEnv - the gym.Env base class of the reference (soccer_2d_env.py:23-446), same public surface,
new internals.

The reference's constructor spawns a gRPC server process, an rcssserver and a proxy, and every `step`
blocks on four multiprocessing queues (soccer_2d_env.py:226-269).  Here the episode lives in GPU memory
inside a one-env `Soccer2DVecEnv` and `step` is one C-ABI call (s2d_step): one fused kernel (decode + server
cycle + reward/done + observation) that reads the action from and writes the results to pinned host memory.

Kept: constructor signature (`render_mode, run_grpc_server, run_rcssserver, run_trainer_player, logger,
log_dir`; the three run_* flags are accepted and ignored - there is nothing to spawn), `metadata`,
`action_space` / `observation_space`, `reset() -> obs`, `step(a) -> (obs, reward, done, info)` (old-gym
4-tuple, soccer_2d_env.py:269), `render`, idempotent `close`, and the four scenario hooks
(soccer_2d_env.py:317-354).

Two ways to define a scenario:
  * fused (ReachBallEnv, ShootEnv, FullGameEnv): decode, reward/done and observation run inside the kernel; the
    hooks are not called.  This is the fast path.
  * hooks: a subclass that overrides the reference's four hooks - `action_to_rpc_actions`, `state_to_observation`,
    `check_trainer_observation`, `trainer_reset_actions` - keeps working as it does on the reference: per step the
    hook's PlayerAction (Dash / Turn / Kick / Body_GoToPoint / Body_TurnToPoint / Body_TurnToBall / Body_TurnToAngle /
    Body_KickOneStep / Body_SmartKick (its first kick) / Body_StopBall / Body_Intercept / Body_HoldBall; `service_pb2` messages or
    soccer2d_b200.pb2_lite ones) becomes one command for the GPU cycle, and the other hooks are fed proto-shaped
    State objects (real `service_pb2.State` when that module is importable, attribute views otherwise).  The physics
    still runs on the GPU; the Python hooks make it the slow, compatible path.
Dropped by construction: queues, cycle-desync repair (`_wait_for_agents`, :141-177), per-step logging.
"""
from __future__ import annotations

import logging
import warnings

import numpy as np
import torch

from soccer2d_b200 import _abi, pb2_lite
from soccer2d_b200.proto_state import state_dict, trainer_state_dict
from soccer2d_b200.spaces import Box, Discrete, Env
from soccer2d_b200.vec_env import Soccer2DVecEnv

_HOOKS = ("action_to_rpc_actions", "state_to_observation", "check_trainer_observation", "trainer_reset_actions")


class Soccer2DEnv(Env):
    metadata = {"render.modes": ["human"]}  # soccer_2d_env.py:28
    scenario = "reachball"

    def __init__(self, render_mode: str = None, run_grpc_server: bool = True, run_rcssserver: bool = True,
                 run_trainer_player: bool = True, logger: logging.Logger = None, log_dir: str = None,
                 *, device="cuda", seed: int = 0, server_param: dict | None = None, use_command_action: bool = False,
                 noise: bool = False, **scenario_kwargs):
        self.log_dir = log_dir
        self.logger = logger
        if self.logger is None:
            self.logger = logging.getLogger(type(self).__name__)
            self.logger.addHandler(logging.NullHandler())
        self.render_mode = render_mode
        self.run_grpc_server = run_grpc_server      # accepted for signature compatibility; nothing is spawned
        self.run_rcssserver = run_rcssserver
        self.run_trainer_player = run_trainer_player
        # defaults of the reference base class (soccer_2d_env.py:58-59); scenario classes replace them
        self.action_space = Discrete(4)
        self.observation_space = Box(low=-1, high=1, shape=(2,), dtype=np.float32)
        # a subclass that overrides the reference's four hooks defines its scenario in Python (module docstring)
        self._hook_mode = all(getattr(type(self), h) is not getattr(Soccer2DEnv, h) for h in _HOOKS)
        if self._hook_mode:
            # the kernel only runs the physics: command actions, its own scoring switched off (never done)
            self._vec = Soccer2DVecEnv(1, scenario="reachball", device=device, seed=seed, substeps=1, auto_reset=False,
                                       server_param=server_param, use_command_action=True, noise=noise, host_mapped_io=True,
                                       goto_dist_thr=scenario_kwargs.pop("goto_dist_thr", 0.5),
                                       min_distance_to_ball=-1.0, max_steps=2**31 - 1)
            # rcssserver gives a player full stamina / effort / recovery when it connects: start from a recovered
            # player even if the subclass's trainer_reset_actions sends no DoRecover
            self._vec.reset_torch()
            torch.cuda.current_stream(self._vec.device).synchronize()
            self._pb2 = self._find_pb2()
            self._latest_player_state = None
            self._latest_trainer_state = None
        else:
            self._vec = Soccer2DVecEnv(1, scenario=self.scenario, device=device, seed=seed, substeps=1, auto_reset=False,
                                       server_param=server_param, use_command_action=use_command_action,
                                       noise=noise, host_mapped_io=True, **scenario_kwargs)
            self.action_space = self._vec.action_space
            self.observation_space = self._vec.observation_space
        self.step_number = 0
        self.logger.info("Soccer2DEnv ready: 1 episode on %s (no rcssserver / proxy / gRPC processes)", self._vec.device)

    # ---- gym API ------------------------------------------------------------------------------------
    def reset(self) -> np.ndarray:
        return self.abs_reset()

    def abs_reset(self) -> np.ndarray:
        player_observation, _trainer_state = self.env_reset()
        return player_observation

    def env_reset(self) -> tuple:
        """Placement, recover, one idle server cycle, reward priming - all inside s2d_reset
        (soccer_2d_env.py:179-206 + reach_ball_env.py:163-197).  Returns (obs, snapshot of the env); in hook mode
        (obs, trainer State) exactly like the reference."""
        if self._hook_mode:
            return self._hook_env_reset()
        obs = self._vec.reset()
        self.step_number = 0
        return obs[0].copy(), self._vec.export_env(0)

    def step(self, action) -> tuple:
        if self._hook_mode:
            return self._hook_step(action)
        a = self._shape_action(action)
        obs, reward, done, result = self._vec.step_host(a)
        self.step_number += 1
        return obs[0].copy(), float(reward[0]), bool(done[0]), {"result": _abi.RESULT_NAMES[int(result[0])]}

    def render(self, mode="human"):
        return None

    def close(self):
        vec = getattr(self, "_vec", None)
        if vec is not None:
            vec.close()

    # ---- hook mode: the reference's control flow (soccer_2d_env.py:179-269) on top of the GPU cycle -----
    @staticmethod
    def _find_pb2():
        try:
            import service_pb2  # the reference's generated module, if the user has it on the path
            from google.protobuf import json_format  # noqa: F401
            return service_pb2
        except Exception:  # noqa: BLE001
            return None

    def _states(self):
        snap = self._vec.export_env(0)
        player, trainer = state_dict(snap, unum=1, side=1), trainer_state_dict(snap)
        if self._pb2 is not None:
            from google.protobuf import json_format
            return (json_format.ParseDict(player, self._pb2.State()), json_format.ParseDict(trainer, self._pb2.State()))
        return pb2_lite.View(player), pb2_lite.View(trainer)

    def _command_from(self, action) -> np.ndarray:
        """proto PlayerAction (or a list with one) -> {cmd, a, b, c}"""
        if isinstance(action, (list, tuple)):
            action = action[0] if action else None
        cmd = np.zeros((1, 1, 4), np.float32)
        which = action.WhichOneof("action") if action is not None else None
        if which == "dash":
            cmd[0, 0] = [_abi.CMD_DASH, float(action.dash.power), float(action.dash.relative_direction), 0.0]
        elif which == "turn":
            cmd[0, 0] = [_abi.CMD_TURN, float(action.turn.relative_direction), 0.0, 0.0]
        elif which == "kick":
            cmd[0, 0] = [_abi.CMD_KICK, float(action.kick.power), float(action.kick.relative_direction), 0.0]
        elif which == "body_go_to_point":
            g = action.body_go_to_point
            thr = float(g.distance_threshold)
            if thr and abs(thr - self._vec.cfg.goto_dist_thr) > 1e-6:
                warnings.warn(f"Body_GoToPoint.distance_threshold {thr} ignored: the handle was created with "
                              f"goto_dist_thr={self._vec.cfg.goto_dist_thr}", stacklevel=3)
            cmd[0, 0] = [_abi.CMD_GOTO, float(g.target_point.x), float(g.target_point.y), float(g.max_dash_power) or 100.0]
        elif which == "body_turn_to_point":
            t = action.body_turn_to_point
            cmd[0, 0] = [_abi.CMD_TURN_TO_POINT, float(t.target_point.x), float(t.target_point.y), float(t.cycle) or 1.0]
        elif which == "body_turn_to_ball":
            cmd[0, 0] = [_abi.CMD_TURN_TO_BALL, float(action.body_turn_to_ball.cycle) or 1.0, 0.0, 0.0]
        elif which == "body_turn_to_angle":
            cmd[0, 0] = [_abi.CMD_TURN_TO_ANGLE, float(action.body_turn_to_angle.angle), 0.0, 0.0]
        elif which == "body_kick_one_step":
            k = action.body_kick_one_step  # (force_mode semantics: the kick is made even if first_speed cannot be reached)
            cmd[0, 0] = [_abi.CMD_KICK_ONE_STEP, float(k.target_point.x), float(k.target_point.y), float(k.first_speed)]
        elif which == "body_smart_kick":
            k = action.body_smart_kick  # staged over 2-3 cycles when one kick cannot reach first_speed (include/soccer2d.h)
            cmd[0, 0] = [_abi.CMD_SMART_KICK, float(k.target_point.x), float(k.target_point.y), float(k.first_speed)]
        elif which == "body_stop_ball":
            cmd[0, 0] = [_abi.CMD_STOP_BALL, 0.0, 0.0, 0.0]
        elif which == "body_intercept":
            cmd[0, 0] = [_abi.CMD_INTERCEPT, 0.0, 0.0, 0.0]
        elif which not in (None, "body_hold_ball"):
            warnings.warn(f"PlayerAction.{which} is not simulated; the player does nothing this cycle", stacklevel=3)
        return cmd

    def _apply_trainer_actions(self, actions) -> None:
        """DoMoveBall / DoMovePlayer / DoRecover / DoChangeMode on env 0 (applied on receipt, before the cycle)"""
        if not isinstance(actions, (list, tuple)):
            actions = [actions]
        f, _ = self._vec.state_planes()
        sp = self._vec.cfg.sp
        torch.cuda.current_stream(self._vec.device).synchronize()
        for a in actions:
            which = a.WhichOneof("action")
            if which == "do_move_ball":
                m = a.do_move_ball
                f[2, 0] = torch.tensor([float(m.position.x), float(m.position.y), float(m.velocity.x), float(m.velocity.y)],
                                       device=f.device)
            elif which == "do_move_player":
                m = a.do_move_player
                body = float(m.body_direction)
                body = body - 360.0 if body > 180.0 else body + 360.0 if body < -180.0 else body
                f[0, 0] = torch.tensor([float(m.position.x), float(m.position.y), 0.0, 0.0], device=f.device)
                f[1, 0, 0] = body
            elif which == "do_recover":
                f[1, 0, 1:] = torch.tensor([sp.stamina_max, sp.effort_max, sp.recover_init], device=f.device)
                f[3, 0, 2] = sp.stamina_capacity
            # do_change_mode(PlayOn): the one-player scenarios are always PlayOn (soccer_2d_env.py:242)

    def _hook_cycle(self, cmd):
        self._vec.step_host(cmd)
        self._latest_player_state, self._latest_trainer_state = self._states()

    def _hook_env_reset(self):
        self._apply_trainer_actions(self.trainer_reset_actions())
        self._hook_cycle(np.zeros((1, 1, 4), np.float32))  # Body_HoldBall: the idle cycle of the reference's reset
        return self.state_to_observation(self._latest_player_state), self._latest_trainer_state

    def _hook_step(self, action):
        cmd = self._command_from(self.action_to_rpc_actions(action, self._latest_player_state))
        self._hook_cycle(cmd)
        player_observation = self.state_to_observation(self._latest_player_state)
        done, reward, info = self.check_trainer_observation(self._latest_trainer_state)
        return player_observation, reward, done, info

    # ---- helpers ------------------------------------------------------------------------------------
    def _shape_action(self, action):
        mode = self._vec.action_mode
        if mode == _abi.ACT_DISCRETE:
            a = int(np.asarray(action).reshape(-1)[0])
            n = self._vec.cfg.action_space_size
            if not 0 <= a < n:
                raise ValueError(f"discrete action {a} outside Discrete({n})")
            return np.array([[a]], dtype=np.uint8)
        a = np.asarray(action, dtype=np.float32).reshape(-1)
        want = 8 if mode == _abi.ACT_PARAMETERIZED else 4 if mode in (_abi.ACT_TURNING, _abi.ACT_COMMAND) else 1
        if a.size != want:
            raise ValueError(f"expected an action with {want} value(s), got shape {np.asarray(action).shape}")
        return a.reshape((1, 1, want) if want > 1 else (1, 1))

    @property
    def distance_to_ball(self) -> float:
        return float(self._vec.export_env(0).mem_distance_to_ball)

    @property
    def body_ball_angle_diff(self) -> float:
        return float(self._vec.export_env(0).mem_body_ball_angle_diff)

    # ---- the reference's scenario hooks (soccer_2d_env.py:317-354): names kept for subclasses that
    # ---- introspect them; the GPU path does not call them -------------------------------------------
    def action_to_rpc_actions(self, action, player_state=None):
        raise NotImplementedError("action decode is fused into the step kernel (csrc/s2d_scenarios.cuh)")

    def state_to_observation(self, state=None):
        raise NotImplementedError("observation build is fused into the step kernel (csrc/s2d_scenarios.cuh)")

    def check_trainer_observation(self, observation=None):
        raise NotImplementedError("reward/done is fused into the step kernel (csrc/s2d_scenarios.cuh)")

    def trainer_reset_actions(self):
        raise NotImplementedError("reset placement is drawn inside the reset kernel (csrc/s2d_scenarios.cuh)")
