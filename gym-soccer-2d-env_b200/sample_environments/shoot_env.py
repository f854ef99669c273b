"""ShootEnv - 1v0 shoot-on-goal (BASELINE configs[2]): one player has to take the ball and score in the right goal.

Not part of the reference (whose only scenario is ReachBall); it exists to exercise the kick model, the
kickable-area test and goal / ball-out detection behind the same gym API.  The scenario contract (reset, reward,
done, result names) is specified in include/soccer2d.h and implemented in csrc/s2d_scenarios.cuh (check_shoot).
Observation: the same 10 values as ReachBall.  Actions: Discrete(action_space_size) = dashes + `kick_actions` kicks,
proto-style commands with use_command_action=True (Dash / Turn / Kick / Body_GoToPoint), or with
use_parameterized_action=True HFO's parameterized Box(8): weights of dash / turn / kick and their continuous arguments.
"""
from __future__ import annotations

from soccer_2d_env import Soccer2DEnv
from soccer2d_b200.vec_env import SHOOT_DEFAULTS


class ShootEnv(Soccer2DEnv):
    scenario = "shoot"

    def __init__(self, render_mode=None, logger=None, log_dir=None, *, device="cuda", seed: int = 0,
                 server_param: dict | None = None, use_command_action: bool = False, noise: bool = False,
                 **kwargs):
        known = {k: kwargs[k] for k in SHOOT_DEFAULTS if k in kwargs}
        super().__init__(render_mode, logger=logger, log_dir=log_dir, device=device, seed=seed,
                         server_param=server_param, use_command_action=use_command_action, noise=noise, **known)
        for k, v in dict(SHOOT_DEFAULTS, **known).items():
            setattr(self, k, v)
