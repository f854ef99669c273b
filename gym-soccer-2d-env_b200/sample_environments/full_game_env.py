"""FullGameEnv - a whole match, up to 11 v 11 (BASELINE configs[3]) behind the gym API: every step takes one
proto-style command {cmd, a, b, c} per player (shape [2 * players_per_side, 4]: Dash / Turn / Kick / Body_GoToPoint)
and returns the 120-value global observation (ball, 22 x {x, y, vx, vy, body}, play mode, side, scores, time), the
left team's reward, done at time over and info['result'] in {'Goal' (left wins), 'Out' (right wins), 'Timeout' (draw)}.

scripted_players (None, "left", "right" or a list of player indices) hands players to the built-in script that runs in
the step kernel (include/soccer2d.h, "FULLGAME scripted players"): the action then holds one command per CONTROLLED
player only, shape [n_controlled, 4], the non-scripted players in index order.  The reward is still the left team's
view, whichever team is scripted: to train the right team against a scripted left, negate it.

Not part of the reference (one player, referee off); spec in include/soccer2d.h, kernels in csrc/s2d_fullgame.cuh.
"""
from __future__ import annotations

import numpy as np

from soccer_2d_env import Soccer2DEnv
from soccer2d_b200.spaces import Box
from soccer2d_b200.vec_env import FULLGAME_DEFAULTS


class FullGameEnv(Soccer2DEnv):
    scenario = "fullgame"

    def __init__(self, render_mode=None, logger=None, log_dir=None, *, device="cuda", seed: int = 0,
                 server_param: dict | None = None, noise: bool = False, scripted_players=None, **kwargs):
        known = {k: kwargs[k] for k in FULLGAME_DEFAULTS if k in kwargs}
        super().__init__(render_mode, logger=logger, log_dir=log_dir, device=device, seed=seed,
                         server_param=server_param, noise=noise, **known)
        for k, v in dict(FULLGAME_DEFAULTS, **known).items():
            setattr(self, k, v)
        self._full_action_space = self.action_space
        self.set_scripted_players(scripted_players)

    def set_scripted_players(self, players) -> None:
        """None / "left" / "right" / player indices: who the built-in script plays; action_space shrinks to the others"""
        self._vec.set_scripted_players(players)
        self.scripted_players = self._vec.scripted_players
        self.controlled_players = tuple(j for j in range(self._vec.num_players) if j not in self.scripted_players)
        full = self._full_action_space
        rows = list(self.controlled_players)
        self.action_space = Box(low=full.low[rows], high=full.high[rows], dtype=np.float32)

    def _shape_action(self, action):
        a = np.asarray(action, dtype=np.float32)
        want = (len(self.controlled_players), 4)
        if a.shape != want:
            raise ValueError(f"expected one command per controlled player, shape {want}, got {a.shape}")
        full = np.zeros((1, 1, self._vec.num_players, 4), np.float32)  # (the scripted players' rows are ignored)
        full[0, 0, list(self.controlled_players)] = a
        return full
