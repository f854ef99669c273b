#!/usr/bin/env python
"""DDPG on ReachBall (continuous Dash direction) with the lockstep GPU simulator - the counterpart of the reference's
ddpg_stable_baselines3.py (:18-31 env kwargs: fixed ball at the centre, Box(-1, 1, (1,)) action; :36-62 train / test).
`--scenario shoot`: DDPG on Shoot (1v0 shoot-on-goal) with HFO's parameterized dash / turn / kick action space, Box(8)
(Hausknecht & Stone 2016, PAPERS.md); the test line then carries the goal / out / timeout rates.

    python gym-soccer-2d-env_b200/ddpg_b200.py --envs 4096 --steps 3000
    python gym-soccer-2d-env_b200/ddpg_b200.py --scenario shoot --envs 4096 --steps 3000 --fused 8
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from soccer2d_b200 import Soccer2DVecEnv  # noqa: E402
from soccer2d_b200.vec_env import SHOOT_DEFAULTS  # noqa: E402
from soccer2d_b200.rollout import DDPGConfig, DeviceDDPG  # noqa: E402

# ddpg_stable_baselines3.py:18-31
KWARGS = dict(change_ball_position=False, change_ball_velocity=False, ball_position_x=0, ball_position_y=0, ball_speed=0,
              ball_direction=0, min_distance_to_ball=5.0, max_steps=200, action_space_size=16, use_continuous_action=True,
              use_turning=False)
SHOOT_KWARGS = dict(SHOOT_DEFAULTS, use_parameterized_action=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenario", choices=("reachball", "shoot"), default="reachball")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--test-steps", type=int, default=400)
    ap.add_argument("--report-every", type=int, default=500)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--fused", type=int, default=0, metavar="K",
                    help="collect the rollout with the actor inside the step kernel, K cycles per launch (0: torch actor)")
    args = ap.parse_args()
    kwargs = SHOOT_KWARGS if args.scenario == "shoot" else KWARGS
    env = Soccer2DVecEnv(args.envs, scenario=args.scenario, device=args.device, seed=args.seed, terminal_obs=True, **kwargs)
    agent = DeviceDDPG(env, DDPGConfig(seed=args.seed, learning_starts=min(1 << 16, 16 * args.envs)))
    log = (agent.learn_fused(args.steps, k=args.fused, report_every=args.report_every) if args.fused
           else agent.learn(args.steps, report_every=args.report_every))
    for rep in log:
        print(json.dumps(rep), flush=True)
    print(json.dumps({"test": agent.evaluate(args.test_steps, fused=bool(args.fused))}), flush=True)
    env.close()


if __name__ == "__main__":
    main()
