"""Launch times (CUDA events, ms, median) of the kernels other than the K = 16 ReachBall Discrete(16) step kernel that share
the end-of-episode code (csrc/s2d_scenarios.cuh, end_of_episode), for whichever libsoccer2d build S2D_LIB names (default:
the in-tree build), so that two builds can be timed alternately on the same card in one session:

  box1_k16       ReachBall Box(1) step kernel, 2^20 envs, K = 16
  shoot_k16      Shoot Discrete(24) step kernel, 2^22 envs, K = 16
  shoot_cmd_k1   Shoot command step kernel, 2^22 envs, K = 1
  mlp_tf32_k16   fused DQN policy + step (rollout_mlp, tcgen05 TF32), 2^20 envs, K = 16
  actor_k16      fused DDPG actor + step (rollout_actor, ReachBall Box(4)), 2^20 envs, K = 16

Every timed launch follows 160 untimed ones after a reset (episode ages mixed) and an untimed 256 MB clear of the L2.
Prints one JSON line with the library, the card and its power limit."""
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-soccer-2d-env_b200"))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import torch  # noqa: E402

from soccer2d_b200 import Soccer2DVecEnv, _abi  # noqa: E402
from soccer2d_b200.rollout import Actor, QNetwork, mlp_layers  # noqa: E402
from time_step_ab import card  # noqa: E402

WARM, TIMED = 160, 100
dev = torch.device("cuda:0")
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
gen = torch.Generator(device=dev).manual_seed(7)


def timed(launch):
    """median ms of TIMED launches after WARM untimed ones"""
    for i in range(WARM):
        launch(i)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(TIMED)]
    for i, (a, b) in enumerate(ev):
        flush.zero_()
        a.record()
        launch(i)
        b.record()
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in ev)


def step_launch(env, pool):
    def launch(i):
        env.bind_actions(pool[i % len(pool)])
        env.step_torch()
    return launch


def commands(shape):
    a = torch.zeros(shape + (4,), device=dev)
    cmd = torch.randint(0, 5, shape, device=dev, generator=gen)
    a[..., 0] = cmd.float()
    a[..., 1] = torch.rand(shape, device=dev, generator=gen) * 100
    a[..., 2] = torch.rand(shape, device=dev, generator=gen) * 360 - 180
    a[..., 3] = 100.0
    return a


def main():
    out = {"lib": os.path.relpath(_abi.LIB_PATH, ROOT), "card": card()}
    reach = dict(change_ball_position=True, change_ball_velocity=True)

    env = Soccer2DVecEnv(1 << 20, device=dev, seed=0, substeps=16, use_continuous_action=True, **reach)
    env.reset_torch()
    pool = [torch.rand(env.actions.shape, device=dev, generator=gen) * 2 - 1 for _ in range(4)]
    out["box1_k16"] = timed(step_launch(env, pool))
    env.close()

    for name, k, command in (("shoot_k16", 16, False), ("shoot_cmd_k1", 1, True)):
        n = 1 << 22
        env = Soccer2DVecEnv(n, scenario="shoot", device=dev, seed=0, substeps=k, use_command_action=command)
        env.reset_torch()
        pool = ([commands((n, k)) for _ in range(2)] if command else
                [torch.randint(0, 24, (n, k), dtype=torch.uint8, device=dev, generator=gen) for _ in range(4)])
        out[name] = timed(step_launch(env, pool))
        env.close()
        del pool

    torch.manual_seed(0)
    env = Soccer2DVecEnv(1 << 20, device=dev, seed=0, substeps=16, use_continuous_action=False, action_space_size=16, **reach)
    env.reset_torch()
    layers = mlp_layers(QNetwork(10, 16).to(dev))
    out["mlp_tf32_k16"] = timed(lambda i: env.rollout_mlp(layers, 16, precision="tf32"))
    env.close()

    env = Soccer2DVecEnv(1 << 20, device=dev, seed=0, substeps=16, use_continuous_action=True, use_turning=True, **reach)
    env.reset_torch()
    layers = mlp_layers(Actor(10, 4).to(dev))
    out["actor_k16"] = timed(lambda i: env.rollout_actor(layers, 16, precision="tf32"))
    env.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
