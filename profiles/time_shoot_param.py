"""What the parameterized action space costs on Shoot: CUDA-event time per launch of the step kernel on 2^22 envs, K = 1
and K = 16, for the three encodings of the same scenario - Discrete(24) (uint8 rows), S2D_ACT_COMMAND (16-byte rows)
and S2D_ACT_PARAMETERIZED (32-byte rows, translated to the command row in the kernel).  The COMMAND arm is fed the
command rows the PARAM arm's random rows stand for (translated on the device in float32), so those two simulate the
same cycles.  Then the DDPG actor: the fused tcgen05 kernel (s2d_rollout_actor_collect, K cycles per launch) against a
torch actor followed by the step kernel, once per cycle.

Method: the arms run in rounds, in an order that alternates from round to round; each round times ROUND_LAUNCHES
launches per arm with CUDA events (median reported).  No L2 flush: the state alone (80 B x 2^22 = 335 MB) is larger
than the 126 MB L2.  Algorithmic bytes per env: state read + written (160), the action rows, obs (40), reward, done,
result (6); the achieved rate is those bytes over the kernel time.  The card's name and power limit are read in the
same run.

    python profiles/time_shoot_param.py [out.json]
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-soccer-2d-env_b200"))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from soccer2d_b200 import Soccer2DVecEnv  # noqa: E402
from soccer2d_b200.rollout import Actor, mlp_layers  # noqa: E402

N = int(os.environ.get("SHOOT_ENVS", 1 << 22))
ROUNDS, ROUND_LAUNCHES, WARM = 6, 10, 5
HBM_TBS = 7.7  # HGX B200 data sheet, one GPU
dev = torch.device("cuda:0")
ROW_BYTES = {"discrete": 1, "command": 16, "parameterized": 32}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def to_command(a):
    """device float32 translation of parameterized rows [.., 8] into command rows [.., 4] (include/soccer2d.h)"""
    c = torch.nan_to_num(a, nan=1.0).clamp(-1.0, 1.0)
    dash = (c[..., 0] >= c[..., 1]) & (c[..., 0] >= c[..., 2])
    turn = ~dash & (c[..., 1] >= c[..., 2])
    out = torch.zeros(a.shape[:-1] + (4,), device=a.device)
    out[..., 0] = torch.where(dash, 1.0, torch.where(turn, 2.0, 3.0))
    out[..., 1] = torch.where(dash, (c[..., 3] + 1) * 50, torch.where(turn, c[..., 5] * 180, (c[..., 6] + 1) * 50))
    out[..., 2] = torch.where(dash, c[..., 4] * 180, torch.where(turn, torch.zeros_like(c[..., 0]), c[..., 7] * 180))
    return out


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def step_arms(k):
    gen = torch.Generator(device=dev).manual_seed(7)
    envs, pools = {}, {}
    for name in ("discrete", "command", "parameterized"):
        envs[name] = Soccer2DVecEnv(N, scenario="shoot", device=dev, seed=0, substeps=k, max_steps=200,
                                    use_command_action=name == "command", use_parameterized_action=name == "parameterized")
        envs[name].reset_torch()
    par = [torch.rand((N, k, 8), device=dev, generator=gen) * 2 - 1 for _ in range(2)]
    pools["parameterized"] = par
    pools["command"] = [to_command(p) for p in par]
    pools["discrete"] = [torch.randint(0, 24, (N, k), device=dev, dtype=torch.uint8, generator=gen) for _ in range(2)]
    names = list(envs)
    for name in names:
        bench.time_launches(envs[name], pools[name], WARM, None)
    times = {name: [] for name in names}
    for r in range(ROUNDS):
        order = names if r % 2 == 0 else names[::-1]
        for name in order:
            times[name] += bench.time_launches(envs[name], pools[name], ROUND_LAUNCHES, None)
    rows = []
    for name in names:
        ms = median(times[name])
        nbytes = 160 + k * ROW_BYTES[name] + 46
        rows.append(dict(arm="step", action=name, k=k, envs=N, ms_per_launch=round(ms, 4),
                         ns_per_env_cycle=round(ms * 1e6 / (N * k), 4), bytes_per_env_launch=nbytes,
                         achieved_tb_s=round(nbytes * N / (ms * 1e-3) / 1e12, 3),
                         frac_of_hbm_peak=round(nbytes * N / (ms * 1e-3) / 1e12 / HBM_TBS, 3)))
        envs[name].close()
    return rows


def actor_arms(k):
    """fused: one rollout_actor launch plays k cycles; torch: k x (actor forward on the obs, copy into the action
    tensor, s2d_step with K = 1).  Neither writes a trajectory."""
    torch.manual_seed(0)
    actor = Actor(10, 8).to(dev)
    layers = mlp_layers(actor)
    fused = Soccer2DVecEnv(N, scenario="shoot", device=dev, seed=0, substeps=k, use_parameterized_action=True)
    plain = Soccer2DVecEnv(N, scenario="shoot", device=dev, seed=0, substeps=1, use_parameterized_action=True)
    fused.reset_torch()
    plain.reset_torch()

    @torch.no_grad()
    def torch_loop():
        for _ in range(k):
            plain.actions.view(N, 8).copy_(actor(plain.obs))
            plain.step_torch()

    def fused_loop():
        fused.rollout_actor(layers, k)

    arms = {"fused_tcgen05": fused_loop, "torch_actor_then_step": torch_loop}
    for f in arms.values():
        for _ in range(WARM):
            f()
    times = {name: [] for name in arms}
    for r in range(ROUNDS):
        for name in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            for _ in range(ROUND_LAUNCHES):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                arms[name]()
                e.record()
                torch.cuda.synchronize()
                times[name].append(s.elapsed_time(e))
    rows = [dict(arm="actor", path=name, k=k, envs=N, ms_per_k_cycles=round(median(times[name]), 4),
                 ns_per_env_cycle=round(median(times[name]) * 1e6 / (N * k), 4)) for name in arms]
    fused.close()
    plain.close()
    return rows


def main():
    gpu = card()
    out = []
    for k in (1, 16):
        for row in step_arms(k) + actor_arms(k):
            row["gpu"] = gpu
            print(json.dumps(row), flush=True)
            out.append(row)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
