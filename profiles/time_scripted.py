"""What scripted players cost: CUDA-event time per launch of the 11 v 11 step kernel on 2^18 matches, K = 1 and K = 16,
for three workloads - (a) nobody scripted, every player on bench.commands (bench.py's random mix); (b) the right team
scripted, the left on bench.commands; (c) all 22 players scripted.  Every workload first plays WARM_CYCLES cycles (past
the first 400 of a match: formation, kick-off and first goals are behind), then is timed; then it plays on while goals
and play modes are counted.  Prints one JSON line per workload, with the card's name and power limit.

    python profiles/time_scripted.py [out.json]
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

N = int(os.environ.get("FG_MATCHES", 1 << 18))
WARM_CYCLES, TIMED_CYCLES, COUNT_CYCLES = 480, 320, 800
dev = torch.device("cuda:0")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def run(workload, k):
    gen = torch.Generator(device=dev).manual_seed(99)
    # half_time_cycles large: no match ends inside the window, so every cycle is a match-cycle of play
    env = Soccer2DVecEnv(N, scenario="fullgame", device=dev, seed=0, substeps=k, half_time_cycles=100000,
                         scripted_players={"a": None, "b": "right", "c": "left"}[workload])
    if workload == "c":
        env.set_scripted_players(range(22))
    pool = [bench.commands(torch, gen, dev, (N, k, 22)) for _ in range(2)]
    env.reset_torch()
    bench.time_launches(env, pool, WARM_CYCLES // k, None)  # warm-up: modules loaded, matches well under way
    ms = bench.time_launches(env, pool, max(TIMED_CYCLES // k, 20), None)
    us = sorted(x * 1e3 for x in ms)
    median = us[len(us) // 2]
    g0 = env.fullgame_planes()["ej"][:, :2].long().sum()
    hist = torch.zeros(9, dtype=torch.long, device=dev)
    for _ in range(COUNT_CYCLES // k):
        env.bind_actions(pool[0])
        env.step_torch()
        hist += torch.bincount((env.fullgame_planes()["ei"][:, 3] & 0xff).long(), minlength=9)[:9]
    goals = int(env.fullgame_planes()["ej"][:, :2].long().sum() - g0)
    counted = N * (COUNT_CYCLES // k) * k
    out = dict(workload=workload, k=k, matches=N, us_per_launch_median=round(median, 1),
               us_per_launch_mean=round(sum(us) / len(us), 1),
               match_cycles_per_s=round(N * k / (median * 1e-6)),
               goals_per_1000_match_cycles=round(goals * 1000.0 / counted, 4),
               play_modes_at_launch_end={name: int(v) for name, v in zip(
                   ["BeforeKickOff", "TimeOver", "PlayOn", "KickOff", "KickIn", "FreeKick", "CornerKick", "GoalKick",
                    "AfterGoal"], hist.tolist())})
    env.close()
    return out


def main():
    rows = []
    gpu = card()
    for k in (1, 16):
        for w in ("a", "b", "c"):
            r = dict(run(w, k), gpu=gpu)
            print(json.dumps(r), flush=True)
            rows.append(r)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
