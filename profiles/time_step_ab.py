"""K = 16 ReachBall step launch time (CUDA events, ms) in three regimes, for whichever libsoccer2d build S2D_LIB names
(default: the in-tree build), so that two builds can be timed alternately on the same card in one session:

  steady   the bench configuration, launches 160 .. 359 after a reset (episode ages mixed as in the benchmark)
  young    the bench configuration, the first 10 launches after a reset, over 8 resets (every episode young)
  no_end   episodes that never end by goal or time-out (min_distance_to_ball = 0, max_steps = 2^30), launches 160 .. 359

The actions cycle through a pool of four random [N][K] byte tensors and a 256 MB buffer is cleared before every timed
launch (untimed), as in bench.py.  Prints one JSON line: median and mean per regime, the library, the card and its
power limit."""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-soccer-2d-env_b200"))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from soccer2d_b200 import Soccer2DVecEnv, _abi  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0)


def summary(ms):
    return {"median_ms": statistics.median(ms), "mean_ms": statistics.fmean(ms), "launches": len(ms)}


def main():
    n, k = 1 << 20, 16
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(1234)
    pool = [torch.randint(0, 16, (n, k), dtype=torch.uint8, device=dev, generator=gen) for _ in range(4)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"lib": os.path.relpath(_abi.LIB_PATH, ROOT), "card": card(), "n_envs": n, "k": k}

    env = Soccer2DVecEnv(n, device=dev, seed=0, substeps=k, **bench.SCENARIO_KW)
    young = []
    for _ in range(8):
        env.reset_torch()
        young += bench.time_launches(env, pool, 10, flush)
    env.reset_torch()
    bench.time_launches(env, pool, 160, flush)
    out["steady"] = summary(bench.time_launches(env, pool, 200, flush))
    out["young"] = summary(young)
    env.close()

    env = Soccer2DVecEnv(n, device=dev, seed=0, substeps=k, **dict(bench.SCENARIO_KW, min_distance_to_ball=0.0, max_steps=1 << 30))
    env.reset_torch()
    bench.time_launches(env, pool, 160, flush)
    out["no_end"] = summary(bench.time_launches(env, pool, 200, flush))
    env.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
