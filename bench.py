#!/usr/bin/env python
"""bench.py - env-steps/sec of the lockstep ReachBall step path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one launch of the fused step kernel over one batch of synthetic actions: 2^20 ReachBall episodes per
GPU x 16 fused cycles (BASELINE.json configs[1]); weak scaling: every rank holds its own 2^20 episodes (global
env ids rank*2^20 ...), no data-path collective, one NCCL all-reduce of the episode statistics after the timed
region.  One JSON line is printed by rank 0.

  value      env-steps/s with actions and state resident in HBM, sum of per-launch CUDA-event durations
             (L2 flushed between launches, flush not timed), max over ranks
  e2e        the same workload through the host-buffer calls of the C ABI (s2d_submit_host / s2d_wait_host): pinned
             host actions -> H2D -> kernel -> ONE D2H of the packed obs/reward/done/result block, three steps in
             flight, the host reads every step's result; wall clock between barriers, max over ranks.
             `pcie_probe` = plain cudaMemcpyAsync of the same byte counts (both directions at once, all ranks at once):
             the ceiling this box gives that path; `frac_of_probe` = e2e / probe
  roofline   the step kernel at the bench workload (K = 16): algorithmic bytes / launch time vs the measured
             HBM copy peak; `roofline_k1` is the same kernel in its HBM-bound regime (closed loop, K = 1)
  shoot, fullgame   BASELINE configs[2] / [3] (4M shoot-on-goal envs, 256K 11v11 matches, sharded over the ranks):
             value, launch time, roofline fraction and e2e of each, measured in the same run
  cpu_baseline  the C oracle (oracle/s2d_oracle.c, f64, OpenMP) on this box's host cores, bounded sample

--impl reference times that CPU oracle alone on the SAME workload (2^20 envs x 16 cycles per step).  The reference's own
step path needs rcssserver + the C++ proxy, external binaries that cannot run offline; the oracle is the CPU restatement
of the same path.  That arm imports neither the product package nor libsoccer2d.so.

--dump-outputs DIR writes what the last timed launch of the B200 arm returned (rank 0's envs): obs.npy, reward.npy,
done.npy, result.npy as float32, and env_index.npy (float64), the env of each row.  Actions and the env seed are fixed,
so two builds run with the same arguments can be compared output for output.  Above 64 MB a fixed, seeded sample of
the envs is written.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "gym-soccer-2d-env_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
ENVS_PER_GPU = 1 << 20
SUBSTEPS = 16
# ReachBall as the reference's DQN script configures it (dqn_stable_baselines3.py:17-31), noise off
SCENARIO_KW = dict(use_continuous_action=False, action_space_size=16, change_ball_position=True,
                   change_ball_velocity=True, min_distance_to_ball=5.0, max_steps=200)
STATE_BYTES, OBS_BYTES, OUT_BYTES = 80, 40, 6  # per env: state planes; obs row; reward + done + result
FG_STATE_BYTES, FG_OBS_BYTES = 22 * 36 + 80, 480  # per 11v11 match: 22 players x 9 words + 16 match words + 16 B of tackle / catch counters
DUMP_BYTES = 64 * 10**6 - 4096  # --dump-outputs budget, less room for the .npy headers


def algorithmic_bytes_per_env(k):
    """state read + state write + k action bytes + obs/reward/done/result written once per launch (DESIGN.md)"""
    return 2 * STATE_BYTES + k + OBS_BYTES + OUT_BYTES


def workload_config(n_gpus, envs, k):
    """The `config` of the JSON line - the same dict, key for key, in the B200 arm and in the reference arm."""
    return {"workload": f"ReachBall {envs} lockstep envs per GPU (1 player + ball, dash only, Discrete(16)), "
                        f"fused K={k} substeps per launch, noise off, auto-reset",
            "envs_per_gpu": envs, "substeps": k, "global_envs": envs * n_gpus,
            "scenario_kwargs": SCENARIO_KW, "parallelism": f"episode-shard x{n_gpus}",
            "l2": "B200 arm: L2 flushed between timed launches (256 MiB memset, not timed), the K=1 run uses a working "
                  "set >> L2; CPU arm: 2^20 envs of state (>> last-level cache) streamed every step",
            "timing": "B200 arm: sum of per-launch CUDA-event durations on the launching stream, max over ranks; CPU arm: "
                      "wall clock around the timed steps"}


def load_traffic(key, envs, field="traffic_bytes"):
    """DRAM bytes per launch (or another recorded ncu figure) of the step kernel from the committed ncu capture
    (profiles/traffic.json); None if the capture was taken at another size."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)[f"{key}_envs_{envs}"][field]
    except Exception:  # noqa: BLE001
        return None


def load_parity():
    """fp32-vs-f64 flag-flip rate measured over ALL seeds (profiles/flag_flips.py -> profiles/parity_flips.json)"""
    try:
        with open(os.path.join(ROOT, "profiles", "parity_flips.json")) as f:
            return json.load(f)
    except Exception:  # noqa: BLE001
        return None


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock + throttle reasons of one GPU while the timed regions run (NVML)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.mask, self.max_mhz, self.stop_flag, self.error = index, [], 0, None, False, None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = None
            try:
                import torch
                uuid = "GPU-" + str(torch.cuda.get_device_properties(self.index).uuid)
            except Exception:  # noqa: BLE001
                pass
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID(uuid) if uuid else pynvml.nvmlDeviceGetHandleByIndex(self.index)
            except Exception:  # noqa: BLE001
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self.stop_flag:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=2)
        s = sorted(self.samples)
        out = {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
               "reasons": [n for b, n in self.REASONS.items() if self.mask & b], "samples": len(s)}
        if self.error:
            out["error"] = self.error
        return out


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


# ---- the CPU arm: oracle only (tests/oracle_lib.py -> oracle/_build/liboracle_f64.so); no product import ---------
def time_cpu_oracle(envs, k, min_seconds, max_launches=10**9, warmup=1, fixed_launches=None):
    """env-steps/s of the C oracle (f64 build, OpenMP over all host cores) on `envs` episodes x k cycles per call."""
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm is meant to use every host thread it can
    os.environ["OMP_NUM_THREADS"] = str(host_threads())
    import numpy as np

    import oracle_lib as OL
    cfg = OL.default_config(envs, 0, action_mode=OL.ACT_DISCRETE, seed=0, change_ball_velocity=1,
                            change_ball_position=1, max_steps=SCENARIO_KW["max_steps"],
                            min_distance_to_ball=SCENARIO_KW["min_distance_to_ball"],
                            action_space_size=SCENARIO_KW["action_space_size"])
    sim = OL.OracleSim(cfg, "f64")
    OL.lib("f64").s2do_set_threads(host_threads())
    sim.reset()
    rng = np.random.default_rng(0)
    pool = [rng.integers(0, 16, size=(envs, k)).astype(np.uint8) for _ in range(2)]
    for i in range(warmup):
        sim.step(pool[i % 2], k)
    launches, t0 = 0, time.perf_counter()
    while True:
        sim.step(pool[launches % 2], k)
        launches += 1
        dt = time.perf_counter() - t0
        if fixed_launches is not None:
            if launches >= fixed_launches:
                break
        elif dt >= min_seconds or launches >= max_launches:
            break
    sim.close()
    return envs * k * launches / dt, launches, dt


def run_reference(args, rank):
    if rank != 0:
        return
    envs, k = args.envs, args.substeps
    value, launches, dt = time_cpu_oracle(envs, k, 0, warmup=args.warmup, fixed_launches=args.steps)
    cores = host_threads()
    sample = (f"oracle/s2d_oracle.c (f64, OpenMP, {cores} threads): {envs} envs x {k} cycles per step "
              f"({envs * k} env-steps), {launches} steps, {dt:.1f} s")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / launches * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.gpus, envs, k),
            "reference_note": "the reference's Soccer2DEnv.step needs rcssserver + soccer-simulation-proxy (external "
                              "binaries, not available offline); this arm times oracle/s2d_oracle.c, the CPU restatement "
                              "of that path, OpenMP over the host cores, on one GPU's share of the workload",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
def time_launches(env, pool, steps, flush):
    """per-launch CUDA-event durations (ms) of `steps` s2d_step launches; optional L2 flush between (untimed)"""
    import torch
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for i in range(steps):
        env.bind_actions(pool[i % len(pool)])
        if flush is not None:
            flush.zero_()
        starts[i].record()
        env.step_torch()
        stops[i].record()
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in zip(starts, stops)]


def dump_outputs(out_dir, obs, reward, done, result):
    """the step's (obs, reward, done, result) as float32 .npy files under out_dir, with the env index of every row;
    a seeded sample of the envs (the same rows in every file) when all of them would exceed DUMP_BYTES"""
    import numpy as np
    n = reward.shape[0]
    per_env = 4 * (obs[0].numel() + 3) + 8
    rows = np.arange(n)
    if n * per_env > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // per_env, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("obs", obs), ("reward", reward), ("done", done), ("result", result)):
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy()[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))


class Ranks:
    """barrier / max-over-ranks of the timing contract"""

    def __init__(self, world, dev):
        self.world, self.dev = world, dev

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, x):
        if self.world == 1:
            return x
        import torch
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, x):
        """list of one float per rank (on every rank)"""
        if self.world == 1:
            return [x]
        import torch
        import torch.distributed as dist
        t = torch.zeros(self.world, dtype=torch.float64, device=self.dev)
        t[dist.get_rank()] = x
        dist.all_reduce(t)
        return [float(v) for v in t.tolist()]


def e2e_pipelined(env, host_pool, steps, ranks, slots=3):
    """`steps` steps through submit_host / wait_host with `slots` in flight; the host reads every step's reward.
    Returns seconds (max over ranks)."""
    import torch
    env.enable_pipeline(slots=slots)
    pend = [env.submit_host(host_pool[i % len(host_pool)]) for i in range(slots)]  # warm every slot once
    for t in pend:
        env.wait_host(t)
    ranks.barrier()
    t0 = time.perf_counter()
    pend, checksum, sent = [], 0.0, 0
    while sent < min(slots - 1, steps):
        pend.append(env.submit_host(host_pool[sent % len(host_pool)]))
        sent += 1
    for _ in range(steps):
        if sent < steps:
            pend.append(env.submit_host(host_pool[sent % len(host_pool)]))
            sent += 1
        _, reward, _, _ = env.wait_host(pend.pop(0))
        checksum += float(reward[0])
    torch.cuda.synchronize()
    dt = ranks.max(time.perf_counter() - t0)
    ranks.barrier()
    return dt, checksum


def pcie_probe(env, h2d_bytes, d2h_bytes, steps, ranks):
    """The ceiling of the host-buffer path on THIS box: plain cudaMemcpyAsync of one step's byte counts, pinned host
    memory (allocated like the env's staging blocks), no kernel; all ranks at the same time.  Three measurements:
    device-to-host alone, host-to-device alone, both directions concurrently (what the pipeline does)."""
    import torch
    dev = env.device
    d_in, d_out = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev), torch.zeros(d2h_bytes, dtype=torch.uint8, device=dev)
    h_in, h_out = env.pinned_bytes(h2d_bytes), env.pinned_bytes(d2h_bytes)
    h_in.zero_()
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(do_in, do_out):
        for rep in range(2):  # first pass warms up
            ranks.barrier()
            t0 = time.perf_counter()
            for _ in range(steps if rep else 3):
                if do_in:
                    with torch.cuda.stream(s_in):
                        d_in.copy_(h_in, non_blocking=True)
                if do_out:
                    with torch.cuda.stream(s_out):
                        h_out.copy_(d_out, non_blocking=True)
            s_in.synchronize()
            s_out.synchronize()
            dt = time.perf_counter() - t0
        return ranks.max(dt), ranks.gather(dt)

    t_out, per_out = run(False, True)
    t_in, _ = run(True, False)
    t_both, per_both = run(True, True)
    ranks.barrier()
    return {"steps": steps, "d2h_only_gbs_per_rank": d2h_bytes * steps / t_out / 1e9,
            "h2d_only_gbs_per_rank": h2d_bytes * steps / t_in / 1e9,
            "both_d2h_gbs_per_rank": d2h_bytes * steps / t_both / 1e9, "both_h2d_gbs_per_rank": h2d_bytes * steps / t_both / 1e9,
            "both_seconds": t_both, "d2h_only_gbs_each_rank": [d2h_bytes * steps / t / 1e9 for t in per_out],
            "both_d2h_gbs_each_rank": [d2h_bytes * steps / t / 1e9 for t in per_both],
            "what": "cudaMemcpyAsync pinned<->device of one step's bytes (no kernel), all ranks concurrently, slowest rank"}


def commands(torch, gen, dev, shape):
    """synthetic proto-style commands {cmd, a, b, c}: none / dash / turn / kick / go-to-point, uniformly"""
    a = torch.zeros(shape + (4,), device=dev)
    cmd = torch.randint(0, 5, shape, device=dev, generator=gen)
    u = lambda: torch.rand(shape, device=dev, generator=gen)  # noqa: E731
    a[..., 0] = cmd.float()
    a[..., 1] = torch.where(cmd == 4, u() * 100 - 50, u() * 100)
    a[..., 2] = torch.where(cmd == 4, u() * 60 - 30, u() * 360 - 180)
    a[..., 3] = 100.0
    return a


def measure_scenario(kind, total, k, steps, warmup, rank, world, dev, ranks, numa_node, with_e2e=True, dump_dir=None):
    """BASELINE configs[2] (kind = "shoot": 1v0 shoot-on-goal, `total` envs) / configs[3] ("fullgame": 11v11, `total`
    matches), sharded over the ranks (strong scaling, shard_range), command actions resident in HBM.  Same timing rules
    as the main arm; `dump_dir`: see dump_outputs.  Returns the section dict (identical on every rank)."""
    import torch

    from soccer2d_b200 import Soccer2DVecEnv, shard_range
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    off, n = shard_range(rank, world, total)
    if kind == "shoot":
        env = Soccer2DVecEnv(n, scenario="shoot", device=dev, seed=0, substeps=k, env_id_offset=off, use_command_action=True,
                             host_numa_node=numa_node)
        pool = [commands(torch, gen, dev, (n, k)) for _ in range(2)]
        per_env = 2 * STATE_BYTES + 16 * k + OBS_BYTES + OUT_BYTES
        name = f"1v0 shoot-on-goal, {total} envs in total, proto-style command actions (dash/turn/kick/go-to-point), K={k}"
        kernel = "s2d::step_kernel<SHOOT, COMMAND, default ServerParam>"
    else:
        env = Soccer2DVecEnv(n, scenario="fullgame", device=dev, seed=0, substeps=k, env_id_offset=off, host_numa_node=numa_node)
        # a fresh command for every player in every cycle of the timed window.  (Rounds 1 and 2 alternated TWO command
        # tensors: every player then repeats the same two commands for ever, drifts in one direction and the teams
        # pile up - 2.6 % of the matches collide per cycle by cycle 30.  That workload is still timed below, as
        # `repeating_commands`.)
        pool = [commands(torch, gen, dev, (n, k, 22)) for _ in range(8 if k == 1 else 2)]
        per_env = 2 * FG_STATE_BYTES + 22 * 16 * k + FG_OBS_BYTES + OUT_BYTES
        name = (f"11v11 full game, {total} matches in total, one command per player per cycle (8 command tensors in turn: "
                f"no player repeats a command within 8 cycles), K={k}")
        kernel = "s2d::fullgame_step_kernel<default ServerParam, 11v11>"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    env.reset_torch()
    time_launches(env, pool, max(warmup, 3), flush)
    ranks.barrier()
    ms = time_launches(env, pool, steps, flush)
    ranks.barrier()
    total_ms = ranks.max(sum(ms))
    launch_ms = sum(ms) / len(ms)
    if dump_dir:
        dump_outputs(dump_dir, env.obs, env.reward, env.done, env.result)
    out = {"workload": name, "value": total * k * steps / (total_ms * 1e-3), "unit": UNIT, "scaling": "strong",
           "envs_per_gpu": n, "global_envs": total, "substeps": k, "steps": steps, "launch_ms": launch_ms,
           "ms_per_step": total_ms / steps, "gpu_launches": steps}
    peak, peak_src = load_peaks()
    ach = per_env * n / (launch_ms * 1e-3) / 1e9
    key = f"fullgame_k{k}"
    out["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                       "traffic": load_traffic(key, n) if kind == "fullgame" else None,
                       "issue_slots_busy_pct_ncu": load_traffic(key, n, "issue_active_pct") if kind == "fullgame" else None,
                       "kernel": kernel, "launch_ms": launch_ms, "algorithmic_bytes_per_launch": per_env * n,
                       "peak_source": peak_src}
    if kind == "fullgame" and len(pool) > 2:  # the workload of rounds 1 and 2: two command tensors in turn
        env.reset_torch()
        time_launches(env, pool[:2], max(warmup, 3), flush)
        ms2 = time_launches(env, pool[:2], steps, flush)
        l2 = ranks.max(sum(ms2)) / steps
        out["repeating_commands"] = {
            "launch_ms": l2, "value": total * k / (l2 * 1e-3), "roofline_frac": per_env * n / (l2 * 1e-3) / 1e9 / peak,
            "what": "two command tensors alternating (every player repeats two commands, drifts and piles up with the others: "
                    "the pair scan and the collision resolver run in nearly every warp); same window (cycles 4-23)"}
        pool = pool[:3]
    if with_e2e:
        host_pool = [env.pinned_like(p) for p in pool]
        for hp, p in zip(host_pool, pool):
            hp.copy_(p)
        e2e_steps = max(3, min(steps, 20))
        e2e_s, _ = e2e_pipelined(env, host_pool, e2e_steps, ranks)
        h2d = pool[0].numel() * pool[0].element_size()
        out["e2e"] = {"value": total * k * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": int(env.layout.step_bytes), "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3,
                      "d2h_copies_per_step": env.pipeline_info()["d2h_copies_last_step"],
                      "path": "Soccer2DVecEnv.submit_host / wait_host (s2d_submit_host / s2d_wait_host), pinned host buffers, "
                              "3 slots in flight"}
    out["episode_stats"] = env.allreduce_stats()
    env.close()
    del env, pool, flush
    torch.cuda.empty_cache()
    return out


def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 arm has no CPU fallback (use --impl reference)")
    from soccer2d_b200 import Soccer2DVecEnv, numa

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # the rank's host side next to its GPU: CPU affinity and the pinned staging buffers on the GPU's NUMA node
    placement = numa.bind_process_to_gpu(local_rank) if args.numa else {"disabled": True, "node": None}
    numa_node = placement.get("node")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ranks = Ranks(world, dev)

    if args.workload != "reachball":
        total = args.envs if args.envs != ENVS_PER_GPU else (1 << 22 if args.workload == "shoot" else 1 << 18)
        sampler = ClockSampler(local_rank)
        sampler.start()
        sec = measure_scenario(args.workload, total, args.substeps, args.steps, args.warmup, rank, world, dev, ranks, numa_node,
                               dump_dir=args.dump_outputs if rank == 0 else None)
        clocks = sampler.summary()
        if rank == 0:
            line = {"metric": METRIC, "value": sec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": max(args.warmup, 3), "ms_per_step": sec["ms_per_step"], "higher_is_better": True,
                    "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": {"workload": sec["workload"], "envs_per_gpu": sec["envs_per_gpu"], "substeps": sec["substeps"],
                               "global_envs": sec["global_envs"], "parallelism": f"episode-shard x{world}",
                               "l2": "flushed between timed launches (256 MiB memset, not timed)"},
                    "e2e": sec["e2e"], "gpu_launches": sec["gpu_launches"], "roofline": sec["roofline"], "clocks": clocks,
                    "episode_stats": sec["episode_stats"], "host_placement": placement}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    n, k = args.envs, args.substeps
    env = Soccer2DVecEnv(n, device=dev, seed=0, substeps=k, env_id_offset=rank * n, host_numa_node=numa_node, **SCENARIO_KW)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = [torch.randint(0, 16, (n, k), dtype=torch.uint8, device=dev, generator=gen) for _ in range(4)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # 2x the 126 MB L2
    env.reset_torch()
    time_launches(env, pool, max(args.warmup, 3), flush)

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- value: device-resident inputs --------------------------------------------------------------
    ranks.barrier()
    ms = time_launches(env, pool, args.steps, flush)
    ranks.barrier()
    total_ms = ranks.max(sum(ms))
    value = world * n * k * args.steps / (total_ms * 1e-3)
    launch_ms = sum(ms) / len(ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env.obs, env.reward, env.done, env.result)  # what the last step_torch returned

    # ---- e2e: host buffers, every step's actions H2D and results D2H inside the timed region --------------
    host_pool = [env.pinned_like(p) for p in pool[:3]]
    for hp, p in zip(host_pool, pool):
        hp.copy_(p)
    e2e_steps = max(3, min(args.steps, 30))
    h2d = pool[0].numel() * pool[0].element_size()
    d2h = int(env.layout.step_bytes)
    # (a) synchronous call: s2d_step_host, one step at a time (H2D -> kernel -> D2H -> host reads the reward)
    for i in range(3):
        env.step_host(host_pool[i % 3])
    ranks.barrier()
    t0 = time.perf_counter()
    checksum = 0.0
    for i in range(e2e_steps):
        _, reward, _, _ = env.step_host(host_pool[i % 3])
        checksum += float(reward[0])
    torch.cuda.synchronize()
    e2e_sync_s = ranks.max(time.perf_counter() - t0)
    ranks.barrier()
    # (b) pipelined call: s2d_submit_host / s2d_wait_host, three steps in flight - the D2H of step i, the kernel of
    #     step i+1 and the H2D of step i+2 overlap; the host still reads every step's result
    e2e_s, c2 = e2e_pipelined(env, host_pool, e2e_steps, ranks, slots=3)
    d2h_copies = env.pipeline_info()["d2h_copies_last_step"]
    e2e_value = world * n * k * e2e_steps / e2e_s
    e2e_sync_value = world * n * k * e2e_steps / e2e_sync_s
    # (c) what the box gives plain copies of the same sizes
    probe = pcie_probe(env, h2d, d2h, e2e_steps, ranks)
    probe_value = world * n * k * e2e_steps / probe["both_seconds"]
    kernel_s = launch_ms * 1e-3
    copy_s = probe["both_seconds"] / e2e_steps
    limiter = ("host<->device copies: the D2H of 46 bytes of results per env and launch at the box's concurrent PCIe rate "
               f"({probe['both_d2h_gbs_per_rank']:.1f} GB/s per rank with {world} rank(s) copying)" if copy_s > kernel_s
               else "the step kernel")

    stats = env.allreduce_stats()  # NCCL all-reduce of the episode statistics (the only collective)
    env.close()
    del env, pool, host_pool
    torch.cuda.empty_cache()

    # ---- the same kernel in its HBM-bound regime: closed loop, K = 1, working set >> L2 -------------
    n1 = args.envs_k1
    env1 = Soccer2DVecEnv(n1, device=dev, seed=0, substeps=1, env_id_offset=rank * n1, **SCENARIO_KW)
    pool1 = [torch.randint(0, 16, (n1, 1), dtype=torch.uint8, device=dev, generator=gen) for _ in range(4)]
    env1.reset_torch()
    k1_steps = max(10, min(args.steps, 100))
    time_launches(env1, pool1, 5, None)
    ranks.barrier()
    ms1 = time_launches(env1, pool1, k1_steps, None)
    ranks.barrier()
    k1_total_ms = ranks.max(sum(ms1))
    k1_launch_ms = sum(ms1) / len(ms1)
    k1_value = world * n1 * k1_steps / (k1_total_ms * 1e-3)
    env1.close()
    del env1, pool1

    # ---- BASELINE configs[2] and [3] in the same run (short): 4M shoot envs / 256K 11v11 matches over the ranks ----
    extra_steps = max(3, min(args.steps, 20))
    shoot = fullgame = None
    if not args.no_extras:
        shoot = measure_scenario("shoot", 1 << 22, 1, extra_steps, 3, rank, world, dev, ranks, numa_node)
        fullgame = measure_scenario("fullgame", 1 << 18, 1, extra_steps, 3, rank, world, dev, ranks, numa_node)

    # ---- closed-loop policy rollout (configs[4]): obs -> 64-64 MLP -> argmax -> step, all on the device ----
    from soccer2d_b200.rollout import QNetwork, measure_fused_rollout, measure_rollout
    rollout, rollout_fused = {}, {}
    for nr in (1 << 16, 1 << 20):
        envr = Soccer2DVecEnv(nr, device=dev, seed=0, substeps=1, env_id_offset=rank * nr, **SCENARIO_KW)
        envr.reset_torch()
        torch.manual_seed(0)
        qnet = QNetwork(envr.obs_dim, 16).to(dev)
        try:
            rollout[str(nr)] = measure_rollout(envr, qnet, steps=max(10, min(args.steps, 50)), use_graph=True)
        except Exception as exc:  # noqa: BLE001 - graph capture refused: time the eager loop
            rollout[str(nr)] = measure_rollout(envr, qnet, steps=max(10, min(args.steps, 50)), use_graph=False)
            rollout["note"] = f"CUDA graph capture failed ({type(exc).__name__}); eager launches"
        # the same loop with the Q-network inside the step kernel: 16 cycles per launch (s2d_rollout_mlp)
        rollout_fused[str(nr)] = measure_fused_rollout(envr, qnet, launches=max(5, min(args.steps, 20)), k=SUBSTEPS)
        envr.close()
        del envr
    clocks = sampler.summary()

    # ---- configs[0]: ONE env behind the reference's gym API (reset / step -> 4-tuple), host round trip every step ----
    single = None
    if rank == 0 and world == 1:
        from sample_environments.environment_factory import EnvironmentFactory
        genv = EnvironmentFactory().create("ReachBall", None, None, None, device=dev, seed=0, **SCENARIO_KW)
        import numpy as _np
        arng = _np.random.default_rng(0)
        acts = arng.integers(0, 16, size=4000)
        genv.reset()
        for a in acts[:200]:
            if genv.step(int(a))[2]:
                genv.reset()
        t0 = time.perf_counter()
        episodes = 0
        for a in acts[200:]:
            if genv.step(int(a))[2]:
                genv.reset()
                episodes += 1
        dt = time.perf_counter() - t0
        genv.close()
        single = {"value": (len(acts) - 200) / dt, "unit": "env-steps/s", "steps": len(acts) - 200, "episodes": episodes,
                  "path": "EnvironmentFactory().create('ReachBall').step(a): s2d_step_host on 1 env, stream sync, numpy 4-tuple"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = load_peaks()
    bytes16 = algorithmic_bytes_per_env(k) * n
    bytes1 = algorithmic_bytes_per_env(1) * n1
    ach16 = bytes16 / (launch_ms * 1e-3) / 1e9
    ach1 = bytes1 / (k1_launch_ms * 1e-3) / 1e9
    cpu_line = None
    if world == 1:
        cv, cl, cdt = time_cpu_oracle(n, k, args.cpu_seconds)
        cpu_line = {"value": cv, "unit": UNIT, "cores": host_threads(), "kind": "port",
                    "sample": f"oracle/s2d_oracle.c (f64, OpenMP): {n} envs x {k} cycles x {cl} launches, {cdt:.1f} s"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(world, n, k),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3,
                "d2h_gbs": d2h * e2e_steps / e2e_s / 1e9, "h2d_gbs": h2d * e2e_steps / e2e_s / 1e9,
                "d2h_copies_per_step": d2h_copies, "slots_in_flight": 3,
                "pcie_probe": dict(probe, value=probe_value, unit=UNIT), "frac_of_probe": e2e_value / probe_value,
                "limiter": limiter,
                "path": "Soccer2DVecEnv.submit_host / wait_host -> s2d_submit_host / s2d_wait_host: pinned host actions in, "
                        "ONE packed obs|reward|done|result block out, three steps in flight (copies overlap the kernel)",
                "synchronous": {"value": e2e_sync_value, "ms_per_step": e2e_sync_s / e2e_steps * 1e3,
                                "path": "Soccer2DVecEnv.step_host -> s2d_step_host, one step at a time"}},
        "gpu_launches": args.steps,
        "roofline": {"bound": "hbm", "achieved": ach16, "peak": peak, "unit": "GB/s", "frac": ach16 / peak,
                     "traffic": load_traffic(f"k{k}", n),
                     "issue_slots_busy_pct_ncu": load_traffic(f"k{k}", n, "issue_active_pct"),
                     "warp_instructions_per_env_step_ncu": load_traffic(f"k{k}", n, "warp_instructions_per_env_step"),
                     "kernel": "s2d::step_kernel<REACHBALL, DISCRETE, default ServerParam>", "launch_ms": launch_ms,
                     "algorithmic_bytes_per_launch": bytes16, "peak_source": peak_src,
                     "note": "K=16 keeps 16 cycles in registers: HBM traffic is 222 B per 16 env-steps by construction, "
                             "this regime is instruction-issue bound; see roofline_k1 for the HBM-bound regime"},
        "roofline_k1": {"bound": "hbm", "achieved": ach1, "peak": peak, "unit": "GB/s", "frac": ach1 / peak,
                        "traffic": load_traffic("k1", n1),
                        "kernel": "s2d::step_kernel<REACHBALL, DISCRETE, default ServerParam>", "launch_ms": k1_launch_ms, "envs_per_gpu": n1,
                        "substeps": 1, "algorithmic_bytes_per_launch": bytes1, "env_steps_per_sec": k1_value,
                        "peak_source": peak_src},
        "shoot": shoot, "fullgame": fullgame,
        "rollout_dqn": {"unit": UNIT + " per GPU", "policy": "64-64 ReLU MLP (SB3 DQN MlpPolicy shape), greedy, K=1, zero-copy obs/action "
                        "tensors, loop body replayed as a CUDA graph (torch fp32 matmuls for the policy, not part of the "
                        "step path)",
                        "envs_to_value": rollout,
                        "fused_policy_kernel": {
                            "envs_to_value": rollout_fused, "substeps": SUBSTEPS,
                            "path": "Soccer2DVecEnv.rollout_mlp -> s2d_rollout_mlp: observe -> Q-network (tcgen05.mma kind::tf32, one "
                                    "M=128 tile per block, accumulators and layer-2/3 activations in tensor memory, weights "
                                    "in shared memory) -> argmax -> step, K cycles per launch; observation and action never "
                                    "leave the SM"}},
        "single_env_gym_api": single,
        "clocks": clocks,
        "episode_stats": stats,
        "host_placement": placement,
        "parity": load_parity(),
    }
    if cpu_line:
        line["cpu_baseline"] = cpu_line
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed launches (default 200; 25 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="reachball", choices=["reachball", "shoot", "fullgame"],
                    help="reachball = BASELINE configs[1] (the contract line, with short shoot / fullgame sections); "
                         "shoot / fullgame = configs[2] / [3] as the whole line")
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="episodes per GPU (default 2^20, configs[1])")
    ap.add_argument("--substeps", type=int, default=None, help="fused cycles per launch (default: 16 for reachball, 1 for shoot / fullgame)")
    ap.add_argument("--envs-k1", type=int, default=1 << 23, help="episodes per GPU of the K=1 roofline run")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="bound on the cpu_baseline sample")
    ap.add_argument("--no-extras", action="store_true", help="skip the shoot / fullgame sections of the default line")
    ap.add_argument("--no-numa", dest="numa", action="store_false", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed launch as .npy files under DIR (B200 arm)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm's timed path; use it with --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        args.substeps = args.substeps or SUBSTEPS
        if args.steps is None:  # the default K of the B200 arm would take minutes on the CPU: keep it bounded
            args.steps = 25  # (2.6 s timed)
        run_reference(args, rank)
        return
    if args.steps is None:
        args.steps = 200
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun: python -m torch.distributed.run --nproc-per-node {args.gpus} "
                         f"--master-addr 127.0.0.1 bench.py --gpus {args.gpus} ...")
    if args.substeps is None:
        args.substeps = SUBSTEPS if args.workload == "reachball" else 1
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
