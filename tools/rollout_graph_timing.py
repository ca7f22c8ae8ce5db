"""Time one T-step rollout three ways on the same env and print one JSON line:

  eager   body(0) .. body(T-1) launched directly (what a runner without graphs does)
  run     RolloutGraph.run(): the captured graph replayed with fresh Philox keys and the per-step episode logging
  frozen  the same body captured once and replayed as is (bench.py's form: every replay repeats the capture's keys)

body(k) = step_device(actions) on the aliengo flat task with the terrain curriculum attached (so the per-step
terrain_level reduction of the episode logging runs); pushes, disturbances and the command curriculum are off, as in
bench.py, so every window replays.  The modes alternate over --repeats rounds of --iters rollouts each; the JSON
holds per-mode medians and spreads in us per env-step, the cost of the terrain_level reduction alone, and the card
name and power limit the numbers were taken at.

    python tools/rollout_graph_timing.py [--envs 65536 4096] [--steps 24] [--repeats 7] [--iters 10] [--out FILE]

--schedule reference times the training schedule instead: T = 100 with the presets' disturbance (8 steps), push (800)
and command-curriculum (1000) intervals, over whole 4,000-step cycles (40 windows), with the default run() (push and
curriculum windows eager) against run() of capture_rollout(..., capture_schedule=True), alternating per cycle over
--repeats rounds after one unmeasured cycle (warm-up and first captures).  Per mode: the mean us per env-step over a
cycle (host clock around the 40 run() calls; each ends in a device sync), the share of windows replayed and the
number of cached graphs.

    python tools/rollout_graph_timing.py --schedule reference [--envs 4096 65536] [--repeats 5]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                              f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:           # no nvidia-smi / unparsable: the field stays empty
        return None


def make_env(n, seed=1, schedule=False):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from oracle.make_goldens import reset_inputs
    cfg, hf, state, _, ter, _ = reset_inputs(dict(task="flat", n=n, seed=seed))
    if schedule:              # the presets' schedule (every AlienGo task enables all three)
        cfg.reset.push_robots = cfg.reset.disturbance = cfg.reset.commands_curriculum = True
    else:
        cfg.reset.push_robots = cfg.reset.disturbance = cfg.reset.commands_curriculum = False
    env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", seed=seed)
    env.custom_origins = True
    env.env_origins = ter["env_origins"].cuda().contiguous()
    env.terrain_origins, env.terrain_types = ter["origins"].cuda().contiguous(), ter["types"].cuda().contiguous()
    env.max_terrain_level = cfg.num_rows
    env.refresh_buffers()
    return env


def timed_ms(fn, iters):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def measure(n, t_len, repeats, iters):
    env = make_env(n)
    acts = 0.3 * torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(5))

    def body(k):
        env.step_device(acts)

    def eager():
        for k in range(t_len):
            body(k)

    rg = env.capture_rollout(body, t_len)
    rg.run()                                     # warm-up (eager)
    rg.run()                                     # capture + replay
    frozen = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(frozen, stream=s):
        eager()
    torch.cuda.current_stream().wait_stream(s)
    # the per-step terrain_level reduction of the episode logging, on its own (T of them in one graph)
    tsum = torch.zeros(t_len, dtype=torch.long, device="cuda")
    red = torch.cuda.CUDAGraph()
    with torch.cuda.graph(red, stream=s):
        for k in range(t_len):
            torch.sum(env.terrain_levels, dim=0, out=tsum[k])
    torch.cuda.current_stream().wait_stream(s)
    modes = {"eager": eager, "run": rg.run, "frozen": frozen.replay}
    per = {m: [] for m in modes}
    red_us = []
    for _ in range(repeats):
        for m, fn in modes.items():
            per[m].append(1e3 * timed_ms(fn, iters) / t_len)
        red_us.append(1e3 * timed_ms(red.replay, iters) / t_len)
    out = {m: {"median_us_per_step": statistics.median(v), "min": min(v), "max": max(v)} for m, v in per.items()}
    out["terrain_level_reduction_us_per_step"] = statistics.median(red_us)
    out["run_modes"] = dict(rg.stats)
    out["envs"], out["rollout_len"] = n, t_len
    return out


def measure_schedule(n, repeats, t_len=100):
    """The reference schedule over whole cycles: default run() vs capture_schedule=True, alternating per cycle."""
    from isaacgymloco_b200.rollout_graph import env_schedule
    runs = {}
    for mode in ("default", "capture_schedule"):
        env = make_env(n, schedule=True)
        acts = 0.3 * torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
        body = (lambda e, a: lambda k: e.step_device(a))(env, acts)
        runs[mode] = env.capture_rollout(body, t_len, capture_schedule=(mode == "capture_schedule"))
    sched = env_schedule(runs["default"].env)
    cycle = math.lcm(*(m for m in sched.values() if m > 0), t_len) // t_len
    per = {m: [] for m in runs}
    replayed = {m: [] for m in runs}
    for rnd in range(repeats + 1):
        for m, rg in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            modes = []
            for _ in range(cycle):
                rg.run()
                modes.append(rg.last_mode)
            dt = time.perf_counter() - t0
            if rnd > 0:           # round 0: warm-up and the first captures
                per[m].append(1e6 * dt / (cycle * t_len))
                replayed[m].append(sum(x != "eager" for x in modes) / cycle)
    out = {m: {"mean_us_per_step": statistics.mean(v), "median": statistics.median(v), "min": min(v), "max": max(v),
               "replayed_share": statistics.mean(replayed[m]), "cached_graphs": len(runs[m]._graphs),
               "run_modes": dict(runs[m].stats)} for m, v in per.items()}
    out["envs"], out["rollout_len"], out["windows_per_cycle"], out["schedule"] = n, t_len, cycle, sched
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--schedule", choices=["none", "reference"], default="none")
    ap.add_argument("--envs", type=int, nargs="+", default=None)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.schedule == "reference":
        envs = args.envs or [4096, 65536]
        res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "schedule": "reference",
               "results": [measure_schedule(n, args.repeats) for n in envs]}
    else:
        envs = args.envs or [65536, 4096]
        res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
               "results": [measure(n, args.steps, args.repeats, args.iters) for n in envs]}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
