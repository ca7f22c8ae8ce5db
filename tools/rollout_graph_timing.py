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
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                              f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:           # no nvidia-smi / unparsable: the field stays empty
        return None


def make_env(n, seed=1):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from oracle.make_goldens import reset_inputs
    cfg, hf, state, _, ter, _ = reset_inputs(dict(task="flat", n=n, seed=seed))
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[65536, 4096])
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
           "results": [measure(n, args.steps, args.repeats, args.iters) for n in args.envs]}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
