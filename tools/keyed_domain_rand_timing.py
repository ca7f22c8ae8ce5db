"""Time keyed domain randomisation (ResetCfg.keyed_domain_rand) against the torch hooks and print one JSON line (card
name and power limit included).

(a) clip + delay: step()'s torch.clamp + the torch _delay_actions (torch.randint, arange, mask, sub, mul, add) against
    one hl_delay_actions launch, each as --copies back-to-back copies captured in one CUDA graph, timed with CUDA events
    over 20 replays, at --kernel-envs envs (aliengo flat, decimation 4).  Bytes from shapes: 96 read (actions and
    last_actions) + 240 written (actions and delayed_actions) per env, over the time of one copy.
(b) run(): microseconds per env-step of RolloutGraph.run(capture_schedule=True) with body = step_device(), on the flat
    preset with its delay, disturbance (every 8 steps), push (every 800) and command-curriculum (every 1000) intervals,
    flag on against flag off: two envs, --warmup rollouts each (captures), then the two modes alternated over --repeats
    rounds of --iters rollouts.  Every rollout is timed on its own with CUDA events; the median is the steady state (a
    window that meets a new push / curriculum position captures a graph first, which only the max shows).

    python tools/keyed_domain_rand_timing.py [--kernel-envs 4096 65536] [--loop 4096:100 65536:24] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from rollout_graph_timing import make_env, power_limit_w, timed_ms  # noqa: E402

READ_B, WRITE_B = 96, 240          # per env at decimation 4


def spread(v):
    return {"median_us": statistics.median(v), "min_us": min(v), "max_us": max(v)}


# ----------------------------------------------------------------------------------------------------------- (a)
def measure_delay(n, copies, replays):
    env = make_env(n)
    assert env.cfg_hot.decimation == 4 and env.cfg_hot.reset.delay
    acts = 150.0 * torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    env.last_actions.copy_(torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(4)))
    graphs, outs = {}, {}
    for mode in ("torch", "kernel"):
        env.cfg_hot.reset.keyed_domain_rand = mode == "kernel"
        env._clip_and_delay(acts)                   # warm-up: modules loaded, allocator pools set up
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for _ in range(copies):
                env._clip_and_delay(acts)
        torch.cuda.current_stream().wait_stream(s)
        g.replay()
        graphs[mode] = g
        outs[mode] = env.actions.clone()
    assert torch.equal(outs["torch"], outs["kernel"])          # the clip is the same either way
    per = {m: [] for m in graphs}
    for _ in range(replays):
        for m, g in graphs.items():
            per[m].append(1e3 * timed_ms(g.replay, 1) / copies)
    res = {"envs": n, "copies_per_graph": copies, "replays": replays, "bytes": (READ_B + WRITE_B) * n}
    for m, v in per.items():
        res[m] = spread(v)
        res[m]["gb_per_s"] = res["bytes"] / (res[m]["median_us"] * 1e-6) / 1e9
    res["saved_us_per_step"] = res["torch"]["median_us"] - res["kernel"]["median_us"]
    env.cfg_hot.reset.keyed_domain_rand = False
    return res


# ----------------------------------------------------------------------------------------------------------- (b)
def measure_run(n, t_len, warmup, repeats, iters):
    runs = {}
    for mode in ("off", "on"):
        env = make_env(n, schedule=True)
        env.cfg_hot.reset.keyed_domain_rand = mode == "on"
        acts = 0.3 * torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(5))

        def body(k, env=env, acts=acts):
            env.step_device(acts)
        runs[mode] = env.capture_rollout(body, t_len, capture_schedule=True, max_graphs=16)
        for _ in range(warmup):
            runs[mode].run()
    per = {m: [] for m in runs}
    before = {m: dict(rg.stats) for m, rg in runs.items()}
    for _ in range(repeats):
        for m, rg in runs.items():
            for _ in range(iters):
                per[m].append(1e3 * timed_ms(rg.run, 1) / t_len)
    out = {"envs": n, "rollout_len": t_len, "rollouts_per_mode": repeats * iters}
    for m, v in per.items():
        out[m] = spread(v)
        out[m]["mean_us"] = statistics.fmean(v)
        out[m]["timed_captures"] = runs[m].stats["captures"] - before[m]["captures"]
        out[m]["run_modes"] = dict(runs[m].stats)
    out["on_vs_off"] = out["on"]["median_us"] / out["off"]["median_us"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel-envs", type=int, nargs="*", default=[4096, 65536])
    ap.add_argument("--copies", type=int, default=50)
    ap.add_argument("--loop", nargs="*", default=["4096:100", "65536:24"], help="envs:T pairs for (b)")
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("keyed_domain_rand_timing.py needs a CUDA device")
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "read_bytes_per_env": READ_B,
           "write_bytes_per_env": WRITE_B, "delay": [], "run": []}
    for n in args.kernel_envs:
        res["delay"].append(measure_delay(n, args.copies, 20))
        torch.cuda.empty_cache()
    for spec in args.loop:
        n, t = (int(x) for x in spec.split(":"))
        res["run"].append(measure_run(n, t, args.warmup, args.repeats, args.iters))
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
