"""Time the runners' episode statistics on the device (EpisodeStats / hl_episode_stats) and print one JSON line (card
name and power limit included).

(a) kernel: --launches back-to-back EpisodeStats.record() calls (step_device()'s id form, ~2 % of the envs done, a
    100-entry ring) captured in one CUDA graph, timed with CUDA events over 20 replays, at --kernel-envs envs.
    Bytes from shapes: 21 per env (rewards, dones, the two running sums read and written) over the kernel time.
(b) run(): microseconds per env-step of RolloutGraph.run() with body = step_device() and with body = step_device() +
    record(), on the aliengo flat task of tools/rollout_graph_timing.py (pushes, disturbances and the curriculum off, so
    every window replays), two identical envs, the modes alternated over --repeats rounds of --iters rollouts each.
    Next to it, the host clock of collect() alone (the two copies, a sync, the deque extension) and of a bare sync:
    their difference is what run() adds once per rollout besides the T launches.
(c) eager loop: microseconds per env-step of T public step() calls followed by the runners' block with its two .cpu()
    syncs, against T step() calls with record() and one collect() per rollout; same envs sizes, same alternation.

    python tools/episode_stats_timing.py [--kernel-envs 4096 65536] [--loop 4096:100 65536:24] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time
from collections import deque

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from rollout_graph_timing import make_env, power_limit_w, timed_ms  # noqa: E402

BYTES_PER_ENV = 21


def spread(v):
    return {"median_us": statistics.median(v), "min_us": min(v), "max_us": max(v)}


def host_us(fn, calls=200):
    v = []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        v.append(1e6 * (time.perf_counter() - t0))
    return statistics.median(v)


# ----------------------------------------------------------------------------------------------------------- (a)
def measure_kernel(n, launches, repeats):
    from isaacgymloco_b200.episode_stats import EpisodeStats
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(n)
    rewards = torch.randn(n, device=dev, generator=g)
    dones = torch.rand(n, device=dev, generator=g) < 0.02
    found = dones.nonzero().flatten()
    m = found.numel()
    ids = torch.zeros(n, dtype=torch.long, device=dev)
    ids[:m] = found
    cnt = torch.tensor([m], dtype=torch.int32, device=dev)
    stats = EpisodeStats(n, dev)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr, stream=s):
        for _ in range(launches):
            stats.record(rewards, dones, ids, cnt)
    torch.cuda.current_stream().wait_stream(s)
    gr.replay()
    us = [1e3 * timed_ms(gr.replay, 1) / launches for _ in range(repeats)]
    res = {"envs": n, "done_envs": m, "launches_per_replay": launches, "kernel": spread(us),
           "bytes": BYTES_PER_ENV * n}
    res["gb_per_s"] = res["bytes"] / (res["kernel"]["median_us"] * 1e-6) / 1e9
    return res


# ----------------------------------------------------------------------------------------------------------- (b)
def measure_run(n, t_len, repeats, iters):
    from isaacgymloco_b200.episode_stats import EpisodeStats
    runs, stats = {}, {}
    for mode in ("without", "with"):
        env = make_env(n)
        acts = 0.3 * torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
        st = EpisodeStats(n, env.device) if mode == "with" else None

        def body(k, env=env, acts=acts, st=st):
            _, _, rew, done, _, ids, n_dev, _, _ = env.step_device(acts)
            if st is not None:
                st.record(rew, done, ids, n_dev)
        runs[mode] = env.capture_rollout(body, t_len, episode_stats=st)
        stats[mode] = st
        runs[mode].run()                          # warm-up (eager)
        runs[mode].run()                          # capture + replay
    per = {m: [] for m in runs}
    for _ in range(repeats):
        for m, rg in runs.items():
            per[m].append(1e3 * timed_ms(rg.run, iters) / t_len)
    out = {m: spread(v) for m, v in per.items()}
    for m, rg in runs.items():
        out[m]["run_modes"] = dict(rg.stats)
    out["with"]["episodes_logged"] = stats["with"]._seen
    out["with"]["collect_us"] = host_us(stats["with"].collect)
    out["with"]["sync_us"] = host_us(torch.cuda.current_stream().synchronize)
    out["envs"], out["rollout_len"] = n, t_len
    out["delta_us_per_step"] = out["with"]["median_us"] - out["without"]["median_us"]
    return out


# ----------------------------------------------------------------------------------------------------------- (c)
def measure_eager(n, t_len, repeats):
    from isaacgymloco_b200.episode_stats import EpisodeStats
    loops = {}
    for mode in ("block", "record"):
        env = make_env(n)
        acts = 0.3 * torch.randn(n, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
        if mode == "block":
            state = dict(rewbuffer=deque(maxlen=100), lenbuffer=deque(maxlen=100),
                         cur_reward_sum=torch.zeros(n, dtype=torch.float, device=env.device),
                         cur_episode_length=torch.zeros(n, dtype=torch.float, device=env.device))

            def rollout(env=env, acts=acts, s=state):
                rewbuffer, lenbuffer = s["rewbuffer"], s["lenbuffer"]
                cur_reward_sum, cur_episode_length = s["cur_reward_sum"], s["cur_episode_length"]
                for _ in range(t_len):
                    _, _, rewards, dones, _, _, _ = env.step(acts)
                    cur_reward_sum += rewards
                    cur_episode_length += 1
                    new_ids = (dones > 0).nonzero(as_tuple=False)
                    rewbuffer.extend(cur_reward_sum[new_ids][:, 0].cpu().numpy().tolist())
                    lenbuffer.extend(cur_episode_length[new_ids][:, 0].cpu().numpy().tolist())
                    cur_reward_sum[new_ids] = 0
                    cur_episode_length[new_ids] = 0
        else:
            st = EpisodeStats(n, env.device)

            def rollout(env=env, acts=acts, st=st):
                for _ in range(t_len):
                    _, _, rewards, dones, _, ids, _ = env.step(acts)
                    st.record(rewards, dones, ids)
                st.collect()
        loops[mode] = rollout
        rollout()                                 # warm-up
    per = {m: [] for m in loops}
    for _ in range(repeats):
        for m, fn in loops.items():
            per[m].append(1e3 * timed_ms(fn, 1) / t_len)
    out = {m: spread(v) for m, v in per.items()}
    out["envs"], out["rollout_len"] = n, t_len
    out["record_vs_block"] = out["record"]["median_us"] / out["block"]["median_us"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel-envs", type=int, nargs="*", default=[4096, 65536])
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--loop", nargs="*", default=["4096:100", "65536:24"], help="envs:T pairs for (b) and (c)")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("episode_stats_timing.py needs a CUDA device")
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "bytes_per_env": BYTES_PER_ENV,
           "kernel": [measure_kernel(n, args.launches, 20) for n in args.kernel_envs], "run": [], "eager": []}
    for spec in args.loop:
        n, t = (int(x) for x in spec.split(":"))
        res["run"].append(measure_run(n, t, args.repeats, args.iters))
        torch.cuda.empty_cache()
        res["eager"].append(measure_eager(n, t, args.repeats))
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
