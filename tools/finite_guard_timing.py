"""Time the non-finite guard (FiniteGuard / hl_finite_scan) and print one JSON line (card name and power limit
included, read in the same run).

(a) launch: --launches back-to-back FiniteGuard.record() calls with the default fields (the env's root_states,
    dof_state and contact_forces; a HIMRolloutStorage slot's actions, mu, sigma, values, actions_log_prob and rewards)
    captured in one CUDA graph, timed with CUDA events over 20 replays, at --kernel-envs envs.  Bytes from shapes: the
    fields' widths x 4 per env, over the kernel time.  The fields are written by the step just before the scan, so the
    repeated launches read them from L2 as the scan inside a rollout does (they fit the 126 MB L2 at 65,536 envs).
(b) run(): microseconds per env-step of RolloutGraph.run() with body = step_device() + record_env_step() and with the
    same body + FiniteGuard.record(k), on the aliengo flat task of tools/rollout_graph_timing.py (pushes, disturbances
    and the curriculum off, so every window replays), two identical envs, the modes alternated over --repeats rounds of
    --iters rollouts each.

    python tools/finite_guard_timing.py [--kernel-envs 4096 65536] [--loop 4096:100 65536:24] [--out FILE]
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


def spread(v):
    return {"median_us": statistics.median(v), "min_us": min(v), "max_us": max(v)}


def make_loop(n, t_len, guarded):
    """An env, a storage and the runner's body (fixed actions), with or without a guard over the default fields."""
    from isaacgymloco_b200.finite_guard import FiniteGuard
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    env = make_env(n)
    dev = env.device
    st = HIMRolloutStorage(n, t_len, [270], [env.num_privileged_obs], [12], device=dev)
    tr = HIMRolloutStorage.Transition()
    acts = 0.3 * torch.randn(n, 12, device=dev, generator=torch.Generator(dev).manual_seed(5))
    values, logp, sigma = torch.full((n, 1), 0.1, device=dev), torch.zeros(n, device=dev), torch.ones(n, 12, device=dev)
    guard = FiniteGuard(env, t_len, storage=st) if guarded else None

    def body(k):
        tr.observations, tr.critic_observations, tr.actions = env.obs_buf, env.privileged_obs_buf, acts
        tr.values, tr.actions_log_prob, tr.action_mean, tr.action_sigma = values, logp, acts, sigma
        _, priv, rew, done, extras, ids, n_dev, term, _ = env.step_device(acts)
        st.record_env_step(tr, rew, done, extras, priv, ids, term, 0.99, termination_count=n_dev)
        if guard is not None:
            guard.record(k)
    return env, st, guard, body


# ----------------------------------------------------------------------------------------------------------- (a)
def measure_kernel(n, launches, repeats):
    env, st, guard, body = make_loop(n, 1, True)
    body(0)                                       # real step outputs in the fields
    widths = dict(zip(guard.fields, guard.widths))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr, stream=s):
        for _ in range(launches):
            guard.record(0)
    torch.cuda.current_stream().wait_stream(s)
    gr.replay()
    us = [1e3 * timed_ms(gr.replay, 1) / launches for _ in range(repeats)]
    flagged = int(guard.table[0, :, 0].sum())
    res = {"envs": n, "launches_per_replay": launches, "fields": widths, "kernel": spread(us),
           "bytes": 4 * n * sum(widths.values()), "flagged": flagged}
    res["gb_per_s"] = res["bytes"] / (res["kernel"]["median_us"] * 1e-6) / 1e9
    return res


# ----------------------------------------------------------------------------------------------------------- (b)
def measure_run(n, t_len, repeats, iters):
    runs, stores = {}, {}
    for mode in ("without", "with"):
        env, st, guard, body = make_loop(n, t_len, mode == "with")
        rg = env.capture_rollout(body, t_len, storage=st, finite_guard=guard)
        runs[mode], stores[mode] = rg, st
        for _ in range(2):                        # warm-up (eager), then capture + replay
            rg.run()
            st.clear()
    per = {m: [] for m in runs}
    for _ in range(repeats):
        for m, rg in runs.items():
            st = stores[m]
            per[m].append(1e3 * timed_ms(lambda: (rg.run(), st.clear()), iters) / t_len)
    out = {m: spread(v) for m, v in per.items()}
    for m, rg in runs.items():
        out[m]["run_modes"] = dict(rg.stats)
    out["envs"], out["rollout_len"] = n, t_len
    out["delta_us_per_step"] = out["with"]["median_us"] - out["without"]["median_us"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel-envs", type=int, nargs="*", default=[4096, 65536])
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--loop", nargs="*", default=["4096:100", "65536:24"], help="envs:T pairs for (b)")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("finite_guard_timing.py needs a CUDA device")
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
           "kernel": [measure_kernel(n, args.launches, 20) for n in args.kernel_envs], "run": []}
    torch.cuda.empty_cache()
    for spec in args.loop:
        n, t = (int(x) for x in spec.split(":"))
        res["run"].append(measure_run(n, t, args.repeats, args.iters))
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
