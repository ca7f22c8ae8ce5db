"""Time the keyed policy sampling (policy_sampling.keyed_act) against torch's sampling and print one JSON line (card name
and power limit included).

(a) sampling: torch's composition -- Normal(mean, mean*0. + std, validate_args=False), rsample(), log_prob().sum(-1),
    mean and stddev -- plus the record launch that copies the four into the rollout slots (add_transitions with only
    those fields), against one keyed_act launch writing the slots; each as --copies back-to-back copies captured in one
    CUDA graph, timed with CUDA events over 20 replays, at --kernel-envs envs, A = 12.
(b) run(): microseconds per env-step of RolloutGraph.run(capture_schedule=True) on the flat preset with
    keyed_domain_rand on, body = actor MLP -> sampling -> critic -> step_device() -> record_env_step(), with torch's
    sampling (validate_args=False, rsample) against keyed_act.  Two envs, --warmup rollouts each (captures), then the
    two bodies alternated over --repeats rounds of --iters rollouts, each timed on its own with CUDA events.
(c) the eager public-step() loop with the same body, torch's default (validating) Normal.sample() against keyed_act,
    per env-step over whole rollouts, alternated the same way.

The actor is HIMActorCritic-sized (270 -> 512 -> 256 -> 128 -> 12, ELU), the critic 512 -> 256 -> 128 -> 1.

    python tools/policy_sampling_timing.py [--kernel-envs 4096 65536] [--loop 4096:100 65536:24] [--out FILE]
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

GAMMA, LAM = 0.99, 0.95


def spread(v):
    return {"median_us": statistics.median(v), "min_us": min(v), "max_us": max(v)}


def mlp(dims, dev):
    layers = []
    for i in range(len(dims) - 1):
        layers.append(torch.nn.Linear(dims[i], dims[i + 1]))
        if i < len(dims) - 2:
            layers.append(torch.nn.ELU())
    return torch.nn.Sequential(*layers).to(dev)


def torch_sample(mean, std, tr, validate):
    """HIMPPO.act's sampling as HIMActorCritic does it (validate=None: torch's default argument validation)."""
    dist = torch.distributions.Normal(mean, mean * 0. + std, **({} if validate is None else {"validate_args": validate}))
    tr.actions = dist.sample() if validate is None else dist.rsample()
    tr.actions_log_prob = dist.log_prob(tr.actions).sum(dim=-1)
    tr.action_mean, tr.action_sigma = dist.mean, dist.stddev
    return tr.actions


# ----------------------------------------------------------------------------------------------------------- (a)
def measure_sampling(n, copies, replays):
    from isaacgymloco_b200.policy_sampling import keyed_act
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    env = make_env(n)
    g = torch.Generator("cuda").manual_seed(3)
    mean = torch.randn(n, 12, device="cuda", generator=g)
    std = torch.nn.Parameter(torch.full((12,), 0.8, device="cuda"))
    st = HIMRolloutStorage(n, 1, [45], [None], [12], device="cuda")
    tr = HIMRolloutStorage.Transition()

    def torch_path():
        st.step = 0
        with torch.no_grad():
            torch_sample(mean, std, tr, False)
        st.add_transitions(tr)

    def kernel_path():
        st.step = 0
        with torch.no_grad():
            keyed_act(env, mean, std, tr, st)

    graphs = {}
    for mode, fn in (("torch", torch_path), ("kernel", kernel_path)):
        fn()                                         # warm-up: modules loaded, allocator pools set up
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            for _ in range(copies):
                fn()
        torch.cuda.current_stream().wait_stream(s)
        gr.replay()
        graphs[mode] = gr
    torch.cuda.synchronize()
    per = {m: [] for m in graphs}
    for _ in range(replays):
        for m, gr in graphs.items():
            per[m].append(1e3 * timed_ms(gr.replay, 1) / copies)
    res = {"envs": n, "copies_per_graph": copies, "replays": replays}
    for m, v in per.items():
        res[m] = spread(v)
    res["saved_us_per_step"] = res["torch"]["median_us"] - res["kernel"]["median_us"]
    return res


# ----------------------------------------------------------------------------------------------------------- (b), (c)
class Loop:
    """One env + storage + policy; body(k) = the runner's step with the given sampling."""

    def __init__(self, n, t_len, sampling, eager):
        from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
        self.env = env = make_env(n, schedule=True)
        env.cfg_hot.reset.keyed_domain_rand = True
        torch.manual_seed(0)
        self.actor = mlp([env.obs_buf.shape[1], 512, 256, 128, 12], env.device)
        self.critic = mlp([env.num_privileged_obs, 512, 256, 128, 1], env.device)
        self.std = torch.nn.Parameter(torch.full((12,), 0.8, device=env.device))
        env.extras["time_outs"] = env.time_out_buf
        self.st = HIMRolloutStorage(n, t_len, [env.obs_buf.shape[1]], [env.num_privileged_obs], [12], device=env.device,
                                    env_writes_slots=True)
        env.bind_rollout(self.st)
        self.tr = HIMRolloutStorage.Transition()
        self.sampling, self.eager, self.t_len = sampling, eager, t_len
        self.last_values = torch.zeros(n, 1, device=env.device)

    def body(self, k):
        from isaacgymloco_b200.policy_sampling import keyed_act
        env, tr, st = self.env, self.tr, self.st
        with torch.no_grad():
            mean = self.actor(env.obs_buf)
            if self.sampling == "kernel":
                keyed_act(env, mean, self.std, tr, st)
            else:
                torch_sample(mean, self.std, tr, None if self.eager else False)
            tr.values = self.critic(env.privileged_obs_buf)
        tr.observations, tr.critic_observations = env.obs_buf, env.privileged_obs_buf
        if self.eager:
            obs, priv, rew, done, extras, ids, term = env.step(tr.actions)
            st.record_env_step(tr, rew, done, extras, priv, ids, term, GAMMA)
        else:
            obs, priv, rew, done, extras, ids, n_dev, term, _ = env.step_device(tr.actions)
            st.record_env_step(tr, rew, done, extras, priv, ids, term, GAMMA, termination_count=n_dev)

    def finish(self):
        self.st.compute_returns(self.last_values, GAMMA, LAM)

    def rollout_eager(self):
        for k in range(self.t_len):
            self.body(k)
        self.finish()
        self.st.clear()


def measure_loop(n, t_len, warmup, repeats, iters, eager):
    loops, fns = {}, {}
    for mode in ("torch", "kernel"):
        lp = loops[mode] = Loop(n, t_len, mode, eager)
        if eager:
            fns[mode] = lp.rollout_eager
        else:
            rg = lp.rg = lp.env.capture_rollout(lp.body, t_len, storage=lp.st, finish=lp.finish, capture_schedule=True,
                                                max_graphs=16)
            fns[mode] = lambda rg=rg, lp=lp: (rg.run(), lp.st.clear())
        for _ in range(warmup):
            fns[mode]()
    per = {m: [] for m in loops}
    for _ in range(repeats):
        for m, fn in fns.items():
            for _ in range(iters):
                per[m].append(1e3 * timed_ms(fn, 1) / t_len)
    out = {"envs": n, "rollout_len": t_len, "rollouts_per_mode": repeats * iters}
    for m, v in per.items():
        out[m] = spread(v)
        out[m]["mean_us"] = statistics.fmean(v)
        if not eager:
            out[m]["run_modes"] = dict(loops[m].rg.stats)
    out["kernel_vs_torch"] = out["kernel"]["median_us"] / out["torch"]["median_us"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel-envs", type=int, nargs="*", default=[4096, 65536])
    ap.add_argument("--copies", type=int, default=50)
    ap.add_argument("--loop", nargs="*", default=["4096:100", "65536:24"], help="envs:T pairs for (b) and (c)")
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("policy_sampling_timing.py needs a CUDA device")
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "sampling": [], "run": [], "eager": []}
    for n in args.kernel_envs:
        res["sampling"].append(measure_sampling(n, args.copies, 20))
        torch.cuda.empty_cache()
    for spec in args.loop:
        n, t = (int(x) for x in spec.split(":"))
        res["run"].append(measure_loop(n, t, args.warmup, args.repeats, args.iters, eager=False))
        torch.cuda.empty_cache()
        res["eager"].append(measure_loop(n, t, 2, args.repeats, 2, eager=True))
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
