"""Time the AMP env-step of the hybrid runner and print one JSON line (card name and power limit included).

(a) kernel: one hl_amp_transition launch against the launches it replaces -- get_amp_observations into a fresh tensor,
    clone, index_put of the terminal rows, AMPDiscriminator.assemble_input (hl_amp_disc_input), ReplayBuffer.insert
    (hl_ring_insert), clone -- at --kernel-envs envs with a --ring-rows replay ring.  Both are captured as --launches
    back-to-back copies in one CUDA graph and timed with CUDA events over --repeats replays (device time per step, no
    host launch cost).  Inputs: random AMP state with ~2.5 % of the envs resetting.  The kernel's bytes from shapes
    (841 B per env + 128 B per reset env) over its time, as a share of the measured HBM peak.  The env-side inputs
    (about 16 MB at 65,536 envs) stay in L2 across launches; the ring rows are new on every launch.
(b) hybrid loop: microseconds per env-step of the runner's rollout on the aliengo "amp" preset (disturbance, push and
    command-curriculum intervals as configured) with a [1024, 512] discriminator: the eager composition (public step(),
    the runner's AMP block, record_env_step) against RolloutGraph.run() of AMPRolloutStep + capture_rollout(...,
    capture_schedule=True, amp=...).  Whole schedule cycles (every push / curriculum position once), one unmeasured
    cycle first (warm-up, captures), then --loop-repeats cycles per mode, alternating; host clock around each cycle,
    which ends in a device sync.  The discriminator MLP alone (T forwards in one graph) is reported next to it.

    python tools/amp_rollout_timing.py [--kernel-envs 16384 65536] [--loop 4096:100 16384:24] [--out FILE]
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

PEAK_GBS = 6535.7          # measured HBM copy peak of the B200 (DESIGN §3: the roofline denominator)


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                              f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:           # no nvidia-smi / unparsable: the field stays empty
        return None


def graph_of(fn, copies):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()                    # warm-up outside the capture (library handles, allocator)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for _ in range(copies):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    return g


def events_ms(fn, repeats):
    out = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


# ----------------------------------------------------------------------------------------------------------- (a)
def measure_kernel(n, ring_rows, launches, repeats):
    from types import SimpleNamespace
    from isaacgymloco_b200.amp_discriminator import AMPDiscriminator, Normalizer
    from isaacgymloco_b200.amp_rollout import AMPRolloutStep
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from isaacgymloco_b200.replay_buffer import ReplayBuffer
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(n)
    env = SimpleNamespace(num_envs=n, device=dev, dof_state=torch.randn(n, 24, device=dev, generator=g),
                          base_lin_vel=torch.randn(n, 3, device=dev, generator=g),
                          base_ang_vel=torch.randn(n, 3, device=dev, generator=g))
    env.reset_buf = torch.rand(n, device=dev, generator=g) < 0.025
    ids_host = env.reset_buf.nonzero().flatten()
    m = int(ids_host.numel())
    ids = torch.zeros(n, dtype=torch.long, device=dev)
    ids[:m] = ids_host
    n_dev = torch.tensor([m], dtype=torch.int32, device=dev)
    term = torch.randn(n, 30, device=dev, generator=g)
    disc = AMPDiscriminator(60, 2.0, [1024, 512], dev, task_reward_lerp=0.3)
    norm = Normalizer(30, device=dev)
    norm.update(torch.randn(4096, 30, device=dev, generator=g))
    rb_k, rb_c = ReplayBuffer(30, ring_rows, dev), ReplayBuffer(30, ring_rows, dev)
    amp = AMPRolloutStep(env, disc, norm, rb_k)
    amp.begin()
    amp.refresh()
    from isaacgymloco_b200 import _lib as L

    def kernel():
        L.check(L.lib.hl_amp_transition(
            L.ptr(env.dof_state), L.ptr(env.base_lin_vel), L.ptr(env.base_ang_vel), L.ptr(env.reset_buf), L.ptr(ids),
            L.ptr(n_dev), L.ptr(term), L.ptr(amp._stats), float(norm.epsilon), float(norm.clip_obs), L.ptr(amp.amp_obs),
            L.ptr(amp.x), L.ptr(rb_k.states), L.ptr(rb_k.next_states), ring_rows, L.ptr(amp._cursor), n, L.stream()))

    state = {"amp_obs": FusedLeggedRobot.get_amp_observations(env)}
    term_m = term[:m]

    def composition():
        next_amp_obs = FusedLeggedRobot.get_amp_observations(env)
        nwt = next_amp_obs.clone()
        nwt[ids_host] = term_m
        disc.assemble_input(state["amp_obs"], nwt, norm)
        rb_c.insert(state["amp_obs"], nwt)
        state["amp_obs"] = next_amp_obs.clone()

    res = {"envs": n, "ring_rows": ring_rows, "reset_envs": m, "launches_per_replay": launches}
    kg = graph_of(kernel, launches)
    cg = graph_of(composition, launches)
    for name, gr in (("kernel", kg), ("composition", cg), ("kernel", kg), ("composition", cg)):
        res.setdefault(name + "_us", []).extend(1e3 * t / launches for t in events_ms(gr.replay, repeats))
    for name in ("kernel", "composition"):
        v = res.pop(name + "_us")
        res[name] = {"median_us": statistics.median(v), "min_us": min(v), "max_us": max(v)}
    nbytes = 841 * n + 128 * m
    res["kernel_bytes"] = nbytes
    res["kernel_share_of_peak"] = nbytes / (res["kernel"]["median_us"] * 1e-6) / (PEAK_GBS * 1e9)
    res["speedup"] = res["composition"]["median_us"] / res["kernel"]["median_us"]
    del kg, cg
    return res


# ----------------------------------------------------------------------------------------------------------- (b)
class HybridLoop:
    """HybridPolicyRunner's rollout over one env: eager = public step() + the runner's AMP block; otherwise
    step_device() + AMPRolloutStep.step() inside a RolloutGraph."""

    def __init__(self, n, t_len, eager, ring_rows=1_000_000, seed=1):
        from isaacgymloco_b200.amp_discriminator import AMPDiscriminator, Normalizer
        from isaacgymloco_b200.amp_rollout import AMPRolloutStep
        from isaacgymloco_b200.legged_robot import FusedLeggedRobot
        from isaacgymloco_b200.replay_buffer import ReplayBuffer
        from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
        from oracle.make_goldens import reset_inputs
        cfg, hf, state, _, ter, _ = reset_inputs(dict(task="amp", n=n, seed=seed))
        env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", seed=seed)
        env.custom_origins = True
        env.env_origins = ter["env_origins"].cuda().contiguous()
        env.terrain_origins, env.terrain_types = ter["origins"].cuda().contiguous(), ter["types"].cuda().contiguous()
        env.max_terrain_level = cfg.num_rows
        env.refresh_buffers()
        dev = env.device
        self.env, self.eager, self.t_len = env, eager, t_len
        torch.manual_seed(seed)
        self.disc = AMPDiscriminator(60, 2.0, [1024, 512], dev, task_reward_lerp=0.3)
        self.norm = Normalizer(30, device=dev)
        self.rb = ReplayBuffer(30, ring_rows, dev)
        env.extras["time_outs"] = env.time_out_buf
        self.st = HIMRolloutStorage(n, t_len, [270], [env.num_privileged_obs], [12], device=dev, env_writes_slots=True)
        env.bind_rollout(self.st)
        self.tr = HIMRolloutStorage.Transition()
        self.acts = 0.3 * torch.randn(n, 12, device=dev, generator=torch.Generator(dev).manual_seed(5))
        self.values, self.logp, self.sigma = torch.full((n, 1), 0.1, device=dev), torch.zeros(n, device=dev), torch.ones(n, 12, device=dev)
        self.last_values = torch.zeros(n, 1, device=dev)
        if eager:
            self.amp_obs = env.get_amp_observations()
        else:
            self.amp = AMPRolloutStep(env, self.disc, self.norm, self.rb)
            self.amp.begin()
            self.rg = env.capture_rollout(self.body, t_len, storage=self.st, finish=self.finish, capture_schedule=True,
                                          amp=self.amp, max_graphs=1024)

    def body(self, k):
        env, tr = self.env, self.tr
        tr.observations, tr.critic_observations, tr.actions = env.obs_buf, env.privileged_obs_buf, self.acts
        tr.values, tr.actions_log_prob, tr.action_mean, tr.action_sigma = self.values, self.logp, self.acts, self.sigma
        if self.eager:
            obs, priv, rew, done, extras, ids, term, term_amp = env.step(self.acts)
            next_amp_obs = env.get_amp_observations()
            next_amp_obs_with_term = next_amp_obs.clone()
            next_amp_obs_with_term[ids] = term_amp
            rewards = self.disc.predict_amp_reward(self.amp_obs, next_amp_obs_with_term, rew, self.norm)[0]
            self.rb.insert(self.amp_obs, next_amp_obs_with_term)
            self.amp_obs = next_amp_obs.clone()
            self.st.record_env_step(tr, rewards, done, extras, priv, ids, term, 0.99)
        else:
            obs, priv, rew, done, extras, ids, n_dev, term, term_amp = env.step_device(self.acts)
            rewards = self.amp.step(rew, ids, n_dev, term_amp)
            self.st.record_env_step(tr, rewards, done, extras, priv, ids, term, 0.99, termination_count=n_dev)

    def finish(self):
        self.st.compute_returns(self.last_values, 0.99, 0.95)

    def rollout(self):
        if self.eager:
            for k in range(self.t_len):
                self.body(k)
            self.finish()
        else:
            self.rg.run()
        self.st.clear()


def measure_loop(n, t_len, repeats):
    from isaacgymloco_b200.rollout_graph import env_schedule
    loops = {"eager": HybridLoop(n, t_len, True), "run": HybridLoop(n, t_len, False)}
    sched = env_schedule(loops["run"].env)
    cycle = math.lcm(*(m for m in sched.values() if m > 0), t_len) // t_len
    per = {m: [] for m in loops}
    for rnd in range(repeats + 1):
        for m, lp in loops.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(cycle):
                lp.rollout()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if rnd > 0:           # round 0: warm-up and the captures
                per[m].append(1e6 * dt / (cycle * t_len))
    out = {m: {"mean_us_per_step": statistics.mean(v), "min": min(v), "max": max(v)} for m, v in per.items()}
    rg = loops["run"].rg
    out["run"].update(run_modes=dict(rg.stats), cached_graphs=len(rg._graphs))
    # the discriminator MLP alone: T forwards on the (N, 60) input in one graph
    lp = loops["run"]

    def mlp():
        with torch.no_grad():
            lp.disc.amp_linear(lp.disc.trunk(lp.amp.x))
    g = graph_of(mlp, t_len)
    out["mlp_us_per_step"] = statistics.median(1e3 * t / t_len for t in events_ms(g.replay, 20))
    out["envs"], out["rollout_len"], out["windows_per_cycle"], out["schedule"] = n, t_len, cycle, sched
    out["run_vs_eager"] = out["run"]["mean_us_per_step"] / out["eager"]["mean_us_per_step"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel-envs", type=int, nargs="*", default=[16384, 65536])
    ap.add_argument("--ring-rows", type=int, default=1_000_000)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--loop", nargs="*", default=["4096:100", "16384:24"], help="envs:T pairs for (b)")
    ap.add_argument("--loop-repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("amp_rollout_timing.py needs a CUDA device")
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "peak_gbs": PEAK_GBS,
           "kernel": [measure_kernel(n, args.ring_rows, args.launches, args.repeats) for n in args.kernel_envs],
           "loop": []}
    for spec in args.loop:
        n, t = (int(x) for x in spec.split(":"))
        res["loop"].append(measure_loop(n, t, args.loop_repeats))
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
