#!/usr/bin/env python
"""bench.py -- post-physics + GAE env-steps/s (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference --steps K --warmup W    (the reference arm: CPU torch)

One *step* = one rollout iteration of the hot path for this rank's env shard:
    T x { 4 x PD torques (decimation) ; fused post-physics ; reset-id compaction ; terminal rows ;
          post-reset fix-up }  +  HIMRolloutStorage.compute_returns (GAE scan + normalisation)
on synthetic, seeded PhysX state (SURVEY.md §8d).  One *env-step* = one env through one of the T
inner steps (+ 1/T of the GAE).  Rank r owns a contiguous shard of the global env set (weak
scaling: --envs per GPU); for N>1 the advantage moments are all-reduced every step and the 20
flat PPO-gradient all-reduces of one update (545,660 fp32) run on a side stream.

JSON line (rank 0): see the driver contract; extra keys `roofline` (dominant kernel, CUDA-event
timed inside the timed region) and `cpu_baseline` (the torch oracle port on the host cores).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "post_physics_gae_env_steps_per_s"
UNIT = "env-steps/s"
AC_PARAMS = 545_660          # HIMActorCritic incl. estimator (SURVEY.md §2 #20)
EST_PARAMS = 59_875          # HIMEstimator's own optimiser step (him_estimator.py:111-114)
DISC_PARAMS = 587_777        # AMPDiscriminator (hybrid_ppo.py:271)


def bind_to_gpu_numa(local_rank):
    """Pin this process to the CPUs of the GPU's NUMA node (NVML's ideal affinity) so pinned staging buffers and the
    copy-issuing thread are socket-local.  Returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local_rank])
                                              if os.environ.get("CUDA_VISIBLE_DEVICES") else local_rank)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        return {"cpus": len(cpus), "first": cpus[0], "last": cpus[-1]}
    except Exception as ex:  # pragma: no cover
        return {"error": str(ex)[:80]}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arm
def _reference_root():
    """Where the reference's own Python sources are, if anywhere (this container: /root/reference; the GPU box has
    neither -- the reference needs the proprietary isaacgym wheel and is not pip-installable: DESIGN.md §7)."""
    for cand in (os.environ.get("HIMLOCO_REFERENCE_ROOT"), "/root/reference", os.path.join(ROOT, "baseline", "_ref")):
        if cand and os.path.isdir(os.path.join(cand, "legged_gym", "legged_gym")) and os.path.isdir(os.path.join(cand, "rsl_rl", "rsl_rl")):
            return cand
    return None


def cpu_rollout_runner(n_envs, t_len, seed=1234):
    """The reference's torch implementation of the path on all host cores: the reference's OWN classes under the
    stub harness (oracle/ref_harness.py) when its sources are present (kind "reference"), else the restatement
    oracle/torch_oracle.py (kind "port": the Python reference cannot travel to the GPU box).  Returns
    (callable running ONE rollout = T x {4 torques, post_physics_step} + compute_returns, threads, kind)."""
    from isaacgymloco_b200 import config as C, synthetic as S
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = C.aliengo("flat", num_envs=n_envs, index_math=C.INDEX_MATH_TORCH_CPU)
    hf = S.make_terrain(cfg, seed=1)
    state = S.make_state(cfg, n_envs, hf, seed=seed)
    roll = S.make_rollout(n_envs, t_len, seed)
    ref_root = _reference_root()
    if ref_root is not None:
        try:
            os.environ["HIMLOCO_REFERENCE_ROOT"] = ref_root
            import types
            from oracle import ref_harness as H
            H.REFERENCE_ROOT = ref_root
            env = H.build_reference_env("flat", state, hf, sum_names=cfg.episode_sum_names(), hot_cfg=cfg)
            from rsl_rl.storage import HIMRolloutStorage as RefStorage
            rc = env.cfg
            env.custom_origins = True
            env.env_origins = torch.zeros(n_envs, 3)
            env.terrain_origins = torch.zeros(cfg.num_rows, cfg.num_cols, 3)
            env.terrain_types = torch.zeros(n_envs, dtype=torch.long)
            env.max_terrain_level = cfg.num_rows
            env.base_init_state = torch.tensor(rc.init_state.pos + rc.init_state.rot + rc.init_state.lin_vel + rc.init_state.ang_vel,
                                               dtype=torch.float)
            noop = lambda self, *a, **k: None
            # PhysX-facing / host-curriculum hooks are outside the path (and need a live sim): no-ops, as on the GPU arm
            for name in ("refresh_actor_rigid_shape_props", "update_command_curriculum", "_push_robots", "_disturbance_robots"):
                setattr(env, name, types.MethodType(noop, env))
            st = RefStorage(n_envs, t_len, [270], [238], [12], "cpu")
            st.rewards.copy_(roll["rewards"]); st.values.copy_(roll["values"]); st.dones.copy_(roll["dones"])
            delayed = env.actions.view(n_envs, 1, 12).repeat(1, 4, 1)

            def one_rollout_ref():
                for _ in range(t_len):
                    for k in range(4):
                        env.torques = env._compute_torques(delayed[:, k]).view(env.torques.shape)
                    env.post_physics_step()
                st.compute_returns(roll["last_values"], 0.99, 0.95)

            one_rollout_ref()
            return one_rollout_ref, torch.get_num_threads(), "reference"
        except Exception as ex:  # pragma: no cover
            sys.stderr.write(f"[bench] reference under the stub harness failed ({type(ex).__name__}: {ex}); timing the port\n")
    from oracle import torch_oracle as O
    env = O.OracleEnv(cfg, state, hf)
    delayed = env.actions.view(n_envs, 1, 12).repeat(1, 4, 1)

    def one_rollout():
        for _ in range(t_len):
            for k in range(4):
                env.torques = env._compute_torques(delayed[:, k])
            noise = dict(term45=torch.rand(n_envs, 45), term187=torch.rand(n_envs, 187),
                         obs45=torch.rand(n_envs, 45), obs187=torch.rand(n_envs, 187))
            env.post_physics_step(noise, None)
        O.compute_returns(roll["rewards"], roll["values"], roll["dones"], roll["last_values"], 0.99, 0.95)

    return one_rollout, torch.get_num_threads(), "port"


CPU_SAMPLE_ENVS = 4096      # bounded sample of the workload for the CPU arms (configs[0]: the reference's own CPU-runnable case)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_envs, t_len = CPU_SAMPLE_ENVS, args.rollout
    fn, cores, kind = cpu_rollout_runner(n_envs, t_len)
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = time.perf_counter() - t0
    value = n_envs * t_len * args.steps / dt
    src = "the reference's own LeggedRobot / HIMRolloutStorage under oracle/ref_harness.py" if kind == "reference" else "oracle/torch_oracle.py"
    sample = (f"each step = one {t_len}-step rollout of {n_envs} envs (a {n_envs}-of-{args.envs} env sample of the workload; "
              f"throughput per env-step is size-independent on the CPU), {src}, torch CPU, {cores} threads")
    cfgd = workload_config(args, world=args.gpus)
    cfgd["sample_envs"] = n_envs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfgd,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"aliengo flat, {args.envs} envs/GPU x {args.rollout}-step synthetic rollout: 4x PD torque + fused "
                        f"post-physics (45-dim obs, 6-step history, 187-pt scan, 21 reward terms) per env-step, GAE per rollout",
            "baseline_config": "configs[4] at N GPUs (65,536 envs/GPU; the roofline-target size, inputs 323 MB/step > 126 MB L2); "
                               "configs[1] (4096 envs) is L2-resident and reported under `latency_4096`",
            "envs_per_gpu": args.envs, "global_envs": args.envs * world, "rollout_len": args.rollout,
            "l2_policy": "inputs larger than L2 (no flush needed)" if args.envs >= 32768 else "L2-resident (latency regime)",
            "noise": "in-kernel Philox", "parallelism": f"env-shard x{world}"}


# ----------------------------------------------------------------------------- GPU arm
class Workload:
    def __init__(self, envs, t_len, rank, world, device, seed=1234, task="flat"):
        from isaacgymloco_b200 import config as C, synthetic as S
        from isaacgymloco_b200.legged_robot import FusedLeggedRobot
        from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
        self.envs, self.t_len, self.world, self.device = envs, t_len, world, device
        self.cfg = C.aliengo(task, num_envs=envs * world, env_id_offset=rank * envs)
        # the torch-RNG / PhysX-facing interval hooks (pushes, disturbances, the host-side command curriculum) are
        # outside the path (SURVEY.md §2); everything else of post_physics_step runs, reset_idx included
        self.cfg.reset.push_robots = False
        self.cfg.reset.disturbance = False
        self.cfg.reset.commands_curriculum = False
        hf = S.make_terrain(self.cfg, seed=1)
        state = S.make_state(self.cfg, envs, hf, seed=seed + rank, env_id_offset=rank * envs)
        self.host_state = state
        self.env = FusedLeggedRobot(self.cfg, state, hf, device=device, seed=seed)
        self.env.disturbance[:, 0, :] = 0.0
        self.storage = HIMRolloutStorage(envs, t_len, [270], [self.env.num_privileged_obs], [12], device=device,
                                         shard_statistics=world > 1)
        roll = S.make_rollout(envs, t_len, seed + rank)
        self.storage.rewards.copy_(roll["rewards"]); self.storage.values.copy_(roll["values"])
        self.storage.dones.copy_(roll["dones"])
        self.last_values = roll["last_values"].to(device)
        self.env._delay_actions()
        self.fused_ms = []            # CUDA-event pairs around the dominant kernel
        self.launches = 0
        self.exchange_cb = None       # N>1: called with the env-step index right after the fused launch is queued

    def env_step(self, time_fused=False, k_step=0):
        env = self.env
        for k in range(env.cfg_hot.decimation):
            env._compute_torques_into(env.delayed_actions[:, k], env.torques)
        cb = self.exchange_cb
        if time_fused or cb is not None:
            def hook():
                if time_fused:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()

                def after():
                    if time_fused:
                        e1.record()
                        self.fused_ms.append((e0, e1))
                    if cb is not None:
                        cb(k_step)
                return after
            env._fused_event_hook = hook
        else:
            env._fused_event_hook = None
        # the whole of post_physics_step as one chain of launches, no host sync: the fused kernel (pre-step command resampling folded in),
        # reset ids + terminal rows, then ONE launch for reset_idx (Philox re-draws, episode-logging means) + post-reset fix-up
        env.post_physics_step_device()
        self.launches += env.cfg_hot.decimation + (2 if env.single_launch else 3)

    def rollout(self, time_fused=False, finish=True):
        for k in range(self.t_len):
            self.env_step(time_fused, k)
        # compute_returns = GAE scan, [all-reduce of the 3 moments when sharded], normalisation
        self.storage.gae_scan(self.last_values, self.cfg.gamma, self.cfg.lam)
        if finish:
            self.finish()
        self.launches += 2

    def finish(self):
        self.storage.normalize_advantages()


def timed(fn, iters, sync_dist):
    """K calls of fn bracketed by barrier + synchronize, timed with CUDA events on the launch stream."""
    import torch.distributed as dist
    if sync_dist:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if sync_dist:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if sync_dist:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def run_gpu_arm(args):
    import torch.distributed as dist
    from isaacgymloco_b200 import dist as D
    from isaacgymloco_b200 import roofline as R
    rank, world, local = D.init_from_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    affinity = bind_to_gpu_numa(local)           # before any pinned allocation: H2D/D2H staging stays on the GPU's socket
    if world > 1:
        # env kernels on a high-priority stream: the (persistent, few-CTA) NCCL kernels of the side stream get the SM
        # slots the env grid leaves, not the other way round
        torch.cuda.set_stream(torch.cuda.Stream(device=device, priority=-1))
    wl = Workload(args.envs, args.rollout, rank, world, device)
    bytes_tab = R.per_env_step_bytes(wl.cfg, args.rollout)

    # multi-GPU exchange steps of one PPO update (SURVEY.md §8e), on a side stream, synthetic payloads of the real sizes:
    # per minibatch (5 epochs x 4) the estimator's own step (him_estimator.py:111-114, 59,875 fp32), the flat
    # HIMActorCritic gradient (him_ppo.py:182, 545,660 fp32) and the adaptive-KL scalar (him_ppo.py:148); with --amp
    # also the discriminator gradient (hybrid_ppo.py:271, 587,777 fp32) and the 61-double normaliser merge
    # (hybrid_ppo.py:279-281).  The 3-double advantage moments ride inside the rollout (storage.normalize_advantages).
    comm_stream = torch.cuda.Stream() if world > 1 and not args.no_comm else None
    if world > 1:
        # the in-rollout statistics get their own communicator: collectives of one communicator execute in issue order,
        # so on a shared one the 3-double moments would queue behind every gradient message still in flight
        wl.storage.process_group = dist.new_group(backend="nccl")
    if comm_stream is not None:
        grad_group = dist.new_group(backend="nccl")
        grads = torch.randn(AC_PARAMS + 1, device=device)      # + the adaptive-KL scalar: needed by the same optimiser step, same message
        est_grads = torch.randn(EST_PARAMS, device=device)
        disc_grads = torch.randn(DISC_PARAMS, device=device) if args.amp else None
        norm_stats = torch.zeros(61, dtype=torch.float64, device=device) if args.amp else None
        fork = torch.cuda.Event()

    N_MSG = 20                                       # 5 epochs x 4 minibatches

    def exchange():
        """All messages of one update, forked onto the side stream at the start of the rollout.  (Queuing pair k behind
        env-step k's fused kernel instead was measured too: 3.88 vs 3.76 ms per rollout on 8 GPUs, tools/scale_probe.py.)"""
        fork.record()
        comm_stream.wait_event(fork)
        with torch.cuda.stream(comm_stream):
            for _ in range(N_MSG):
                dist.all_reduce(est_grads, op=dist.ReduceOp.AVG, group=grad_group)
                dist.all_reduce(grads, op=dist.ReduceOp.AVG, group=grad_group)
                if args.amp:
                    dist.all_reduce(disc_grads, op=dist.ReduceOp.AVG, group=grad_group)
                    dist.all_reduce(norm_stats, op=dist.ReduceOp.SUM, group=grad_group)

    def step():
        if comm_stream is not None:
            exchange()
        wl.rollout(time_fused=True)
        if comm_stream is not None:
            torch.cuda.current_stream().wait_stream(comm_stream)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    # ---- pass A: direct launches, CUDA-event pair around every launch of the dominant kernel
    wl.fused_ms.clear()
    wl.launches = 0
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_direct = timed(step, args.steps, world > 1)
    launches = wl.launches
    fused = [a.elapsed_time(b) for a, b in wl.fused_ms]
    ms, mode = ms_direct, "direct_launch"

    # ---- pass B: the same K rollouts replayed from ONE captured CUDA graph -- the form the
    # library is meant to be driven in (every entry point is capture-safe); launch overhead gone
    graph_info = None
    if not args.no_graph:
        try:
            g = torch.cuda.CUDAGraph()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                wl.rollout()
                torch.cuda.synchronize()
                moments_in_graph = True
                try:
                    # world > 1: the collectives are captured too -- the 3-double moments on the rollout's own branch,
                    # the gradient messages as a forked branch that joins before the graph ends
                    with torch.cuda.graph(g, stream=s):
                        if comm_stream is not None:
                            exchange()
                        wl.rollout(finish=True)
                        if comm_stream is not None:
                            s.wait_stream(comm_stream)
                except Exception:
                    moments_in_graph = False             # NCCL build that cannot be captured: keep the collectives outside
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=s):
                        wl.rollout(finish=(world == 1))
            torch.cuda.current_stream().wait_stream(s)

            def graph_step():
                if comm_stream is not None and not moments_in_graph:
                    exchange()
                g.replay()
                if world > 1 and not moments_in_graph:
                    wl.finish()
                    if comm_stream is not None:
                        torch.cuda.current_stream().wait_stream(comm_stream)

            for _ in range(3):
                graph_step()
            gms = timed(graph_step, args.steps, world > 1)
            graph_info = {"value": world * args.envs * args.rollout * args.steps / (gms * 1e-3), "unit": UNIT,
                          "ms_per_step": gms / args.steps, "moments_allreduce_in_graph": bool(moments_in_graph) if world > 1 else None}
            if gms < ms_direct:
                ms, mode = gms, "cuda_graph_replay"
        except Exception as ex:  # pragma: no cover
            graph_info = {"error": str(ex)[:200]}
    clocks = sampler.stop() if sampler else None
    value = world * args.envs * args.rollout * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)

    # ---- e2e runs on EVERY rank (it contains collectives: moment all-reduce, barriers)
    wl.env._fused_event_hook = None
    e2e = None if args.no_e2e else measure_e2e(wl, args, world)
    if rank != 0:
        return
    peak, peak_src = peaks()
    fused_avg_ms = sum(fused) / max(len(fused), 1)
    alg_bytes = bytes_tab["post_physics"] * args.envs
    achieved = alg_bytes / (fused_avg_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "hl_post_physics_fused_kernel", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": args.traffic,
                "traffic_source": "ncu dram__bytes_read+write of one launch of this kernel build (profiles/fused_traffic.json; --traffic overrides), not re-measured in this run",
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": fused_avg_ms,
                "bytes_per_env_step": bytes_tab,
                "whole_step_frac": (bytes_tab["total"] * args.envs * args.rollout * args.steps / (ms * 1e-3) / 1e9) / peak}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, world), "clocks": clocks,
        "gpu_launches": launches, "roofline": roofline, "timing_mode": mode, "cpu_affinity": affinity,
        "exchange": None if world == 1 else ("off (--no-comm)" if args.no_comm else
                                             "20 x {estimator 59,875 fp32; actor-critic 545,660 fp32 grads + KL scalar (one message)}" +
                                             (" + {discriminator 587,777 fp32 + 61-double normaliser}" if args.amp else "") +
                                             " all-reduces per rollout on a side stream (own communicator, captured in the graph with the rollout); 3-double advantage moments inside the rollout on a second communicator"),
        "direct_launch": {"value": world * args.envs * args.rollout * args.steps / (ms_direct * 1e-3), "unit": UNIT,
                          "ms_per_step": ms_direct / args.steps},
    }
    if graph_info:
        line["cuda_graph"] = graph_info

    # ---- e2e: the public API with HOST buffers (pinned), H2D of the PhysX tensors + actions and
    # D2H of obs / privileged obs / rewards / dones every env-step, inside the timed region
    if e2e is not None:
        line["e2e"] = e2e
    # ---- 4096-env latency regime (configs[1]) and the CPU baseline: rank 0, N=1 only
    if world == 1:
        if not args.no_latency:
            line["latency_4096"] = measure_latency_4096(args)
            line["next_rows"] = {"record_transition": measure_record_transition(args, peak),
                                 "minibatch_gather": measure_minibatch_gather(args, peak)}
            line["other_configs"] = {"stairs16384": measure_stairs16384(args, peak), "amp16384": measure_amp16384(args, peak)}
        if not args.no_cpu:
            fn, cores, kind = cpu_rollout_runner(CPU_SAMPLE_ENVS, args.rollout)
            fn()
            t0 = time.perf_counter()
            reps = 3
            for _ in range(reps):
                fn()
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": CPU_SAMPLE_ENVS * args.rollout * reps / dt, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": f"{reps} rollouts of {CPU_SAMPLE_ENVS} envs x {args.rollout} steps (configs[0]) after 1 warm-up, "
                                              + ("the reference's own classes under oracle/ref_harness.py" if kind == "reference"
                                                 else "oracle/torch_oracle.py") + " on torch CPU"}
    print(json.dumps(line), flush=True)


DUMP_ROWS = 4096        # envs (and resets) sampled for --dump-outputs


def dump_outputs(wl, out_dir):
    """What the caller of the timed rollout receives after its last step, as DIR/<name>.npy: the last env-step's
    observations, privileged observations, rewards, reset / time-out flags, the reset count, reset ids with their
    terminal privileged rows, and the rollout's returns and advantages.  Per-env outputs are taken at DUMP_ROWS envs and
    the reset outputs at DUMP_ROWS resets, picked by a fixed seed and stored too (`env_rows`, `reset_rows`), so two builds
    are compared on the same rows whatever --envs is: about 13 MB at --rollout 24.  Integer and boolean outputs are
    stored as float64 (exact)."""
    import numpy as np
    env, st = wl.env, wl.storage
    torch.cuda.synchronize()

    def sample(count):
        return torch.randperm(count, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values

    rows = sample(env.num_envs)
    n_reset = int(env._n_reset.item())
    reset_rows = sample(n_reset)
    out = {"env_rows": rows, "obs_buf": env.obs_buf.cpu()[rows], "privileged_obs_buf": env.privileged_obs_buf.cpu()[rows],
           "rew_buf": env.rew_buf.cpu()[rows], "reset_buf": env.reset_buf.cpu()[rows], "time_out_buf": env.time_out_buf.cpu()[rows],
           "n_reset": torch.tensor([n_reset]), "reset_rows": reset_rows, "reset_ids": env._reset_ids[:n_reset].cpu()[reset_rows],
           "termination_privileged_obs": env._term_priv[:n_reset].cpu()[reset_rows],
           "returns": st.returns.cpu()[:, rows], "advantages": st.advantages.cpu()[:, rows]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), (t if t.dtype in (torch.float32, torch.float64) else t.double()).numpy())


def measure_e2e(wl, args, world):
    import torch.distributed as dist
    env = wl.env
    # the host ships the four foot records packed ((N,4,13): 208 B/env) instead of all 17 bodies (884 B/env)
    names_in = ("root_states", "dof_state", "contact_forces", "foot_records", "actions")
    nb = env.num_bodies
    feet = wl.host_state["rigid_body_states"].view(-1, nb, 13)[:, list(wl.cfg.feet_indices), :].contiguous()
    env.foot_records = feet.to(env.device)
    env.refresh_buffers()
    host_src = dict(wl.host_state, foot_records=feet)
    host_in = {k: host_src[k].contiguous().pin_memory() for k in names_in}
    dev_in = {k: getattr(env, k) for k in names_in}
    outs = {"obs_buf": env.obs_buf, "privileged_obs_buf": env.privileged_obs_buf, "rew_buf": env.rew_buf, "reset_buf": env.reset_buf}
    host_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in outs.items()}
    h2d = sum(v.numel() * v.element_size() for v in host_in.values())
    d2h = sum(v.numel() * v.element_size() for v in host_out.values())

    # Three streams: H2D of step t+1 and D2H of step t overlap (PCIe is full duplex); the step itself
    # goes through the public API, including post_physics_step's host sync on the reset count.
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    main = torch.cuda.current_stream()
    ev = {"in": torch.cuda.Event(), "compute": torch.cuda.Event(), "out": torch.cuda.Event()}
    ev["compute"].record(main)
    ev["out"].record(main)

    def e2e_step():
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev["compute"])               # previous step has consumed the input tensors
            for k in names_in:
                dev_in[k].view(-1).copy_(host_in[k].view(-1), non_blocking=True)
            ev["in"].record(s_in)
        main.wait_event(ev["in"])
        main.wait_event(ev["out"])                       # previous results are on the host: outputs may be overwritten
        env._delay_actions()
        for k in range(env.cfg_hot.decimation):
            env._compute_torques_into(env.delayed_actions[:, k], env.torques)
        env.post_physics_step()
        ev["compute"].record(main)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev["compute"])
            for k, v in outs.items():
                host_out[k].copy_(v, non_blocking=True)
            ev["out"].record(s_out)

    def e2e_rollout():
        for _ in range(wl.t_len):
            e2e_step()
        wl.storage.compute_returns(wl.last_values, wl.cfg.gamma, wl.cfg.lam)
        s_out.synchronize()
        main.synchronize()

    e2e_rollout()
    iters = max(1, min(args.steps, 3))
    ms = timed(e2e_rollout, iters, world > 1)
    return {"value": world * args.envs * wl.t_len * iters / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * wl.t_len,
            "d2h_bytes_per_step": d2h * wl.t_len, "rollouts": iters, "ms_per_step": ms / iters,
            "api": "FusedLeggedRobot._compute_torques x4 + post_physics_step per env-step, HIMRolloutStorage.compute_returns per rollout",
            "h2d_per_env": h2d // args.envs, "d2h_per_env": d2h // args.envs}


def measure_record_transition(args, peak_gbs):
    """SURVEY.md §8f rank 1 (runner patch + process_env_step + add_transitions as one launch): a pure
    HBM copy, reported beside the headline as its own roofline line (not part of `value`)."""
    from isaacgymloco_b200 import roofline as R, synthetic as S
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    n, t_len, dev = args.envs, 4, torch.device("cuda", torch.cuda.current_device())
    st = HIMRolloutStorage(n, t_len, [270], [238], [12], device=dev)
    tr = {k: v.to(dev) for k, v in S.make_transition(n, 3).items()}
    tt = HIMRolloutStorage.Transition()
    tt.observations, tt.critic_observations, tt.actions, tt.values = tr["obs"], tr["critic_obs"], tr["actions"], tr["values"]
    tt.actions_log_prob, tt.action_mean, tt.action_sigma = tr["log_prob"], tr["mu"], tr["sigma"]
    cnt = torch.tensor([tr["termination_ids"].numel()], dtype=torch.int32, device=dev)

    def one():
        st.step = st.step % t_len
        st.record_env_step(tt, tr["rewards"], tr["dones"], {"time_outs": tr["time_outs"]}, tr["privileged_obs"],
                           tr["termination_ids"], tr["termination_privileged_obs"], 0.99, termination_count=cnt)
    for _ in range(3):
        one()
    iters = 20
    ms = timed(one, iters, False) / iters
    bytes_env = R.record_transition_bytes()["total"]
    gbs = bytes_env * n / (ms * 1e-3) / 1e9
    return {"envs": n, "us_per_step": 1e3 * ms, "bytes_per_env": bytes_env, "achieved_GBps": gbs, "peak_GBps": peak_gbs,
            "frac": gbs / peak_gbs, "note": "slots rotate over 4 steps: 1.65 GB working set per pass, larger than L2"}


def measure_minibatch_gather(args, peak_gbs):
    """SURVEY.md §8f rank 3: one minibatch (T*N/4 random rows of all ten rollout fields) gathered by
    one fused launch; 16,384 envs x 24 steps (configs[3] sizes), beside torch's ten index gathers."""
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    n, t_len, dev = 16384, 24, torch.device("cuda", torch.cuda.current_device())
    st = HIMRolloutStorage(n, t_len, [270], [238], [12], device=dev)
    for x in st._batch_fields():
        x.normal_()
    perm = torch.randperm(n * t_len, device=dev)
    mb = n * t_len // 4
    fields = st._batch_fields()
    chunks = [perm[i * mb:(i + 1) * mb] for i in range(4)]

    def fused():
        for c in chunks:
            st.gather_batch(c, fields)

    def eager():
        for c in chunks:
            for x in fields:
                x[c]
    for _ in range(2):
        fused(); eager()
    ms = timed(fused, 5, False) / 5 / 4
    ms_t = timed(eager, 5, False) / 5 / 4
    row_bytes = 2 * 4 * sum(int(x[0].numel()) for x in fields) + 8
    gbs = row_bytes * mb / (ms * 1e-3) / 1e9
    return {"rows": mb, "us_per_minibatch": 1e3 * ms, "bytes_per_row": row_bytes, "achieved_GBps": gbs, "peak_GBps": peak_gbs,
            "frac": gbs / peak_gbs, "torch_index_us_per_minibatch": 1e3 * ms_t}


def measure_stairs16384(args, peak_gbs):
    """BASELINE.json configs[2] (SURVEY.md §8d config 3): aliengo_stairs, 16,384 envs, 1300 x 2300 synthetic stair /
    slope / rough field, the 20-term stairs reward set + termination, all five termination clauses.  16,384 envs touch
    81 MB per env-step -- less than the 126 MB L2 -- so 277 MB are written between timed replays to flush it."""
    from isaacgymloco_b200 import roofline as R
    dev = torch.device("cuda", torch.cuda.current_device())
    n = 16384
    wl = Workload(n, args.rollout, 0, 1, dev, task="stairs")
    bytes_tab = R.per_env_step_bytes(wl.cfg, args.rollout)
    flush = torch.empty(277 * 1024 * 1024 // 4, device=dev)
    for _ in range(2):
        wl.rollout()
    # direct launches with an L2 flush before every env-step: CUDA-event pairs around the fused kernel
    wl.fused_ms.clear()
    for _ in range(8):
        flush.fill_(1.0)
        wl.env_step(time_fused=True)
    torch.cuda.synchronize()
    fus = [a.elapsed_time(b) for a, b in wl.fused_ms][2:]
    fused_ms = sum(fus) / len(fus)
    wl.env._fused_event_hook = None
    g = torch.cuda.CUDAGraph()
    s_ = torch.cuda.Stream()
    s_.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s_):
        wl.rollout()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s_):
            wl.rollout()
    torch.cuda.current_stream().wait_stream(s_)
    for _ in range(3):
        g.replay()
    iters = 10
    ms = timed(g.replay, iters, False) / iters
    alg = bytes_tab["post_physics"] * n
    gbs = alg / (fused_ms * 1e-3) / 1e9
    return {"workload": "aliengo_stairs, 16384 envs x 24-step rollout, 21-row stairs reward set, 187-pt scan on the 1300x2300 field",
            "value": n * args.rollout / (ms * 1e-3), "unit": UNIT, "ms_per_rollout_graph": ms, "l2_policy": "fused-kernel timing: 277 MB flush "
            "write before every env-step; rollout value: graph replay, 81 MB working set (L2-resident)",
            "roofline": {"bound": "hbm", "kernel": "hl_post_physics_fused_kernel", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s",
                         "frac": gbs / peak_gbs, "avg_launch_ms": fused_ms, "algorithmic_bytes_per_launch": alg,
                         "bytes_per_env_step": bytes_tab}}


def measure_amp16384(args, peak_gbs):
    """BASELINE.json configs[3] (SURVEY.md §8d config 4): the 7 aliengo clips (from tests/golden/amp.npz: the mocap
    files live in the reference tree), 16,384 samples per get_full_frame_at_time_batch, a 2e6-transition preload,
    expert-pair gathers of 16384*24/4 rows, discriminator-input assembly + reward epilogue for 16,384 envs; the MLP
    (cuBLAS) is timed separately."""
    import numpy as np
    from isaacgymloco_b200.amp_discriminator import AMPDiscriminator, Normalizer
    from isaacgymloco_b200.motion_loader import AMPLoader
    dev = torch.device("cuda", torch.cuda.current_device())
    gold = dict(np.load(os.path.join(ROOT, "tests", "golden", "amp.npz"), allow_pickle=False))
    k = len(gold["frame_durations"])
    tabs = dict(frames=[gold[f"clip{i}"] for i in range(k)], frame_durations=gold["frame_durations"], weights=gold["weights_raw"],
                names=[str(x) for x in gold["clip_names"]])
    np.random.seed(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ld = AMPLoader(str(dev), 0.02, preload_transitions=True, num_preload_transitions=2_000_000, clip_tables=tabs)
    torch.cuda.synchronize()
    preload_s = time.perf_counter() - t0
    n = 16384
    idx = ld.weighted_traj_idx_sample_batch(n)
    tm = ld.traj_time_sample_batch(idx)
    idx_t, tm_t = torch.as_tensor(idx).to(dev), torch.as_tensor(tm).to(dev)
    blend = lambda: ld.get_full_frame_at_time_batch_device(idx_t, tm_t)
    for _ in range(3):
        blend()
    ms_blend = timed(blend, 50, False) / 50
    mb = n * 24 // 4
    pidx = torch.as_tensor(np.random.choice(ld.preloaded_s.shape[0], size=mb)).to(dev)
    pairs = lambda: ld.gather_pairs(pidx)
    for _ in range(3):
        pairs()
    ms_pairs = timed(pairs, 50, False) / 50
    torch.manual_seed(0)
    disc = AMPDiscriminator(60, 0.01, [1024, 512], str(dev), task_reward_lerp=0.3).to(dev)
    norm = Normalizer(30, device=str(dev))
    s0, s1 = ld.gather_pairs(pidx[:n])
    norm.update(s0)
    task_r = torch.rand(n, device=dev)
    asm = lambda: disc.assemble_input(s0, s1, norm)
    full = lambda: disc.predict_amp_reward(s0, s1, task_r, normalizer=norm)
    for _ in range(3):
        asm(); full()
    ms_asm = timed(asm, 50, False) / 50
    ms_full = timed(full, 50, False) / 50
    gb = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9
    return {"workload": "aliengo AMP: 7 clips / 658 frames, 16384-sample frame blend, 2e6 preload, 98304-row pair gather, 16384-env "
                        "discriminator input + reward",
            "frame_blend": {"samples": n, "us": 1e3 * ms_blend, "samples_per_s": n / (ms_blend * 1e-3),
                            "GBps_written": gb(n * 49 * 4, ms_blend), "note": "table (129 KB) is L2/L1-resident; output 3.2 MB"},
            "preload_2e6": {"seconds": preload_s, "note": "host numpy sampling (RNG, as in the reference) + 2 blend launches of 2e6 samples"},
            "pair_gather": {"rows": mb, "us": 1e3 * ms_pairs, "GBps": gb(mb * (2 * 30 * 4 + 2 * 30 * 4 + 8), ms_pairs),
                            "frac_of_hbm_peak": gb(mb * (2 * 30 * 4 + 2 * 30 * 4 + 8), ms_pairs) / peak_gbs,
                            "note": "random 196-B rows of two 392 MB tables: sector-granular gathers (algorithmic bytes counted, not sectors)"},
            "disc_input": {"envs": n, "us": 1e3 * ms_asm, "GBps": gb(n * (60 * 4 + 60 * 4), ms_asm)},
            "predict_amp_reward": {"envs": n, "us_total": 1e3 * ms_full, "us_mlp_cublas": 1e3 * (ms_full - ms_asm),
                                   "note": "assembly + 60-1024-512-1 MLP (cuBLAS, out of scope) + reward epilogue"}}


def measure_latency_4096(args):
    """configs[1]: 4096 envs on one B200 -- the working set (20 MB) is L2-resident, so this is a
    latency number (CUDA-graph replay of one rollout), not a roofline one."""
    wl = Workload(4096, args.rollout, 0, 1, torch.device("cuda", torch.cuda.current_device()))
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        wl.rollout()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            wl.rollout()
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(5):
        g.replay()
    iters = 20
    ms = timed(g.replay, iters, False)
    direct = timed(wl.rollout, 5, False)
    return {"envs": 4096, "rollout_len": args.rollout, "us_per_env_step_graph": 1e3 * ms / iters / args.rollout,
            "value_graph": 4096 * args.rollout * iters / (ms * 1e-3), "value_direct_launch": 4096 * args.rollout * 5 / (direct * 1e-3),
            "unit": UNIT}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--rollout", type=int, default=24, help="T: env-steps per rollout")
    ap.add_argument("--traffic", type=float, default=None, help="ncu dram bytes per fused launch (from profiles/)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-comm", action="store_true", help="N>1: leave out the gradient / statistics exchanges (attribution runs)")
    ap.add_argument("--amp", action="store_true", help="N>1: add the AMP discriminator-gradient and normaliser exchanges")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's shard) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    if args.traffic is None:
        p = os.path.join(ROOT, "profiles", "fused_traffic.json")
        if os.path.exists(p):
            args.traffic = json.load(open(p)).get("dram_bytes_per_launch")
    run_gpu_arm(args)
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
