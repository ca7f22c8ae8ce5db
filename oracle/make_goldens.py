"""TEST INFRASTRUCTURE ONLY.  Mint tests/golden/*.npz by executing the REAL reference classes
(/root/reference, via oracle/ref_harness.py) on seeded synthetic inputs.

Run in the build container only:   python -m oracle.make_goldens
The GPU box has no /root/reference; it consumes the committed fixtures.  Inputs are regenerated
from seeds by isaacgymloco_b200.synthetic (an `input_checksum` guards against generator drift);
only reference OUTPUTS are stored.
"""
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from isaacgymloco_b200 import config as C          # noqa: E402
from isaacgymloco_b200 import synthetic as S       # noqa: E402
from oracle import ref_harness as H                # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# (case name, reference task, N, seed, overrides of reward scales / cfg)
ENV_CASES = [
    dict(name="flat", task="flat", n=192, seed=11),
    dict(name="stairs", task="stairs", n=192, seed=12),
    dict(name="recover", task="recover", n=128, seed=13),
    dict(name="allterms", task="stairs", n=128, seed=14, all_terms=True),
    dict(name="plane", task="flat", n=64, seed=15, plane=True),
    dict(name="flat_noreset", task="flat", n=64, seed=16, no_reset=True),
    dict(name="amp", task="amp", n=96, seed=33),     # no `termination` cfg class: contact + time-out clauses only
]


def all_term_scales():
    """Every one of the 51 reward terms with a distinct non-zero scale."""
    sc = {}
    for i, name in enumerate(C.REWARD_TERMS):
        sc[name] = (-1.0 if i % 2 else 1.0) * (0.01 + 0.003 * i)
    return sc


def case_cfg(case) -> C.HotPathCfg:
    cfg = C.aliengo(case["task"], num_envs=case["n"], index_math=C.INDEX_MATH_TORCH_CPU)
    if case.get("all_terms"):
        cfg.reward_scales = all_term_scales()
    if case.get("plane"):
        # with mesh_type 'plane' the reference never builds self.terrain (LR:470-482), so a valid
        # plane cfg has out_of_border off (check_termination would raise otherwise, LR:276)
        cfg.mesh_type = "plane"
        cfg.out_of_border = False
    return cfg


def input_checksum(state):
    tot = 0.0
    for k in sorted(state):
        tot += float(state[k].double().abs().sum())
    return np.float64(tot)


def _patch_reference_env(env, case, targets, noise):
    n = env.num_envs
    calls = {"resample": 0}

    def resample(self, env_ids):
        calls["resample"] += 1
        if calls["resample"] % 2 == 0:           # 2nd call of a step comes from reset_idx
            self.commands[env_ids] = targets["commands"][env_ids]

    def reset_dofs(self, env_ids):
        self.dof_state.view(n, 12, 2)[env_ids] = targets["dof_state"].view(n, 12, 2)[env_ids]

    def reset_root(self, env_ids):
        self.root_states[env_ids] = targets["root_states"][env_ids]

    noop = lambda self, *a, **k: None
    for name, fn in (("_resample_commands", resample), ("_reset_dofs", reset_dofs),
                     ("_reset_root_states", reset_root), ("_update_terrain_curriculum", noop),
                     ("update_command_curriculum", noop), ("_push_robots", noop),
                     ("_disturbance_robots", noop), ("refresh_actor_rigid_shape_props", noop)):
        setattr(env, name, types.MethodType(fn, env))
    if case.get("no_reset"):
        env.reset_idx = types.MethodType(noop, env)


def mint_env_case(case):
    cfg = case_cfg(case)
    n = case["n"]
    hf = S.make_terrain(cfg, seed=case["seed"])
    state = S.make_state(cfg, n, hf, seed=case["seed"])
    noise = S.make_noise(n, seed=case["seed"] + 1000)
    targets = S.make_reset_targets(cfg, state, hf, seed=case["seed"] + 2000)

    # -------- the reference's own cfg object, edited the way a user would edit the cfg file
    H.install_stubs()
    from legged_gym.envs.base.legged_robot import LeggedRobot
    orig_cfg_fn = H.reference_cfg

    def cfg_fn(task):
        rc = orig_cfg_fn(task)
        if case.get("all_terms"):
            for k, v in all_term_scales().items():
                setattr(rc.rewards.scales, k, v)
        if case.get("plane"):
            rc.terrain.mesh_type = "plane"
            rc.termination.out_of_border = False
        return rc

    H.reference_cfg = cfg_fn
    try:
        env = H.build_reference_env(case["task"], state, hf, sum_names=cfg.episode_sum_names(), hot_cfg=cfg)
    finally:
        H.reference_cfg = orig_cfg_fn
    assert list(env.reward_names) == cfg.active_terms()[0], (env.reward_names, cfg.active_terms()[0])
    np.testing.assert_allclose([env.reward_scales[k] for k in env.reward_names], cfg.active_terms()[1],
                               rtol=1e-15)
    np.testing.assert_array_equal(env.noise_scale_vec.numpy(), cfg.noise_scale_vec())
    assert int(env.max_episode_length) == cfg.max_episode_length
    _patch_reference_env(env, case, targets, noise)

    out = {"input_checksum": input_checksum(state)}
    # a1: torques for the 4 substeps of a delayed-action tensor
    g = torch.Generator().manual_seed(case["seed"] + 3000)
    delayed = 0.5 * torch.randn(n, 4, 12, generator=g)
    out["torques4"] = torch.stack([env._compute_torques(delayed[:, k]) for k in range(4)], dim=1).numpy()

    # rand_like queue
    queue = [noise["term45"], noise["term187"], noise["obs45"], noise["obs187"]]
    if cfg.is_plane:
        pass
    real_rand_like = torch.rand_like

    def fake_rand_like(t, *a, **k):
        u = queue.pop(0)
        assert u.shape == t.shape, (u.shape, t.shape)
        return u.clone()

    torch.rand_like = fake_rand_like
    try:
        # a5 indices straight from the reference arithmetic (before the step mutates anything)
        if not cfg.is_plane:
            from legged_gym.utils.math import quat_apply_yaw
            pts = quat_apply_yaw(env.base_quat.repeat(1, 187), env.height_points) + env.root_states[:, :3].unsqueeze(1)
            pts += cfg.border_size
            pts = (pts / cfg.horizontal_scale).long()
            out["px"] = torch.clip(pts[:, :, 0], 0, hf.shape[0] - 2).numpy().astype(np.int16)
            out["py"] = torch.clip(pts[:, :, 1], 0, hf.shape[1] - 2).numpy().astype(np.int16)
        env_ids, term_obs, term_amp = env.post_physics_step()
        clip = cfg.clip_observations                      # LR:167-171 (end of step())
        env.obs_buf = torch.clip(env.obs_buf, -clip, clip)
        env.privileged_obs_buf = torch.clip(env.privileged_obs_buf, -clip, clip)
    finally:
        torch.rand_like = real_rand_like

    out["env_ids"] = env_ids.numpy()
    out["term_obs"] = term_obs.numpy()
    out["term_amp"] = term_amp.numpy()
    for k in ("base_lin_vel", "base_ang_vel", "projected_gravity", "measured_heights", "reset_buf",
              "time_out_buf", "rew_buf", "contact_filt", "last_contacts", "feet_air_time", "commands",
              "episode_length_buf", "obs_buf", "privileged_obs_buf", "last_actions",
              "last_last_actions", "last_dof_pos", "last_dof_vel", "last_torques", "last_root_vel"):
        out[k] = getattr(env, k).numpy().copy()
    out["episode_sums"] = np.stack([env.episode_sums[k].numpy() for k in cfg.episode_sum_names()]) \
        if cfg.episode_sum_names() else np.zeros((0, n), np.float32)
    if "episode" in env.extras:
        out["extras_names"] = np.array(sorted(k for k in env.extras["episode"] if k.startswith("rew_")))
        out["extras_vals"] = np.array([float(env.extras["episode"][k]) for k in out["extras_names"]],
                                      dtype=np.float32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, f"env_{case['name']}.npz"), **out)
    print(f"[golden] env_{case['name']}: n={n} resets={len(env_ids)} terms={len(cfg.active_terms()[0])}")


def mint_gae():
    H.install_stubs()
    from rsl_rl.storage import HIMRolloutStorage
    out = {}
    for name, n, t, seed, gamma, lam in (("a", 96, 24, 21, 0.99, 0.95), ("b", 33, 100, 22, 0.99, 0.95),
                                         ("c", 1, 5, 23, 0.9, 0.8), ("alldone", 8, 6, 24, 0.99, 0.95)):
        r = S.make_rollout(n, t, seed)
        if name == "alldone":
            r["dones"][:] = 1
        st = HIMRolloutStorage(n, t, [270], [238], [12], device="cpu")
        st.rewards.copy_(r["rewards"])
        st.values.copy_(r["values"])
        st.dones.copy_(r["dones"])
        st.compute_returns(r["last_values"], gamma, lam)
        out[f"{name}_returns"] = st.returns.numpy().copy()
        out[f"{name}_advantages"] = st.advantages.numpy().copy()
        out[f"{name}_meta"] = np.array([n, t, seed, gamma, lam], dtype=np.float64)
        out[f"{name}_checksum"] = np.float64(float(r["rewards"].double().abs().sum() + r["values"].double().abs().sum()))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "gae.npz"), **out)
    print("[golden] gae")


def mint_record():
    """Rollout-step recording (SURVEY.md §8f rank 1) through the reference's own classes:
    HIMPPO.process_env_step (him_ppo.py:104-115) on a real HIMRolloutStorage; the runner's
    two-line terminal patch (him_on_policy_runner.py:122-123) is applied as the runner does."""
    H.install_stubs()
    from rsl_rl.storage import HIMRolloutStorage
    from rsl_rl.algorithms import HIMPPO

    class _AC:
        def reset(self, dones=None):
            pass

    out = {}
    for name, n, t, seed, gamma in (("a", 40, 2, 41, 0.99), ("b", 67, 2, 42, 0.99), ("one", 1, 2, 43, 0.9)):
        alg = HIMPPO.__new__(HIMPPO)
        alg.device, alg.gamma, alg.actor_critic = "cpu", gamma, _AC()
        alg.transition = HIMRolloutStorage.Transition()
        alg.storage = HIMRolloutStorage(n, t, [270], [238], [12], device="cpu")
        for step in range(t):
            tr = S.make_transition(n, seed * 10 + step, reset_frac=(1.0 if name == "one" and step == 1 else 0.05))
            # HIMPPO.act (him_ppo.py:90-102) stores these on the transition
            alg.transition.actions, alg.transition.values = tr["actions"], tr["values"]
            alg.transition.actions_log_prob, alg.transition.action_mean = tr["log_prob"], tr["mu"]
            alg.transition.action_sigma = tr["sigma"]
            alg.transition.observations, alg.transition.critic_observations = tr["obs"], tr["critic_obs"]
            next_critic_obs = tr["privileged_obs"].clone().detach()
            next_critic_obs[tr["termination_ids"]] = tr["termination_privileged_obs"].clone().detach()
            alg.process_env_step(tr["rewards"], tr["dones"], {"time_outs": tr["time_outs"]}, next_critic_obs)
        st = alg.storage
        for f in ("observations", "privileged_observations", "next_privileged_observations", "actions", "rewards", "dones",
                  "values", "actions_log_prob", "mu", "sigma"):
            out[f"{name}_{f}"] = getattr(st, f).numpy().copy()
        out[f"{name}_meta"] = np.array([n, t, seed, gamma], dtype=np.float64)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "record.npz"), **out)
    print("[golden] record")


def mint_minibatch():
    """mini_batch_generator (SURVEY.md §8f rank 3) of the reference's own HIMRolloutStorage on CPU; the
    permutation it drew is recovered by re-seeding torch (same call, same generator state)."""
    H.install_stubs()
    from rsl_rl.storage import HIMRolloutStorage
    n, t, nmb, epochs, seed = 6, 5, 2, 2, 77
    st = HIMRolloutStorage(n, t, [270], [238], [12], device="cpu")
    for k_, v in S.make_filled_storage(n, t, seed).items():
        getattr(st, k_).copy_(v)
    torch.manual_seed(seed)
    batches = list(st.mini_batch_generator(nmb, epochs))
    torch.manual_seed(seed)
    indices = torch.randperm(nmb * ((n * t) // nmb))
    out = {"meta": np.array([n, t, nmb, epochs, seed], dtype=np.int64), "indices": indices.numpy()}
    for bi, b in enumerate(batches):
        for fi, x in enumerate(b):
            out[f"b{bi}_f{fi}"] = x.numpy().copy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "minibatch.npz"), **out)
    print(f"[golden] minibatch: {len(batches)} batches")


REPLAY_INSERTS = (5, 9, 4, 12, 1, 17, 3)   # rows per insert into a 16-row ring: plain, wrapping, > buffer_size


def replay_inputs(obs_dim=30, seed=88):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(k, obs_dim, generator=g), torch.randn(k, obs_dim, generator=g)) for k in REPLAY_INSERTS]


def mint_replay():
    """The reference's ReplayBuffer (replay_buffer.py) on CPU: a sequence of inserts with wrap-around,
    then sampled minibatches under a fixed numpy seed."""
    H.install_stubs()
    from rsl_rl.storage.replay_buffer import ReplayBuffer
    rb = ReplayBuffer(30, 16, "cpu")
    out = {}
    for i, (a, b) in enumerate(replay_inputs()):
        rb.insert(a, b)
        out[f"states_{i}"], out[f"next_{i}"] = rb.states.numpy().copy(), rb.next_states.numpy().copy()
        out[f"meta_{i}"] = np.array([rb.step, rb.num_samples], dtype=np.int64)
    np.random.seed(123)
    for j, (s_, n_) in enumerate(rb.feed_forward_generator(3, 7)):
        out[f"mb_s{j}"], out[f"mb_n{j}"] = s_.numpy().copy(), n_.numpy().copy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "replay.npz"), **out)
    print("[golden] replay")


def mint_amp():
    H.install_stubs()
    np.random.seed(31)
    loader = H.load_reference_amp_loader(preload=True, num_preload=1024, dt=0.02)
    out = {}
    nclips = len(loader.trajectories_full)
    out["clip_names"] = np.array([os.path.basename(p) for p in H.default_aliengo_motion_files()])
    for i in range(nclips):
        out[f"clip{i}"] = loader.trajectories_full[i].numpy()
    out["frame_durations"] = np.asarray(loader.trajectory_frame_durations, dtype=np.float64)
    out["weights_raw"] = np.asarray([1.0, 1.0, 1.0, 1.5, 1.5, 1.5, 1.5][:nclips])
    out["weights"] = np.asarray(loader.trajectory_weights, dtype=np.float64)
    out["lens"] = np.asarray(loader.trajectory_lens, dtype=np.float64)
    out["num_frames"] = np.asarray(loader.trajectory_num_frames, dtype=np.float64)

    # a16: frame blends at random + adversarial times
    rng = np.random.default_rng(32)
    b = 2048
    idx = rng.integers(0, nclips, size=b)
    times = loader.trajectory_lens[idx] * rng.uniform(size=b)
    # adversarial: t=0, exact frame multiples (blend==0 / ==1 neighbourhoods), near the clip end
    k = 256
    fd = loader.trajectory_frame_durations[idx[:k]]
    times[:k] = np.floor(times[:k] / fd) * fd
    times[k:k + 32] = 0.0
    times[k + 32:k + 64] = loader.trajectory_lens[idx[k + 32:k + 64]] * (1 - 1.0 / loader.trajectory_num_frames[idx[k + 32:k + 64]]) * 0.999999
    p = times / loader.trajectory_lens[idx]
    ok = np.ceil(p * loader.trajectory_num_frames[idx]) < loader.trajectory_num_frames[idx]
    idx, times = idx[ok], times[ok]
    frames = loader.get_full_frame_at_time_batch(idx, times)
    out["blend_idx"], out["blend_times"], out["blend_frames"] = idx, times, frames.numpy()

    # a17: pair gather from the preloaded tables
    out["pre_s"] = loader.preloaded_s.numpy()
    out["pre_s_next"] = loader.preloaded_s_next.numpy()
    np.random.seed(33)
    state = np.random.get_state()
    gen = loader.feed_forward_generator(2, 512)
    pairs = list(gen)
    np.random.set_state(state)
    out["pair_idx0"] = np.random.choice(loader.preloaded_s.shape[0], size=512)
    out["pair_idx1"] = np.random.choice(loader.preloaded_s.shape[0], size=512)
    out["pair_s0"], out["pair_sn0"] = pairs[0][0].numpy(), pairs[0][1].numpy()
    out["pair_s1"], out["pair_sn1"] = pairs[1][0].numpy(), pairs[1][1].numpy()

    # a19/a20: normaliser + discriminator reward
    from rsl_rl.algorithms.amp_discriminator import AMPDiscriminator
    from rsl_rl.utils.utils import Normalizer
    torch.manual_seed(34)
    disc = AMPDiscriminator(60, 0.01, [64, 32], "cpu", task_reward_lerp=0.3)
    norm = Normalizer(30)
    norm.update(pairs[0][0].numpy())
    norm.update(pairs[1][0].numpy())
    out["norm_mean"], out["norm_var"], out["norm_count"] = norm.mean, norm.var, np.float64(norm.count)
    s, sn = pairs[0][0][:256] * 1.5, pairs[0][1][:256] * 1.5
    task_r = torch.randn(256)
    r, d = disc.predict_amp_reward(s, sn, task_r, normalizer=norm)
    with torch.no_grad():
        x = torch.cat([norm.normalize_torch(s, "cpu"), norm.normalize_torch(sn, "cpu")], dim=-1)
    for k_, v in disc.state_dict().items():
        out["disc_" + k_.replace(".", "_")] = v.numpy()
    out["disc_s"], out["disc_sn"], out["disc_task_r"] = s.numpy(), sn.numpy(), task_r.numpy()
    out["disc_x"], out["disc_d"], out["disc_r"] = x.numpy(), d.numpy(), r.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "amp.npz"), **out)
    print(f"[golden] amp: clips={nclips} frames={sum(loader.trajectories_full[i].shape[0] for i in range(nclips))} blends={len(idx)}")

# --------------------------------------------------------------------------- f2: reset_idx with its draws
RESET_CASES = [dict(name="flat", task="flat", n=256, seed=51), dict(name="stairs", task="stairs", n=192, seed=52)]


def reset_inputs(case):
    """Seeded inputs of a reset golden: state, uniforms (N, 44), terrain-curriculum tables, the reset id list."""
    cfg = C.aliengo(case["task"], num_envs=case["n"])
    n = case["n"]
    hf = S.make_terrain(cfg, seed=case["seed"])
    state = S.make_state(cfg, n, hf, seed=case["seed"])
    g = torch.Generator().manual_seed(case["seed"] + 7000)
    u = torch.rand(n, C.RESET_NU, generator=g)
    origins = torch.zeros(cfg.num_rows, cfg.num_cols, 3)
    origins[..., 0] = (torch.arange(cfg.num_rows).float()[:, None] + 0.5) * cfg.terrain_length
    origins[..., 1] = (torch.arange(cfg.num_cols).float()[None, :] + 0.5) * cfg.terrain_width
    origins[..., 2] = 0.1 * torch.rand(cfg.num_rows, cfg.num_cols, generator=g)
    types_ = torch.div(torch.arange(n), (n / cfg.num_cols), rounding_mode="floor").to(torch.long)      # LR:1234
    levels = state["terrain_levels"].clone()
    levels[: n // 8] = cfg.num_rows - 1                    # some at the top level: move_up sends them to a random one
    env_origins = origins[levels, types_].clone()
    # half of the envs walked far (move up), a quarter barely moved (move down)
    state["root_states"][: n // 2, 0:2] = env_origins[: n // 2, 0:2] + cfg.terrain_length
    state["root_states"][n // 2: 3 * n // 4, 0:2] = env_origins[n // 2: 3 * n // 4, 0:2] + 0.01
    state["terrain_levels"] = levels
    ids = (torch.rand(n, generator=g) < 0.4).nonzero(as_tuple=False).flatten()
    return cfg, hf, state, u, dict(origins=origins, types=types_, env_origins=env_origins), ids


def mint_reset():
    H.install_stubs()
    import legged_gym.envs.base.legged_robot as LRM
    for case in RESET_CASES:
        cfg, hf, state, u, ter, ids = reset_inputs(case)
        n = case["n"]
        env = H.build_reference_env(case["task"], state, hf, sum_names=cfg.episode_sum_names(), hot_cfg=cfg)
        env.custom_origins = True
        env.env_origins = ter["env_origins"].clone()
        env.terrain_origins, env.terrain_types = ter["origins"].clone(), ter["types"].clone()
        env.max_terrain_level = cfg.num_rows
        rc = env.cfg
        base = rc.init_state.pos + rc.init_state.rot + rc.init_state.lin_vel + rc.init_state.ang_vel
        env.base_init_state = torch.tensor(base, dtype=torch.float)
        env.refresh_actor_rigid_shape_props = types.MethodType(lambda self, *a, **k: None, env)
        env.update_command_curriculum = types.MethodType(lambda self, *a, **k: None, env)
        assert rc.terrain.curriculum and env.init_done
        # the uniform columns in the reference's call order (include/himloco_b200.h: HL_RESET_NU)
        plan = []
        plan.append(("rand12", 0))                        # _reset_dofs: torch_rand_float(..., (len, 12))
        for k in (24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, 36, 37, 38):
            plan.append(("col", k))
        plan.append(("high", 39))                         # _resample_commands: the high-speed prefix of env_ids
        for k in (40, 41, 42):
            plan.append(("col", k))
        cursor = {"i": 0}

        def fake_rand_float(lower, upper, shape, device):
            kind, k = plan[cursor["i"]]
            cursor["i"] += 1
            if kind == "rand12":
                assert tuple(shape) == (len(ids), 12)
                uu = u[ids, 0:12]
            elif kind == "high":
                uu = u[ids[: shape[0]], 39:40]
            else:
                assert tuple(shape) == (len(ids), 1), (shape, k)
                uu = u[ids, k:k + 1]
            return (upper - lower) * uu + lower

        real_rf, real_rl, real_ri = LRM.torch_rand_float, torch.rand_like, torch.randint_like
        LRM.torch_rand_float = fake_rand_float
        torch.rand_like = lambda t, *a, **k: u[ids, 12:24].clone()
        torch.randint_like = lambda t, hi, *a, **k: (u[ids, 43] * hi).long().clamp(max=hi - 1)
        try:
            env.reset_idx(ids)
        finally:
            LRM.torch_rand_float, torch.rand_like, torch.randint_like = real_rf, real_rl, real_ri
        assert cursor["i"] == len(plan), (cursor["i"], len(plan))
        out = {"input_checksum": input_checksum(state), "ids": ids.numpy(), "u_checksum": np.float64(u.double().sum())}
        for k in ("root_states", "dof_state", "commands", "Kp_factors", "Kd_factors", "motor_strength_factors", "terrain_levels",
                  "env_origins", "last_actions", "last_last_actions", "last_dof_pos", "last_dof_vel", "last_torques",
                  "feet_air_time", "episode_length_buf", "reset_buf", "measured_heights"):
            out[k] = getattr(env, k).numpy().copy()
        out["episode_sums"] = np.stack([env.episode_sums[k].numpy() for k in cfg.episode_sum_names()])
        out["extras_names"] = np.array(sorted(k for k in env.extras["episode"] if k.startswith("rew_")))
        out["extras_vals"] = np.array([float(env.extras["episode"][k]) for k in out["extras_names"]], dtype=np.float32)
        np.savez_compressed(os.path.join(GOLDEN_DIR, f"reset_{case['name']}.npz"), **out)
        print(f"[golden] reset_{case['name']}: n={n} resets={len(ids)} levels moved={(out['terrain_levels'] != state['terrain_levels'].numpy()).sum()}")


def cfg_record(hc):
    """What tests/test_cpu_host.py compares of a HotPathCfg, JSON-safe and exact (fp32 fields as their double values):
    every HlCfg field, the reward table, the episode-sum rows, the noise vector and the reset / resampling ranges."""
    import ctypes
    import dataclasses
    import json
    c = hc.to_c()
    fields = {}
    for name, _ in C.HlCfg._fields_:
        v = getattr(c, name)
        fields[name] = list(v) if isinstance(v, ctypes.Array) else v
    names, scales = hc.active_terms()
    rec = dict(hlcfg=fields, terms=list(names), scales=[float(x) for x in scales], episode_sum_names=list(hc.episode_sum_names()),
               noise_scale_vec=[float(x) for x in hc.noise_scale_vec()], reset=dataclasses.asdict(hc.reset))
    return json.loads(json.dumps(rec))


def dof_record(reference_root):
    """aliengo.urdf's revolute-joint limits (LR:565-580 read them through Isaac Gym's asset loader) and the reference's
    default joint angles, keyed by joint name."""
    import xml.etree.ElementTree as ET
    root = ET.parse(os.path.join(reference_root, "legged_gym", "resources", "robots", "aliengo", "urdf", "aliengo.urdf")).getroot()
    limits = {j.get("name"): {k: float(v) for k, v in j.find("limit").attrib.items()}
              for j in root.findall("joint") if j.get("type") == "revolute"}
    dflt = {k: float(v) for k, v in H.reference_cfg("flat").init_state.default_joint_angles.items()}
    return dict(limits=limits, default_joint_angles=dflt)


REFERENCE_CFG_TASKS = ("flat", "stairs", "amp", "recover")


def mint_reference_cfg():
    """tests/golden/reference_cfg.json: cfg_record() of from_reference_cfg() for each of the reference's AlienGo*Cfg
    classes, and dof_record() of its URDF."""
    import json
    out = {task: cfg_record(C.from_reference_cfg(H.reference_cfg(task), num_envs=4096, sim_dt=0.005)) for task in REFERENCE_CFG_TASKS}
    out["aliengo_dof"] = dof_record(H.REFERENCE_ROOT)
    with open(os.path.join(GOLDEN_DIR, "reference_cfg.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


def main():
    assert H.reference_available(), "run in the build container (needs /root/reference)"
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(1)
    for case in ENV_CASES:
        mint_env_case(case)
    mint_gae()
    mint_record()
    mint_minibatch()
    mint_replay()
    mint_amp()
    mint_reset()
    mint_reference_cfg()


if __name__ == "__main__":
    main()
