"""-m gpu: every reward term of the CUDA path against a float64 reference on the reward probe state
(tests/reward_probe.py), and the compile-time reward lists (`hl_reward_fast<MASK>`) against the generic
`hl_eval_term` loop bit for bit.

Bound for row k: |got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[k]|.  The episode sums start at zero, so each
row is the scaled term of this step (one IEEE add onto 0 is exact).  feet_air_time and last_contacts, which the
terms mutate, are compared exactly (against the fp32 oracle for feet_air_time)."""
import functools

import pytest
import torch

import reward_probe as P
from isaacgymloco_b200 import config as C

pytestmark = pytest.mark.gpu

CUDA, CPU = C.INDEX_MATH_TORCH_CUDA, C.INDEX_MATH_TORCH_CPU

# the two compile-time reward lists of csrc/hl_math.cuh (HL_MASK_FLAT also serves the AMP task)
_COMMON = ["action_rate", "ang_vel_xy", "base_height", "calf_pose", "dof_acc", "feet_air_time", "feet_contact_forces",
           "feet_slide", "hip_pos", "joint_power", "lin_vel_z", "orientation", "stand_still", "stuck", "thigh_pose",
           "torques", "tracking_ang_vel", "tracking_lin_vel"]
FAST_LISTS = {"flat": sorted(_COMMON + ["feet_mirror", "foot_clearance_base", "smoothness"]),
              "amp": sorted(_COMMON + ["feet_mirror", "foot_clearance_base", "smoothness"]),
              "stairs": sorted(_COMMON + ["collision", "feet_stumble"])}


@functools.lru_cache(maxsize=3)
def _probe(task, n, index_math, only_positive=False):
    kw = dict(only_positive_rewards=True) if only_positive else {}
    cfg = P.probe_cfg(task, n, index_math=index_math, **kw)
    state, hf = P.make_probe(cfg, n)
    return cfg, state, hf, P.reference64(cfg, state, hf), P.reference32(cfg, state, hf)


def _outputs(env):
    torch.cuda.synchronize()
    r = len(env.episode_sums)
    return dict(rew_buf=env.rew_buf.cpu().clone(), episode_sums=env._episode_sums_buf[:r].cpu().clone(),
                feet_air_time=env.feet_air_time.cpu().clone(), last_contacts=env.last_contacts.cpu().clone())


def _fused(cfg, state, hf, single=None):
    from gpu_helpers import make_env
    env = make_env(cfg, state, hf)
    if single is not None:
        env.single_launch = single
        env.refresh_buffers()
    env.fused_pre_reset()
    return _outputs(env)


def _stages(cfg, state, hf):
    """The drop-in methods in the reference's order (LR:193-222)."""
    from gpu_helpers import make_env
    env = make_env(cfg, state, hf)
    env.episode_length_buf += 1
    env.update_base_frame()
    env.update_heading_command()
    env.measured_heights = env._get_heights()
    env.check_termination()
    env.compute_reward()
    return _outputs(env)


def _check_vs_reference(cfg, got, ref64, ref32, what):
    P.check_bound(got["episode_sums"], P.rows64(ref64), cfg.episode_sum_names(), f"{what}: episode_sums")
    P.check_bound(got["rew_buf"], ref64.rew_buf, ["rew_buf"], f"{what}: rew_buf")
    assert torch.equal(got["last_contacts"], ref64.last_contacts), f"{what}: last_contacts"
    assert torch.equal(got["feet_air_time"], ref32.feet_air_time), f"{what}: feet_air_time"


@pytest.mark.parametrize("n", [4099, 65536])
@pytest.mark.parametrize("path,index_math", [("fused", CPU), ("fused", CUDA), ("stages", CPU), ("stages", CUDA)],
                         ids=["fused-cpu_math", "fused-cuda_math", "stages-cpu_math", "stages-cuda_math"])
def test_all_terms_generic_loop_vs_float64(path, index_math, n):
    """All 51 terms (the generic hl_eval_term loop: this list has no compile-time form) through the fused step and
    through the drop-in stage sequence, every episode_sums row and rew_buf within the bound of the float64 reference."""
    cfg, state, hf, ref64, ref32 = _probe("allterms", n, index_math)
    got = _fused(cfg, state, hf) if path == "fused" else _stages(cfg, state, hf)
    _check_vs_reference(cfg, got, ref64, ref32, f"allterms {path} n={n}")


def _form(monkeypatch, cfg, state, hf, impl, epb, single):
    from isaacgymloco_b200 import _lib as L
    monkeypatch.delenv("HL_FUSED_GENERIC_REWARD", raising=False)
    monkeypatch.setenv("HL_FUSED_IMPL", impl)
    if epb:
        monkeypatch.setenv("HL_FUSED_EPB", epb)
    else:
        monkeypatch.delenv("HL_FUSED_EPB", raising=False)
    out = _fused(cfg, state, hf, single)
    return out, int(L.lib.hl_fused_last_impl())


@pytest.mark.parametrize("n", [4096, 16385, 65536])
@pytest.mark.parametrize("task", P.TASKS)
def test_fast_reward_list_equals_generic_loop(monkeypatch, task, n):
    """hl_reward_fast<MASK> (torch-CUDA index arithmetic) in every kernel form -- the tile the size picks (32 at 4,096
    envs, 52 at 65,536), HL_FUSED_EPB=64, single-launch and separate compaction, the persistent kernel -- equals the
    tiled kernel running the generic loop (HL_FUSED_GENERIC_REWARD=1) on identical inputs, bit for bit; and is within
    the bound of the float64 reference."""
    from isaacgymloco_b200 import _lib as L
    cfg, state, hf, ref64, ref32 = _probe(task, n, CUDA)
    assert cfg.active_terms()[0] == FAST_LISTS[task], "the task's list is no longer a compile-time list"
    monkeypatch.setenv("HL_FUSED_IMPL", "tiled")
    monkeypatch.setenv("HL_FUSED_GENERIC_REWARD", "1")
    want = _fused(cfg, state, hf)
    assert int(L.lib.hl_fused_last_impl()) == 0
    _check_vs_reference(cfg, want, ref64, ref32, f"{task} generic n={n}")
    for impl, epb in (("tiled", None), ("tiled", "64"), ("persist", None)):
        for single in (True, False):
            got, used = _form(monkeypatch, cfg, state, hf, impl, epb, single)
            what = f"{task} n={n} {impl} epb={epb or 'auto'} single_launch={single}"
            assert used == (1 if impl == "persist" else 0), f"{what}: kernel form {used} ran"   # 1 = persistent
            rows = [f"{nm} ({int((g != w).sum())} envs)" for nm, g, w in
                    zip(cfg.episode_sum_names(), got["episode_sums"], want["episode_sums"]) if not torch.equal(g, w)]
            assert not rows, f"{what}: episode_sums rows differ from the generic loop: {', '.join(rows)}"
            for k in want:
                assert torch.equal(got[k], want[k]), f"{what}: {k} differs from the generic loop"


@pytest.mark.parametrize("path", ["fused-fast", "fused-generic", "stages"])
def test_clip_then_termination(monkeypatch, path):
    """only_positive_rewards with a termination scale (LR:376-380): on envs whose loop sum is negative,
    rew_buf == max(sum, 0) + termination == the termination row, exactly -- for resets without time-out (the
    termination term), resets with time-out and envs that do not reset (both 0)."""
    n = 4099
    cfg, state, hf, ref64, ref32 = _probe("stairs", n, CUDA, only_positive=True)
    assert cfg.only_positive_rewards and cfg.termination_scale is not None
    monkeypatch.setenv("HL_FUSED_IMPL", "tiled")
    if path == "fused-generic":
        monkeypatch.setenv("HL_FUSED_GENERIC_REWARD", "1")
    got = _stages(cfg, state, hf) if path == "stages" else _fused(cfg, state, hf)
    _check_vs_reference(cfg, got, ref64, ref32, f"clip {path}")
    neg = P.loop_sum(ref64) < -1e-6
    term = got["episode_sums"][-1]
    cats = {"reset without time-out": ref64.reset_buf & ~ref64.time_out_buf,
            "reset with time-out": ref64.reset_buf & ref64.time_out_buf,
            "no reset": ~ref64.reset_buf}
    for name, m in cats.items():
        sel = neg & m
        assert int(sel.sum()) >= n // 50, f"{name}: only {int(sel.sum())} envs with a negative sum"
        assert torch.equal(got["rew_buf"][sel], term[sel]), f"{name}: rew_buf != max(sum, 0) + termination"
    assert (term[cats["reset without time-out"]] == float(torch.tensor(cfg.termination_scale, dtype=torch.float32))).all()
    assert (term[~cats["reset without time-out"]] == 0).all()
