"""-m gpu: PD torques and observations of the CUDA path against float64 references on the probes of
tests/torque_obs_probe.py, where every clip and control branch is taken on both sides.

Bound for column k: |got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[:, k]| (reward_probe.bound).  Beyond it, exact:
clipped torques equal +-torque_limits[d]; T-mode torques (pure products and a clip, nothing to contract) equal the
fp32 oracle on the same device; a height entry where the +-1 clip binds equals +-obs_height (no noise); an entry
where clip_observations binds equals +-clip_observations; the observation history shift equals the old rows."""
import functools

import numpy as np
import pytest
import torch

import torque_obs_probe as TP
from isaacgymloco_b200 import config as C

pytestmark = pytest.mark.gpu

CUDA, CPU = C.INDEX_MATH_TORCH_CUDA, C.INDEX_MATH_TORCH_CPU
DOFS = [f"dof {d}" for d in range(12)]


# ----------------------------------------------------------------------------- torques
@functools.lru_cache(maxsize=4)
def _torque_probe(ctl, n):
    cfg = TP.torque_cfg(ctl, n, CPU)
    state, hf = TP.make_torque_probe(cfg, n)
    return (state, hf) + TP.reference64_torques(cfg, state, hf)


def _actions_view(actions, how):
    """The (N, 12) actions as the caller passes them: contiguous, a column slice of a (N, 4, 12) delay buffer, or
    one float into a buffer with row stride 13 (the scalar-kernel path)."""
    n = actions.shape[0]
    if how == "contiguous":
        return actions.cuda()
    if how == "delayed":
        buf = torch.zeros(n, 4, 12, device="cuda")
        buf[:, 2] = actions.cuda()
        return buf[:, 2]
    buf = torch.zeros(n * 13 + 1, device="cuda")
    view = buf[1:].as_strided((n, 12), (13, 1))
    view.copy_(actions.cuda())
    return view


@pytest.mark.parametrize("n", [1, 3, 4099, 65536 + 3])
@pytest.mark.parametrize("index_math", [CPU, CUDA], ids=["cpu_math", "cuda_math"])
@pytest.mark.parametrize("method,how", [("compute", "contiguous"), ("compute", "delayed"), ("into", "delayed"),
                                        ("into", "strided13")])
@pytest.mark.parametrize("ctl", TP.CONTROL_TYPES)
def test_torques_vs_float64(ctl, method, how, index_math, n):
    """_compute_torques / _compute_torques_into: torques and joint_pos_target within the bound of the float64
    reference; clipped entries exactly +-limit; T mode bit-equal to the fp32 oracle on the device.  The 65,539-env
    case ends in a partial float4 group of threads; the stride-13 view is routed to the scalar kernel."""
    from gpu_helpers import make_env
    from oracle import torch_oracle as O
    from isaacgymloco_b200 import synthetic as S
    state, hf, tq64, tg64, raw = _torque_probe(ctl, n)
    cfg = TP.torque_cfg(ctl, n, index_math)
    env = make_env(cfg, state, hf)
    actions = _actions_view(state["actions"], how)
    if how == "strided13":
        assert actions.data_ptr() % 16 != 0 and actions.stride(0) % 4 != 0, "the view would take the float4 kernel"
    env.joint_pos_target.fill_(float("nan"))
    if method == "compute":
        got = env._compute_torques(actions)
    else:
        got = torch.full((n, 12), float("nan"), device="cuda")
        assert env._compute_torques_into(actions, got) is got
    torch.cuda.synchronize()
    got, target = got.cpu(), env.joint_pos_target.cpu()
    what = f"{ctl} {method}({how}) n={n}"
    TP.check_bound(got.T, tq64.T, DOFS, f"{what}: torques")
    TP.check_bound(target.T, tg64.T, DOFS, f"{what}: joint_pos_target")
    lim = torch.from_numpy(cfg.dof_tables()["torque_limits"]).expand(n, 12)
    gates = TP.torque_gates(cfg, raw)
    assert torch.equal(got[gates["raw torque > +limit"]], lim[gates["raw torque > +limit"]]), f"{what}: +clip"
    assert torch.equal(got[gates["raw torque < -limit"]], -lim[gates["raw torque < -limit"]]), f"{what}: -clip"
    oenv = O.OracleEnv(cfg, S.to_device(state, "cuda"), hf.cuda())
    want = oenv._compute_torques(state["actions"].cuda()).cpu()
    if ctl == "T":
        assert torch.equal(got, want), f"{what}: {int((got != want).sum())} T-mode torques differ from the fp32 oracle"
    else:
        inside = gates["inside the limits"]
        print(f"\n[{what}] bit-equal to the fp32 oracle: {float((got == want).double().mean()):.1%} of all entries, "
              f"{float((got[inside] == want[inside]).double().mean()):.1%} of the unclipped ones")


def test_compute_torques_into_rejects_bad_views():
    """A transposed or column-strided actions view and an `out` that is not a contiguous fp32 (N, 12) CUDA tensor
    raise ValueError instead of being read or written wrong."""
    from gpu_helpers import make_env
    n = 64
    state, hf, _, _, _ = _torque_probe("P", n)
    env = make_env(TP.torque_cfg("P", n), state, hf)
    good_a, good_out = state["actions"].cuda(), torch.empty(n, 12, device="cuda")
    bad_actions = [torch.empty(12, n, device="cuda").T, torch.empty(n, 24, device="cuda")[:, ::2],
                   good_a.double(), good_a[:32]]
    bad_outs = [torch.empty(12, n, device="cuda").T, torch.empty(n, 24, device="cuda")[:, ::2],
                torch.empty(n, 12, device="cuda", dtype=torch.float64), torch.empty(n, 12), torch.empty(n, 13, device="cuda")]
    for a in bad_actions:
        with pytest.raises(ValueError):
            env._compute_torques_into(a, good_out)
    for o in bad_outs:
        with pytest.raises(ValueError):
            env._compute_torques_into(good_a, o)
    env._compute_torques_into(good_a, good_out)


# ----------------------------------------------------------------------------- observations
@functools.lru_cache(maxsize=2)
def _obs_probe(task, variant, n):
    cfg = TP.obs_cfg(task, variant, n)
    state, hf, noise = TP.make_obs_probe(cfg, n)
    return (cfg, state, hf, noise) + TP.reference64_obs(cfg, state, hf, noise)


PATHS = ["tiled-single", "tiled-separate", "tiled-epb64", "persist", "stages"]


def _run(monkeypatch, path, cfg, state, hf, noise):
    """One step without resets applied -> (ids, obs_buf, privileged_obs_buf, terminal rows, terminal AMP rows, form)."""
    from gpu_helpers import make_env
    from isaacgymloco_b200 import _lib as L
    monkeypatch.delenv("HL_FUSED_EPB", raising=False)
    monkeypatch.setenv("HL_FUSED_IMPL", "persist" if path == "persist" else "tiled")
    if path == "tiled-epb64":
        monkeypatch.setenv("HL_FUSED_EPB", "64")
    env = make_env(cfg, state, hf, noise=noise)
    form = None
    if path == "stages":
        clip = cfg.clip_observations
        env.episode_length_buf += 1
        env.update_base_frame()
        env.update_heading_command()
        env.measured_heights = env._get_heights()
        env.check_termination()
        env.compute_reward()
        ids = env.reset_buf.nonzero(as_tuple=False).flatten()
        term = env.compute_termination_observations(ids).clone()
        amp = env.get_amp_observations()[ids]
        env.compute_observations()
        env.obs_buf.clamp_(-clip, clip)
        env.privileged_obs_buf.clamp_(-clip, clip)
    else:
        if path in ("tiled-single", "tiled-separate"):
            env.single_launch = path == "tiled-single"
            env.refresh_buffers()
        ids, term, amp = env.post_physics_step()
        form = int(L.lib.hl_fused_last_impl())
    torch.cuda.synchronize()
    return ids.cpu(), env.obs_buf.cpu(), env.privileged_obs_buf.cpu(), term.cpu(), amp.cpu(), form


def _cols(what, width):
    return [f"{what}[{i}]" for i in range(width)]


@pytest.mark.parametrize("n", [4099, 65536])
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("variant", TP.OBS_VARIANTS)
@pytest.mark.parametrize("task", TP.OBS_TASKS)
def test_observations_vs_float64(monkeypatch, task, variant, path, n):
    """obs_buf[:, :45], privileged_obs_buf, the terminal rows and the terminal AMP rows within the bound of the
    float64 reference; the clips exact where they bind; the history shift bit-exact.  The persistent kernel covers
    the heightfield configs whose clip_observations cannot bind (plane meshes and a binding clip run the tiled kernel,
    which the test checks too)."""
    cfg, state, hf, noise, e64, ids64, term64, amp64 = _obs_probe(task, variant, n)
    ids, obs, priv, term, amp, form = _run(monkeypatch, path, cfg, state, hf, noise)
    what = f"{task} {variant} {path} n={n}"
    if path == "persist":
        assert form == (1 if task != "plane" and variant != "clip" else 0), f"{what}: kernel form {form} ran"
    elif form is not None:
        assert form == 0, f"{what}: kernel form {form} ran"
    assert torch.equal(ids, ids64), f"{what}: reset ids"
    pw = priv.shape[1]
    TP.check_bound(obs[:, :45].T, e64.obs_buf[:, :45].T, _cols("obs", 45), f"{what}: obs_buf")
    TP.check_bound(priv.T, e64.privileged_obs_buf.T, _cols("priv", pw), f"{what}: privileged_obs_buf")
    TP.check_bound(term.T, term64.T, _cols("term", pw), f"{what}: terminal rows")
    TP.check_bound(amp.T, amp64.T, _cols("amp", 30), f"{what}: terminal AMP rows")
    clip = cfg.clip_observations
    assert torch.equal(obs[:, 45:], state["obs_buf"][:, :225].clamp(-clip, clip)), f"{what}: history shift"

    gates = TP.obs_gates(cfg, e64)
    if variant == "plain":
        s = np.float32(cfg.obs_height)
        for key, sign in (("height z-0.5-h > +1", 1.0), ("height z-0.5-h < -1", -1.0)):
            m = gates[key]
            assert (priv[:, 51:][m] == sign * s).all(), f"{what}: {key}: height obs != {sign * s}"
            assert (term[:, 51:][m[ids64]] == sign * s).all(), f"{what}: {key}: terminal height != {sign * s}"
    if variant == "clip":
        cl = np.float32(clip)
        for grp in ("ang_vel", "dof_vel", "heights"):
            for side, sign in ((">", 1.0), ("<", -1.0)):
                m = gates[f"{grp} {side} {'+' if sign > 0 else '-'}clip_observations"]
                sl = TP.GROUPS[grp]
                assert (priv[:, sl][m] == sign * cl).all(), f"{what}: {grp} {side}: privileged obs != {sign * cl}"
                if sl.stop is not None and sl.stop <= 45:
                    assert (obs[:, sl][m] == sign * cl).all(), f"{what}: {grp} {side}: obs != {sign * cl}"
