"""Shared helpers of the -m gpu parity tests (imported lazily: needs the CUDA library)."""
import numpy as np
import torch

RTOL, ATOL = 1e-5, 2e-6     # north_star: floats within rel 1e-5 in fp32 (atol for values near 0)

EXACT = ("reset_buf", "time_out_buf", "contact_filt", "last_contacts", "episode_length_buf")
FLOATS = ("base_lin_vel", "base_ang_vel", "projected_gravity", "measured_heights", "rew_buf", "feet_air_time",
          "commands", "obs_buf", "privileged_obs_buf", "last_actions", "last_last_actions", "last_dof_pos",
          "last_dof_vel", "last_torques", "last_root_vel", "episode_sums")


def make_env(cfg, state, hf, targets=None, noise=None, no_reset=False, device="cuda:0"):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot

    class Env(FusedLeggedRobot):
        def _reset_dofs(self, ids):
            n = self.num_envs
            self.dof_state.view(n, 12, 2)[ids] = self._t["dof_state"].view(n, 12, 2)[ids]

        def _reset_root_states(self, ids):
            self.root_states[ids] = self._t["root_states"][ids]

        def _resample_commands(self, ids):
            self.commands[ids] = self._t["commands"][ids]

        def reset_idx(self, ids):
            if self._no_reset:
                return
            # the replayed targets carry no gain factors: keep them as they were (reset_idx would re-draw them)
            factors = [t.clone() for t in (self.Kp_factors, self.Kd_factors, self.motor_strength_factors)]
            super().reset_idx(ids)
            for t, old in zip((self.Kp_factors, self.Kd_factors, self.motor_strength_factors), factors):
                t.copy_(old)

        def _pre_step_callbacks(self):
            # these tests replay the step without its RNG-driven callbacks (pre-step command resampling,
            # disturbances; LR:612-613,631-632) -- tests/test_gpu_reset.py covers those
            return None

    env = Env(cfg, state, hf, device=device)
    env.push_interval = 0                       # no pushes (LR:627-628) in the replayed step either
    env._no_reset = no_reset or targets is None
    env._t = {k: v.to(device) for k, v in (targets or {}).items()}
    if noise is not None:
        env.set_noise_tensors(**noise)
    return env


def assert_close(a, b, name, rtol=RTOL, atol=ATOL):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=name)


def assert_equal(a, b, name):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_array_equal(a, b, err_msg=name)


def compare_snapshots(got, want, heights_exact=True):
    for k in EXACT:
        assert_equal(got[k], want[k], k)
    for k in FLOATS:
        if k == "measured_heights" and heights_exact:
            assert_equal(got[k], want[k], k)      # same cell index => same int16 => same float
        else:
            assert_close(got[k], want[k], k)
