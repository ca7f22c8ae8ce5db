"""CPU (-m "not gpu"): the C-ABI library loads and exports every symbol the header declares,
struct layouts match, the host-side config logic follows the reference's rules, the mocap parser
matches the reference loader, and the product path refuses to run without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden


def test_library_exports_every_declared_symbol():
    from isaacgymloco_b200 import _lib as L
    header = open(os.path.join(ROOT, "include", "himloco_b200.h")).read()
    declared = set(re.findall(r"\b(hl_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    raw = ctypes.CDLL(L.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(raw, name), f"{name} declared in include/himloco_b200.h but not exported"
    assert declared == set(L.EXPORTS), (declared ^ set(L.EXPORTS))
    assert L.lib.hl_version() == 102
    assert L.lib.hl_sizeof_cfg() == ctypes.sizeof(L.HlCfg)
    assert L.lib.hl_sizeof_env_buffers() == ctypes.sizeof(L.HlEnvBuffers)


def test_high_speed_slice_count_is_the_references():
    """The integer the kernels compare global env ids with equals the size of the reference's slice
    `env_ids < num_envs * 0.2` (LR:649) for every num_envs up to 300,000.  Since arange is increasing, the
    reference's count is fixed by the comparison on the ids next to the boundary; it is checked there for every size,
    and on the whole arange for every size up to 2,000 and for the sizes the tests and the benchmark use."""
    from isaacgymloco_b200.config import high_vel_env_count
    for n in range(1, 300001):
        c = high_vel_env_count(n)
        lo, hi = max(c - 2, 0), min(c + 2, n)
        w = torch.arange(lo, hi) < n * 0.2            # the reference's comparison on ids lo .. hi-1
        k = int(w.sum())
        assert lo + k == c and (lo == 0 or bool(w[0])) and (hi == n or not bool(w[-1])), n
    for n in list(range(1, 2001)) + [4096, 4100, 16384, 16385, 65536, 262144, 299995, 300000]:
        assert high_vel_env_count(n) == int((torch.arange(n) < n * 0.2).sum()), n
    assert [high_vel_env_count(n) for n in (20, 4100, 5000, 16385)] == [4, 820, 1000, 3277]


def test_abi_guards_reject_bad_structs():
    from isaacgymloco_b200 import _lib as L
    from isaacgymloco_b200 import config as C
    c = C.aliengo("flat").to_c()
    c.struct_bytes = 12
    b = L.HlEnvBuffers()
    rc = L.lib.hl_post_physics_fused(ctypes.byref(c), ctypes.byref(b), 16, None)
    assert rc == 1 and b"size mismatch" in L.lib.hl_last_error()
    with pytest.raises(RuntimeError):
        L.check(rc)
    with pytest.raises(RuntimeError):
        L.ptr(torch.zeros(4))            # CPU tensor: no fallback


def test_no_cpu_fallback():
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    from isaacgymloco_b200.motion_loader import AMPLoader
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from isaacgymloco_b200 import config as C, synthetic as S
    with pytest.raises(RuntimeError):
        HIMRolloutStorage(8, 4, [270], [238], [12], device="cpu")
    with pytest.raises(RuntimeError):
        AMPLoader("cpu", 0.02, clip_tables=dict(frames=[np.zeros((3, 61))], frame_durations=[0.02], weights=[1]))
    cfg = C.aliengo("flat", num_envs=8)
    hf = S.make_terrain(cfg)
    with pytest.raises(RuntimeError):
        FusedLeggedRobot(cfg, S.make_state(cfg, 8, hf), hf, device="cpu")


def test_reward_term_tables_follow_reference_rules():
    from isaacgymloco_b200 import config as C
    flat = C.aliengo("flat")
    names, scales = flat.active_terms()
    assert names == sorted(names) and len(names) == 21 and "termination" not in names
    assert names[:3] == ["action_rate", "ang_vel_xy", "base_height"]
    assert abs(scales[names.index("tracking_lin_vel")] - 1.5 * 0.02) < 1e-12
    assert flat.termination_scale is None and flat.max_episode_length == 1000
    st = C.aliengo("stairs", num_envs=16384)
    n2, _ = st.active_terms()
    assert len(n2) == 20 and abs(st.termination_scale + 50 * 0.02) < 1e-12
    assert st.terrain_shape == (1300, 2300) and flat.terrain_shape == (1100, 1900)
    sr = st.stumble_ranges()
    assert (sr["stairsup_start"], sr["stairsup_end"], sr["pit_start"], sr["gap_end"]) == (3277, 8192, 16384, 16384)
    assert st.episode_sum_names()[-1] == "termination"
    nv = flat.noise_scale_vec()
    assert nv.shape == (232,) and np.allclose(nv[3:6], 0.05) and np.allclose(nv[21:33], 0.075) and np.allclose(nv[45:], 0.5)
    with pytest.raises(AttributeError):
        C.aliengo("flat", reward_scales={"foot_clearance_base_terrain": -1.0}).active_terms()
    with pytest.raises(NameError):
        C.aliengo("flat", control_type="X").to_c()
    c = st.to_c()
    assert c.n_terms == 20 and c.has_termination_term == 1 and c.term_base_vel_violate == 1
    assert [c.term_id[k] for k in range(3)] == [C.TERM_ID[n] for n in n2[:3]]
    assert len(C.REWARD_TERMS) == 51 and C.REWARD_TERMS == sorted(C.REWARD_TERMS)


def test_synthetic_state_is_deterministic_and_shaped():
    from isaacgymloco_b200 import config as C, synthetic as S
    cfg = C.aliengo("stairs", num_envs=64)
    hf = S.make_terrain(cfg, seed=2)
    assert hf.dtype == torch.int16 and tuple(hf.shape) == (1300, 2300) and int(hf.abs().max()) > 0
    a, b = S.make_state(cfg, 64, hf, seed=3), S.make_state(cfg, 64, hf, seed=3)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert a["root_states"].shape == (64, 13) and a["dof_state"].shape == (768, 2)
    assert a["rigid_body_states"].shape == (64 * 17, 13) and a["contact_forces"].shape == (64 * 17, 3)
    assert a["episode_length_buf"].dtype == torch.long and a["last_contacts"].dtype == torch.bool


@pytest.mark.skipif(not os.path.isdir("/root/reference/datasets/mocap_motions_aliengo"), reason="needs the reference's mocap clips (build container only)")
def test_mocap_parser_matches_reference_loader():
    from isaacgymloco_b200.motion_loader import AMPLoader
    gold = load_golden("amp.npz")
    d = "/root/reference/datasets/mocap_motions_aliengo"
    for i, name in enumerate(gold["clip_names"]):
        data, dur, w = AMPLoader._parse_motion_file(os.path.join(d, str(name)))
        np.testing.assert_array_equal(data[:, :49].astype(np.float32), gold[f"clip{i}"])
        assert dur == gold["frame_durations"][i] and w == gold["weights_raw"][i]


def test_mocap_binary_cache_round_trip(tmp_path):
    """SURVEY.md §8f rank 4: the binary clip cache holds exactly what the JSON parse produces."""
    from isaacgymloco_b200.motion_loader import AMPLoader
    gold = load_golden("amp.npz")
    k = len(gold["frame_durations"])
    tabs = dict(frames=[gold[f"clip{i}"].astype(np.float64) for i in range(k)], frame_durations=list(gold["frame_durations"]),
                weights=list(gold["weights_raw"]), names=[str(x) for x in gold["clip_names"]])
    path = str(tmp_path / "clips.npz")
    AMPLoader._write_cache(path, tabs)
    back = AMPLoader.read_cache(path)
    assert back["names"] == tabs["names"]
    np.testing.assert_array_equal(back["frame_durations"], tabs["frame_durations"])
    np.testing.assert_array_equal(back["weights"], tabs["weights"])
    for a, b in zip(back["frames"], tabs["frames"]):
        np.testing.assert_array_equal(a, b)
    d = "/root/reference/datasets/mocap_motions_aliengo"
    if os.path.isdir(d):   # build container: straight from the reference's JSON clips
        files = [os.path.join(d, str(n)) for n in gold["clip_names"]]
        AMPLoader.build_cache(files, path)
        back = AMPLoader.read_cache(path)
        for i, fr in enumerate(back["frames"]):
            np.testing.assert_array_equal(fr[:, :49].astype(np.float32), gold[f"clip{i}"])


def _reference_cfg_golden():
    """tests/golden/reference_cfg.json: what the reference's config classes and URDF give (oracle/make_goldens.py::
    mint_reference_cfg), stored so the comparisons below run without the reference sources."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_cfg.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("task", ["flat", "stairs", "amp", "recover"])
def test_presets_equal_the_reference_config_classes(task):
    """config.aliengo(task) (the constants that travel to the GPU box) == from_reference_cfg() of the
    reference's own AlienGo*Cfg class: every field of the C struct, the reward table, the noise vector and the
    reset_idx / resampling / domain-rand ranges.  Against the stored record, and against the reference's classes
    themselves where its sources are present."""
    from oracle import ref_harness as H
    from oracle.make_goldens import cfg_record
    from isaacgymloco_b200 import config as C
    wants = [_reference_cfg_golden()[task]]
    if H.reference_available():
        wants.append(cfg_record(C.from_reference_cfg(H.reference_cfg(task), num_envs=4096, sim_dt=0.005)))
    got = cfg_record(C.aliengo(task, num_envs=4096))
    for want in wants:
        for name, _ in C.HlCfg._fields_:
            assert got["hlcfg"][name] == want["hlcfg"][name], name
        for k in ("terms", "scales", "episode_sum_names", "noise_scale_vec", "reset"):
            assert got[k] == want[k], k


def test_aliengo_dof_constants_equal_the_urdf():
    """The joint limits / efforts / velocities the reference reads through Isaac Gym's asset loader
    (LR:565-580) come from aliengo.urdf; the constants in config.py must be those numbers, in the
    reference's DOF order (FL, FR, RL, RR x hip, thigh, calf: LR:1145).  Against the stored record, and
    against the URDF itself where the reference sources are present."""
    from oracle import ref_harness as H
    from oracle.make_goldens import dof_record
    from isaacgymloco_b200 import config as C
    sources = [_reference_cfg_golden()["aliengo_dof"]]
    if H.reference_available():
        sources.append(dof_record(H.REFERENCE_ROOT))
    cfg = C.aliengo("flat")
    cfg.soft_dof_pos_limit = 1.0        # raw limits
    t = cfg.dof_tables()
    for src in sources:
        lim, dflt = src["limits"], src["default_joint_angles"]
        k = 0
        for leg in ("FL", "FR", "RL", "RR"):
            for joint in ("hip", "thigh", "calf"):
                a = lim[f"{leg}_{joint}_joint"]
                assert np.float32(a["effort"]) == t["torque_limits"][k]
                assert np.float32(a["velocity"]) == t["dof_vel_limits"][k]
                np.testing.assert_allclose([t["dof_pos_lo"][k], t["dof_pos_hi"][k]], [a["lower"], a["upper"]], rtol=1e-6)
                assert np.float32(dflt[f"{leg}_{joint}_joint"]) == t["default_dof_pos"][k]
                k += 1


@pytest.mark.skipif(not os.path.isdir("/root/reference/legged_gym"), reason="needs the reference sources (build container only)")
def test_integration_mixin_resolves_as_documented():
    """INTEGRATION.md §2: class LeggedRobotB200(FusedLeggedRobot, LeggedRobot) -- the hot-path methods, the reset
    hooks and step()/post_physics_step() come from FusedLeggedRobot; construction, sim creation and the config
    system stay the reference's.  (Class-level check: building a live env needs Isaac Gym.)"""
    from oracle import ref_harness as H
    H.install_stubs()
    from legged_gym.envs.base.legged_robot import LeggedRobot
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot

    class LeggedRobotB200(FusedLeggedRobot, LeggedRobot):
        def __init__(self, *a, **k):
            LeggedRobot.__init__(self, *a, **k)

    for name in ("step", "post_physics_step", "_compute_torques", "_get_heights", "_get_base_heights", "check_termination",
                 "compute_reward", "compute_observations", "compute_termination_observations", "get_amp_observations",
                 "reset_idx", "_reset_dofs", "_reset_root_states", "_resample_commands", "_push_robots", "_disturbance_robots",
                 "_update_terrain_curriculum", "update_command_curriculum"):
        assert getattr(LeggedRobotB200, name) is getattr(FusedLeggedRobot, name), name
        assert hasattr(LeggedRobot, name), f"the reference has no {name} to replace"
    for name in ("create_sim", "_create_envs", "_init_buffers", "_parse_cfg", "_get_env_origins", "_prepare_reward_function",
                 "refresh_actor_rigid_shape_props", "_process_rigid_shape_props", "_get_noise_scale_vec"):
        assert getattr(LeggedRobotB200, name) is getattr(LeggedRobot, name), name
    assert LeggedRobotB200.__mro__[1] is FusedLeggedRobot


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the contract's
    keys, the real env count of the sample, no GPU launches, and `kind` saying which CPU implementation was timed."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    proc = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, timeout=600, cwd=root)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "post_physics_gae_env_steps_per_s" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    if os.path.isdir("/root/reference"):
        assert cb["kind"] == "reference"          # the reference's own classes under the stub harness
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["sample_envs"] == 4096     # the env count actually timed, stated in the line


def test_library_holds_sm_100a_code_only():
    """The in-tree build is native Blackwell code (no PTX-only JIT path, no other arch): every embedded ELF is sm_100a."""
    import shutil
    import subprocess
    from isaacgymloco_b200 import _lib as L
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-lelf", L.LIB_PATH], capture_output=True, text=True, timeout=120).stdout
    elfs = [l for l in out.splitlines() if "ELF file" in l]
    assert elfs and all("sm_100a" in l for l in elfs), out
