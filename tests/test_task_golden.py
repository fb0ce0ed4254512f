"""Oracle task layer vs the golden vectors produced by executing the reference's own Python
(tests/golden/make_golden.py): utils/quaternion.py, Ultrasound.reward/_post_action/_check_terminated/
get_trajectory.  float64, tolerance = round-off only."""
import numpy as np
import pytest

from rui_b200 import abi
from rui_b200.env import probe_torso_contact


def test_quaternion(golden, O):
    for c in golden["quaternion"]:
        q1, q2 = np.array(c["q1"]), np.array(c["q2"])
        np.testing.assert_allclose(O.difference_quat(q1, q2), c["difference"], atol=1e-14)
        d = O.distance_quat(q1, q2)
        if c["distance"] is None:  # the reference raises (quaternion.py:51) when q1*conj(q2) == (-1,0,0,0): treated as 0
            assert d == 0.0
        else:
            assert abs(d - c["distance"]) < 1e-12


def test_reward(golden, O):
    assert len(golden["reward"]) >= 50
    for c in golden["reward"]:
        r, pe, oe = O.reward(c["eef_pos"], c["eef_quat_xyzw"], c["traj_pt"], c["vel_mean"], c["fz_mean"], c["dfz"], c["in_contact"])
        assert abs(r - c["reward"]) < 1e-12
        np.testing.assert_allclose(pe, c["pos_error"], rtol=1e-12, atol=1e-15)
        assert abs(oe - c["ori_error"]) < 1e-12
        assert 0.0 <= r <= 12.0


def test_post_action_sequences(golden, O):
    jr = np.zeros(14)  # joint limits unused here: check_q_limits is stubbed to False in the golden generator
    for seq in golden["post_action"]:
        ts = np.zeros(abi.TASK_DIM)
        ts[abi.TS_TRAJ_START:abi.TS_TRAJ_START + 3] = seq["start"]
        ts[abi.TS_TRAJ_END:abi.TS_TRAJ_END + 3] = seq["end"]
        ts[abi.TS_U0] = seq["u0"]
        u = min(max(seq["u0"], 0.0), 1.0)
        ts[abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3] = np.array(seq["start"]) + u * (np.array(seq["end"]) - np.array(seq["start"]))
        ts[abi.TS_FZ_MEAN] = seq["fz_mean0"]
        n_done = 0
        for t, s in enumerate(seq["steps"]):
            ts[abi.TS_TIMESTEP] = t + 1
            r, d = O.post_action(ts, seq["horizon"], seq["control_freq"], seq["early_termination"], jr, s["eef_pos"], s["eef_quat_xyzw"],
                                 s["hand_vel"], s["fz"], s["in_contact"], None)
            assert abs(r - s["reward"]) < 1e-11, (t, r, s["reward"])
            assert d == s["done"], t
            np.testing.assert_allclose(ts[abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3], s["traj_pt"], atol=1e-14)
            np.testing.assert_allclose(ts[abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3], s["controller_traj_pos"], atol=1e-14)
            assert abs(ts[abi.TS_VEL_MEAN] - s["vel_mean"]) < 1e-13
            assert abs(ts[abi.TS_DFZ] - s["dfz"]) < 1e-9
            assert abs(ts[abi.TS_FZ_MEAN] - s["fz_mean"]) < 1e-12
            assert bool(ts[abi.TS_TOUCHED]) == s["touched"]
            n_done += d
        assert n_done <= 1
    # the four sequences exercise: orientation termination, horizon, lost contact, trajectory deviation
    assert [s["steps"][-1]["done"] for s in golden["post_action"]] == [True, True, True, True]


def test_contact_query(golden):
    for c in golden["contact_query"]:
        assert probe_torso_contact(c["names"]) == c["in_contact"]


def test_trajectory_grid(golden, O):
    g = golden["trajectory"]
    t = g["torso_xpos"]
    gx = [O.grid_point(t, i, 0)[0] for i in range(50)]
    gy = [O.grid_point(t, 0, i)[1] for i in range(50)]
    np.testing.assert_allclose(gx, g["grid_x"], atol=1e-15)
    np.testing.assert_allclose(gy, g["grid_y"], atol=1e-15)
    for d in g["draws_seed3"]:  # every reference draw is a grid point at z = torso z + 0.039
        for p in (d["start"], d["end"]):
            assert min(abs(np.array(g["grid_x"]) - p[0])) < 1e-15 and min(abs(np.array(g["grid_y"]) - p[1])) < 1e-15
            assert abs(p[2] - O.grid_point(t, 0, 0)[2]) < 1e-15
    assert g["deterministic"]["start"] == [0.062, -0.020, 0.896] and g["deterministic"]["end"] == [-0.032, -0.075, 0.896]


def test_constants(golden):
    c = golden["constants"]
    np.testing.assert_allclose(c["goal_quat"], abi.GOAL_QUAT_XYZW, atol=0)
    assert (c["pos_error_mul"], c["ori_error_mul"], c["vel_error_mul"], c["force_error_mul"], c["der_force_error_mul"]) == (90, 0.2, 45, 0.7, 0.01)
    assert (c["pos_reward_mul"], c["ori_reward_mul"], c["vel_reward_mul"], c["force_reward_mul"], c["der_force_reward_mul"]) == (5, 1, 1, 3, 2)
    assert (c["goal_velocity"], c["goal_contact_z_force"], c["alpha"], c["pos_error_threshold"], c["ori_error_threshold"]) == (0.04, 5, 0.1, 1.0, 0.10)
    assert (c["top_torso_offset"], c["x_range"], c["y_range"], c["grid_pts"], c["sigma"]) == (0.039, 0.15, 0.09, 50, 0.010)


def test_reset_noise_and_draws(golden, O, soft_model):
    """Seeded Philox reset: integer draws in range, probe noise matches the reference's sigmas (ultrasound.py:880-881)."""
    from conftest import CC_TRACK
    g = golden["trajectory"]
    cfg = abi.make_config(1, CC_TRACK, control_freq=500, torso_solref_randomization=True, initial_probe_pos_randomization=True, seed=11,
                          reset_eef_bias=(0, 0, 0))
    dev, ks, bs = [], [], []
    for gid in range(160):
        e = O.OracleEnv(soft_model, cfg, gid)
        obs = e.reset()
        ts = e.get_state()[3]
        ks.append(ts[abi.TS_STIFFNESS]); bs.append(ts[abi.TS_DAMPING])
        assert 1300 <= ts[abi.TS_STIFFNESS] < 1600 and ts[abi.TS_STIFFNESS] == int(ts[abi.TS_STIFFNESS])
        assert 17 <= ts[abi.TS_DAMPING] < 41 and ts[abi.TS_DAMPING] == int(ts[abi.TS_DAMPING])
        assert 0 <= ts[abi.TS_U0] < 1
        for k in (abi.TS_TRAJ_START, abi.TS_TRAJ_END):
            assert min(abs(np.array(g["grid_x"]) - ts[k])) < 1e-12 and min(abs(np.array(g["grid_y"]) - ts[k + 1])) < 1e-12
        dev.append(obs[12:15])  # eef - traj_pt = noise (IK converged, zero bias)
    std = np.std(dev, axis=0)
    np.testing.assert_allclose(std, g["noise_std"], rtol=0.25)
    assert len(set(ks)) > 50 and len(set(bs)) > 15


def test_cylinder_torso_constants(golden):
    """use_box_torso=False (ultrasound.py:184-186, soft_human_torso.xml): trajectory-grid constants of the cylinder model."""
    from rui_b200.model import build_model, cylinder_torso_params
    c = golden["constants_cylinder"]
    p = cylinder_torso_params()
    assert c["use_box_torso"] is False
    assert (p.top_torso_offset, p.traj_x_range, p.traj_y_range) == (c["top_torso_offset"], c["x_range"], c["y_range"]) == (0.041, 0.15, 0.05)
    m = build_model(p)
    assert (m.nq, m.nv, len(m.eq_pairs)) == (284, 283, 536)  # same topology as the box, projected geometry
    pos = m.part_pos
    assert np.hypot(pos[:, 0], pos[:, 1]).max() <= 0.14 + 1e-12  # (x, y) inside the L2 ball of the largest half extent
    assert abs(np.abs(pos[:, 2]).max() - 0.175) < 1e-12
    assert abs(p.torso_pos[2] - (0.8 + 0.005 + 0.05)) < 1e-12


def _reward_from_obs_row(O, o, in_contact):
    """reward() (ultrasound.py:230-269) evaluated from ONE 19-float observation row: the eef quaternion is recovered from
    obs[15:19] = difference_quat(eef_xquat, goal_quat) (xyzw arrays through the wxyz routine, :390 -> eef = obs ⊗ goal for unit goal)."""
    g = np.asarray(abi.GOAL_QUAT_XYZW, dtype=np.float64)
    g = g / np.linalg.norm(g)
    a, b = np.asarray(o[15:19], dtype=np.float64), g
    eef_xyzw = np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                         a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])
    # eef_pos - traj_pt = obs[12:15]: only the difference enters the reward
    r, _, _ = O.reward(o[12:15], eef_xyzw, np.zeros(3), o[11] + 0.04, o[9] + 5.0, o[10], in_contact)
    return r


def test_art_reward_is_reproduced_by_its_observation_row(art, O):
    """Reference-produced pin of the OBSERVATION TIMING.  The shipped VecNormalize pickles hold the last raw (obs, reward) batch of
    training (`old_obs`, `old_reward`, 64 envs x 3 models).  reward() at step t reads the task state of step t-1 (ultrasound.py:525
    runs before :528-546).  In every one of the 192 rows the reward is reproduced, to float32 round-off, from the SAME step's
    observation row -- so the observation returned for step t also carries the t-1 task state (traj_pt, running means, dFz):
    robosuite samples the observables inside the substep loop, before _post_action, and returns the cached values.  The oracle
    and the CUDA kernel follow that (oracle_step: write_obs before post_action; soft.cuh K9)."""
    n = 0
    for name, a in art.items():
        obs, rew = np.array(a["old_obs"]), np.array(a["old_reward"])
        assert obs.shape == (64, 19) and rew.shape == (64,)
        for o, r in zip(obs, rew):
            with_c, without_c = _reward_from_obs_row(O, o, True), _reward_from_obs_row(O, o, False)
            err = min(abs(r - with_c), abs(r - without_c))  # in_contact itself is not an observation channel
            assert err < 2e-5, (name, r, with_c, without_c)
            n += 1
    assert n == 192


def test_oracle_step_returns_the_observation_reward_was_computed_from(O, soft_model):
    """The same identity on the oracle's own rollouts: reward_t == reward(obs_t) with the step's contact flag."""
    from conftest import CC_TRACK
    e = O.OracleEnv(soft_model, abi.make_config(1, CC_TRACK, control_freq=500, seed=5, torso_solref_randomization=True,
                                                initial_probe_pos_randomization=True), 0)
    e.reset()
    rng = np.random.default_rng(1)
    for s in range(25):
        o, r, d = e.step(rng.uniform(0, 1, 6))
        inc = bool(e.get_state()[3][abi.TS_IN_CONTACT])
        assert abs(r - _reward_from_obs_row(O, o, inc)) < 2e-5, s  # (acos near -1 amplifies the 1e-8 norm error of the 8-digit goal_quat)


def test_scene_params_match_the_reference_mjcf():
    """SceneParams (what the kernels are compiled against) vs the reference's in-tree MJCF (soft_box.xml, soft_human_torso.xml,
    ultrasound_arena.xml + ultrasound_arena.py placement, ultrasound_probe_gripper.xml), parsed by the package's own reader.  The
    committed parse (tests/golden/mjcf_golden.json, written by make_golden.py) is checked always; where RUI_REFERENCE names a
    checkout of the reference the files are re-read and must give the same parse."""
    import json
    import os

    from rui_b200 import mjcf
    from rui_b200.model import SceneParams, cylinder_torso_params
    here = os.path.dirname(os.path.abspath(__file__))
    with open(os.path.join(here, "golden", "mjcf_golden.json")) as f:
        gold = json.load(f)

    def norm(x):  # JSON turns tuples into lists
        return json.loads(json.dumps(x))

    for key, params, box in (("soft_box", SceneParams(), True), ("soft_human_torso", cylinder_torso_params(), False)):
        assert mjcf.check_scene_params(params, gold[key]) == {}, key
        f = mjcf.scene_fields(gold[key])
        assert f["comp_count"] == (9, 4, 11) and f["solref_smooth"] == (-1324.17, -17.59) and f["probe_pos"] == (-0.004, -0.063, 0.128)
        if os.environ.get("RUI_REFERENCE"):
            ref = os.path.join(os.environ["RUI_REFERENCE"], "src", "my_models")
            assert norm(mjcf.read_assets(ref, box)) == gold[key]
            assert mjcf.scene_params_from_mjcf(ref, box) == params
    # a deliberately wrong constant is caught
    import dataclasses
    assert "cap_radius" in mjcf.check_scene_params(dataclasses.replace(SceneParams(), cap_radius=0.008), gold["soft_box"])
    assert gold["soft_box"]["gripper"]["mesh_file"] == "meshes/ultrasound_probe_mesh.stl"  # (missing from the reference: A-PROBE-1)
    assert gold["soft_box"]["arena"]["colliding_geoms"] == ["floor", "table_collision"]


def test_error_metrics_match_the_reference_files(tmp_path):
    """SURVEY 8(f) rank 3, second half: `rui_b200.error_metrics.calculate_error_metrics` over the save_data CSV stream writes the
    files `src/utils/error.py:calculate_error_metrics` writes (error_data/<model>/<metric>.csv) with the same numbers.  Golden:
    the reference's own module executed on a synthetic episode (tests/golden/make_golden.py -> error_metrics_golden.json)."""
    import json
    import os

    import pandas as pd

    from rui_b200.error_metrics import calculate_error_metrics
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "error_metrics_golden.json")) as f:
        g = json.load(f)
    for fld in ("simulation_data", "reward_data"):
        os.makedirs(tmp_path / fld)
        for k, v in g[fld].items():
            pd.DataFrame(np.array(v)).to_csv(tmp_path / fld / f"{k}_7.csv", header=None, index=None)
    m = calculate_error_metrics("7", root=str(tmp_path))
    files = sorted(os.listdir(tmp_path / "error_data" / "7"))
    assert files == sorted(k + ".csv" for k in g["error_data_files"]) and len(files) == 13
    for k, text in g["error_data_files"].items():
        ref = float(text)
        got = float(open(tmp_path / "error_data" / "7" / (k + ".csv")).read())
        assert abs(got - ref) <= 1e-12 * max(1.0, abs(ref)), (k, got, ref)
        assert abs(m[k] - ref) <= 1e-12 * max(1.0, abs(ref))
