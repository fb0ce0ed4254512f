#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by EXECUTING the reference's own Python.

Needs a checkout of the reference, named by the RUI_REFERENCE environment variable; the JSON files it
writes are committed, so the tests never need the reference.  What is executed unmodified from the reference checkout:

  * src/utils/quaternion.py ............ q_log, difference_quat, distance_quat
  * src/my_environments/ultrasound.py .. Ultrasound.__init__ constants, reward, _post_action,
    _check_terminated, _check_probe_contact_with_torso, _get_contacts_objects, get_trajectory,
    _get_torso_grid, _get_waypoint, _convert_robosuite_to_toolbox_xpos, _add_noise_to_pos

Its third-party imports are NOT installed here (robosuite fork, mujoco-py, klampt, roboticstoolbox,
spatialmath, transforms3d; SURVEY.md §8c), so they are replaced by the minimal stubs below.  Each stub
restates documented upstream behaviour [EXT-recall]; everything in the reference tree itself runs as is.

Also decodes the statistics shipped in src/trained_rl_models/ (SURVEY.md App. D) into art_stats.json.

  RUI_REFERENCE=<checkout> python tests/golden/make_golden.py
"""
import base64
import importlib.util
import io
import json
import math
import os
import pickle
import sys
import types
import zipfile

import numpy as np

REF = os.path.join(os.environ["RUI_REFERENCE"], "src")
OUT = os.path.dirname(os.path.abspath(__file__))


# ----------------------------------------------------------------------------- stubs of un-vendored deps
class _Dummy:
    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Dummy()

    def __getattr__(self, n):
        return _Dummy()


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        t = type(name, (_Dummy,), {})
        setattr(self, name, t)
        return t


def _mod(name, **attrs):
    m = _StubModule(name)
    m.__path__ = []
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent:
        setattr(sys.modules[parent], child, m)
    return m


# transforms3d.quaternions (w,x,y,z)
def qconjugate(q):
    return np.array(q) * np.array([1.0, -1, -1, -1])


def qmult(q1, q2):
    w1, x1, y1, z1 = q1
    w2, x2, y2, z2 = q2
    return np.array([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                     w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2])


# robosuite.utils.transform_utils
def convert_quat(q, to="xyzw"):
    if to == "xyzw":
        return np.asarray(q)[[1, 2, 3, 0]]
    if to == "wxyz":
        return np.asarray(q)[[3, 0, 1, 2]]
    raise Exception("convert_quat: choose a valid `to` argument (xyzw or wxyz)")


def quat2mat_xyzw(q):
    x, y, z, w = np.asarray(q, dtype=np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def quat2axisangle(q):
    q = np.array(q, dtype=np.float64)
    q[3] = min(max(q[3], -1.0), 1.0)
    den = np.sqrt(1.0 - q[3] * q[3])
    if math.isclose(den, 0.0):
        return np.zeros(3)
    return (q[:3] * 2.0 * math.acos(q[3])) / den


class Trajectory:
    """klampt.model.trajectory.Trajectory: piecewise-linear, default times 0..n-1, end behaviour 'halt'."""

    def __init__(self, times=None, milestones=None):
        self.milestones = [np.asarray(m, dtype=np.float64) for m in milestones]
        self.times = list(range(len(self.milestones))) if times is None else list(times)

    def eval(self, t):
        if t <= self.times[0]:
            return self.milestones[0].tolist()
        if t >= self.times[-1]:
            return self.milestones[-1].tolist()
        i = int(np.searchsorted(self.times, t, side="right")) - 1
        u = (t - self.times[i]) / (self.times[i + 1] - self.times[i])
        return (self.milestones[i] + u * (self.milestones[i + 1] - self.milestones[i])).tolist()

    def deriv(self, t):
        if t <= self.times[0] or t >= self.times[-1]:
            return [0.0] * len(self.milestones[0])
        i = int(np.searchsorted(self.times, t, side="right")) - 1
        return ((self.milestones[i + 1] - self.milestones[i]) / (self.times[i + 1] - self.times[i])).tolist()


class SingleArmEnv:
    """robosuite SingleArmEnv/MujocoEnv slice used by the task code."""

    def __init__(self, **kwargs):
        self.control_freq = kwargs["control_freq"]
        self.horizon = kwargs["horizon"]
        self.ignore_done = kwargs["ignore_done"]
        self.control_timestep = 1.0 / self.control_freq
        self.timestep = 0
        self.deterministic_reset = False

    def _post_action(self, action):  # robosuite MujocoEnv._post_action
        reward = self.reward(action)
        self.done = (self.timestep >= self.horizon) and not self.ignore_done
        return reward, self.done, {}


class MujocoModel:
    pass


def install_stubs():
    _mod("transforms3d")
    _mod("transforms3d.quaternions", qconjugate=qconjugate, qmult=qmult)
    _mod("klampt")
    _mod("klampt.model")
    _mod("klampt.model.trajectory", Trajectory=Trajectory)
    _mod("roboticstoolbox")
    _mod("spatialmath")
    _mod("mujoco_py")
    _mod("robosuite")
    _mod("robosuite.utils")
    _mod("robosuite.utils.transform_utils", convert_quat=convert_quat, quat2mat=quat2mat_xyzw, quat2axisangle=quat2axisangle)
    _mod("robosuite.utils.mjcf_utils")
    _mod("robosuite.utils.placement_samplers")
    _mod("robosuite.utils.observables")
    _mod("robosuite.environments")
    _mod("robosuite.environments.manipulation")
    _mod("robosuite.environments.manipulation.single_arm_env", SingleArmEnv=SingleArmEnv)
    _mod("robosuite.models")
    _mod("robosuite.models.tasks")
    _mod("robosuite.models.tasks.task")
    _mod("robosuite.models.base", MujocoModel=MujocoModel)
    _mod("robosuite.models.objects")
    _mod("robosuite.models.arenas")
    _mod("robosuite.models.grippers")
    _mod("robosuite.models.grippers.gripper_model")


def load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


# ----------------------------------------------------------------------------- fake sim objects
class _Contact:
    def __init__(self, g1, g2):
        self.geom1, self.geom2, self.frame = g1, g2, np.array([0, 0, 1.0, 1, 0, 0, 0, 1, 0])


class _SimModel:
    def __init__(self, names):
        self.names = names

    def geom_id2name(self, i):
        return self.names[i]


class _SimData:
    pass


class _Sim:
    pass


class _Gripper(MujocoModel):
    contact_geoms = ["gripper0_probe_collision"]


class _Robot:
    name = "Panda"


def make_env(Ultrasound, early_termination=True, horizon=1000, control_freq=500):
    env = Ultrasound(robots="Panda", controller_configs={"type": "OSC_POSE"}, control_freq=control_freq, horizon=horizon,
                     early_termination=early_termination, use_camera_obs=False, use_object_obs=False, has_offscreen_renderer=False)
    geom_names = ["floor", "table_collision", "gripper0_probe_collision", "torso_Gcenter"] + [f"torso_G{i}_{j}_{k}" for i in range(2) for j in range(2) for k in range(3)]
    env.sim = _Sim()
    env.sim.model = _SimModel(geom_names)
    env.sim.data = _SimData()
    env.sim.data.contact = []
    env.sim.data.ncon = 0
    env.probe_id = 0
    env.sim.data.cfrc_ext = np.zeros((1, 6))
    r = _Robot()
    r.gripper = _Gripper()
    r._hand_vel = np.zeros(3)
    r.controller = types.SimpleNamespace(traj_pos=None)
    r.check_q_limits = lambda: False
    env.robots = [r]
    return env, geom_names


def jl(x):
    return np.asarray(x, dtype=np.float64).tolist()


def main():
    install_stubs()
    sys.path.insert(0, REF)
    quat = load(os.path.join(REF, "utils", "quaternion.py"), "utils.quaternion")
    _mod("utils", quaternion=quat)
    sys.modules["utils.quaternion"] = quat
    us = load(os.path.join(REF, "my_environments", "ultrasound.py"), "ref_ultrasound")
    Ultrasound = us.Ultrasound
    rng = np.random.default_rng(20261017)
    G = {}

    # ---------------- quaternion.py
    cases = []
    qs = rng.normal(size=(40, 2, 4))
    qs /= np.linalg.norm(qs, axis=-1, keepdims=True)
    extra = [(np.array([1.0, 0, 0, 0]), np.array([1.0, 0, 0, 0])), (np.array([0.0, 1, 0, 0]), np.array([0.0, -1, 0, 0])),
             (np.array([0.5, 0.5, 0.5, 0.5]), np.array([0.5, 0.5, 0.5, -0.5]))]
    for q1, q2 in [(a, b) for a, b in qs] + extra:
        try:
            dist = float(quat.distance_quat(q1, q2))
        except ValueError:  # quaternion.py:51 compares an array in a boolean context when q1*conj(q2) == (-1,0,0,0) exactly
            dist = None
        cases.append({"q1": jl(q1), "q2": jl(q2), "difference": jl(quat.difference_quat(q1, q2)), "distance": dist,
                      "log_q1": jl(quat.q_log(q1))})
    G["quaternion"] = cases

    # ---------------- constants + reward()
    env, names = make_env(Ultrasound)
    G["constants"] = {k: (jl(v) if isinstance(v, np.ndarray) else v) for k, v in vars(env).items()
                      if isinstance(v, (int, float, bool, np.ndarray)) and not k.startswith("_")}
    env_c, _ = make_env(Ultrasound)
    env_c.__init__(robots="Panda", controller_configs={"type": "OSC_POSE"}, control_freq=500, horizon=1000, use_camera_obs=False,
                   use_object_obs=False, has_offscreen_renderer=False, use_box_torso=False)
    G["constants_cylinder"] = {k: getattr(env_c, k) for k in ("top_torso_offset", "x_range", "y_range", "grid_pts", "use_box_torso")}
    rew = []
    for i in range(60):
        eef = np.array([0.0, 0.0, 0.9]) + rng.normal(scale=[0.02, 0.02, 0.01])
        traj = np.array([0.0, 0.0, 0.896]) + rng.normal(scale=[0.02, 0.02, 0.0])
        q = env.goal_quat + rng.normal(scale=0.05 if i % 3 else 0.6, size=4)
        q = q / np.linalg.norm(q)
        if q[3] < 0:
            q = -q  # robosuite mat2quat returns w >= 0
        env._eef_xpos, env._eef_xquat, env.traj_pt = eef, q, traj
        env.vel_running_mean = float(abs(rng.normal(0.04, 0.03)))
        env.z_contact_force_running_mean = float(rng.normal(6, 6))
        env.der_z_contact_force = float(rng.normal(0, 300))
        contact = bool(i % 4)
        env.sim.data.contact = [_Contact(2, 5)] if contact else [_Contact(1, 6)]
        env.sim.data.ncon = 1
        r = env.reward()
        rew.append({"eef_pos": jl(eef), "eef_quat_xyzw": jl(q), "traj_pt": jl(traj), "vel_mean": env.vel_running_mean,
                    "fz_mean": env.z_contact_force_running_mean, "dfz": env.der_z_contact_force, "in_contact": contact,
                    "reward": float(r), "pos_error": jl(env.pos_error), "ori_error": float(env.ori_error),
                    "terms": [float(env.pos_reward), float(env.ori_reward), float(env.vel_reward), float(env.force_reward), float(env.der_force_reward)]})
    G["reward"] = rew

    # ---------------- contact query (ultrasound.py:673-736)
    cq = []
    for pairs in ([], [(1, 5)], [(2, 1)], [(5, 2)], [(2, 3)], [(1, 4), (1, 6), (9, 2)], [(0, 2), (2, 1)]):
        env.sim.data.contact = [_Contact(a, b) for a, b in pairs] + [_Contact(2, 7)]  # one stale entry beyond ncon
        env.sim.data.ncon = len(pairs)
        env.has_touched_torso = False
        res = env._check_probe_contact_with_torso()
        cq.append({"pairs": pairs, "names": [[names[a], names[b]] for a, b in pairs], "in_contact": bool(res), "touched": bool(env.has_touched_torso)})
    G["contact_query"] = cq

    # ---------------- _post_action / _check_terminated sequences
    seqs = []
    for s, (early, horizon) in enumerate([(True, 1000), (False, 30), (True, 1000), (True, 1000)]):
        env, names = make_env(Ultrasound, early_termination=early, horizon=horizon)
        start, end = np.array([0.05, -0.02, 0.896]), np.array([-0.03, 0.04, 0.896])
        env.trajectory = Trajectory(milestones=np.array([start, end]))
        env.num_waypoints = 2
        env.initial_traj_step = float(rng.uniform(0, 1)) if s != 2 else 0.97
        env.traj_step = env.initial_traj_step
        env.traj_pt = env.trajectory.eval(env.traj_step)
        env.has_touched_torso = False
        env.prev_z_contact_force = 0
        env.der_z_contact_force = 0
        env.vel_running_mean = 0.0
        env.z_contact_force_running_mean = 3.0
        steps = []
        eef = np.array(env.traj_pt) + np.array([0.002, -0.001, 0.004])
        for t in range(40):
            env.timestep += 1
            eef = eef + rng.normal(scale=[0.0005, 0.0005, 0.0002]) + (np.array([0.02, 0.0, 0.0]) if (s == 3 and t >= 25) else 0)
            q = env.goal_quat + rng.normal(scale=0.01 if not (s == 0 and t >= 30) else 0.5, size=4)
            q /= np.linalg.norm(q)
            if q[3] < 0:
                q = -q
            hv = rng.normal(scale=0.03, size=3)
            fz = float(max(0.0, rng.normal(8, 4)))
            contact = (t >= 3) and not (s == 2 and t >= 20)
            if not contact:
                fz = 0.0
            env._eef_xpos, env._eef_xquat = eef.copy(), q
            env.robots[0]._hand_vel = hv
            env.sim.data.cfrc_ext = np.array([[0, 0, 0, 0.1, -0.2, fz]])
            env.sim.data.contact = [_Contact(1, 5), _Contact(2, 6)] if contact else [_Contact(1, 5)]
            env.sim.data.ncon = len(env.sim.data.contact)
            import contextlib
            with contextlib.redirect_stdout(io.StringIO()):
                reward, done, _ = env._post_action(np.zeros(6))
            steps.append({"eef_pos": jl(eef), "eef_quat_xyzw": jl(q), "hand_vel": jl(hv), "fz": fz, "in_contact": bool(contact),
                          "reward": float(reward), "done": bool(done), "traj_pt": jl(env.traj_pt), "vel_mean": float(env.vel_running_mean),
                          "dfz": float(env.der_z_contact_force), "fz_mean": float(env.z_contact_force_running_mean),
                          "touched": bool(env.has_touched_torso), "controller_traj_pos": jl(env.robots[0].controller.traj_pos)})
            if done:
                break
        seqs.append({"early_termination": early, "horizon": horizon, "control_freq": 500, "u0": env.initial_traj_step, "start": jl(start),
                     "end": jl(end), "fz_mean0": 3.0, "steps": steps})
    G["post_action"] = seqs

    # ---------------- trajectory / grid / noise / frame conversion
    env, _ = make_env(Ultrasound)
    env.torso_body_id = 0
    env.sim.data.body_xpos = np.array([[0.0, 0.0, 0.8572]])
    grid = env._get_torso_grid()
    np.random.seed(3)
    draws = []
    for _ in range(6):
        tr = env.get_trajectory()
        draws.append({"start": jl(tr.milestones[0]), "end": jl(tr.milestones[1])})
    env.deterministic_trajectory = True
    det = env.get_trajectory()
    np.random.seed(3)
    noise = [jl(env._add_noise_to_pos(np.array([0.1, -0.02, 0.896]))) for _ in range(2000)]
    env.robots[0].robot_model = types.SimpleNamespace(base_xpos_offset={"table": lambda L: (-0.16 - L / 2, 0, 0)}, top_offset=np.array([0, 0, 1.0]))
    G["trajectory"] = {"torso_xpos": [0.0, 0.0, 0.8572], "grid_x": jl(grid[0]), "grid_y": jl(grid[1]), "draws_seed3": draws,
                       "deterministic": {"start": jl(det.milestones[0]), "end": jl(det.milestones[1])},
                       "noise_mean": jl(np.mean(noise, axis=0)), "noise_std": jl(np.std(noise, axis=0)), "noise_base": [0.1, -0.02, 0.896],
                       "toolbox_xpos_of_[0.1,-0.02,0.896]": jl(env._convert_robosuite_to_toolbox_xpos(np.array([0.1, -0.02, 0.896]))),
                       "traj_ori_axisangle": jl(quat2axisangle(env.goal_quat))}
    with open(os.path.join(OUT, "task_golden.json"), "w") as f:
        json.dump(G, f, indent=1)
    print("wrote task_golden.json:", {k: len(v) for k, v in G.items()})

    # ---------------- shipped training artifacts (SURVEY App. D)
    class _U(pickle.Unpickler):
        def find_class(self, module, name):
            if module.startswith("numpy") or module in ("collections", "builtins", "_codecs"):
                return super().find_class(module, name)
            return type(name, (), {"__setstate__": lambda self, st: self.__dict__.update(st if isinstance(st, dict) else {})})

    art = {}
    mdir = os.path.join(os.path.dirname(REF), "src", "trained_rl_models")
    for model in ("tracking", "variable_z", "wrench"):
        z = zipfile.ZipFile(os.path.join(mdir, model + ".zip"))
        data = json.loads(z.read("data"))

        def dec(key):
            return _U(io.BytesIO(base64.b64decode(data[key][":serialized:"]))).load()

        ep = list(dec("ep_info_buffer"))
        entry = {"num_timesteps": data["num_timesteps"], "n_envs": data["n_envs"], "n_steps": data["n_steps"], "batch_size": data["batch_size"],
                 "n_epochs": data["n_epochs"], "gamma": data["gamma"], "gae_lambda": data["gae_lambda"], "ent_coef": data["ent_coef"],
                 "vf_coef": data["vf_coef"], "max_grad_norm": data["max_grad_norm"],
                 "last_original_obs": jl(dec("_last_original_obs")),
                 "ep_returns": [float(e["r"]) for e in ep], "ep_lengths": [int(e["l"]) for e in ep], "ep_t_max": float(max(e["t"] for e in ep)),
                 "action_low": jl(dec("action_space").low), "action_high": jl(dec("action_space").high)}
        with open(os.path.join(mdir, f"vec_normalize_{model}.pkl"), "rb") as f:
            vn = _U(f).load()
        entry.update({"obs_mean": jl(vn.obs_rms.mean), "obs_var": jl(vn.obs_rms.var), "obs_count": float(vn.obs_rms.count),
                      "ret_mean": float(vn.ret_rms.mean), "ret_var": float(vn.ret_rms.var), "old_obs": jl(vn.old_obs),
                      "old_reward": jl(vn.old_reward), "clip_obs": float(vn.clip_obs), "gamma_vn": float(vn.gamma)})
        art[model] = entry
    with open(os.path.join(OUT, "art_stats.json"), "w") as f:
        json.dump(art, f)
    # weights of the shipped `tracking` policy (76,941 fp32 parameters) + its normaliser: the closed-loop behavioural probe
    import torch
    z = zipfile.ZipFile(os.path.join(mdir, "tracking.zip"))
    sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=False)
    np.savez_compressed(os.path.join(OUT, "tracking_policy.npz"), **{k: v.numpy() for k, v in sd.items()},
                        obs_mean=np.array(art["tracking"]["obs_mean"]), obs_var=np.array(art["tracking"]["obs_var"]))
    print("wrote art_stats.json:", {k: (v["num_timesteps"], len(v["ep_returns"])) for k, v in art.items()})
    # the in-tree MJCF scene files, parsed by the package's own reader (robotic-ultrasound-imaging_b200/mjcf.py): SceneParams is
    # asserted against this parse (tests/test_task_golden.py::test_scene_params_match_the_reference_mjcf)
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    from rui_b200 import mjcf
    models = os.path.join(REF, "my_models")
    with open(os.path.join(OUT, "mjcf_golden.json"), "w") as f:
        json.dump({"soft_box": mjcf.read_assets(models, True), "soft_human_torso": mjcf.read_assets(models, False)}, f, indent=1)
    print("wrote mjcf_golden.json")
    # utils/error.py (the consumer of the save_data CSV stream): run the reference's own calculate_error_metrics on a small synthetic
    # episode and keep inputs + outputs (rui_b200/error_metrics.py must write the same files with the same numbers)
    import tempfile
    import pandas as pd
    err = load(os.path.join(REF, "utils", "error.py"), "ref_error")
    rng = np.random.default_rng(11)
    H = 40
    sim = {"ee_pos": rng.normal(size=(H, 3)), "ee_goal_pos": rng.normal(size=(H, 3)), "ee_vel": 0.05 * rng.normal(size=(H, 3)),
           "ee_goal_vel": np.full(H, 0.04), "ee_running_mean_vel": 0.04 + 0.01 * rng.normal(size=H),
           "ee_z_contact_force": 5 + 3 * rng.normal(size=H), "ee_z_goal_contact_force": np.full(H, 5.0),
           "ee_z_running_mean_contact_force": 5 + rng.normal(size=H), "ee_z_derivative_contact_force": 100 * rng.normal(size=H),
           "ee_z_goal_derivative_contact_force": np.zeros(H), "ee_diff_quat": np.abs(0.1 * rng.normal(size=H))}
    rew = {k: rng.uniform(0, 3, size=H) for k in ("pos", "ori", "force", "derivative_force", "vel")}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)
        try:
            for fld, d in (("simulation_data", sim), ("reward_data", rew)):
                os.makedirs(fld)
                for k, v in d.items():
                    pd.DataFrame(v).to_csv(os.path.join(fld, f"{k}_7.csv"), header=None, index=None)
            err.calculate_error_metrics("7")
            outs = {f[:-4]: open(os.path.join("error_data", "7", f)).read() for f in sorted(os.listdir(os.path.join("error_data", "7")))}
        finally:
            os.chdir(cwd)
    with open(os.path.join(OUT, "error_metrics_golden.json"), "w") as f:
        json.dump({"simulation_data": {k: jl(v) for k, v in sim.items()}, "reward_data": {k: jl(v) for k, v in rew.items()},
                   "error_data_files": outs}, f, indent=1)
    print("wrote error_metrics_golden.json:", sorted(outs))


if __name__ == "__main__":
    main()
