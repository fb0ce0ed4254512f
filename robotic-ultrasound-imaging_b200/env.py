"""Host-side mirror of the reference env API over the CUDA library.

Three stacked APIs, as in the reference (SURVEY.md §8b):

* :class:`BatchedUltrasound` — the native batched env (torch CUDA tensors in / out).
* :class:`Ultrasound` + :func:`make` — robosuite-style single env
  (``suite.make("Ultrasound", **rl_config["robosuite"])``, rl.py:38;
  ``reset() -> OrderedDict``, ``step(a) -> (obs, reward, done, info)``).
* :class:`GymWrapper` — robosuite ``GymWrapper`` (rl.py:38,173): flat 19-float observation.
* :class:`UltrasoundVecEnv` — SB3 ``VecEnv``-shaped batched env with auto-reset,
  ``terminal_observation`` and Monitor-style ``episode`` infos (rl.py:130,140).

PyTorch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes as C
import re
import time
from collections import OrderedDict
from typing import Any, Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .abi import (ARM_RECORD_DIM, DIAG_DIM, MAX_CONTACTS, OBS_DIM, TASK_DIM, PackedModel, action_bounds, action_dim, make_config)
from .model import SceneParams, UltrasoundModel, build_model, cylinder_torso_params

SENSOR_NAMES = (  # ultrasound.py:394-401, dims App. A.4
    ("eef_contact_force", 3),
    ("eef_torque", 3),
    ("eef_vel", 3),
    ("eef_contact_force_z_diff", 1),
    ("eef_contact_derivative_force_z_diff", 1),
    ("eef_vel_diff", 1),
    ("eef_pose_diff", 7),
)
PROPRIO_KEY = "robot0_proprio-state"

_TORSO_GEOM_RE = re.compile(r"[G]\d+[_]\d+[_]\d+$")  # ultrasound.py:724


def probe_torso_contact(name_pairs, probe_geoms=("gripper0_probe_collision",)) -> bool:
    """ultrasound.py:673-736 on a list of (geom1 name, geom2 name) of the active contacts."""
    for n1, n2 in name_pairs:
        if n1 in probe_geoms or n2 in probe_geoms:
            if _TORSO_GEOM_RE.search(n1) is not None or _TORSO_GEOM_RE.search(n2) is not None:
                return True
    return False


_MODEL_CACHE: Dict[bool, PackedModel] = {}


def packed_model(soft_torso: bool = True, params: Optional[SceneParams] = None) -> PackedModel:
    if params is not None:
        return PackedModel(build_model(params))
    if soft_torso not in _MODEL_CACHE:
        _MODEL_CACHE[soft_torso] = PackedModel(build_model(SceneParams(soft_torso=soft_torso)))
    return _MODEL_CACHE[soft_torso]


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class BatchedUltrasound:
    """N independent Ultrasound envs stepped by one C-ABI call on one GPU."""

    def __init__(
        self,
        num_envs: int,
        device: int | str | torch.device = 0,
        soft_torso: bool = True,
        controller_configs: Optional[Dict[str, Any]] = None,
        control_freq: float = 500,
        horizon: int = 1000,
        early_termination: bool = False,
        torso_solref_randomization: bool = False,
        initial_probe_pos_randomization: bool = False,
        deterministic_trajectory: bool = False,
        seed: int = 0,
        env_id_offset: int = 0,
        solver_iterations: int = 40,
        solver_tolerance: float = 3e-5,
        scene_params: Optional[SceneParams] = None,
        record_contacts: bool = False,
        **cfg_kwargs,
    ):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedUltrasound needs a CUDA device: the env step has no CPU fallback")
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        self.packed = packed_model(soft_torso, scene_params)
        self.model: UltrasoundModel = self.packed.model
        self.cfg = make_config(
            num_envs, controller_configs, control_freq=control_freq, horizon=horizon, early_termination=early_termination,
            torso_solref_randomization=torso_solref_randomization, initial_probe_pos_randomization=initial_probe_pos_randomization,
            deterministic_trajectory=deterministic_trajectory, seed=seed, env_id_offset=env_id_offset,
            solver_iterations=solver_iterations, solver_tolerance=solver_tolerance, **cfg_kwargs)
        self.num_envs = int(num_envs)
        self.nq, self.nv = self.model.nq, self.model.nv
        self.action_dim = action_dim(self.cfg)
        self.horizon = int(horizon)
        self.control_freq = float(control_freq)
        L = _lib.lib()
        h = C.c_void_p()
        _lib.check(L.usim_create(C.byref(self.packed.struct), C.byref(self.cfg), self.device.index or 0, C.byref(h)))
        self._h = h
        N, dev = self.num_envs, self.device
        self.obs = torch.zeros(N, OBS_DIM, device=dev)
        self.term_obs = torch.zeros(N, OBS_DIM, device=dev)
        self.rew = torch.zeros(N, device=dev)
        self.done = torch.zeros(N, dtype=torch.uint8, device=dev)
        if record_contacts:
            self.set_contact_record(True)

    # -- lifecycle ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().usim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def action_spec(self):
        return action_bounds(self.cfg)

    # -- core --------------------------------------------------------------
    def reset(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_reset(self._h, _ptr(mask), _ptr(self.obs), self._stream()))
        return self.obs

    def step(self, actions: torch.Tensor, auto_reset: bool = True):
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        assert a.shape == (self.num_envs, self.action_dim), a.shape
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_step(self._h, _ptr(a), _ptr(self.obs), _ptr(self.rew), _ptr(self.done), _ptr(self.term_obs),
                                            int(auto_reset), self._stream()))
        return self.obs, self.rew, self.done, self.term_obs

    def forward(self, mask: Optional[torch.Tensor] = None, ctrl: Optional[torch.Tensor] = None, qacc: bool = False):
        """``sim.forward()`` (MuJoCo ``mj_forward``) at the current state of the envs selected by ``mask`` (None: all), with joint
        torques ``ctrl`` [N, 7] clipped to the actuator ranges (None: zero; UR5e: column 6 is ignored).  Refreshes :meth:`diag`,
        :meth:`contacts` and :meth:`contact_forces` of the selected envs and writes their observation into ``self.obs`` (returned);
        the state, the task record, :meth:`arm_record` and everything a later step reads are left as they were.  With
        ``qacc=True`` returns ``(obs, qacc [N, nv])`` (rows of unselected envs are zero)."""
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            assert mask.shape == (self.num_envs,), mask.shape
        if ctrl is not None:
            ctrl = torch.as_tensor(ctrl, dtype=torch.float32, device=self.device).contiguous()
            assert ctrl.shape == (self.num_envs, 7), ctrl.shape
        qa = torch.zeros(self.num_envs, self.nv, device=self.device) if qacc else None
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_forward(self._h, _ptr(mask), _ptr(ctrl), _ptr(self.obs), _ptr(qa), self._stream()))
        return (self.obs, qa) if qacc else self.obs

    def step_host(self, actions: np.ndarray, auto_reset: bool = True):
        """End-to-end call with HOST buffers (copies inside the library)."""
        a = np.ascontiguousarray(actions, dtype=np.float32)
        assert a.shape == (self.num_envs, self.action_dim), a.shape
        if not hasattr(self, "_h_obs"):
            # page-locked result buffers: the library DMAs straight into them (pageable caller buffers are staged inside the library)
            N = self.num_envs
            pin = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, pin_memory=True).numpy()
            self._h_obs, self._h_tobs = pin(N, OBS_DIM), pin(N, OBS_DIM)
            self._h_rew, self._h_done = pin(N), pin(N, dtype=torch.uint8)
        p = lambda x: C.c_void_p(x.ctypes.data)
        _lib.check(_lib.lib().usim_step_host(self._h, p(a), p(self._h_obs), p(self._h_rew), p(self._h_done), p(self._h_tobs), int(auto_reset)))
        return self._h_obs, self._h_rew, self._h_done, self._h_tobs

    # -- parity hooks --------------------------------------------------------
    def get_state(self):
        N, dev = self.num_envs, self.device
        q, v, w = torch.empty(N, self.nq, device=dev), torch.empty(N, self.nv, device=dev), torch.empty(N, self.nv, device=dev)
        t = torch.empty(N, TASK_DIM, device=dev)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_get_state(self._h, _ptr(q), _ptr(v), _ptr(w), _ptr(t), self._stream()))
        return q, v, w, t

    def set_state(self, qpos=None, qvel=None, warm=None, task=None):
        def prep(x, d):
            if x is None:
                return None
            x = torch.as_tensor(x, dtype=torch.float32, device=self.device).contiguous()
            assert x.shape == (self.num_envs, d), (x.shape, d)
            return x

        q, v, w, t = prep(qpos, self.nq), prep(qvel, self.nv), prep(warm, self.nv), prep(task, TASK_DIM)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_set_state(self._h, _ptr(q), _ptr(v), _ptr(w), _ptr(t), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()  # inputs may be temporaries

    def contacts(self):
        N, dev = self.num_envs, self.device
        ncon = torch.empty(N, dtype=torch.int32, device=dev)
        g1 = torch.empty(N, MAX_CONTACTS, dtype=torch.int32, device=dev)
        g2 = torch.empty(N, MAX_CONTACTS, dtype=torch.int32, device=dev)
        dist = torch.empty(N, MAX_CONTACTS, device=dev)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_get_contacts(self._h, _ptr(ncon), _ptr(g1), _ptr(g2), _ptr(dist), self._stream()))
        return ncon, g1, g2, dist

    def set_contact_record(self, enable: bool = True):
        """Record position, frame and force of every contact from the next step / reset on (read with :meth:`contact_forces`).
        Off by default: the record costs one store pass over the contacts per step and USIM_MAX_CONTACTS * 36 bytes per env."""
        _lib.check(_lib.lib().usim_set_contact_record(self._h, int(enable)))

    def contact_forces(self):
        """``sim.data.contact[:ncon].pos / .frame`` and ``mj_contactForce`` of the last forward pass (the one :meth:`contacts`
        lists): pos [N, MAX_CONTACTS, 3], frame [N, MAX_CONTACTS, 3, 3] (rows: normal geom1 -> geom2, two tangents) and force
        [N, MAX_CONTACTS, 3] on geom2 in that frame (normal, tangent 1, tangent 2).  Rows at or beyond ncon are zero."""
        N, dev = self.num_envs, self.device
        pos = torch.empty(N, MAX_CONTACTS, 3, device=dev)
        frame = torch.empty(N, MAX_CONTACTS, 3, 3, device=dev)
        force = torch.empty(N, MAX_CONTACTS, 3, device=dev)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_get_contact_forces(self._h, _ptr(pos), _ptr(frame), _ptr(force), self._stream()))
        return pos, frame, force

    def diag(self):
        d = torch.empty(self.num_envs, DIAG_DIM, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_get_diag(self._h, _ptr(d), self._stream()))
        return d

    def arm_record(self):
        """[N][180] arm record of the last physics step (M, qfrc_smooth, torques, Jacobians, site pose ...: usim.h)."""
        d = torch.empty(self.num_envs, ARM_RECORD_DIM, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().usim_get_arm_record(self._h, _ptr(d), self._stream()))
        return d

    @property
    def launch_count(self) -> int:
        return int(_lib.lib().usim_launch_count(self._h))

    @property
    def divergence_count(self) -> int:
        c = C.c_int64()
        _lib.check(_lib.lib().usim_divergence_count(self._h, C.byref(c)))
        return int(c.value)

    @property
    def contact_overflow_count(self) -> int:
        """env steps in which more than MAX_CONTACTS contacts were found (the surplus is dropped, never silently)."""
        c = C.c_int64()
        _lib.check(_lib.lib().usim_contact_overflow_count(self._h, C.byref(c)))
        return int(c.value)

    @property
    def substeps(self) -> int:
        return int(_lib.lib().usim_substeps(self._h))

    def set_timing(self, enable: bool = True):
        """Opt in to per-launch CUDA-event timing of the dominant kernel (read with :meth:`kernel_time`)."""
        _lib.check(_lib.lib().usim_set_timing(self._h, int(enable)))

    def kernel_time(self, reset: bool = True):
        ms, n = C.c_double(), C.c_int64()
        _lib.check(_lib.lib().usim_kernel_time(self._h, int(reset), C.byref(ms), C.byref(n)))
        return ms.value, n.value


# ----------------------------------------------------------------------------
# robosuite-style single env
# ----------------------------------------------------------------------------
class _Controller:
    """``robots[0].controller`` as the task code uses it (ultrasound.py:451-465,535): name, trajectory goal, null-space reference."""

    name = "OSC_POSE"

    def __init__(self, env: "Ultrasound"):
        self._env = env

    @property
    def traj_pos(self):
        from .abi import TS_TRAJ_PT
        return self._env._task_state()[TS_TRAJ_PT:TS_TRAJ_PT + 3]

    @property
    def traj_ori(self):
        """axis-angle of ``goal_quat`` (T.quat2axisangle, ultrasound.py:456)"""
        from .abi import GOAL_QUAT_XYZW
        q = np.asarray(GOAL_QUAT_XYZW, dtype=np.float64)
        w = float(np.clip(q[3], -1.0, 1.0))
        den = np.sqrt(1.0 - w * w)
        return np.zeros(3) if den < 1e-12 else q[:3] * 2.0 * np.arccos(w) / den

    @property
    def initial_joint(self):
        from .abi import TS_INIT_JOINT
        return self._env._task_state()[TS_INIT_JOINT:TS_INIT_JOINT + 7]

    def update_initial_joints(self, q):
        """ultrasound.py:465: new null-space reference; the OSC goal is re-initialised at the current eef pose by the next reset forward."""
        from .abi import TS_INIT_JOINT
        t = self._env.core.get_state()[3]
        t[0, TS_INIT_JOINT:TS_INIT_JOINT + 7] = torch.as_tensor(np.asarray(q, dtype=np.float32), device=t.device)
        self._env.core.set_state(task=t)


class _RobotModel:
    """``robots[0].robot_model`` constants the task code reads (ultrasound.py:279-280,346,858-859)."""

    naming_prefix = "robot0_"
    top_offset = np.array((0.0, 0.0, 1.0))
    base_xpos_offset = {"table": lambda table_length: (-0.16 - table_length / 2, 0, 0), "bins": (-0.5, -0.1, 0), "empty": (-0.6, 0, 0)}


class _Gripper:
    """``robots[0].gripper`` (ultrasound_probe_gripper.py:26-29, .xml:6-8)."""

    naming_prefix = "gripper0_"
    root_body = "gripper0_gripper_base"
    contact_geoms = ["gripper0_probe_collision"]
    important_geoms = {"probe": ["gripper0_probe_collision"]}


class _Robot:
    """The slice of robosuite's robot object the task code reads (SURVEY §8b, last row)."""

    def __init__(self, env: "Ultrasound"):
        self._env = env
        self.name = env.robot_name
        self.dof = len(env.core.model.params.link_pos)  # 7 (Panda) / 6 (UR5e)
        self.init_qpos = np.array(env.core.model.params.init_qpos)
        self.controller = _Controller(env)
        self.robot_model = _RobotModel()
        self.gripper = _Gripper()

    @property
    def action_dim(self):
        return self._env.core.action_dim

    @property
    def _joint_positions(self):
        return self._env.core.get_state()[0][0, :self.dof].cpu().numpy().astype(np.float64)

    @property
    def _joint_velocities(self):
        return self._env.core.get_state()[1][0, :self.dof].cpu().numpy().astype(np.float64)

    @property
    def torques(self):
        return self._env.core.diag()[0, 13:13 + self.dof].cpu().numpy().astype(np.float64)

    @property
    def ee_torque(self):
        return self._env.core.diag()[0, 3:6].cpu().numpy().astype(np.float64)

    @property
    def ee_force(self):
        return self._env.core.diag()[0, 0:3].cpu().numpy().astype(np.float64)

    @property
    def _hand_vel(self):
        """linear eef velocity of the last step (ultrasound.py:373,474,538)"""
        return self._env.core.obs[0, 6:9].cpu().numpy().astype(np.float64)

    def check_q_limits(self) -> bool:
        """robosuite ``Robot.check_q_limits``: any joint within 0.1 rad of a limit (ultrasound.py:651)."""
        q = self._joint_positions
        rng = np.asarray(self._env.core.model.g_jnt_range, dtype=np.float64)[:self.dof]
        return bool(np.any(~((rng[:, 0] + 0.1 < q) & (q < rng[:, 1] - 0.1))))

    def set_robot_joint_positions(self, jpos):
        """ultrasound.py:462: overwrite the arm joint positions (velocities are left as they are), then ``sim.forward()``, as
        robosuite does: eef pose, contacts and forces describe the new pose."""
        q = self._env.core.get_state()[0]
        q[0, :self.dof] = torch.as_tensor(np.asarray(jpos, dtype=np.float32), device=q.device)
        self._env.core.set_state(qpos=q)
        self._env.sim.forward()


class _Sim:
    """``env.sim`` as far as the task code uses it: ``forward()`` (ultrasound.py:431)."""

    def __init__(self, env: "Ultrasound"):
        self._env = env

    def forward(self):
        """``sim.forward()`` with ``data.ctrl`` as MuJoCo keeps it: the torques last applied (diag[13:20]; zero after a reset)."""
        core = self._env.core
        core.forward(ctrl=core.diag()[:, 13:20])


class Ultrasound:
    """robosuite-style ``Ultrasound`` env (kwargs of ultrasound.py:99-133)."""

    def __init__(
        self,
        robots="Panda",
        env_configuration="default",
        controller_configs=None,
        gripper_types="UltrasoundProbeGripper",
        initialization_noise="default",
        table_full_size=(0.8, 0.8, 0.05),
        table_friction=100 * (1.0, 5e-3, 1e-4),
        use_camera_obs=False,
        use_object_obs=True,
        reward_scale=1.0,
        reward_shaping=False,
        placement_initializer=None,
        has_renderer=False,
        has_offscreen_renderer=False,
        render_camera="frontview",
        render_collision_mesh=False,
        render_visual_mesh=True,
        render_gpu_device_id=-1,
        control_freq=20,
        horizon=1000,
        ignore_done=False,
        hard_reset=True,
        camera_names="agentview",
        camera_heights=256,
        camera_widths=256,
        camera_depths=False,
        early_termination=False,
        save_data=False,
        deterministic_trajectory=False,
        torso_solref_randomization=False,
        initial_probe_pos_randomization=False,
        use_box_torso=True,
        seed=0,
        device=0,
        soft_torso=True,
        scene_params=None,
    ):
        assert gripper_types == "UltrasoundProbeGripper", "Tried to specify gripper other than UltrasoundProbeGripper in Ultrasound environment!"
        if isinstance(robots, (list, tuple)):
            assert len(robots) == 1, "Ultrasound is a single-arm env"
            robots = robots[0]
        assert robots in ("Panda", "UR5e"), "Robot must be either Panda or UR5e!"  # ultrasound.py:137
        if use_camera_obs or has_renderer or has_offscreen_renderer:
            raise NotImplementedError("rendering / camera observations are out of scope of the hot path (SURVEY §2.1 #4, §8f rank 4)")
        # kwargs the reference stores but never uses are accepted and ignored exactly as there: table_friction (never forwarded,
        # ultrasound.py:107,283), initialization_noise (forced to None, :211), reward_scale / reward_shaping (unused by reward()),
        # placement_initializer (overwritten, :304).  Those that WOULD change the scene are refused instead of silently dropped:
        if tuple(table_full_size) != (0.8, 0.8, 0.05):
            raise NotImplementedError("table_full_size other than (0.8, 0.8, 0.05): the arm base offset and the IK frame conversion "
                                      "(ultrasound.py:279,858) are compiled for the reference's table")
        if not hard_reset:
            raise NotImplementedError("hard_reset=False: the device reset always re-draws the torso solref (hard-reset semantics, ultrasound.py:122,291-297)")
        self.robot_name = robots
        self.save_data = bool(save_data)
        self.use_camera_obs, self.use_object_obs = use_camera_obs, use_object_obs
        self.reward_scale, self.reward_shaping = reward_scale, reward_shaping
        self.horizon, self.control_freq = horizon, control_freq
        self.control_timestep = 1.0 / control_freq
        self.ignore_done = ignore_done
        self.early_termination = early_termination
        self.table_full_size = tuple(table_full_size)
        if scene_params is None and not use_box_torso:
            scene_params = cylinder_torso_params(soft_torso=soft_torso)
        if robots == "UR5e":  # ultrasound.py:137,833-839: six joints, the seventh arm slot of the state is inert
            from .model import ur5e_params
            scene_params = ur5e_params(scene_params if scene_params is not None else SceneParams(soft_torso=soft_torso))
        self.core = BatchedUltrasound(
            1, device=device, soft_torso=soft_torso, controller_configs=controller_configs, control_freq=control_freq,
            horizon=horizon, early_termination=early_termination, torso_solref_randomization=torso_solref_randomization,
            initial_probe_pos_randomization=initial_probe_pos_randomization, deterministic_trajectory=deterministic_trajectory,
            seed=seed, ignore_done=ignore_done, scene_params=scene_params, record_contacts=True)
        self.robots = [_Robot(self)]
        self.sim = _Sim(self)
        self.timestep = 0
        self.done = True

    @property
    def action_spec(self):
        return self.core.action_spec

    @property
    def action_dim(self):
        return self.core.action_dim

    def _obs_dict(self, flat: np.ndarray) -> "OrderedDict[str, np.ndarray]":
        od: "OrderedDict[str, np.ndarray]" = OrderedDict()
        k = 0
        for name, dim in SENSOR_NAMES:
            od[name] = flat[k : k + dim].copy()
            k += dim
        od[PROPRIO_KEY] = flat.copy()
        return od

    def reset(self):
        flat = self.core.reset()[0].cpu().numpy().astype(np.float64)
        self.timestep, self.done = 0, False
        if self.save_data:
            self._init_data_collection()
        return self._obs_dict(flat)

    def step(self, action):
        if self.done:
            raise ValueError("executing action in terminated episode")
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1))
        obs, rew, done, _ = self.core.step(a, auto_reset=False)
        self.timestep += 1
        d = bool(done[0].item())  # with ignore_done the device does not end the episode at the horizon (early termination still does)
        self.done = d
        flat = obs[0].cpu().numpy().astype(np.float64)
        if self.save_data:
            self._collect(np.asarray(action, dtype=np.float64).reshape(-1), flat, float(rew[0].item()), d)
        return self._obs_dict(flat), float(rew[0].item()), d, {}

    # -- save_data: the per-episode CSV stream of ultrasound.py:479-509 (allocation), :552-614 (collection), :890-910 (files)
    _SIM_FILES = ("ee_pos", "ee_goal_pos", "ee_vel", "ee_goal_vel", "ee_running_mean_vel", "ee_quat", "ee_goal_quat", "ee_diff_quat",
                  "ee_z_contact_force", "ee_z_goal_contact_force", "ee_z_running_mean_contact_force", "ee_z_derivative_contact_force",
                  "ee_z_goal_derivative_contact_force", "is_contact", "q_pos", "q_torques", "time")
    _REWARD_FILES = ("pos", "ori", "vel", "force", "derivative_force")

    def _task_state(self):
        return self.core.get_state()[3][0].cpu().numpy().astype(np.float64)

    def _init_data_collection(self):
        H, A = self.horizon, self.core.action_dim
        dims = {"ee_pos": 3, "ee_goal_pos": 3, "ee_vel": 3, "ee_quat": 4, "ee_goal_quat": 4, "q_pos": 7, "q_torques": 7}
        self._data = {k: np.zeros((H, dims[k])) if k in dims else np.zeros(H) for k in self._SIM_FILES}
        self._data.update({"reward_" + k: np.zeros(H) for k in self._REWARD_FILES})
        self._data["action"] = np.zeros((H, A))
        self._prev_ts = self._task_state()  # reward() at step t uses the task state of step t-1 (ultrasound.py:525)

    def _collect(self, action, flat, reward, done):
        from .abi import GOAL_QUAT_XYZW, TS_DFZ, TS_FZ_MEAN, TS_IN_CONTACT, TS_ORI_ERR, TS_POS_ERR, TS_TRAJ_PT, TS_VEL_MEAN
        ts, prev, dg = self._task_state(), self._prev_ts, self.core.diag()[0].cpu().numpy().astype(np.float64)
        i, D = self.timestep - 1, self._data
        D["ee_pos"][i], D["ee_goal_pos"][i], D["ee_vel"][i] = dg[6:9], ts[TS_TRAJ_PT:TS_TRAJ_PT + 3], flat[6:9]
        D["ee_goal_vel"][i], D["ee_running_mean_vel"][i] = 0.04, ts[TS_VEL_MEAN]
        D["ee_quat"][i], D["ee_goal_quat"][i], D["ee_diff_quat"][i] = dg[9:13], GOAL_QUAT_XYZW, ts[TS_ORI_ERR] / 0.2
        D["ee_z_contact_force"][i], D["ee_z_goal_contact_force"][i] = flat[2], 5
        D["ee_z_running_mean_contact_force"][i], D["ee_z_derivative_contact_force"][i] = ts[TS_FZ_MEAN], ts[TS_DFZ]
        D["ee_z_goal_derivative_contact_force"][i], D["is_contact"][i] = 0, ts[TS_IN_CONTACT]
        D["q_pos"][i], D["q_torques"][i] = self.robots[0]._joint_positions, dg[13:20]
        D["time"][i] = (self.timestep - 1) / self.horizon * 100
        c = ts[TS_IN_CONTACT] != 0
        D["reward_pos"][i] = 5 * np.exp(-np.hypot(ts[TS_POS_ERR], ts[TS_POS_ERR + 1]))
        D["reward_ori"][i] = np.exp(-ts[TS_ORI_ERR])
        D["reward_vel"][i] = np.exp(-np.square(45 * (prev[TS_VEL_MEAN] - 0.04)))
        D["reward_force"][i] = 3 * np.exp(-np.square(0.7 * (prev[TS_FZ_MEAN] - 5))) if c else 0
        D["reward_derivative_force"][i] = 2 * np.exp(-np.square(0.01 * prev[TS_DFZ])) if c else 0
        D["action"][i] = action
        self._prev_ts = ts
        if done:
            for k in self._SIM_FILES:
                self._save_data(D[k], "simulation_data", k)
            for k in self._REWARD_FILES:
                self._save_data(D["reward_" + k], "reward_data", k)
            self._save_data(D["action"], "policy_data", "action")

    @staticmethod
    def _save_data(data, fldr, filename):
        """ultrasound.py:890-910: first free `<filename>_<idx>.csv`, no header, no index."""
        import os

        import pandas as pd
        os.makedirs(fldr, exist_ok=True)
        idx = 1
        path = os.path.join(fldr, filename + "_" + str(idx) + ".csv")
        while os.path.exists(path):
            idx += 1
            path = os.path.join(fldr, filename + "_" + str(idx) + ".csv")
        pd.DataFrame(data).to_csv(path, header=None, index=None)

    @property
    def _eef_xpos(self):
        return self.core.diag()[0, 6:9].cpu().numpy().astype(np.float64)

    @property
    def _eef_xquat(self):
        """(x, y, z, w), w >= 0 (robosuite mat2quat)"""
        return self.core.diag()[0, 9:13].cpu().numpy().astype(np.float64)

    @property
    def _torso_xpos(self):
        """ultrasound.py:913-921: world position of the torso root body"""
        q = self.core.get_state()[0][0].cpu().numpy().astype(np.float64)
        return q[7:10] if self.core.model.params.soft_torso else np.array([0.0, 0.0, 0.8 + 0.005 + 0.0522])

    def check_contact(self, geoms_1, geoms_2=None) -> bool:
        """robosuite ``MujocoEnv.check_contact`` on geom names / models with ``contact_geoms`` (ultrasound.py:746)."""
        def names(g):
            if g is None:
                return None
            if isinstance(g, str):
                return {g}
            return set(getattr(g, "contact_geoms", g))
        a, b = names(geoms_1), names(geoms_2)
        ncon, g1, g2, _ = self.core.contacts()
        n, m = int(ncon[0].item()), self.core.model
        for x, y in zip(g1[0, :n].tolist(), g2[0, :n].tolist()):
            nx, ny = m.geom_name(x), m.geom_name(y)
            if (nx in a and (b is None or ny in b)) or (ny in a and (b is None or nx in b)):
                return True
        return False

    def get_contacts(self) -> List[Dict[str, Any]]:
        """The active contacts of the last forward pass, as a mujoco-py user reads them: for each of ``sim.data.contact[:ncon]``
        the geom names, ``dist``, ``pos``, ``frame`` (3x3, rows: normal geom1 -> geom2, two tangents) and ``force``, the
        first three components of ``mj_contactForce`` (normal, tangent 1, tangent 2: the force on geom2 in that frame)."""
        ncon, g1, g2, dist = self.core.contacts()
        pos, frame, force = self.core.contact_forces()
        n, m = int(ncon[0].item()), self.core.model
        g1, g2, dist = g1[0, :n].tolist(), g2[0, :n].tolist(), dist[0, :n].cpu().numpy().astype(np.float64)
        pos, frame, force = [x[0, :n].cpu().numpy().astype(np.float64) for x in (pos, frame, force)]
        return [dict(geom1=m.geom_name(g1[c]), geom2=m.geom_name(g2[c]), dist=float(dist[c]), pos=pos[c], frame=frame[c], force=force[c])
                for c in range(n)]

    def _check_probe_contact_with_table(self) -> bool:
        """ultrasound.py:739-746"""
        return self.check_contact(self.robots[0].gripper, "table_collision")

    def _check_probe_contact_with_torso(self) -> bool:
        """ultrasound.py:714-736: any active contact between probe_collision and a geom named G\\d+_\\d+_\\d+."""
        ncon, g1, g2, _ = self.core.contacts()
        n = int(ncon[0].item())
        names = self.core.model
        return probe_torso_contact([(names.geom_name(a), names.geom_name(b)) for a, b in zip(g1[0, :n].tolist(), g2[0, :n].tolist())])

    def close(self):
        self.core.close()


_REGISTERED = {"Ultrasound": Ultrasound}


def make(env_name: str, *args, **kwargs):
    """``robosuite.make`` for the one env this framework provides."""
    if env_name not in _REGISTERED:
        raise Exception(f"Environment {env_name} not found. Registered: {', '.join(_REGISTERED)}")
    return _REGISTERED[env_name](*args, **kwargs)


class _Box:
    """Minimal ``gym.spaces.Box`` stand-in (gym is not a dependency)."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        self.low = np.broadcast_to(np.asarray(low, dtype=dtype), shape if shape is not None else np.shape(low)).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=dtype), self.low.shape).copy()
        self.shape, self.dtype = self.low.shape, np.dtype(dtype)

    def sample(self, rng: Optional[np.random.Generator] = None):
        rng = rng or np.random.default_rng()
        return rng.uniform(self.low, self.high).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

    def __repr__(self):
        return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"


class GymWrapper:
    """robosuite ``GymWrapper``: flattens ``keys`` (default: the proprio modality) into one vector."""

    def __init__(self, env: Ultrasound, keys: Optional[Sequence[str]] = None):
        self.env = env
        self.keys = list(keys) if keys is not None else [PROPRIO_KEY]
        self.name = "Panda_" + type(env).__name__
        self.reward_range = (0, env.reward_scale)
        low, high = env.action_spec
        self.action_space = _Box(low.astype(np.float32), high.astype(np.float32))
        self.obs_dim = sum(dict(SENSOR_NAMES, **{PROPRIO_KEY: OBS_DIM})[k] for k in self.keys)
        self.observation_space = _Box(-np.inf, np.inf, (self.obs_dim,), np.float32)

    def _flatten_obs(self, obs_dict):
        return np.concatenate([np.asarray(obs_dict[k]).flatten() for k in self.keys])

    def reset(self):
        return self._flatten_obs(self.env.reset())

    def step(self, action):
        od, reward, done, info = self.env.step(action)
        return self._flatten_obs(od), reward, done, info

    def seed(self, seed=None):
        if seed is not None:
            np.random.seed(seed)

    def close(self):
        self.env.close()


class UltrasoundVecEnv:
    """SB3 ``VecEnv``-shaped batched env (SubprocVecEnv + Monitor semantics, rl.py:36-41,130)."""

    def __init__(self, num_envs: int, env_options: Optional[Dict[str, Any]] = None, seed: int = 0, device=0, env_id_offset: int = 0):
        opts = dict(env_options or {})
        robots = opts.pop("robots", "Panda")
        robots = robots[0] if isinstance(robots, (list, tuple)) else robots
        assert robots in ("Panda", "UR5e"), "Robot must be either Panda or UR5e!"
        for k in ("env_id", "use_camera_obs", "use_object_obs", "has_renderer", "has_offscreen_renderer", "render_camera",
                  "camera_names", "camera_heights", "camera_widths", "camera_depths", "reward_shaping", "save_data", "gripper_types"):
            opts.pop(k, None)
        if not opts.pop("use_box_torso", True):
            opts["scene_params"] = cylinder_torso_params()
        if robots == "UR5e":
            from .model import ur5e_params
            opts["scene_params"] = ur5e_params(opts.get("scene_params"))
        self.core = BatchedUltrasound(num_envs, device=device, seed=seed, env_id_offset=env_id_offset, **opts)
        self.num_envs = num_envs
        self.seed_value = int(seed)
        low, high = self.core.action_spec
        self.action_space = _Box(low.astype(np.float32), high.astype(np.float32))
        self.observation_space = _Box(-np.inf, np.inf, (OBS_DIM,), np.float32)
        self._actions = None
        self._t0 = time.time()
        self._ep_ret = np.zeros(num_envs, np.float64)
        self._ep_len = np.zeros(num_envs, np.int64)
        self._ep_hist_r: List[List[float]] = [[] for _ in range(num_envs)]  # Monitor.get_episode_rewards / _lengths
        self._ep_hist_l: List[List[int]] = [[] for _ in range(num_envs)]
        self._views: Optional[List[_EnvView]] = None

    def reset(self) -> np.ndarray:
        self._ep_ret[:] = 0
        self._ep_len[:] = 0
        return self.core.reset().cpu().numpy()

    def step_async(self, actions):
        self._actions = np.clip(np.asarray(actions, dtype=np.float32), self.action_space.low, self.action_space.high)

    def step_wait(self):
        obs, rew, done, tobs = self.core.step_host(self._actions, auto_reset=True)
        obs, rew, done = obs.copy(), rew.copy(), done.astype(bool)
        self._ep_ret += rew
        self._ep_len += 1
        infos: List[Dict[str, Any]] = [{} for _ in range(self.num_envs)]
        for i in np.nonzero(done)[0]:
            infos[i]["terminal_observation"] = tobs[i].copy()
            infos[i]["episode"] = {"r": float(self._ep_ret[i]), "l": int(self._ep_len[i]), "t": round(time.time() - self._t0, 6)}
            self._ep_hist_r[i].append(float(self._ep_ret[i]))
            self._ep_hist_l[i].append(int(self._ep_len[i]))
            self._ep_ret[i] = 0
            self._ep_len[i] = 0
        return obs, rew, done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self):
        self.core.close()

    # -- the rest of SB3's VecEnv surface (rl.py never calls these; SB3's own wrappers and utilities do) ----------------
    def _view(self, i):
        if self._views is None:
            self._views = [_EnvView(self, k) for k in range(self.num_envs)]
        return self._views[i]

    def _idx(self, indices):
        if indices is None:
            return list(range(self.num_envs))
        return [indices] if isinstance(indices, int) else list(indices)

    def seed(self, seed=None):
        return [self._view(i).seed(None if seed is None else seed + i)[0] for i in range(self.num_envs)]

    def get_attr(self, attr_name, indices=None):
        return [getattr(self._view(i), attr_name) for i in self._idx(indices)]

    def set_attr(self, attr_name, value, indices=None):
        if attr_name in ("horizon", "control_freq", "action_dim", "action_spec", "observation_space", "action_space"):
            raise AttributeError(f"{attr_name} is fixed at construction of the batched env")
        for i in self._idx(indices):
            setattr(self._view(i), attr_name, value)

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        return [getattr(self._view(i), method_name)(*method_args, **method_kwargs) for i in self._idx(indices)]

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [getattr(wrapper_class, "__name__", "") == "Monitor"] * len(self._idx(indices))


# ----------------------------------------------------------------------------
# stable-baselines3 adapter (rl.py:130,140,143: SubprocVecEnv -> VecNormalize -> PPO)
# ----------------------------------------------------------------------------
def _gym_box(low, high, shape=None):
    """``gym.spaces.Box`` when gym / gymnasium is installed (SB3 type-checks its spaces), else the stand-in."""
    for mod in ("gym", "gymnasium"):
        try:
            spaces = __import__(mod + ".spaces", fromlist=["Box"])
        except ImportError:
            continue
        if shape is not None:
            return spaces.Box(low=low, high=high, shape=shape, dtype=np.float32)
        return spaces.Box(low=np.asarray(low, np.float32), high=np.asarray(high, np.float32), dtype=np.float32)
    return _Box(low, high, shape, np.float32)


class _EnvView:
    """What ``get_attr`` / ``env_method`` see as "env i" of the vectorised env: the GymWrapper-level attributes of rl.py's workers."""

    def __init__(self, vec: "UltrasoundVecEnv", index: int):
        self._vec, self.index = vec, index
        c = vec.core
        self.horizon, self.control_freq, self.action_dim = c.horizon, c.control_freq, c.action_dim
        self.action_spec = c.action_spec
        self.observation_space, self.action_space = vec.observation_space, vec.action_space
        self.reward_range = (0.0, 12.0)  # ultrasound.py:230-269: five terms, maxima 5 + 1 + 1 + 3 + 2
        self.spec, self.metadata, self.render_mode = None, {"render.modes": []}, None

    def seed(self, seed=None):
        """GymWrapper.seed (rl.py:40).  The device streams are keyed by (seed, global env id, episode) at construction."""
        return [self._vec.seed_value + self.index if seed is None else seed]

    def get_episode_rewards(self):  # Monitor
        return list(self._vec._ep_hist_r[self.index])

    def get_episode_lengths(self):  # Monitor
        return list(self._vec._ep_hist_l[self.index])

    def get_state(self):
        """(qpos, qvel) of this env (mujoco-py ``sim.get_state()``-like, numpy)"""
        q, v, _, _ = self._vec.core.get_state()
        return q[self.index].cpu().numpy(), v[self.index].cpu().numpy()


def sb3_vec_env_class():
    """``class SB3UltrasoundVecEnv(stable_baselines3.common.vec_env.VecEnv)``, created on demand: stable-baselines3 is not a
    dependency of this package (and is not installed where the tests run), so the subclass exists only when SB3 imports.
    An instance passes SB3's ``isinstance(env, VecEnv)`` checks (``VecNormalize(env)``, ``PPO("MlpPolicy", env)``, rl.py:140-143),
    carries gym ``Box`` spaces, auto-resets with ``terminal_observation`` / Monitor ``episode`` infos, and implements the whole
    abstract surface (``get_attr / set_attr / env_method / env_is_wrapped / seed``)."""
    from stable_baselines3.common.vec_env import VecEnv  # ImportError if SB3 is absent: the caller decides

    class SB3UltrasoundVecEnv(VecEnv):
        def __init__(self, num_envs: int, env_options: Optional[Dict[str, Any]] = None, seed: int = 0, device=0, env_id_offset: int = 0):
            self._impl = UltrasoundVecEnv(num_envs, env_options, seed=seed, device=device, env_id_offset=env_id_offset)
            lo, hi = self._impl.core.action_spec
            VecEnv.__init__(self, num_envs, _gym_box(-np.inf, np.inf, (OBS_DIM,)), _gym_box(lo, hi))
            self._impl.observation_space, self._impl.action_space = self.observation_space, self.action_space
            self._views = [_EnvView(self._impl, i) for i in range(num_envs)]
            self._overlay: List[Dict[str, Any]] = [{} for _ in range(num_envs)]

        # -- the abstract surface of VecEnv ---------------------------------
        def reset(self):
            return self._impl.reset()

        def step_async(self, actions):
            self._impl.step_async(actions)

        def step_wait(self):
            return self._impl.step_wait()

        def close(self):
            self._impl.close()

        def _idx(self, indices):
            if indices is None:
                return list(range(self.num_envs))
            return [indices] if isinstance(indices, int) else list(indices)

        def get_attr(self, attr_name, indices=None):
            return [self._overlay[i][attr_name] if attr_name in self._overlay[i] else getattr(self._views[i], attr_name) for i in self._idx(indices)]

        def set_attr(self, attr_name, value, indices=None):
            # per-env Python-side attributes only: anything that shapes the device step is fixed at construction
            if attr_name in ("horizon", "control_freq", "action_dim", "action_spec", "observation_space", "action_space"):
                raise AttributeError(f"{attr_name} is fixed at construction of the batched env")
            for i in self._idx(indices):
                self._overlay[i][attr_name] = value

        def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
            return [getattr(self._views[i], method_name)(*method_args, **method_kwargs) for i in self._idx(indices)]

        def env_is_wrapped(self, wrapper_class, indices=None):
            # the batched env itself provides what rl.py:39 wraps around each worker: Monitor episode statistics
            return [getattr(wrapper_class, "__name__", "") == "Monitor"] * len(self._idx(indices))

        def seed(self, seed=None):
            return [v.seed(None if seed is None else seed + i)[0] for i, v in enumerate(self._views)]

        def get_images(self):
            raise NotImplementedError("rendering is out of scope of the hot path")

        def render(self, mode="human"):
            raise NotImplementedError("rendering is out of scope of the hot path")

    return SB3UltrasoundVecEnv


def make_sb3_vec_env(num_envs: int, env_options: Optional[Dict[str, Any]] = None, seed: int = 0, device=0, env_id_offset: int = 0):
    """Drop-in for ``SubprocVecEnv([make_robosuite_env(...)] * num_cpu)`` of rl.py:130 when stable-baselines3 is installed."""
    return sb3_vec_env_class()(num_envs, env_options, seed=seed, device=device, env_id_offset=env_id_offset)
