"""The device forward pass (usim_forward, BatchedUltrasound.forward) on identical inputs, judged by the float64 oracle's forward.

Both sides get the same float32 states (solve_util.trajectory_batches) and the same joint torques: zero, and random within
ctrl_range.  The device runs forward(qacc=True); the oracle runs oracle_forward at that state with the torques the device applied
(diag[13:20]) and is evaluated at the device's qacc (solve_util.compare: stopping rule, contact list, contact forces, probe wrench,
F/T torque).  On top of that, the 19 observation channels against oracle_observation() and the eef pose against oracle_eef.

Used by tests/test_forward.py (asserts the bounds) and scripts/forward_parity_report.py (measures the maxima the bounds come from;
profiles/forward_parity.json).
"""
from __future__ import annotations

import numpy as np
import torch

import solve_util as su
from rui_b200 import abi

SCENES = ("soft", "rigid", "cylinder", "ur5e")
CTRLS = ("zero", "random")
FORWARD_CAP = 2 * su.DEFAULT["solver_iterations"]  # a forward pass solves with the reset forward's cap


def ctrl_range(env):
    """the actuator ranges as the device holds them (float32), [7]; the UR5e's inert seventh slot is 0"""
    return np.asarray(env.model.g_ctrl_range, dtype=np.float32)


def clipped(env, ctrl):
    """what the device applies for `ctrl` [N, 7]: clipped to ctrl_range in float32, the UR5e's seventh column zero"""
    r = ctrl_range(env)
    out = np.clip(np.asarray(ctrl, np.float32), -r, r)
    out[:, len(env.model.params.link_pos):] = 0
    return out


def oracle_observation(O, orc):
    """The observation robosuite's _get_observations(force_update=True) gives after sim.forward(), from the oracle's last forward
    pass (ultrasound.py:363-401): probe wrench and F/T torque (diag[0:6]); the hand body's linear velocity, its Jacobian at the
    forward's kinematics times the current qvel; the task record's statistics as they stand; the grip-site pose against the trajectory
    point and the goal orientation.  The hand Jacobian follows from the grip-site Jacobian (oracle_eef): the grip site is the origin
    of the probe body, which sits at probe_pos in the hand frame with the hand's orientation, so the hand origin is
    r = -R_site probe_pos from the site and each column is Jp_j + Jr_j x r."""
    d = orc.diag()
    J, pos, mat = orc.eef()
    _, v, _, t = orc.get_state()
    r = -mat @ np.asarray(orc.packed.model.params.probe_pos, dtype=np.float64)
    jh = J[:3] + np.cross(J[3:].T, r).T
    obs = np.zeros(abi.OBS_DIM)
    obs[0:6] = d[0:6]
    obs[6:9] = jh @ v[:7]
    obs[9:12] = t[abi.TS_FZ_MEAN] - 5, t[abi.TS_DFZ], t[abi.TS_VEL_MEAN] - 0.04
    obs[12:15] = pos - t[abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3]
    obs[15:19] = O.difference_quat(d[9:13], abi.GOAL_QUAT_XYZW)  # xyzw arrays through a wxyz routine (ultrasound.py:390)
    return obs


def make_ctrl(env, kind, n, seed):
    if kind == "zero":
        return None
    r = ctrl_range(env)
    return np.random.default_rng(seed).uniform(-1, 1, size=(n, 7)).astype(np.float32) * r


def device_forward(env, batch, ctrl):
    """set the batch's state, run one forward pass; what the comparison needs, as float64 numpy"""
    q, v, w, t, _ = batch
    env.set_state(q, v, w, t)
    obs, qacc = env.forward(ctrl=None if ctrl is None else torch.as_tensor(ctrl), qacc=True)
    ncon, g1, g2, _ = [x.cpu().numpy() for x in env.contacts()]
    _, _, force = [x.cpu().numpy().astype(np.float64) for x in env.contact_forces()]
    return dict(qacc=qacc.cpu().numpy().astype(np.float64), diag=env.diag().cpu().numpy().astype(np.float64),
                obs=obs.cpu().numpy().astype(np.float64), ncon=ncon, g1=g1, g2=g2, force=force)


def obs_metrics(d_obs, o_obs, fsum):
    """the observation of one env against the oracle's: force and torque channels relative as solve_util.compare measures them,
    the others absolute"""
    return dict(obs_force_rel=float(np.abs(d_obs[0:3] - o_obs[0:3]).max() / fsum),
                obs_torque_rel=float(np.abs(d_obs[3:6] - o_obs[3:6]).max() / max(0.1, float(np.abs(o_obs[3:6]).max()))),
                obs_vel=float(np.abs(d_obs[6:9] - o_obs[6:9]).max()), obs_task=float(np.abs(d_obs[9:12] - o_obs[9:12]).max()),
                obs_pose=float(np.abs(d_obs[12:19] - o_obs[12:19]).max()))


def eef_metrics(O, orc, d):
    """eef position and quaternion (diag[6:13]) against oracle_eef"""
    _, pos, mat = orc.eef()
    return dict(eef_pos=float(np.abs(d[6:9] - pos).max()), eef_quat=float(np.abs(d[9:13] - O.mat2quat_xyzw(mat)).max()))


def run(O, name, kind, seed=5):
    """Every trajectory batch of the scene through one forward pass with torques of `kind`, every env against the oracle: a record
    per (batch, env) -- solve_util.compare's metrics (cap = the forward's), the observation and eef metrics, and whether diag[13:20]
    is the clipped ctrl bit for bit."""
    params, cc = su.scene(name)
    batches = su.trajectory_batches(O, name)
    n = batches[0][0].shape[0]
    env = su.make_env(params, cc, n, seed)
    env.reset()
    orcs = [su.make_oracle(O, env.packed, cc, seed, i) for i in range(n)]
    out = []
    for bi, b in enumerate(batches):
        ctrl = make_ctrl(env, kind, n, 100 + bi)
        dev = device_forward(env, b, ctrl)
        want_tau = clipped(env, np.zeros((n, 7)) if ctrl is None else ctrl)
        for i in range(n):
            orc = orcs[i]
            orc.set_state(*(x[i].astype(np.float64) for x in b[:4]))
            orc.forward(dev["diag"][i, 13:20])
            opt = orc.evaluate(orc.qacc)
            opt["qacc"] = orc.qacc
            rec = su.compare(orc, dev, i, {}, opt)
            rec["cap"] = FORWARD_CAP
            o_obs = oracle_observation(O, orc)
            fsum = max(1.0, float(orc.contacts()["force"][:, 0].sum()) if orc.ncon else 0.0)
            rec.update(obs_metrics(dev["obs"][i], o_obs, fsum))
            rec.update(eef_metrics(O, orc, dev["diag"][i]))
            rec["tau_exact"] = bool(np.array_equal(dev["diag"][i, 13:20].astype(np.float32), want_tau[i]))
            out.append(rec)
    env.close()
    return out


OBS_KEYS = ("obs_force_rel", "obs_torque_rel", "obs_vel", "obs_task", "obs_pose", "eef_pos", "eef_quat")


def stats(recs):
    """solve_util.stats plus the maxima of the observation and eef metrics, and the count of records whose torques were not the
    clipped ctrl"""
    s = su.stats(recs)
    ok = [r for r in recs if r["list_ok"]]
    s.update({k: float(max((r[k] for r in ok), default=0.0)) for k in OBS_KEYS})
    s["tau_mismatch"] = sum(not r["tau_exact"] for r in recs)
    return s
