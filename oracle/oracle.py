"""ctypes wrapper of the float64 CPU oracle (oracle/oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product package never
imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(_HERE))

from rui_b200.abi import OBS_DIM, TASK_DIM, MAX_CONTACTS, DIAG_DIM, PackedModel, UsimConfig, UsimModel, action_dim  # noqa: E402

_pd = C.POINTER(C.c_double)
_pi = C.POINTER(C.c_int)


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liboracle.so")
    src = [os.path.join(_HERE, f) for f in ("oracle.c", "oracle.h")] + [os.path.join(_HERE, "..", "include", "usim.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src if os.path.exists(s)):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.oracle_create.restype = C.c_void_p
        L.oracle_create.argtypes = [C.POINTER(UsimModel), C.POINTER(UsimConfig), C.c_int]
        L.oracle_destroy.argtypes = [C.c_void_p]
        L.oracle_reset.argtypes = [C.c_void_p, _pd]
        L.oracle_step.argtypes = [C.c_void_p, _pd, _pd, _pd, _pi]
        L.oracle_step.restype = C.c_int
        L.oracle_set_forward_repeats.argtypes = [C.c_void_p, C.c_int]
        L.oracle_get_state.argtypes = [C.c_void_p, _pd, _pd, _pd, _pd]
        L.oracle_set_state.argtypes = [C.c_void_p, _pd, _pd, _pd, _pd]
        L.oracle_forward.argtypes = [C.c_void_p, _pd]
        L.oracle_ncon.argtypes = [C.c_void_p]
        L.oracle_nefc.argtypes = [C.c_void_p]
        L.oracle_solver_iter.argtypes = [C.c_void_p]
        L.oracle_contacts.argtypes = [C.c_void_p, _pi, _pi, _pd, _pd, _pd, _pd]
        for f in ("oracle_qacc", "oracle_qacc_smooth", "oracle_M", "oracle_bias", "oracle_tau"):
            getattr(L, f).restype = _pd
            getattr(L, f).argtypes = [C.c_void_p]
        L.oracle_evaluate.restype = C.c_int
        L.oracle_evaluate.argtypes = [C.c_void_p, _pd, _pd, _pd, _pd, _pd, _pd, _pd, _pd]
        L.oracle_efc_type.argtypes = [C.c_void_p, _pi]
        L.oracle_diag.argtypes = [C.c_void_p, _pd]
        L.oracle_eef.argtypes = [C.c_void_p, _pd, _pd, _pd]
        L.oracle_controller.argtypes = [C.c_void_p, _pd, _pd]
        L.oracle_ik.argtypes = [C.c_void_p, _pd, _pd]
        L.oracle_distance_quat.restype = C.c_double
        L.oracle_distance_quat.argtypes = [_pd, _pd]
        L.oracle_difference_quat.argtypes = [_pd, _pd, _pd]
        L.oracle_mat2quat_xyzw.argtypes = [_pd, _pd]
        L.oracle_reward.restype = C.c_double
        L.oracle_reward.argtypes = [_pd, _pd, _pd, C.c_double, C.c_double, C.c_double, C.c_int, _pd, _pd]
        L.oracle_post_action.argtypes = [_pd, C.c_int, C.c_double, C.c_int, _pd, _pd, _pd, _pd, C.c_double, C.c_int, _pd, _pd, _pi]
        L.oracle_grid_point.argtypes = [C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, _pd]
        L.oracle_philox.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
        L.oracle_rollout.restype = C.c_long
        L.oracle_rollout.argtypes = [C.POINTER(C.c_void_p), C.c_int, _pd, C.c_int, C.c_int, C.c_int, C.c_int, _pd]
        L.oracle_step_batch.argtypes = [C.POINTER(C.c_void_p), C.c_int, _pd, C.c_int, C.c_int, _pd, _pd, _pi, _pi]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(_pd)


def _f64(x, n=None):
    a = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    if n is not None:
        assert a.size == n, (a.size, n)
    return a


class OracleEnv:
    """One float64 env."""

    def __init__(self, packed: PackedModel, cfg: UsimConfig, global_env_id: int = 0):
        self.packed, self.cfg = packed, cfg
        self.nq, self.nv = packed.model.nq, packed.model.nv
        self.adim = action_dim(cfg)
        self.h = lib().oracle_create(C.byref(packed.struct), C.byref(cfg), int(global_env_id))

    def __del__(self):
        if getattr(self, "h", None):
            lib().oracle_destroy(self.h)
            self.h = None

    def reset(self):
        obs = np.zeros(OBS_DIM)
        lib().oracle_reset(self.h, _p(obs))
        return obs

    def step(self, action):
        a = _f64(action, self.adim)
        obs, rew, done = np.zeros(OBS_DIM), C.c_double(), C.c_int()
        rc = lib().oracle_step(self.h, _p(a), _p(obs), C.byref(rew), C.byref(done))
        if rc != 0:
            raise ValueError("executing action in terminated episode")
        return obs, rew.value, bool(done.value)

    def set_forward_repeats(self, n):
        lib().oracle_set_forward_repeats(self.h, int(n))

    def get_state(self):
        q, v, w, t = np.zeros(self.nq), np.zeros(self.nv), np.zeros(self.nv), np.zeros(TASK_DIM)
        lib().oracle_get_state(self.h, _p(q), _p(v), _p(w), _p(t))
        return q, v, w, t

    def set_state(self, qpos=None, qvel=None, warm=None, task=None):
        args = []
        keep = []
        for x, n in ((qpos, self.nq), (qvel, self.nv), (warm, self.nv), (task, TASK_DIM)):
            if x is None:
                args.append(None)
            else:
                a = _f64(x, n)
                keep.append(a)
                args.append(_p(a))
        lib().oracle_set_state(self.h, *args)

    def forward(self, ctrl=None):
        c = _f64(np.zeros(7) if ctrl is None else ctrl, 7)
        lib().oracle_forward(self.h, _p(c))

    def controller(self, action):
        a, tau = _f64(action, self.adim), np.zeros(7)
        lib().oracle_controller(self.h, _p(a), _p(tau))
        return tau

    def ik(self, target):
        t, q = _f64(target, 3), np.zeros(7)
        lib().oracle_ik(self.h, _p(t), _p(q))
        return q

    def _vec(self, name, n):
        return np.ctypeslib.as_array(getattr(lib(), name)(self.h), shape=(n,)).copy()

    @property
    def qacc(self):
        return self._vec("oracle_qacc", self.nv)

    @property
    def qacc_smooth(self):
        return self._vec("oracle_qacc_smooth", self.nv)

    @property
    def M(self):
        return self._vec("oracle_M", self.nv * self.nv).reshape(self.nv, self.nv)

    @property
    def bias(self):
        return self._vec("oracle_bias", self.nv)

    @property
    def tau(self):
        return self._vec("oracle_tau", 7)

    @property
    def ncon(self):
        return lib().oracle_ncon(self.h)

    @property
    def nefc(self):
        return lib().oracle_nefc(self.h)

    @property
    def solver_iter(self):
        return lib().oracle_solver_iter(self.h)

    def diag(self):
        d = np.zeros(DIAG_DIM)
        lib().oracle_diag(self.h, _p(d))
        return d

    def evaluate(self, qacc):
        """The problem of the last forward() evaluated at ``qacc`` (the env is left unchanged): grad = M (qacc - a0) - J^T f, the
        primal cost, the force of every constraint row and its type (0 equality, 1 joint limit, 2 contact normal, 100 friction),
        the contact forces (as contacts()["force"]), cfrc and the F/T torque (as diag()[0:6]), and the norms of the device
        solver's stopping rule |grad| <= tol (1 + |rhs| + |Hx|)."""
        a = _f64(qacc, self.nv)
        nefc, ncon = self.nefc, self.ncon
        grad, cost, frc = np.zeros(self.nv), C.c_double(), np.zeros(max(nefc, 1))
        cf, cfrc, ft, norms = np.zeros(3 * max(ncon, 1)), np.zeros(3), np.zeros(3), np.zeros(3)
        lib().oracle_evaluate(self.h, _p(a), _p(grad), C.byref(cost), _p(frc), _p(cf), _p(cfrc), _p(ft), _p(norms))
        typ = np.zeros(max(nefc, 1), np.intc)
        lib().oracle_efc_type(self.h, typ.ctypes.data_as(_pi))
        return dict(grad=grad, cost=cost.value, efc_force=frc[:nefc], efc_type=typ[:nefc], contact_force=cf.reshape(-1, 3)[:ncon],
                    cfrc=cfrc, ft_torque=ft, gnorm=norms[0], rhs_norm=norms[1], hx_norm=norms[2], nefc=nefc)

    def eef(self):
        J, pos, mat = np.zeros(42), np.zeros(3), np.zeros(9)
        lib().oracle_eef(self.h, _p(J), _p(pos), _p(mat))
        return J.reshape(6, 7), pos, mat.reshape(3, 3)

    def contacts(self):
        n = self.ncon
        g1, g2 = np.zeros(max(n, 1), np.intc), np.zeros(max(n, 1), np.intc)
        dist, pos, frame, force = np.zeros(max(n, 1)), np.zeros(3 * max(n, 1)), np.zeros(9 * max(n, 1)), np.zeros(3 * max(n, 1))
        lib().oracle_contacts(self.h, g1.ctypes.data_as(_pi), g2.ctypes.data_as(_pi), _p(dist), _p(pos), _p(frame), _p(force))
        return dict(geom1=g1[:n], geom2=g2[:n], dist=dist[:n], pos=pos.reshape(-1, 3)[:n], frame=frame.reshape(-1, 3, 3)[:n],
                    force=force.reshape(-1, 3)[:n])


def rollout(envs, actions, auto_reset=True, threads=1):
    """actions [steps][n][adim] float64; returns (env-steps executed, reward sum)."""
    a = _f64(actions)
    steps, n, adim = a.shape
    arr = (C.c_void_p * n)(*[e.h for e in envs])
    rs = C.c_double()
    tot = lib().oracle_rollout(arr, n, _p(a), steps, adim, int(auto_reset), int(threads), C.byref(rs))
    return tot, rs.value


def step_batch(envs, actions, threads=None):
    """One env step of every env (host threads over envs).  Returns (obs [n,19], rew [n], done [n] bool, stepped [n] bool);
    envs that were already done are not stepped (stepped[i] = False, outputs zero)."""
    a = _f64(actions)
    n, adim = a.shape
    assert n == len(envs)
    arr = (C.c_void_p * n)(*[e.h for e in envs])
    obs, rew = np.zeros((n, OBS_DIM)), np.zeros(n)
    done, rc = np.zeros(n, np.intc), np.zeros(n, np.intc)
    lib().oracle_step_batch(arr, n, _p(a), adim, int(threads or os.cpu_count() or 1), _p(obs), _p(rew), done.ctypes.data_as(_pi),
                            rc.ctypes.data_as(_pi))
    return obs, rew, done.astype(bool), rc == 0


# pure task-layer functions -------------------------------------------------
def distance_quat(q1, q2):
    return lib().oracle_distance_quat(_p(_f64(q1, 4)), _p(_f64(q2, 4)))


def difference_quat(q1, q2):
    out = np.zeros(4)
    lib().oracle_difference_quat(_p(_f64(q1, 4)), _p(_f64(q2, 4)), _p(out))
    return out


def mat2quat_xyzw(mat):
    out = np.zeros(4)
    lib().oracle_mat2quat_xyzw(_p(_f64(mat, 9)), _p(out))
    return out


def reward(eef_pos, eef_quat_xyzw, traj_pt, vel_mean, fz_mean, dfz, in_contact):
    pe, oe = np.zeros(2), C.c_double()
    r = lib().oracle_reward(_p(_f64(eef_pos, 3)), _p(_f64(eef_quat_xyzw, 4)), _p(_f64(traj_pt, 3)), float(vel_mean),
                            float(fz_mean), float(dfz), int(bool(in_contact)), _p(pe), C.byref(oe))
    return r, pe, oe.value


def post_action(ts, horizon, control_freq, early_termination, jnt_range, eef_pos, eef_quat_xyzw, hand_vel, fz, in_contact, qpos7=None):
    """In-place update of the task record ``ts`` (float64[TASK_DIM]); returns (reward, done)."""
    assert ts.dtype == np.float64 and ts.size == TASK_DIM
    rew, done = C.c_double(), C.c_int()
    jr = _f64(jnt_range, 14)
    q = None if qpos7 is None else _f64(qpos7, 7)
    lib().oracle_post_action(_p(ts), int(horizon), float(control_freq), int(bool(early_termination)), _p(jr), _p(_f64(eef_pos, 3)),
                             _p(_f64(eef_quat_xyzw, 4)), _p(_f64(hand_vel, 3)), float(fz), int(bool(in_contact)),
                             None if q is None else _p(q), C.byref(rew), C.byref(done))
    return rew.value, bool(done.value)


def grid_point(torso_xpos, ix, iy):
    out = np.zeros(3)
    lib().oracle_grid_point(float(torso_xpos[0]), float(torso_xpos[1]), float(torso_xpos[2]), int(ix), int(iy), _p(out))
    return out


def philox(seed, c0, c1, c2, c3):
    out = (C.c_uint32 * 4)()
    lib().oracle_philox(int(seed), c0, c1, c2, c3, out)
    return np.array(out[:], dtype=np.uint32)
