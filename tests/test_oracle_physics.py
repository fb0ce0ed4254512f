"""Known-answer tests of the float64 oracle (the parity reference for the CUDA path).

The reference ships no tests and its physics lives in a closed binary (SURVEY.md §4, §8c), so the oracle is
pinned here by physics that has a closed-form answer and by an independent numpy formulation of the inertia."""
import numpy as np
import pytest

from conftest import CC_FIXED, CC_TRACK
from rui_b200 import abi
from rui_b200.model import build_model, forward_kinematics, mass_matrix


# the single-contact closed-form tests use the simplest probe shape: an axial capsule whose tip sphere touches the table in ONE point
# exactly below the grip site (the shipped, calibrated probe is a bar with two end spheres: two table contacts)
AXIAL_PROBE = dict(probe_seg_a=None, probe_seg_b=None, probe_com=None, probe_radius=0.05)


def _cfg(cc, **kw):
    return abi.make_config(1, cc, control_freq=500, horizon=1000, **kw)


def test_philox_known_answers(O):
    # Random123 known-answer vectors for Philox4x32-10
    assert [hex(x) for x in O.philox(0, 0, 0, 0, 0)] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    assert [hex(x) for x in O.philox(0xFFFFFFFFFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF)] == [
        "0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    assert [hex(x) for x in O.philox(0x299F31D0A4093822, 0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344)] == [
        "0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_inertia_matches_numpy_formulation(O, soft_model):
    e = O.OracleEnv(soft_model, _cfg(CC_TRACK, seed=5, initial_probe_pos_randomization=True), 0)
    e.reset()
    q = e.get_state()[0]
    rng = np.random.default_rng(0)
    q[14:] += rng.normal(scale=2e-3, size=270)
    e.set_state(qpos=q)
    e.forward()
    M_np, _, _ = mass_matrix(soft_model.model, e.get_state()[0])
    M = e.M
    assert np.abs(M - M.T).max() < 1e-12
    assert np.abs(M - M_np).max() < 1e-12
    assert np.linalg.eigvalsh(M).min() > 0
    # arrow structure the CUDA kernel relies on: sliders couple only with the free translation and themselves
    S = M[13:, 13:]
    assert np.abs(S - np.diag(np.diag(S))).max() < 1e-14
    assert np.abs(M[10:13, 13:]).max() < 1e-12 and np.abs(M[:7, 7:]).max() == 0


def test_bias_is_gravity_torque_at_rest(O, rigid_model):
    """qfrc_bias at zero velocity = -d(potential)/dq, checked by finite differences of the potential energy."""
    m = rigid_model.model
    e = O.OracleEnv(rigid_model, _cfg(CC_FIXED), 0)
    q0 = np.array(m.params.init_qpos) + 0.1
    e.set_state(qpos=q0, qvel=np.zeros(7))
    e.forward()
    bias = e.bias

    def pot(q):
        xpos, xmat = forward_kinematics(m, q)
        return sum(m.g_body_mass[b] * 9.81 * (xpos[b] + xmat[b] @ m.g_body_ipos[b])[2] for b in range(1, m.nbody))

    for j in range(7):
        dq = np.zeros(7); dq[j] = 1e-6
        assert abs((pot(q0 + dq) - pot(q0 - dq)) / 2e-6 - bias[j]) < 1e-6


def test_free_arm_energy_is_conserved_without_damping(O):
    """No damping, no torque, no contact: semi-implicit Euler keeps total energy within O(h) over 200 steps."""
    from rui_b200.model import SceneParams
    pk = abi.PackedModel(build_model(SceneParams(soft_torso=False, joint_damping=0.0)))
    m = pk.model
    cc = dict(CC_FIXED, impedance_mode="wrench")  # wrench mode with a zero action = zero task-space force
    e = O.OracleEnv(pk, _cfg(cc), 0)
    e.reset()
    q0 = np.array([0.3, -0.4, 0.2, -1.6, 0.1, 1.2, 0.5])
    ts = e.get_state()[3]
    ts[abi.TS_INIT_JOINT:abi.TS_INIT_JOINT + 7] = q0
    e.set_state(qpos=q0, qvel=np.zeros(7), task=ts)

    def energy():
        q, v = e.get_state()[:2]
        M, xpos, xmat = mass_matrix(m, q)
        pe = sum(m.g_body_mass[b] * 9.81 * (xpos[b] + xmat[b] @ m.g_body_ipos[b])[2] for b in range(1, m.nbody))
        return 0.5 * v @ M @ v + pe

    # the wrench-mode torque is bias compensation + null-space PD: remove both by stepping the raw dynamics
    E0 = energy()
    for _ in range(100):
        e.forward(np.zeros(7))
        assert e.nefc == 0  # no contact, no joint limit: pure rigid-body dynamics
        q, v = e.get_state()[:2]
        a = e.qacc
        v = v + 0.002 * a
        e.set_state(qpos=q + 0.002 * v, qvel=v)
    E1 = energy()
    q, v = e.get_state()[:2]
    assert np.abs(v).max() > 0.3  # it really fell
    assert abs(E1 - E0) < 0.02 * abs(0.5 * v @ mass_matrix(m, q)[0] @ v)


def test_ik_reaches_target(O, soft_model):
    e = O.OracleEnv(soft_model, _cfg(CC_TRACK), 0)
    for target in ([0.05, 0.02, 0.9], [-0.1, -0.08, 0.88], [0.14, 0.09, 0.91]):
        q = e.ik(target)
        st = e.get_state()
        st[0][:7] = q
        e.set_state(qpos=st[0])
        e.forward()
        _, pos, mat = e.eef()
        assert np.abs(pos - target).max() < 1e-8
        quat = O.mat2quat_xyzw(mat.reshape(9))
        g = np.array(abi.GOAL_QUAT_XYZW)
        assert min(np.abs(quat - g).max(), np.abs(quat + g).max()) < 1e-6
        lo, hi = soft_model.model.g_jnt_range[:, 0], soft_model.model.g_jnt_range[:, 1]
        assert np.all(q > lo) and np.all(q < hi)


def test_torso_settles_with_contact_force_equal_weight(O, soft_model):
    """Probe far away: after settling, the table normal forces carry the torso's weight."""
    m = soft_model.model
    e = O.OracleEnv(soft_model, _cfg(CC_FIXED), 0)
    e.reset()
    q, v, w, ts = e.get_state()
    q[:7] = m.params.init_qpos
    ts[abi.TS_INIT_JOINT:abi.TS_INIT_JOINT + 7] = q[:7]
    e.set_state(qpos=q, qvel=v, task=ts)
    for _ in range(150):
        e.step(np.zeros(6))
    c = e.contacts()
    assert set(c["geom2"]) == {1} and c["geom1"].min() >= 4  # only particle-table contacts
    # force on geom2 (table) along the contact normal (0,0,-1): weight pushes the table down
    fz_on_table = sum(f[0] * fr[0][2] + f[1] * fr[1][2] + f[2] * fr[2][2] for f, fr in zip(c["force"], c["frame"]))
    weight = (270 * 0.01 + 0.01) * 9.81
    assert abs(-fz_on_table - weight) < 0.03 * weight
    v = e.get_state()[1]
    assert np.abs(v[7:13]).max() < 5e-3


def test_single_soft_contact_closed_form(O):
    """Probe tip pressed into the rigid table at rest, arm locked by a huge gain: compare the contact force of the
    7-DoF solve with the closed-form 1-row answer f = -D (J a - aref) of the regularised constraint."""
    from rui_b200.model import SceneParams
    pk = abi.PackedModel(build_model(SceneParams(soft_torso=False, table_friction=1e-6, probe_friction=1e-6, **AXIAL_PROBE)))  # frictionless
    m = pk.model
    e = O.OracleEnv(pk, _cfg(CC_FIXED), 0)
    e.reset()
    # find a configuration with the probe tip 1 mm inside the table
    e2 = O.OracleEnv(abi.PackedModel(build_model(SceneParams(**AXIAL_PROBE))), _cfg(CC_TRACK), 0)
    q = e2.ik([0.0, 0.0, 0.8 - 0.001])
    e.set_state(qpos=q, qvel=np.zeros(7))
    e.forward(np.zeros(7))
    c = e.contacts()
    assert len(c["dist"]) == 1 and abs(c["dist"][0] + 0.001) < 2e-5  # the goal orientation is a hair off vertical
    depth = -c["dist"][0]
    J, pos, _ = e.eef()
    # contact row: normal (0,0,1), point = contact pos; contact point Jacobian from the site Jacobian
    r = c["pos"][0] - pos
    Jn = J[2] + np.cross(J[3:].T, r)[:, 2]
    M, a0 = e.M, e.qacc_smooth
    dmin, dmax, width = 0.9, 0.95, 0.001
    assert depth / width >= 1
    imp = dmax  # |r| >= width
    tc = 0.02
    K, B = 1 / (dmax ** 2 * tc ** 2), 2 / (dmax * tc)
    aref = -K * imp * (-depth)
    R = (1 - imp) / imp * m.body_invweight0[m.ids[4], 0]
    A = Jn @ np.linalg.solve(M, Jn)
    f = (aref - Jn @ a0) / (A + R)  # frictionless 1-row solution; friction rows carry ~0 at rest
    assert f > 0
    assert abs(c["force"][0][0] - f) < 2e-3 * f


def _cone_force_numpy(j, Dn, Dt, mu, fr):
    """Elliptic-cone (condim 3) constraint force of MuJoCo's primal problem, written independently of oracle.c: j = (J a - aref) in the
    contact frame (normal first); returns (force, zone) with zone 0 = top (no force), 1 = middle (on the cone), 2 = bottom (quadratic)."""
    N, U = j[0] * mu, fr * j[1:]
    T = np.hypot(*U)
    if N >= mu * T or (T <= 0 and N >= 0):
        return np.zeros(3), 0
    if mu * N + T <= 0 or (T <= 0 and N < 0):
        return -np.array([Dn * j[0], Dt * j[1], Dt * j[2]]), 2
    Dm = Dn / (mu * mu * (1 + mu * mu))
    f0 = -Dm * (N - mu * T) * mu
    return np.array([f0, -f0 / T * U[0] * fr, -f0 / T * U[1] * fr]), 1


def test_friction_cone_solution_satisfies_the_optimality_conditions(O):
    """One frictional contact (probe tip 1 mm inside the rigid table) with the tip sticking, sliding and separating: the oracle's
    solution satisfies M (a - a_smooth) = J^T f, and f is the cone force of J a - aref computed by an independent numpy
    restatement of the elliptic-cone formulas -- in all three zones; when sliding, |f_t| = friction * f_n exactly."""
    from rui_b200.model import SceneParams
    pk = abi.PackedModel(build_model(SceneParams(soft_torso=False, **AXIAL_PROBE)))
    m = pk.model
    e = O.OracleEnv(pk, _cfg(CC_FIXED), 0)
    e.reset()
    q = O.OracleEnv(abi.PackedModel(build_model(SceneParams(**AXIAL_PROBE))), _cfg(CC_TRACK), 0).ik([0.0, 0.0, 0.8 - 0.001])
    e.set_state(qpos=q, qvel=np.zeros(7))
    e.forward(np.zeros(7))
    J0 = e.eef()[0]
    dmax, tc = 0.95, 0.02
    K, B = 1 / (dmax ** 2 * tc ** 2), 2 / (dmax * tc)
    fr = max(m.params.table_friction, m.params.probe_friction)
    mu = fr / np.sqrt(m.params.impratio)
    zones = []
    for twist in ([0.001, 0, 0, 0, 0, 0], [3.0, 0, 0, 0, 0, 0], [0, 0, 2.0, 0, 0, 0]):  # site velocity: creep, fast slide, lift-off
        qd = np.linalg.pinv(J0) @ np.array(twist, dtype=float)
        e.set_state(qpos=q, qvel=qd)
        e.forward(np.zeros(7))
        c = e.contacts()
        assert len(c["dist"]) == 1
        F, f, depth = c["frame"][0], c["force"][0], -c["dist"][0]
        J, pos, _ = e.eef()
        Jc = J[:3] + np.cross(J[3:].T, c["pos"][0] - pos).T  # contact-point Jacobian (world), then rows normal / t1 / t2
        Jf = F @ Jc
        a, a0, M = e.qacc, e.qacc_smooth, e.M
        assert np.abs(M @ (a - a0) - Jf.T @ f).max() < 1e-8 * max(1.0, np.abs(f).max())
        imp = dmax  # penetration >= solimp width
        v = Jf @ qd
        aref = np.array([-B * v[0] + K * imp * depth, -B * v[1], -B * v[2]])
        Dn = 1.0 / ((1 - imp) / imp * m.body_invweight0[m.ids[4], 0])
        fe, zone = _cone_force_numpy(Jf @ a - aref, Dn, Dn * m.params.impratio, mu, fr)
        zones.append(zone)
        assert np.abs(f - fe).max() < 1e-7 * max(1.0, np.abs(fe).max()), (twist, f, fe)
        if zone == 1:
            assert abs(np.hypot(f[1], f[2]) / f[0] - fr) < 1e-9
    assert zones == [2, 1, 0]


def test_soft_scene_solution_satisfies_the_optimality_conditions(O, soft_model):
    """Whole soft scene (probe on the torso, torso on the table: ~60 contacts, 807 equality rows).  The oracle assembles explicit
    sparse constraint rows over a generic body tree; here the same forces are written in the FORMULATION THE CUDA KERNEL USES
    (numpy, float64): equality rows as a per-slider stencil (270 "fix", 536 "smooth" pairs with the episode's solrefsmooth, one
    tendon), contacts as rigid-body point wrenches on the free body (world force, body-frame torque) plus the slider axis component,
    probe contacts through the site Jacobian.  At the oracle's solution, M (a - a_smooth) equals the sum of those generalized forces
    to rounding: the two formulations describe the same constrained dynamics."""
    m = soft_model.model
    P, A = m.params, m.arrays
    cfg = _cfg(CC_TRACK, seed=5, torso_solref_randomization=True, initial_probe_pos_randomization=True)
    e = O.OracleEnv(soft_model, cfg, 0)
    e.reset()
    rng = np.random.default_rng(1)
    for _ in range(5):
        e.step(rng.uniform(0, 1, 6))
    q, v, _, ts = e.get_state()
    e.forward(e.tau)
    a, a0, M = e.qacc, e.qacc_smooth, e.M
    c = e.contacts()
    assert len(c["dist"]) > 40 and set(c["geom2"]) == {1, 2}  # table-particle and probe-particle contacts are both present

    def quat2mat(qq):
        w_, x, y, z = qq / np.linalg.norm(qq)
        return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w_ * z), 2 * (x * z + w_ * y)],
                         [2 * (x * y + w_ * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w_ * x)],
                         [2 * (x * z - w_ * y), 2 * (y * z + w_ * x), 1 - 2 * (x * x + y * y)]])

    dmin, dmax, width, mid, power = P.solimp

    def imped(pos):  # MuJoCo solimp sigmoid
        x = abs(pos) / width
        y = 1.0 if x >= 1 else (x ** power / mid ** (power - 1) if x <= mid else 1 - (1 - x) ** power / (1 - mid) ** (power - 1))
        return min(max(dmin + (0.0 if x == 0 else y) * (dmax - dmin), 1e-4), 0.9999)

    def KB(sr):  # positive solref: (timeconst, dampratio); negative: direct (stiffness, damping)
        if sr[0] > 0:
            tc = max(sr[0], 2 * P.timestep)
            return 1 / (dmax ** 2 * tc ** 2 * sr[1] ** 2), 2 / (dmax * tc)
        return -sr[0] / dmax ** 2, -sr[1] / dmax

    R, Pt = quat2mat(q[10:14]), q[7:10]
    ax, iw = np.asarray(A["part_axis"]), np.asarray(A["dof_invweight0"])
    qs, vs, acc = q[14:], v[13:], a[13:]
    g = np.zeros(283)
    K, B = KB(P.solref)
    for i in range(270):  # "fix" rows
        imp = imped(qs[i])
        D = 1 / max(1e-15, (1 - imp) / imp * iw[13 + i])
        g[13 + i] += -D * (acc[i] - (-B * vs[i] - K * imp * qs[i]))
    K2, B2 = KB((-ts[abi.TS_STIFFNESS], -ts[abi.TS_DAMPING]))
    for ia, ib in np.asarray(A["eq_pairs"]):  # "smooth" pair rows
        pos, vel = qs[ia] - qs[ib], vs[ia] - vs[ib]
        imp = imped(pos)
        D = 1 / max(1e-15, (1 - imp) / imp * (iw[13 + ia] + iw[13 + ib]))
        f = -D * ((acc[ia] - acc[ib]) - (-B2 * vel - K2 * imp * pos))
        g[13 + ia] += f
        g[13 + ib] -= f
    imp = imped(qs.sum())  # tendon row
    Dt = 1 / max(1e-15, (1 - imp) / imp * float(np.asarray(A["tendon_invweight0"])[0]))
    g[13:] += -Dt * (acc.sum() - (-B * vs.sum() - K * imp * qs.sum()))
    J, spos, _ = e.eef()
    for k in range(len(c["dist"])):  # contacts: +F on geom2, -F on geom1
        Fw, pos = c["frame"][k].T @ c["force"][k], c["pos"][k]
        for geom, sgn in ((c["geom2"][k], 1.0), (c["geom1"][k], -1.0)):
            if geom == 1:    # table: static
                continue
            if geom == 2:    # probe: arm dofs through the site Jacobian moved to the contact point
                g[:7] += sgn * (J[:3] + np.cross(J[3:].T, pos - spos).T).T @ Fw
            else:            # particle geom - 4: free body (world force, body-frame torque) + its slider
                i = geom - 4
                g[7:10] += sgn * Fw
                g[10:13] += sgn * R.T @ np.cross(pos - Pt, Fw)
                g[13 + i] += sgn * (R @ ax[i]) @ Fw
    lhs = M @ (a - a0)
    assert np.abs(lhs).max() > 1.0
    assert np.abs(lhs - g).max() < 1e-9 * np.abs(lhs).max()


def _osc_numpy(J, M, bias, q, qd, eef_pos, eef_mat, goal_pos, goal_R, kp, kd, q_init, ctrl_lim, uncouple=True):
    """robosuite OSC_POSE torque (SURVEY App. C.2/C.3) with numpy primitives: Lambda = pinv(J M^-1 J^T), decoupled position /
    orientation wrench, gravity-and-Coriolis compensation, null-space posture term N^T M (10 (q0 - q) - 2 sqrt(10) qd), clip."""
    eo = 0.5 * sum(np.cross(eef_mat[:, i], goal_R[:, i]) for i in range(3))
    vel = J @ qd
    F = np.r_[kp[:3] * (goal_pos - eef_pos) - kd[:3] * vel[:3], kp[3:] * eo - kd[3:] * vel[3:]]
    Mi = np.linalg.inv(M)
    Lf, Lp, Lo = np.linalg.pinv(J @ Mi @ J.T), np.linalg.pinv(J[:3] @ Mi @ J[:3].T), np.linalg.pinv(J[3:] @ Mi @ J[3:].T)
    W = np.r_[Lp @ F[:3], Lo @ F[3:]] if uncouple else Lf @ F
    N = np.eye(7) - (Mi @ J.T @ Lf) @ J
    t = J.T @ W + bias + N.T @ (M @ (10 * (q_init - q) - 2 * np.sqrt(10) * qd))
    return np.clip(t, -ctrl_lim, ctrl_lim)


def test_osc_pose_torques_match_numpy_restatement(O, soft_model):
    """The oracle's OSC_POSE controller (tracking mode: gains from the action, goal = trajectory point + goal quaternion; fixed mode:
    delta-pose goal with an axis-angle orientation delta) against a numpy restatement built from its own M, bias and site Jacobian."""
    m = soft_model.model
    lim = np.asarray(m.params.ctrl_range, dtype=float)
    rng = np.random.default_rng(3)

    def xyzw2mat(qx):
        x, y, z, w = np.asarray(qx) / np.linalg.norm(qx)
        return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                         [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                         [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])

    for cc in (CC_TRACK, CC_FIXED):
        e = O.OracleEnv(soft_model, _cfg(cc, seed=5, torso_solref_randomization=True, initial_probe_pos_randomization=True), 0)
        e.reset()
        lo, hi = (0, 1) if cc is CC_TRACK else (-1, 1)
        for _ in range(7):
            e.step(rng.uniform(lo, hi, 6))
        act = rng.uniform(lo, hi, 6)
        q, v, _, ts = e.get_state()
        e.forward()  # kinematics at the current state (the controller call below redoes it)
        J, pos, mat = e.eef()
        if cc is CC_TRACK:
            kp = np.clip(act, 0, 1) * 500.0
            kd = 2 * np.sqrt(kp)
            goal_pos, goal_R = ts[abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3], xyzw2mat(abi.GOAL_QUAT_XYZW)
        else:
            kp = np.full(6, float(cc["kp"]))
            kd = 2 * np.sqrt(kp) * float(cc["damping_ratio"])
            delta = np.clip(act, -1, 1) * np.array(cc["output_max"])
            goal_pos = pos + delta[:3]
            ang = np.linalg.norm(delta[3:])
            ax_ = delta[3:] / ang
            Kx = np.array([[0, -ax_[2], ax_[1]], [ax_[2], 0, -ax_[0]], [-ax_[1], ax_[0], 0]])
            goal_R = (np.eye(3) + np.sin(ang) * Kx + (1 - np.cos(ang)) * Kx @ Kx) @ mat  # Rodrigues: R(delta) @ current orientation
        tau = e.controller(act)
        M, bias = e.M[:7, :7], e.bias[:7]
        want = _osc_numpy(J, M, bias, q[:7], v[:7], pos, mat, goal_pos, goal_R, kp, kd, ts[abi.TS_INIT_JOINT:abi.TS_INIT_JOINT + 7], lim)
        assert np.abs(tau - want).max() < 1e-9 * max(1.0, np.abs(want).max()), (cc["impedance_mode"], tau, want)
        assert np.abs(want).max() > 0.5


def test_narrowphase_matches_brute_force(O, soft_model):
    """Probe capsule against the 270 particle capsules: the oracle's closed-form segment-segment narrowphase gives the same contact set
    and penetration depths as a dense sampling of the two segments; table contacts are the capsule end spheres below the table top."""
    m = soft_model.model
    A, P = m.arrays, m.params
    e = O.OracleEnv(soft_model, _cfg(CC_TRACK, seed=5, torso_solref_randomization=True, initial_probe_pos_randomization=True), 0)
    e.reset()
    rng = np.random.default_rng(3)
    for _ in range(30):
        e.step(rng.uniform(0, 1, 6))
    q = e.get_state()[0]
    e.forward(e.tau)
    _, spos, smat = e.eef()
    c = e.contacts()
    w_, x, y, z = q[10:14] / np.linalg.norm(q[10:14])
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w_ * z), 2 * (x * z + w_ * y)],
                  [2 * (x * y + w_ * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w_ * x)],
                  [2 * (x * z - w_ * y), 2 * (y * z + w_ * x), 1 - 2 * (x * x + y * y)]])
    ax, pp, qs, cr, hl = np.asarray(A["part_axis"]), np.asarray(A["part_pos"]), q[14:], P.cap_radius, P.cap_half_len
    eo = q[7:10] + (pp + (qs - cr)[:, None] * ax) @ R.T              # outer / inner end-sphere centres of every particle capsule
    ei = q[7:10] + (pp + (qs - cr - 2 * hl)[:, None] * ax) @ R.T
    seg = np.asarray(A["probe_seg"]).reshape(2, 3)
    ptip, pback, pr = spos + smat @ seg[0], spos + smat @ seg[1], float(np.asarray(A["probe_radius"])[0])
    s = np.linspace(0, 1, 401)
    a_pts = eo[:, None, :] + s[None, :, None] * (ei - eo)[:, None, :]          # [270, 401, 3]
    b_pts = ptip[None, :] + s[:, None] * (pback - ptip)[None, :]               # [401, 3]
    d2 = ((a_pts[:, :, None, :] - b_pts[None, None, :, :]) ** 2).sum(-1)       # [270, 401, 401]
    dist_bf = np.sqrt(d2.reshape(270, -1).min(1)) - cr - pr
    probe = {int(g1) - 4: float(d) for g1, g2, d in zip(c["geom1"], c["geom2"], c["dist"]) if g2 == 2 and g1 >= 4}
    assert len(probe) >= 2
    for i in range(270):
        if i in probe:
            assert abs(probe[i] - dist_bf[i]) < 2e-5, (i, probe[i], dist_bf[i])  # sampling error of the brute force
        else:
            assert dist_bf[i] > -2e-5, (i, dist_bf[i])
    # table: one contact per end sphere below the table top (inside the table's footprint), depth = z - radius - table height
    table = sorted(float(d) for g2, d in zip(c["geom2"], c["dist"]) if g2 == 1)
    dz = np.r_[eo[:, 2], ei[:, 2]] - cr - P.table_top_z
    want = sorted(float(d) for d in dz if d < 0)
    assert len(table) == len(want) and np.allclose(table, want, atol=1e-12)


def test_step_is_semi_implicit_euler_of_the_forward_solution(O, soft_model):
    """One oracle step = controller torque, forward solve, then mj_Euler: (M + h D) a' = M a (implicit joint damping), v += h a',
    q += h v_new, free-joint quaternion q <- q * exp(h w / 2) with the body-frame angular velocity; qacc_warmstart <- a."""
    m = soft_model.model
    cfg = _cfg(CC_TRACK, seed=9, torso_solref_randomization=True, initial_probe_pos_randomization=True)
    a_env, b_env = O.OracleEnv(soft_model, cfg, 0), O.OracleEnv(soft_model, cfg, 0)
    rng = np.random.default_rng(4)
    for e in (a_env, b_env):
        e.reset()
    for _ in range(6):
        act = rng.uniform(0, 1, 6)
        a_env.step(act)
        b_env.step(act)
    act = rng.uniform(0, 1, 6)
    q, v, _, _ = b_env.get_state()
    tau = b_env.controller(act)
    b_env.forward(tau)
    a, M, h = b_env.qacc, b_env.M, m.params.timestep
    damp = np.asarray(m.arrays["g_dof_damping"], dtype=float)
    ap = np.linalg.solve(M + h * np.diag(damp), M @ a)
    v_new = v + h * ap
    q_new = q.copy()
    q_new[:7] += h * v_new[:7]
    q_new[7:10] += h * v_new[7:10]
    w3 = v_new[10:13]
    ang = h * np.linalg.norm(w3)
    qr = np.r_[np.cos(ang / 2), np.sin(ang / 2) * w3 / np.linalg.norm(w3)]
    q0 = q[10:14]
    qq = np.array([q0[0] * qr[0] - q0[1:] @ qr[1:], *(q0[0] * qr[1:] + qr[0] * q0[1:] + np.cross(q0[1:], qr[1:]))])
    q_new[10:14] = qq / np.linalg.norm(qq)
    q_new[14:] += h * v_new[13:]
    a_env.step(act)
    qa, va, wa, _ = a_env.get_state()
    assert np.abs(va - v_new).max() < 1e-10 and np.abs(qa - q_new).max() < 1e-12 and np.abs(wa - a).max() < 1e-12
    assert np.abs(v_new - v).max() > 1e-4  # something moved


def test_probe_contact_force_observation_is_the_sum_of_its_contact_forces(O, soft_model):
    """obs[0:3] (sim.data.cfrc_ext[probe][-3:], ultrasound.py:365) = world-frame sum of the contact forces acting on the probe, i.e.
    frame^T f of every contact whose second geom is the probe; obs[9] = running mean of its z component - 5 (ultrasound.py:375,546), as of the PREVIOUS step."""
    e = O.OracleEnv(soft_model, _cfg(CC_TRACK, seed=9, torso_solref_randomization=True, initial_probe_pos_randomization=True), 0)
    e.reset()
    rng = np.random.default_rng(6)
    fz_mean = e.get_state()[3][abi.TS_FZ_MEAN]
    seen = 0
    for _ in range(12):
        o, _, _ = e.step(rng.uniform(0, 1, 6))
        c = e.contacts()
        F = sum((fr.T @ f for fr, f, g2 in zip(c["frame"], c["force"], c["geom2"]) if g2 == 2), np.zeros(3))
        assert np.abs(o[:3] - F).max() < 1e-9 * max(1.0, np.abs(F).max())
        # the observation is sampled before _post_action updates the running mean (robosuite's cached observables; pinned by
        # the artifacts, test_task_golden.py::test_art_reward_is_reproduced_by_its_observation_row): obs[9] lags one step
        assert abs(o[9] - (fz_mean - 5)) < 1e-9
        fz_mean = 0.1 * F[2] + 0.9 * fz_mean
        assert abs(e.get_state()[3][abi.TS_FZ_MEAN] - fz_mean) < 1e-9
        seen += np.abs(F).max() > 1.0
    assert seen >= 10  # the probe really presses on the torso


def test_arm_links_stay_clear_of_torso_and_table(O, soft_model):
    """Assumption A-COLL-2 (DESIGN.md §8): the robosuite Panda link / mount collision geoms (contype 1, SURVEY App. B.1 last row) are
    not built -- only the probe collides.  The task keeps the probe pressed on the torso top with the arm reaching over it from the
    mount at x = -0.56: over random-gain episodes every link segment (joint origin to joint origin, a generous 8 cm collision
    radius) stays well clear of the torso's box and of the table top, so those geoms could never produce a contact here."""
    m = soft_model.model
    ids = m.ids
    link0, hand = int(ids[2]), int(ids[3])
    half = np.array([0.175, 0.14, 0.0525]) + 0.0075  # world half-extents of the composite box (SURVEY App. B.2) + capsule radius
    rng = np.random.default_rng(3)
    worst_torso, worst_table = np.inf, np.inf
    for seed in (3, 4):
        e = O.OracleEnv(soft_model, _cfg(CC_TRACK, seed=seed, torso_solref_randomization=True, initial_probe_pos_randomization=True), seed)
        e.reset()
        for s in range(120):
            e.step(rng.uniform(0, 1, 6))
            if s % 10:
                continue
            q = e.get_state()[0]
            xpos, _ = forward_kinematics(m, q)
            centre = q[7:10]
            pts = [xpos[b] for b in range(link0, hand + 1)]  # link 1..7 origins + hand
            for a, b in zip(pts[:-2], pts[1:-1]):  # segments up to link 7 (the last one carries the probe, which does collide)
                for t in np.linspace(0, 1, 9):
                    p = a + t * (b - a)
                    d = np.maximum(np.abs(p - centre) - half, 0)
                    worst_torso = min(worst_torso, np.linalg.norm(d) - 0.08)
                    worst_table = min(worst_table, p[2] - 0.8 - 0.08)
    assert worst_torso > 0.05 and worst_table > 0.05, (worst_torso, worst_table)


def test_ur5e_model_has_an_inert_seventh_arm_slot(O):
    """robots="UR5e" (ultrasound.py:137,833-839): six joints; the seventh arm slot of the state is a rotor coupled to nothing, so
    the 7-wide arm layout of the kernels is exact for a 6-joint arm.  The reset IK puts the probe on the trajectory point in the
    goal orientation, and the slot never moves."""
    from rui_b200.abi import PackedModel
    from rui_b200.model import ur5e_params
    pk = PackedModel(build_model(ur5e_params()))
    assert pk.struct.narm == 6 and pk.model.nq == 284 and pk.model.nv == 283
    e = O.OracleEnv(pk, _cfg(CC_TRACK, seed=3, torso_solref_randomization=True, initial_probe_pos_randomization=True, reset_eef_bias=(0, 0, 0)), 0)
    obs = e.reset()
    J, pos, mat = e.eef()
    assert np.abs(J[:, 6]).max() == 0.0
    assert np.linalg.norm(obs[12:14]) < 0.01 and abs(obs[14]) < 0.04 and obs[15] < -0.9999  # on the trajectory point (+ reset noise), goal orientation
    M = e.M
    assert abs(M[6, 6] - 1.0) < 1e-12 and np.abs(np.delete(M[6], 6)).max() == 0.0
    rng = np.random.default_rng(0)
    for _ in range(20):
        e.step(rng.uniform(0, 1, 6))
    q, v, _, _ = e.get_state()
    assert q[6] == 0.0 and v[6] == 0.0
    assert np.isfinite(q).all() and np.abs(v[:6]).max() < 5.0


def _arm_scans_numpy(link, tool, q, qd, grav, nj=7):
    """numpy mirror of the lane-per-link formulation of csrc/arm_warp.cuh: every recursion over the chain as a scan over 8 lanes
    (Hillis-Steele prefix product for the kinematics, prefix sums for the velocities, ONE suffix sum of link force / moment / mass /
    first moment / inertia about the grip site), M from the broadcast spatial forces of unit joint accelerations."""
    W = 8
    R = [np.eye(3) for _ in range(W)]
    t = [np.zeros(3) for _ in range(W)]
    for j in range(nj):
        c, s_ = np.cos(q[j]), np.sin(q[j])
        R[j] = link[j, 3:12].reshape(3, 3) @ np.array([[c, -s_, 0], [s_, c, 0], [0, 0, 1.0]])
        t[j] = link[j, 0:3].copy()
    R[nj], t[nj] = tool[3:12].reshape(3, 3).copy(), tool[0:3].copy()  # lane NJ: tool transform -> grip-site pose
    d = 1
    while d < W:  # inclusive prefix product of (R, t): (Ra, ta) o (Rb, tb) = (Ra Rb, ta + Ra tb)
        Rn, tn = [x.copy() for x in R], [x.copy() for x in t]
        for j in range(d, W):
            Rn[j], tn[j] = R[j - d] @ R[j], t[j - d] + R[j - d] @ t[j]
        R, t, d = Rn, tn, 2 * d
    p = np.array(t[:nj]); z = np.array([R[j][:, 2] for j in range(nj)]); site, Rs = t[nj], R[nj]
    shift = lambda a: np.vstack([np.zeros((1, 3)), a[:-1]])
    zq = qd[:nj, None] * z
    w = np.cumsum(zq, 0); wp = shift(w)
    al = np.cumsum(np.cross(wp, zq), 0); alp = shift(al)
    r = p - shift(p)
    ac = np.cumsum(np.cross(alp, r) + np.cross(wp, np.cross(wp, r)), 0) - grav
    m = link[:nj, 15]
    cl = np.array([R[j] @ link[j, 12:15] for j in range(nj)])
    Iw = []
    for j in range(nj):
        I6 = link[j, 16:22]
        I = np.array([[I6[0], I6[3], I6[4]], [I6[3], I6[1], I6[5]], [I6[4], I6[5], I6[2]]])
        Iw.append(R[j] @ I @ R[j].T)
    Iw = np.array(Iw)
    acom = ac + np.cross(al, cl) + np.cross(w, np.cross(w, cl))
    f = m[:, None] * acom
    nn = np.einsum("jab,jb->ja", Iw, al) + np.cross(w, np.einsum("jab,jb->ja", Iw, w))
    dd = p + cl - site
    n0 = nn + np.cross(dd, f)
    Icomp = Iw + m[:, None, None] * (np.einsum("ja,ja->j", dd, dd)[:, None, None] * np.eye(3) - np.einsum("ja,jb->jab", dd, dd))
    suf = lambda a: np.cumsum(a[::-1], 0)[::-1]
    Fs, Ns, cm, hs, Ic = suf(f), suf(n0), suf(m), suf(m[:, None] * dd), suf(Icomp)
    a = p - site
    bias = np.einsum("ja,ja->j", z, Ns - np.cross(a, Fs))
    fj = np.cross(z, hs - cm[:, None] * a)
    njv = np.einsum("jab,jb->ja", Ic, z) - np.cross(hs, np.cross(z, a))
    M = np.eye(7)
    for c in range(nj):
        for i in range(c + 1):
            M[i, c] = M[c, i] = z[i] @ (njv[c] - np.cross(a[i], fj[c]))
    J = np.zeros((6, 7))
    J[:3, :nj] = np.cross(z, site - p).T
    J[3:, :nj] = z.T
    return M, bias, J, site, Rs


@pytest.mark.parametrize("robot", ["panda", "ur5e"])
def test_lane_per_link_formulation_matches_the_generic_tree(O, robot):
    """CPU pin of the arm kernel's algebra: the scan formulation of csrc/arm_warp.cuh (numpy mirror above, on the SAME link / tool
    tables the kernel reads) against the oracle's generic-tree quantities -- joint-space inertia, bias at non-zero velocity
    (Coriolis / centrifugal + gravity), grip-site Jacobian and pose -- for the Panda and the 6-joint UR5e."""
    from rui_b200.env import packed_model
    from rui_b200.model import ur5e_params
    pk = packed_model(False, ur5e_params()) if robot == "ur5e" else packed_model(False)
    m = pk.model
    nj = len(m.params.link_pos)
    e = O.OracleEnv(pk, _cfg(CC_FIXED), 0)
    e.reset()
    q_full, v_full = e.get_state()[0].copy(), e.get_state()[1].copy()
    rng = np.random.default_rng(3)
    for trial in range(5):
        q = np.zeros(7); qd = np.zeros(7)
        q[:nj] = np.array(m.params.init_qpos)[:nj] + rng.uniform(-0.4, 0.4, nj)
        qd[:nj] = rng.uniform(-1.0, 1.0, nj)
        q_full[:7], v_full[:7] = q, qd
        e.set_state(qpos=q_full, qvel=v_full)
        e.forward()
        M, bias, J, site, Rs = _arm_scans_numpy(np.asarray(m.arm_link).reshape(7, 22), np.asarray(m.arm_tool), q, qd, np.array([0, 0, -9.81]), nj)
        Jo, pos, mat = e.eef()
        assert np.abs(M[:nj, :nj] - e.M[:nj, :nj]).max() < 1e-10
        assert np.abs(bias[:nj] - e.bias[:nj]).max() < 1e-9
        assert np.abs(J - Jo).max() < 1e-12 and np.abs(site - pos).max() < 1e-12 and np.abs(Rs - mat).max() < 1e-12


@pytest.mark.parametrize("scene", ["soft", "rigid", "cylinder"])
def test_evaluate_at_the_oracle_optimum(O, scene):
    """oracle_evaluate (the hook the device solve is judged with): at the oracle's own qacc the float64 gradient vanishes, the primal
    cost is a minimum along random directions, and forces, cfrc and the F/T torque are those of the forward pass.  One arm joint
    sits 0.02 rad past its lower limit and moves into it (the limit is moved, so the contacts stay), so a joint-limit row is active.
    The env is left unchanged."""
    import dataclasses
    from rui_b200.abi import PackedModel
    from rui_b200.model import SceneParams, build_model, cylinder_torso_params
    params = cylinder_torso_params() if scene == "cylinder" else SceneParams(soft_torso=scene != "rigid")
    rng = np.random.default_rng(7)
    if scene == "rigid":  # fixed gains, the probe pressed onto the table
        cfg = _cfg(CC_FIXED, seed=2)
        e = O.OracleEnv(PackedModel(build_model(params)), cfg, 0)
        e.reset()
        for _ in range(250):
            e.step(np.array([0, 0, -1, 0, 0, 0.0]))
    else:
        cfg = _cfg(CC_TRACK, seed=5, torso_solref_randomization=True, initial_probe_pos_randomization=True)
        e = O.OracleEnv(PackedModel(build_model(params)), cfg, 0)
        e.reset()
        for _ in range(5):
            e.step(rng.uniform(0, 1, 6))
    q, v, w, t = e.get_state()
    tau = e.tau
    j = 3
    rng_j = [list(r) for r in params.joint_range]
    rng_j[j][0] = q[j] + 0.02
    pk = PackedModel(build_model(dataclasses.replace(params, joint_range=tuple(tuple(r) for r in rng_j))))
    e = O.OracleEnv(pk, cfg, 0)
    e.reset()
    v[j] = -0.3
    e.set_state(q, v, w, t)
    e.forward(tau)
    a = e.qacc
    c, d = e.contacts(), e.diag()
    assert len(c["dist"]) >= (1 if scene == "rigid" else 10)
    r = e.evaluate(a)
    assert r["nefc"] == e.nefc and np.isfinite(r["grad"]).all()
    lim = r["efc_type"] == 1
    assert lim.sum() == 1 and r["efc_force"][lim][0] > 0  # the lower-limit row pushes the joint back
    scale = 1 + r["rhs_norm"] + r["hx_norm"]
    assert r["gnorm"] == pytest.approx(np.linalg.norm(r["grad"]), rel=1e-12) and r["gnorm"] <= 1e-9 * scale, (r["gnorm"], scale)
    assert np.abs(r["contact_force"] - c["force"]).max() <= 1e-12 * max(1.0, np.abs(c["force"]).max())
    assert np.abs(r["cfrc"] - d[0:3]).max() <= 1e-12 * max(1.0, np.abs(d[0:3]).max())
    assert np.abs(r["ft_torque"] - d[3:6]).max() <= 1e-12 * max(1.0, np.abs(d[3:6]).max())
    for _ in range(8):
        dd = rng.standard_normal(e.nv) * 1e-3 * (1 + np.abs(a))
        assert e.evaluate(a + dd)["cost"] > r["cost"] and e.evaluate(a - dd)["cost"] > r["cost"]
    # elsewhere the gradient is M (a - a0) - J^T f, and the F/T torque follows qacc through the probe's acceleration
    b = a + rng.standard_normal(e.nv) * 0.1
    rb = e.evaluate(b)
    assert np.abs(rb["grad"][:7] - (e.M @ (b - e.qacc_smooth))[:7]).max() > 1e-3 and np.abs(rb["ft_torque"] - d[3:6]).max() > 1e-6
    # and the env is unchanged by the evaluations
    assert np.array_equal(e.qacc, a) and np.array_equal(e.diag(), d) and np.array_equal(e.contacts()["force"], c["force"])
    assert np.array_equal(e.evaluate(a)["efc_force"], r["efc_force"])
