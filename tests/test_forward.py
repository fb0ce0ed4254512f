"""usim_forward / BatchedUltrasound.forward: MuJoCo's mj_forward at the live state, without stepping.

1. On identical inputs (tests/forward_util.py) against the float64 oracle's forward: stopping rule, contact list, forces, probe
   wrench and F/T torque at the device's qacc, all 19 observation channels against forward_util.oracle_observation(), eef pose, and the
   applied torques equal to the clipped ctrl bit for bit.  Every bound is <= 4x the maximum measured on a B200 by
   scripts/forward_parity_report.py (profiles/forward_parity.json); the measured maximum is named beside each.
2. Nothing a later step reads changes: two handles with the same seed, one of them forwarding before some steps, step bit for bit
   alike.
3. Idempotence, masks, clipping, ctrl = None.
4. Readouts refreshed after auto-resets and explicit resets.
5. API edges; 6. the single-env API (set_robot_joint_positions, env.sim.forward()).
"""
import numpy as np
import pytest
import torch

import forward_util as fu
from conftest import CC_TRACK
from rui_b200 import _lib, abi

pytestmark = pytest.mark.gpu

# Bounds per scene, both torque kinds (profiles/forward_parity.json "scenes"; the measured maximum in the comment, the bound <= 4x
# it).  gnorm_err, gap_rel, force_rel, cfrc_rel, ft_rel as in test_solve_identical_inputs; obs_force_rel / obs_torque_rel: obs[0:6]
# measured as cfrc_rel / ft_rel; obs_vel, obs_task, obs_pose: max |d| of obs[6:9], obs[9:12], obs[12:19]; eef_pos, eef_quat: max |d|
# of diag[6:9], diag[9:13].
KEYS = ("gnorm_err", "gap_rel", "force_rel", "cfrc_rel", "ft_rel", "obs_force_rel", "obs_torque_rel", "obs_vel", "obs_task", "obs_pose",
        "eef_pos", "eef_quat")
BOUNDS = {
    "soft": (1.4e-4, 4.1e-8, 4.0e-5, 1.15e-4, 6.2e-4, 7.1e-5, 4.2e-4, 3.6e-7, 7.3e-9, 1.6e-6, 1.6e-6, 1.4e-6),
    #        3.55e-5, 1.03e-8, 1.01e-5, 2.88e-5, 1.55e-4, 1.78e-5, 1.05e-4, 9.0e-8, 1.83e-9, 4.17e-7, 4.17e-7, 3.54e-7
    "rigid": (2.7e-3, 2.0e-6, 2.3e-2, 1.6e-2, 1.7e-2, 1.1e-3, 1.1e-3, 8.5e-7, 3.3e-8, 1.5e-6, 1.5e-6, 9.2e-7),
    #        6.82e-4, 5.19e-7, 5.8e-3, 4.1e-3, 4.4e-3, 2.74e-4, 2.74e-4, 2.14e-7, 8.3e-9, 3.91e-7, 3.91e-7, 2.32e-7
    "cylinder": (1.2e-4, 1.18e-7, 8.1e-5, 1.38e-4, 1.17e-3, 7.4e-5, 6.4e-4, 2.4e-7, 4.7e-7, 1.7e-6, 1.7e-6, 1.1e-6),
    #           3.07e-5, 2.96e-8, 2.03e-5, 3.47e-5, 2.94e-4, 1.86e-5, 1.6e-4, 6.0e-8, 1.19e-7, 4.4e-7, 4.4e-7, 2.85e-7
    "ur5e": (1.27e-4, 9.8e-8, 5.7e-5, 1.14e-4, 1.0e-3, 6.0e-5, 7.4e-4, 4.3e-7, 3.5e-9, 1.7e-6, 1.7e-6, 8.5e-7),
    #        3.18e-5, 2.45e-8, 1.43e-5, 2.85e-5, 2.52e-4, 1.5e-5, 1.87e-4, 1.1e-7, 8.9e-10, 4.41e-7, 4.41e-7, 2.14e-7
}
# diag[21] / (tol (1 + |rhs| + |Hx|)_64) of a converged solve (test_solve_identical_inputs.RULE_DEV)
RULE_DEV = 1.01
COST_ROUNDOFF = 1e-12
MIN_CONTACTS = {"soft": 2000, "rigid": 10, "cylinder": 800, "ur5e": 2000}  # per torque kind; measured 2652, 18, 1011, 2625

RAND = dict(torso_solref_randomization=True, initial_probe_pos_randomization=True)


def _bound(scene, key):
    return BOUNDS[scene][KEYS.index(key)]


def _ctx(what, r):
    return what, {k: v for k, v in r.items() if k not in ("x", "grad")}


def _make(n, horizon=1000, seed=7, soft=True, **kw):
    from rui_b200.env import BatchedUltrasound
    return BatchedUltrasound(n, device=0, soft_torso=soft, controller_configs=CC_TRACK, control_freq=500, horizon=horizon, seed=seed,
                             **kw)


def _acts(env, k, seed=0):
    g = torch.Generator(device=env.device).manual_seed(seed)
    return [torch.rand(env.num_envs, env.action_dim, device=env.device, generator=g) for _ in range(k)]


def _ctrl(env, seed, scale=1.0):
    g = torch.Generator(device=env.device).manual_seed(seed)
    r = torch.as_tensor(fu.ctrl_range(env), device=env.device)
    return (torch.rand(env.num_envs, 7, device=env.device, generator=g) * 2 - 1) * r * scale


def _readouts(env, record=True):
    """every readout a forward refreshes, cloned: obs, diag, contact list (rows past ncon zeroed) and, with record, contact forces"""
    ncon, g1, g2, dist = env.contacts()
    live = torch.arange(abi.MAX_CONTACTS, device=env.device)[None] < ncon[:, None]
    out = dict(obs=env.obs.clone(), diag=env.diag(), ncon=ncon, g1=g1 * live, g2=g2 * live, dist=dist * live)
    if record:
        out.update(zip(("pos", "frame", "force"), env.contact_forces()))
    return out


def _assert_rows_equal(a, b, rows, where):
    for k in a:
        assert torch.equal(a[k][rows], b[k][rows]), (where, k)


# ---------------------------------------------------------------------------- 1. parity on identical inputs
_CACHE = {}


def _records(O, name, kind):
    if (name, kind) not in _CACHE:
        _CACHE[(name, kind)] = fu.run(O, name, kind)
    return _CACHE[(name, kind)]


@pytest.mark.parametrize("kind", fu.CTRLS)
@pytest.mark.parametrize("name", fu.SCENES)
def test_forward_matches_oracle_on_identical_states(O, name, kind):
    recs = _records(O, name, kind)
    for r in recs:
        ctx = _ctx((name, kind), r)
        assert r["list_ok"] and r["nefc_dev"] == r["nefc"], ctx
        assert r["finite"] and r["iters"] < r["cap"] and r["tau_exact"], ctx
        assert r["gnorm_err"] <= _bound(name, "gnorm_err") and r["gap_rel"] >= -COST_ROUNDOFF, ctx
        assert r["rule_dev"] <= RULE_DEV and r["gnorm"] <= (r["tol"] + _bound(name, "gnorm_err")) * r["scale"], ctx
        assert r["gap_rel"] <= _bound(name, "gap_rel"), ctx
        for k in KEYS[2:]:
            assert r[k] <= _bound(name, k), (k, ctx)
    assert sum(r["ncon"] for r in recs) >= MIN_CONTACTS[name]


# ---------------------------------------------------------------------------- 2. nothing a later step reads changes
def test_forward_leaves_every_later_step_bitwise_unchanged():
    """4096 envs, auto-reset, horizon 4 (episode ends every 4th step): handle B forwards before most steps (unmasked and masked, with
    and without ctrl, with the qacc output), handle A never; every output of every step, the state, the readouts and the arm record
    stay bit for bit those of A.  The state right after a forward is the state before it."""
    n, horizon = 4096, 4
    A, B = _make(n, horizon, record_contacts=True, **RAND), _make(n, horizon, record_contacts=True, **RAND)
    A.reset(), B.reset()
    acts = _acts(A, 14)
    g = torch.Generator(device=A.device).manual_seed(3)
    ended = 0
    for s, a in enumerate(acts):
        plan = s % 4
        if plan != 2:
            before = [x.clone() for x in B.get_state()]
            mask = (torch.rand(n, device=B.device, generator=g) < 0.5) if plan == 1 else None
            ctrl = _ctrl(B, 10 + s) if plan in (1, 3) else None
            B.forward(mask=mask, ctrl=ctrl, qacc=plan == 3)
            for x, y in zip(B.get_state(), before):
                assert torch.equal(x, y), ("state changed by the forward", s)
        oa = [x.clone() for x in A.step(a, auto_reset=True)]
        ob = [x.clone() for x in B.step(a, auto_reset=True)]
        for name, x, y in zip(("obs", "reward", "done", "terminal obs"), oa, ob):
            assert torch.equal(x, y), (s, name)
        for name, x, y in zip(("qpos", "qvel", "warm", "task"), A.get_state(), B.get_state()):
            assert torch.equal(x, y), (s, name)
        _assert_rows_equal(_readouts(A), _readouts(B), slice(None), ("step", s))
        assert torch.equal(A.arm_record(), B.arm_record()), (s, "arm record")
        ended += int(oa[2].sum())
    assert ended >= 3 * n, ended
    assert A.divergence_count == B.divergence_count and A.contact_overflow_count == B.contact_overflow_count
    A.close(), B.close()


# ---------------------------------------------------------------------------- 3. idempotence, mask, clipping, ctrl = None
def test_forward_idempotent_masked_clipped():
    n = 256
    env = _make(n, record_contacts=True, **RAND)
    env.reset()
    for a in _acts(env, 10):
        env.step(a, auto_reset=False)
    state = [x.clone() for x in env.get_state()]
    arm = env.arm_record()
    ca, cb = _ctrl(env, 1), _ctrl(env, 2)

    def fwd(**kw):
        _, qa = env.forward(qacc=True, **kw)
        return dict(_readouts(env), qacc=qa.clone())

    # twice in a row: bitwise the same
    x1, x2 = fwd(ctrl=ca), fwd(ctrl=ca)
    _assert_rows_equal(x1, x2, slice(None), "second forward")
    # ctrl = None is zero torques
    _assert_rows_equal(fwd(ctrl=None), fwd(ctrl=torch.zeros(n, 7, device=env.device)), slice(None), "ctrl None vs zeros")
    # out-of-range ctrl is clipped to ctrl_range: the torques applied, and every output, are those of the clipped ctrl
    big = _ctrl(env, 3, scale=10.0)
    xb = fwd(ctrl=big)
    want = torch.as_tensor(fu.clipped(env, big.cpu().numpy()), device=env.device)
    assert torch.equal(xb["diag"][:, 13:20], want)
    _assert_rows_equal(xb, fwd(ctrl=want), slice(None), "clipped ctrl")
    # a mask: selected rows are those of an unmasked forward with the same ctrl, every other row is left as it was
    xa = fwd(ctrl=ca)
    xbb = fwd(ctrl=cb)
    mask = torch.zeros(n, dtype=torch.bool, device=env.device)
    mask[::3] = True
    mask[5] = True
    _, qa = env.forward(mask=mask, ctrl=ca, qacc=True)
    xm = dict(_readouts(env), qacc=qa.clone())
    _assert_rows_equal(xm, xa, mask, "selected rows")
    xbb["qacc"] = torch.zeros_like(xbb["qacc"])
    _assert_rows_equal(xm, xbb, ~mask, "unselected rows")
    # the state and the arm record stay as the last step left them
    for x, y in zip(env.get_state(), state):
        assert torch.equal(x, y)
    assert torch.equal(env.arm_record(), arm)
    env.close()


# ---------------------------------------------------------------------------- 4. refresh after resets
def _oracle_at(O, env, gid, key, q, v, w, t, **cfg_kw):
    """The oracle's reset of (gid, key) (as test_reset_paths builds it), checked against the device's record of that reset; then
    the oracle set to the device's fp32 state and forwarded with zero torques: (oracle env, its observation)."""
    e = O.OracleEnv(env.packed, abi.make_config(1, CC_TRACK, control_freq=500, seed=env.cfg.seed, **cfg_kw), int(gid))
    ts = np.zeros(abi.TASK_DIM)
    ts[abi.TS_EPISODE] = key
    e.set_state(task=ts)
    e.reset()
    _, _, _, ot = e.get_state()
    assert t[abi.TS_EPISODE] == key + 1 and t[abi.TS_STIFFNESS] == np.float32(ot[abi.TS_STIFFNESS]), (gid, key)
    np.testing.assert_allclose(t[:7], ot[:7], atol=2e-7)
    e.set_state(q, v, w, t)
    e.forward(np.zeros(7))
    return e, fu.oracle_observation(O, e)


def _check_against(O, orc, o_obs, d_obs, diag, ncon, g1, g2, scene, where):
    c = orc.contacts()
    k = int(ncon)
    assert k == len(c["geom1"]) and (g1[:k] == c["geom1"]).all() and (g2[:k] == c["geom2"]).all(), (where, "contact list")
    fsum = max(1.0, float(c["force"][:, 0].sum()) if k else 0.0)
    m = fu.obs_metrics(d_obs, o_obs, fsum)
    m["cfrc_rel"] = float(np.abs(diag[0:3] - orc.diag()[0:3]).max() / fsum)
    m.update(fu.eef_metrics(O, orc, diag))
    for key, v in m.items():
        assert v <= _bound(scene, key), (where, key, v)


def _obs_close(a, b, scene, where):
    """two device observations of the same state, within the observation bounds of test 1"""
    fsum = np.maximum(1.0, np.abs(b[:, 0:3]).max(1))
    for i in range(a.shape[0]):
        m = fu.obs_metrics(a[i], b[i], fsum[i])
        for key, v in m.items():
            assert v <= _bound(scene, key), (where, i, key, v)


def test_forward_refreshes_readouts_after_resets(O):
    n, horizon = 32, 3
    env = _make(n, horizon, record_contacts=True, **RAND)
    obs_reset = env.reset().cpu().numpy().astype(np.float64)
    diag_reset = env.diag().cpu().numpy().astype(np.float64)
    ncon_r, g1_r, g2_r, _ = [x.cpu().numpy() for x in env.contacts()]
    # explicit reset: forward() reproduces its diag, contact list and observation
    obs_f = env.forward().cpu().numpy().astype(np.float64)
    diag_f = env.diag().cpu().numpy().astype(np.float64)
    ncon_f, g1_f, g2_f, _ = [x.cpu().numpy() for x in env.contacts()]
    assert np.array_equal(ncon_f, ncon_r)
    for i in range(n):
        assert (g1_f[i, :ncon_r[i]] == g1_r[i, :ncon_r[i]]).all() and (g2_f[i, :ncon_r[i]] == g2_r[i, :ncon_r[i]]).all(), i
    _obs_close(obs_f, obs_reset, "soft", "after usim_reset")
    assert np.abs(diag_f[:, 6:13] - diag_reset[:, 6:13]).max() <= _bound("soft", "eef_pos")
    assert np.array_equal(diag_f[:, 13:20], np.zeros((n, 7)))
    fsum = np.maximum(1.0, np.abs(diag_reset[:, 0:3]).max(1, keepdims=True))
    assert (np.abs(diag_f[:, 0:3] - diag_reset[:, 0:3]) / fsum).max() <= _bound("soft", "cfrc_rel")
    # auto-reset: the step's post-reset observation and the oracle's reset of the same (env, episode)
    ended = 0
    for a in _acts(env, 2 * horizon):
        obs, _, done, _ = env.step(a, auto_reset=True)
        if not bool(done.any()):
            continue
        d = done.cpu().numpy().astype(bool)
        ended += int(d.sum())
        obs_step = obs.cpu().numpy().astype(np.float64).copy()
        obs_f = env.forward().cpu().numpy().astype(np.float64)
        _obs_close(obs_f[d], obs_step[d], "soft", "after an auto-reset")
        diag = env.diag().cpu().numpy().astype(np.float64)
        ncon, g1, g2, _ = [x.cpu().numpy() for x in env.contacts()]
        q, v, w, t = [x.cpu().numpy().astype(np.float64) for x in env.get_state()]
        for i in np.nonzero(d)[0][:8]:
            orc, o_obs = _oracle_at(O, env, i, int(t[i, abi.TS_EPISODE]) - 1, q[i], v[i], w[i], t[i], **RAND)
            _check_against(O, orc, o_obs, obs_f[i], diag[i], ncon[i], g1[i], g2[i], "soft", ("auto-reset", int(i)))
    assert ended >= n
    env.close()


# ---------------------------------------------------------------------------- 5. API edges
def test_forward_api_edges():
    env = _make(64, horizon=2, **RAND)
    with pytest.raises(_lib.UsimError, match="usim_reset"):
        env.forward()
    env.reset()
    # NULL outputs (mask, ctrl, obs and qacc all NULL): the readouts still refresh
    env.forward(ctrl=_ctrl(env, 1))
    with torch.cuda.device(env.device):
        _lib.check(_lib.lib().usim_forward(env._h, None, None, None, None, env._stream()))
    torch.cuda.synchronize()
    assert torch.equal(env.diag()[:, 13:20], torch.zeros(64, 7, device=env.device))
    # a terminated env (auto_reset off) is forwarded and stays done
    for a in _acts(env, 2):
        _, _, done, _ = env.step(a, auto_reset=False)
    assert bool(done.all())
    before = [x.clone() for x in env.get_state()]
    c = _ctrl(env, 4)
    obs = env.forward(ctrl=c)
    assert torch.isfinite(obs).all()
    assert torch.equal(env.diag()[:, 13:20], torch.as_tensor(fu.clipped(env, c.cpu().numpy()), device=env.device))
    for x, y in zip(env.get_state(), before):
        assert torch.equal(x, y)
    assert (env.get_state()[3][:, abi.TS_DONE] == 1).all()
    env.close()


def test_forward_ordered_with_step_host():
    """forward on the caller's stream, then step_host on the library's own stream: the step waits for the forward"""
    n = 512
    A, B = _make(n, **RAND), _make(n, **RAND)
    A.reset(), B.reset()
    acts = [a.cpu().numpy() for a in _acts(A, 6)]
    for s, a in enumerate(acts):
        B.forward(ctrl=_ctrl(B, s))
        oa = [x.copy() for x in A.step_host(a, auto_reset=True)]
        ob = [x.copy() for x in B.step_host(a, auto_reset=True)]
        for x, y in zip(oa[:3], ob[:3]):
            assert np.array_equal(x, y), s
        assert torch.equal(A.diag(), B.diag()), s
    A.close(), B.close()


def test_contact_forces_after_unmasked_forward():
    """recording turned on since the last step: a masked forward does not complete the record, an unmasked one does"""
    n = 64
    env = _make(n, **RAND)
    env.reset()
    env.step(_acts(env, 1)[0], auto_reset=False)
    env.set_contact_record(True)
    with pytest.raises(_lib.UsimError):
        env.contact_forces()
    env.forward(mask=torch.arange(n, device=env.device) < n // 2)
    with pytest.raises(_lib.UsimError):
        env.contact_forces()
    env.forward()
    pos, frame, force = env.contact_forces()
    ncon = env.contacts()[0]
    live = torch.arange(abi.MAX_CONTACTS, device=env.device)[None] < ncon[:, None]
    assert int(ncon.sum()) > 0 and torch.isfinite(force).all()
    assert not force[~live].any() and not pos[~live].any()
    env.close()


# ---------------------------------------------------------------------------- 6. single-env API
@pytest.mark.parametrize("robot", ["Panda", "UR5e"])
def test_single_env_set_robot_joint_positions_forwards(O, robot):
    """set_robot_joint_positions runs sim.forward() with the torques last applied, as robosuite does: eef pose, contacts and probe
    force describe the new pose (the oracle's forward at that state)"""
    from rui_b200.env import make
    env = make("Ultrasound", robots=robot, controller_configs=CC_TRACK, control_freq=500, horizon=50, seed=3)
    assert callable(env.sim.forward)
    env.reset()
    for _ in range(5):
        env.step(np.full(6, 0.5))
    rb = env.robots[0]
    tau = env.core.diag()[0, 13:20].cpu().numpy().astype(np.float64)
    q_old = env._eef_xpos
    rb.set_robot_joint_positions(rb._joint_positions + 0.01)
    assert np.abs(env._eef_xpos - q_old).max() > 1e-3
    q, v, w, t = [x[0].cpu().numpy().astype(np.float64) for x in env.core.get_state()]
    orc = O.OracleEnv(env.core.packed, abi.make_config(1, CC_TRACK, control_freq=500, horizon=50, seed=3), 0)
    orc.set_state(q, v, w, t)
    orc.forward(tau)
    _, pos, _ = orc.eef()
    scene = "ur5e" if robot == "UR5e" else "soft"
    assert np.abs(env._eef_xpos - pos).max() <= _bound(scene, "eef_pos")
    assert np.array_equal(env.core.diag()[0, 13:20].cpu().numpy().astype(np.float64), tau)
    got = env.get_contacts()
    c = orc.contacts()
    names = env.core.model.geom_name
    assert [(x["geom1"], x["geom2"]) for x in got] == [(names(a), names(b)) for a, b in zip(c["geom1"], c["geom2"])]
    fsum = max(1.0, float(c["force"][:, 0].sum()) if len(got) else 0.0)
    if got:
        assert np.abs(np.array([x["force"] for x in got]) - c["force"]).max() / fsum <= _bound(scene, "force_rel")
    assert np.abs(rb.ee_force - orc.diag()[0:3]).max() / fsum <= _bound(scene, "cfrc_rel")
    env.close()
