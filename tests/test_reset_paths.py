"""Every reset path against the float64 oracle's reset of the same (seed, global env id, episode key).

usim.h promises that a reset draws stiffness, damping, waypoints, u0 and probe noise from Philox streams keyed by (seed, global env
id, episode).  Auto-resets take over states prepared ahead of time on a side stream, two slots per env (slot E & 1 holds the state of
episode key E), so the promise rests on that bookkeeping.  These tests follow it through state restores (into the same handle and
into a fresh one), masked resets while prepared states are in flight, batch sizes that leave partial CTAs and request lists longer
than the prepare launches' fixed grids, and the other scenes and reset options.

The oracle's reset for key E: its task record gets TS_EPISODE = E, then reset().  Tolerances are those of
test_gpu_parity.test_reset_pipeline_matches_oracle_resets_under_back_to_back_terminations, measured on a B200.
"""
import numpy as np
import pytest
import torch

from conftest import CC_TRACK
from rui_b200 import abi

pytestmark = pytest.mark.gpu

RAND = dict(torso_solref_randomization=True, initial_probe_pos_randomization=True)

# test_gpu_parity.TOL_SOFT (measured on a B200, fp32 vs float64): bounds the steps between a restore and the next episode end, where
# the restored env starts its solves from another warm start than the original run did (the shift of the warm start comes from the
# arm record, which the state does not carry), so the two agree to solver tolerance only.
TOL_SOFT = dict(qpos=3e-5, qvel=1.2e-3, reward=6e-2, force_rel=8e-3, torque_rel=1.5e-2, obs_eef_vel=4e-4, fz_mean_rel=1e-2, dfz_rel=4e-2,
                obs_vel_mean=2e-5, obs_pos_err=2e-5, obs_quat_err=2e-5, ts_traj_pt=1e-7, ts_pos_err=4e-3, ts_ori_err=1e-3)


def _make(n, horizon, seed, soft=True, **kw):
    from rui_b200.env import BatchedUltrasound
    return BatchedUltrasound(n, device=0, soft_torso=soft, controller_configs=CC_TRACK, control_freq=500, horizon=horizon, seed=seed, **kw)


def _np(*xs):
    return [x.cpu().numpy().astype(np.float64) for x in xs]


def _state(env):
    return [x.clone() for x in env.get_state()]


class OracleResets:
    """The oracle's reset of (global env id, episode key) for the scene and seed of `env`: (obs, qpos, task), memoised."""

    def __init__(self, O, env, **cfg_kw):
        self.O, self.packed = O, env.packed
        self.cfg = abi.make_config(1, CC_TRACK, control_freq=500, seed=env.cfg.seed, **cfg_kw)
        self.envs, self.memo = {}, {}

    def __call__(self, gid, key):
        gid, key = int(gid), int(key)
        if (gid, key) not in self.memo:
            if gid not in self.envs:
                self.envs[gid] = self.O.OracleEnv(self.packed, self.cfg, gid)
            e = self.envs[gid]
            ts = np.zeros(abi.TASK_DIM)
            ts[abi.TS_EPISODE] = key
            e.set_state(task=ts)
            obs = e.reset()
            q, _, _, t = e.get_state()
            self.memo[(gid, key)] = (obs, q, t)
        return self.memo[(gid, key)]


def _assert_reset(orc, gid, key, o, q, v, w, t, where, arm_atol=3e-5):
    """One env's rows right after a reset with episode key `key` against the oracle's reset of (gid, key)."""
    oo, oq, ot = orc(gid, key)
    where = f"{where}: env {gid}, key {key}"
    assert t[abi.TS_EPISODE] == key + 1, (where, "episode counter", t[abi.TS_EPISODE])
    assert t[abi.TS_TIMESTEP] == 0 and t[abi.TS_DONE] == 0, where
    # integer Philox draws are bit-exact (the fp32 record holds them exactly); the float draws and the IK agree to fp32 round-off
    assert t[abi.TS_STIFFNESS] == np.float32(ot[abi.TS_STIFFNESS]) and t[abi.TS_DAMPING] == np.float32(ot[abi.TS_DAMPING]), \
        (where, "stiffness / damping", t[abi.TS_STIFFNESS], ot[abi.TS_STIFFNESS], t[abi.TS_DAMPING], ot[abi.TS_DAMPING])
    np.testing.assert_allclose(t[:7], ot[:7], atol=2e-7, err_msg=where + ": waypoints / u0")
    np.testing.assert_allclose(q[:7], oq[:7], atol=arm_atol, err_msg=where + ": arm qpos")
    np.testing.assert_allclose(q[7:], oq[7:], atol=1e-6, err_msg=where + ": torso qpos")
    assert np.all(v == 0) and np.all(w == 0), (where, "qvel / warm start of a reset state")
    np.testing.assert_allclose(o[12:19], oo[12:19], atol=arm_atol, err_msg=where + ": pose error obs")
    np.testing.assert_allclose(o[:3], oo[:3], rtol=3e-2, atol=0.3, err_msg=where + ": contact force obs")
    assert o[10] == 0 and o[11] == pytest.approx(-0.04), (where, o[10], o[11])


def _assert_soft(where, got, want):
    """Two runs of the same envs that agree to solver tolerance, against TOL_SOFT: got / want = (obs, reward) of a step, optionally
    followed by (qpos, qvel, task) after it (parity_util.compare_rollout's measures, over all envs at once)."""
    go, gr, wo, wr = *got[:2], *want[:2]
    d = dict(reward=np.abs(gr - wr).max(),
             force_rel=(np.abs(go[:, 0:3] - wo[:, 0:3]) / np.maximum(1.0, np.abs(wo[:, 0:3]).max(1, keepdims=True))).max(),
             torque_rel=(np.abs(go[:, 3:6] - wo[:, 3:6]) / np.maximum(0.1, np.abs(wo[:, 3:6]).max(1, keepdims=True))).max(),
             obs_eef_vel=np.abs(go[:, 6:9] - wo[:, 6:9]).max(),
             fz_mean_rel=(np.abs(go[:, 9] - wo[:, 9]) / np.maximum(1.0, np.abs(wo[:, 9] + 5.0))).max(),
             dfz_rel=(np.abs(go[:, 10] - wo[:, 10]) / np.maximum(500.0, np.abs(wo[:, 10]))).max(),
             obs_vel_mean=np.abs(go[:, 11] - wo[:, 11]).max(), obs_pos_err=np.abs(go[:, 12:15] - wo[:, 12:15]).max(),
             obs_quat_err=np.abs(go[:, 15:19] - wo[:, 15:19]).max())
    if len(got) > 2:
        (gq, gv, gt), (wq, wv, wt) = got[2:], want[2:]
        d.update(qpos=np.abs(gq - wq).max(), qvel=np.abs(gv - wv).max(),
                 ts_traj_pt=np.abs(gt[:, abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3] - wt[:, abi.TS_TRAJ_PT:abi.TS_TRAJ_PT + 3]).max(),
                 ts_pos_err=np.abs(gt[:, abi.TS_POS_ERR:abi.TS_POS_ERR + 2] - wt[:, abi.TS_POS_ERR:abi.TS_POS_ERR + 2]).max(),
                 ts_ori_err=np.abs(gt[:, abi.TS_ORI_ERR] - wt[:, abi.TS_ORI_ERR]).max())
        for k in (abi.TS_EPISODE, abi.TS_TIMESTEP, abi.TS_DONE):
            assert np.array_equal(gt[:, k], wt[:, k]), (where, "task record entry", k)
    bad = {k: (float(v), TOL_SOFT[k]) for k, v in d.items() if not v <= TOL_SOFT[k]}
    assert not bad, f"{where}: measured > tolerance: {bad}"


# ---------------------------------------------------------------------------- state restores
HORIZON, N_RESTORE, STEPS = 5, 16, 22
SNAPSHOTS = (17, 12)  # two steps into episodes 4 and 3: one and two episodes back from the end, both slot parities


def _record(env, acts):
    """Run every action with auto-reset; per step: the step's outputs and the state rows after it, and the state rows as snapshots."""
    rec = []
    for a in acts:
        o, r, d, tobs = env.step(a, auto_reset=True)
        o, r, d, tobs = o.clone(), r.clone(), d.clone(), tobs.clone()
        rec.append(dict(out=(o, r, d, tobs), state=_state(env)))
    return rec


def _replay_and_check(env, O, rec, acts, s0, where):
    """Restore the state after step s0 of `rec` into `env`, replay steps s0 + 1 ... and compare with the recording: to solver
    tolerance up to the first episode end, bitwise from the reset it takes over on; every reset against the oracle's."""
    n = env.num_envs
    env.set_state(*rec[s0 - 1]["state"])
    orc = OracleResets(O, env, **RAND)
    counter = int(rec[s0 - 1]["state"][3][0, abi.TS_EPISODE])
    assert (rec[s0 - 1]["state"][3][:, abi.TS_EPISODE] == counter).all()
    bitwise = False
    for s in range(s0 + 1, len(acts) + 1):
        o, r, d, tobs = env.step(acts[s - 1], auto_reset=True)
        ro, rr, rd, rtobs = rec[s - 1]["out"]
        q, v, w, t = env.get_state()
        rq, rv, rw, rt = rec[s - 1]["state"]
        here = f"{where}, restored after step {s0}, step {s}"
        assert torch.equal(d, rd), (here, "done")
        ended = bool(d.all())
        assert ended or not bool(d.any()), (here, "episodes of the batch run in lock step")
        if ended:
            # the counters advance by exactly one: a reset taken from a slot prepared for another episode shows up here first
            tn = t.cpu().numpy()
            assert (tn[:, abi.TS_EPISODE] == counter + 1).all(), \
                (here, f"episode counters after the reset of key {counter}", np.unique(tn[:, abi.TS_EPISODE]).tolist())
            on, qn, vn, wn = _np(o, q, v, w)
            for i in range(n):
                _assert_reset(orc, i, counter, on[i], qn[i], vn[i], wn[i], tn[i], here)
            counter += 1
        if bitwise:
            assert torch.equal(r, rr) and torch.equal(tobs[d.bool()], rtobs[rd.bool()]), (here, "reward / terminal obs")
        elif ended:  # the episode's last step: its observation is the terminal one, its state rows are replaced by the reset's
            _assert_soft(here, _np(tobs, r), _np(rtobs, rr))
        else:
            _assert_soft(here, _np(o, r, q, v, t), _np(ro, rr, rq, rv, rt))
        if ended or bitwise:
            # from the first episode end on the restored run IS the original one
            assert torch.equal(o, ro), (here, "obs")
            for name, a, b in (("qpos", q, rq), ("qvel", v, rv), ("warm", w, rw), ("task", t, rt)):
                assert torch.equal(a, b), (here, name, float((a - b).abs().max()))
            bitwise = True
    assert bitwise, "no episode ended after the restore"


def _restore_run(seed):
    env = _make(N_RESTORE, HORIZON, seed, **RAND)
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    acts = [torch.rand(N_RESTORE, 6, device="cuda", generator=gen) for _ in range(STEPS)]
    rec = _record(env, acts)
    assert (rec[-1]["state"][3][:, abi.TS_EPISODE] == 1 + STEPS // HORIZON).all()
    return env, rec, acts


def test_restore_into_the_same_handle_replays_the_original_run(O):
    """Snapshots 1 and 2 episodes back, restored into the handle that ran on past them (its slots hold later episodes)."""
    env, rec, acts = _restore_run(seed=9)
    for s0 in SNAPSHOTS:
        _replay_and_check(env, O, rec, acts, s0, "same handle")
    env.close()


def test_restore_into_a_fresh_handle_replays_the_original_run(O):
    """The snapshots restored into a new handle of the same seed that was reset once (its slots hold episodes 1 and 2)."""
    env, rec, acts = _restore_run(seed=4)
    env.close()
    for s0 in SNAPSHOTS:
        fresh = _make(N_RESTORE, HORIZON, 4, **RAND)
        fresh.reset()
        _replay_and_check(fresh, O, rec, acts, s0, "fresh handle")
        fresh.close()


# ---------------------------------------------------------------------------- masked resets
def test_masked_resets_with_the_auto_reset_pipeline_running(O):
    """Seeded masks on steps that end episodes and on steps that do not, an all-zero mask, and a mask on the very first reset (envs
    that were never reset stay frozen until a later mask picks them): a masked env's new state is the oracle's reset for its old
    counter, its later auto-resets take the next keys, and the rows of the other envs are untouched by the reset call."""
    n, horizon, steps = 40, 4, 18
    env = _make(n, horizon, 6, **RAND)
    orc = OracleResets(O, env, **RAND)
    rng = np.random.default_rng(12)
    gen = torch.Generator(device="cuda").manual_seed(12)
    counter = np.zeros(n, int)  # expected TS_EPISODE
    tstep = np.zeros(n, int)    # expected TS_TIMESTEP
    live = np.zeros(n, bool)    # reset at least once
    # step after which a masked reset follows -> mask (step 0: the first reset; 4: the first cohort's episodes end in that step)
    masks = {0: rng.random(n) < 0.5, 2: rng.random(n) < 0.3, 4: rng.random(n) < 0.5, 5: np.zeros(n, bool), 7: rng.random(n) < 0.4,
             9: None, 12: rng.random(n) < 0.3}
    masks[0][[0, n - 1]] = True
    masks[0][1] = False
    for m in masks.values():
        if m is not None:
            m[2] = False  # env 2 is never reset: frozen to the end
    checked_end_mask = False

    def masked_reset(mask, where):
        nonlocal checked_end_mask
        before = _state(env)
        obs_before = env.obs.clone()
        o = env.reset(torch.as_tensor(mask.astype(np.uint8)))
        after = _state(env)
        keep = torch.as_tensor(~mask, device="cuda")
        for name, a, b in zip(("qpos", "qvel", "warm", "task"), after, before):
            assert torch.equal(a[keep], b[keep]), (where, "rows of an unmasked env changed", name)
        assert torch.equal(o[keep], obs_before[keep]), (where, "obs rows of an unmasked env changed")
        on, qn, vn, wn, tn = _np(o, *after)
        for i in np.nonzero(mask)[0]:
            checked_end_mask |= bool(live[i] and tstep[i] == 0)
            _assert_reset(orc, i, counter[i], on[i], qn[i], vn[i], wn[i], tn[i], where)
        counter[mask] += 1
        tstep[mask] = 0
        live[mask] = True

    masked_reset(masks[0], "first reset (masked)")
    for s in range(1, steps + 1):
        o, r, d, tobs = env.step(torch.rand(n, 6, device="cuda", generator=gen), auto_reset=True)
        tstep[live] += 1
        ends = live & (tstep == horizon)
        dn = d.cpu().numpy().astype(bool)
        assert np.array_equal(dn, ends), (s, np.nonzero(dn != ends)[0])
        on, qn, vn, wn, tn = _np(o, *env.get_state())
        for i in np.nonzero(ends)[0]:  # auto-reset: the key is the counter of the episode that ended
            _assert_reset(orc, i, counter[i], on[i], qn[i], vn[i], wn[i], tn[i], f"auto-reset at step {s}")
        counter[ends] += 1
        tstep[ends] = 0
        assert np.array_equal(tn[:, abi.TS_EPISODE], counter) and np.array_equal(tn[:, abi.TS_TIMESTEP], tstep), s
        assert np.array_equal(tn[:, abi.TS_DONE] != 0, ~live), s  # never-reset envs stay frozen (done until reset)
        if s in masks:
            m = masks[s]
            if m is None:  # pick up the never-reset envs but one
                m = ~live
                m[2] = False
            masked_reset(m, f"masked reset after step {s}")
    assert checked_end_mask, "no masked reset hit an env that had just been auto-reset"
    assert not live[2] and live.sum() == n - 1 and counter.max() >= 5
    env.close()


# ---------------------------------------------------------------------------- batch sizes
BIG = 4097


def _rows(env, acts, n, off):
    """obs, reward, done, terminal obs of done envs, qpos, qvel, warm, task after the first reset and after every step (host copies;
    the env's output buffers are reused by every call)."""
    host = lambda xs: [x.to("cpu", copy=True) for x in xs]
    o = env.reset()
    out = [host([o, torch.zeros(n), torch.zeros(n, dtype=torch.uint8), torch.zeros(n, abi.OBS_DIM)] + list(env.get_state()))]
    for a in acts:
        o, r, d, tobs = env.step(a[off:off + n].contiguous(), auto_reset=True)
        out.append(host([o, r, d, torch.where(d.bool()[:, None], tobs, torch.zeros_like(tobs))] + list(env.get_state())))
    return out


@pytest.mark.parametrize("horizon", [1, 2])
def test_batch_size_edges_are_bitwise_those_of_a_64_env_handle(O, horizon):
    """n = 1, 3, 5, 33, 4097 (partial CTAs of the arm kernel, 4 envs per CTA, and of the reset kernel, 32 per CTA; 4097: the first
    reset queues 8194 requests for the prepare launches' fixed grids, and slot rows (E & 1) * n + env lie far from 0).  At horizon 1
    every step takes over a slot.  The rows of global env e equal those of e in a 64-env handle whose env_id_offset puts e inside
    it; at 4097, 32 envs spread over the batch (the first and the last among them) are compared with the oracle's resets."""
    seed, steps = 8, 4
    gen = torch.Generator(device="cuda").manual_seed(horizon)
    acts = [torch.rand(BIG, 6, device="cuda", generator=gen) for _ in range(steps)]
    windows = {}  # env_id_offset -> rows of a 64-env handle

    def window(off):
        if off not in windows:
            env = _make(64, horizon, seed, env_id_offset=off, **RAND)
            windows[off] = _rows(env, acts, 64, off)
            env.close()
        return windows[off]

    names = ("obs", "reward", "done", "terminal obs", "qpos", "qvel", "warm", "task")
    for n in (1, 3, 5, 33, BIG):
        env = _make(n, horizon, seed, **RAND)
        got = _rows(env, acts, n, 0)
        env.close()
        for s in range(steps + 1):
            if s:
                ends = got[s][2].bool()
                assert bool(ends.all()) == (s % horizon == 0) and (bool(ends.all()) or not bool(ends.any())), (n, s)
            ep = 1 + s // horizon
            assert (got[s][7][:, abi.TS_EPISODE] == ep).all(), (n, s, "episode counters", got[s][7][:, abi.TS_EPISODE].unique().tolist())
        for lo in range(0, n, 64):
            off = min(lo, max(n, 64) - 64)
            ref = window(off)
            k = min(64, n)
            for s in range(steps + 1):
                for name, a, b in zip(names, got[s], ref[s]):
                    assert torch.equal(a[off:off + k] if n > 64 else a, b[:k]), (n, s, name, f"envs {off}..{off + k - 1}")
        if n == BIG:
            orc = OracleResets(O, env, **RAND)
            for s in range(0, steps + 1, horizon):
                o, _, _, _, q, v, w, t = [x.numpy().astype(np.float64) for x in got[s]]
                for i in np.linspace(0, BIG - 1, 32).astype(int):
                    _assert_reset(orc, i, s // horizon, o[i], q[i], v[i], w[i], t[i], f"n {n}, horizon {horizon}, step {s}")


# ---------------------------------------------------------------------------- scenes and options
def _other_paths():
    from rui_b200.model import ur5e_params
    return {
        "ur5e": (dict(scene_params=ur5e_params(), **RAND), dict(), 5e-5),  # UR5e IK: test_gpu_parity.test_ur5e_parity's bound
        "rigid": (dict(soft=False, **RAND), dict(), 3e-5),
        "deterministic_trajectory": (dict(deterministic_trajectory=True, **RAND), dict(deterministic_trajectory=True), 3e-5),
        "no_randomisation": (dict(), dict(), 3e-5),
        "env_id_offset": (dict(env_id_offset=1000, **RAND), dict(), 3e-5),
    }


@pytest.mark.parametrize("path", ["ur5e", "rigid", "deterministic_trajectory", "no_randomisation", "env_id_offset"])
def test_other_reset_paths_match_oracle_under_auto_reset(O, path):
    """The first reset and every auto-reset of a short run, per scene / option: the UR5e arm (reset_kernel<6>), the rigid scene (no
    IK), a deterministic trajectory, both randomisations off, and env ids offset from 0 (sharded runs)."""
    kw, okw, arm_atol = _other_paths()[path]
    n, horizon, steps = 16, 2, 6
    env = _make(n, horizon, 5, **kw)
    off = kw.get("env_id_offset", 0)
    orc = OracleResets(O, env, **{k: v for k, v in kw.items() if k in RAND}, **okw)
    gen = torch.Generator(device="cuda").manual_seed(3)
    o = env.reset()
    for s in range(steps + 1):
        if s:
            o, r, d, tobs = env.step(torch.rand(n, 6, device="cuda", generator=gen), auto_reset=True)
            assert bool(d.all()) == (s % horizon == 0) and (bool(d.all()) or not bool(d.any())), s
            if s % horizon:
                continue
        on, qn, vn, wn, tn = _np(o, *env.get_state())
        for i in range(n):
            _assert_reset(orc, off + i, s // horizon, on[i], qn[i], vn[i], wn[i], tn[i], f"{path}, step {s}", arm_atol)
    if path == "ur5e":
        assert float(np.abs(qn[:, 6]).max()) == 0.0  # the inert seventh slot
    env.close()
