"""Contact record (usim_set_contact_record / usim_get_contact_forces): position, frame and constraint force of every contact,
against the float64 oracle, against the probe wrench the kernel reports, and its opt-in contract (off changes nothing).

Force tolerance (contact_util.contact_parity): per env-step, the largest |df_c| over max(1 N, sum_c f_n,c); the bounds are <= 4x the
maxima measured on a B200 by scripts/contact_force_report.py (profiles/contact_force_parity.json).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import CC_TRACK
from contact_util import PROBE_GEOM, contact_parity, pair_friction

pytestmark = pytest.mark.gpu

# Measured maxima (B200, profiles/contact_force_parity.json): soft pos 4.4e-7 m, frame 8.7e-5, force_rel 1.1e-5; rigid pos 1.9e-7 m,
# frame 0 (the table normal), force_rel 3.7e-4.  The frame error is that of a probe-particle normal: the direction between two closest
# points a few millimetres apart, computed from metre-scale fp32 positions.
TOL = {True: dict(pos=1e-5, frame=3e-4, force_rel=4e-5), False: dict(pos=1e-5, frame=3e-4, force_rel=1.4e-3)}
MIN_CONTACTS = {True: 1000, False: 100}


def _make(n, **kw):
    from rui_b200.env import BatchedUltrasound
    opts = dict(device=0, controller_configs=CC_TRACK, control_freq=500, horizon=1000, torso_solref_randomization=True,
                initial_probe_pos_randomization=True)
    opts.update(kw)
    return BatchedUltrasound(n, **opts)


@pytest.mark.parametrize("soft", [True, False], ids=["soft", "rigid"])
def test_contact_record_matches_oracle_on_identical_states(O, soft):
    r = contact_parity(O, soft)
    assert r["contacts"] > MIN_CONTACTS[soft], r
    assert r["list_mismatch"] <= r["env_steps"] // 20, r
    bad = {k: (r[k], v) for k, v in TOL[soft].items() if not r[k] <= v}
    assert not bad, f"measured > tolerance: {bad} ({r})"


def _probe_sum(frame, force, g2):
    """sum over the contacts whose geom2 is the probe of frame^T force (the world force on the probe); padded rows are zero"""
    world = torch.einsum("ncij,nci->ncj", frame, force)
    return (world * (g2 == PROBE_GEOM).unsqueeze(-1)).sum(1), world.norm(dim=-1).sum(1)


def _check_identity(env):
    ncon, g1, g2, _ = env.contacts()
    pos, frame, force = env.contact_forces()
    s, scale = _probe_sum(frame, force, g2)
    cfrc = env.diag()[:, 0:3]
    err = (s - cfrc).abs().max(1).values
    assert bool((err <= 2e-5 * scale + 1e-6).all()), float((err / (scale + 1e-6)).max())
    return ncon, g1, g2, pos, frame, force


def test_probe_contact_forces_add_up_to_the_probe_wrench():
    """4096 envs, 300 auto-reset steps with a short horizon (resets every step somewhere, prepare launches running alongside):
    the forces on the probe add up to cfrc_ext (diag[0:3]) to fp32 reordering round-off."""
    n = 4096
    env = _make(n, horizon=60, seed=7, record_contacts=True)
    env.reset()
    gen = torch.Generator(device=env.device).manual_seed(1)
    touched = 0
    for s in range(300):
        env.step(torch.rand(n, 6, device=env.device, generator=gen))
        if s % 10 == 0:
            ncon, g1, g2, *_ = _check_identity(env)
            touched += int(((g2 == PROBE_GEOM) & (g1 >= 4)).any(1).sum())
    assert touched > 0, touched
    env.close()


def test_contact_forces_stay_in_the_friction_cone_and_padding_is_zero():
    """f_n >= 0 and |f_t| <= mu f_n (mu: the pair's friction, the kernel's), rows at or beyond ncon zero; after a reset the probe
    identity holds for the reset state's forward pass."""
    from rui_b200.abi import MAX_CONTACTS
    n = 1024
    env = _make(n, horizon=80, seed=11, record_contacts=True)
    env.reset()
    _check_identity(env)
    gen = torch.Generator(device=env.device).manual_seed(2)
    fmax = 0.0
    for s in range(120):
        env.step(torch.rand(n, 6, device=env.device, generator=gen))
        if s % 8:
            continue
        ncon, g1, g2, pos, frame, force = _check_identity(env)
        live = torch.arange(MAX_CONTACTS, device=env.device).unsqueeze(0) < ncon.unsqueeze(1)
        for x in (pos, frame, force):
            assert bool((x[~live] == 0).all())
        mu = torch.as_tensor(pair_friction(env.packed, g1.cpu().numpy(), g2.cpu().numpy()), device=env.device, dtype=torch.float32)
        fn, ft = force[..., 0], force[..., 1:].norm(dim=-1)
        fmax = max(fmax, float(fn[live].max()) if bool(live.any()) else 0.0)
        assert bool((fn[live] >= -1e-6).all()), float(fn[live].min())
        assert bool((ft[live] <= mu[live] * fn[live] * (1 + 1e-4) + 1e-5).all())
        # frames are orthonormal, normal first
        eye = torch.eye(3, device=env.device)
        assert float((frame[live] @ frame[live].transpose(-1, -2) - eye).abs().max()) < 1e-5
    assert fmax > 0.1
    env.reset()
    _check_identity(env)
    env.close()


def test_diverged_env_records_zero_forces():
    """an env whose solve goes non-finite reports zero forces in the record, as it reports a zero probe wrench"""
    env = _make(16, seed=2, record_contacts=True)
    env.reset()
    q, v, w, t = env.get_state()
    v[3, 20] = float("nan")  # one slider velocity of env 3
    v[7, 2] = float("inf")   # one arm joint velocity of env 7
    env.set_state(q, v, w, t)
    _, _, d, _ = env.step(torch.full((16, 6), 0.5), auto_reset=False)
    assert d.tolist() == [0, 0, 0, 1, 0, 0, 0, 1] + [0] * 8
    ncon, g1, g2, pos, frame, force = _check_identity(env)
    assert bool((force[[3, 7]] == 0).all())
    assert bool(torch.isfinite(force).all()) and float(force[:, :, 0].sum()) > 0
    env.close()


def _outputs(env, o, r, d, t):
    return [x.clone() for x in (o, r, d, t)] + list(env.get_state()) + [env.diag()]


def test_recording_off_or_switched_on_changes_no_output():
    """Same seed, 1024 envs, 200 auto-reset steps: an env that never records, one recording from the start and one switched on
    at step 100 return bitwise identical obs, reward, done, terminal obs, state and diagnostics."""
    n = 1024
    envs = [_make(n, horizon=50, seed=4, record_contacts=rec) for rec in (False, True, False)]
    for e in envs:
        e.reset()
    gen = torch.Generator(device=envs[0].device).manual_seed(5)
    for s in range(200):
        if s == 100:
            envs[2].set_contact_record(True)
        a = torch.rand(n, 6, device=envs[0].device, generator=gen)
        outs = [_outputs(e, *e.step(a)) for e in envs]
        for k, ref in enumerate(outs[0]):
            for o in outs[1:]:
                assert torch.equal(ref, o[k]), (s, k)
    _check_identity(envs[1])
    _check_identity(envs[2])
    for e in envs:
        e.close()


def test_contact_force_api():
    """the getter fails before recording is on (and until every env has run with it), accepts NULL outputs; the single-env
    API's get_contacts() names the pairs check_contact() sees."""
    from rui_b200 import _lib
    from rui_b200.env import make
    env = _make(8, seed=3)
    env.reset()
    with pytest.raises(_lib.UsimError, match="never enabled"):
        env.contact_forces()
    env.set_contact_record(True)
    with pytest.raises(_lib.UsimError, match="since contact recording was enabled"):
        env.contact_forces()
    mask = torch.zeros(8, dtype=torch.uint8)
    mask[0] = 1
    env.reset(mask)
    with pytest.raises(_lib.UsimError):
        env.contact_forces()  # a masked reset leaves the other envs' records behind
    env.step(torch.full((8, 6), 0.5))
    pos, frame, force = env.contact_forces()
    f2 = torch.empty_like(force)
    stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
    _lib.check(_lib.lib().usim_get_contact_forces(env._h, None, None, C.c_void_p(f2.data_ptr()), stream))
    _lib.check(_lib.lib().usim_get_contact_forces(env._h, None, None, None, stream))
    assert torch.equal(f2, force)
    env.set_contact_record(False)
    with pytest.raises(_lib.UsimError):
        env.contact_forces()  # the record no longer follows the contact list
    env.close()

    u = make("Ultrasound", robots="Panda", controller_configs=CC_TRACK, control_freq=500, horizon=200, seed=2)
    u.reset()
    seen = 0
    for s in range(150):
        u.step(np.array([0.5, 0.5, 0.0, 0.5, 0.5, 0.5]))
        cs = u.get_contacts()
        ncon = int(u.core.contacts()[0][0])
        assert len(cs) == ncon
        for c in cs:
            assert u.check_contact(c["geom1"], c["geom2"])
            assert c["pos"].shape == (3,) and c["frame"].shape == (3, 3) and c["force"].shape == (3,) and c["force"][0] >= -1e-6
        seen += len(cs)
        if u.done:
            break
    assert seen > 0
    u.close()
