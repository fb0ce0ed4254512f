"""The oracle's observation at a forward pass (forward_util.oracle_observation): the reference the device's usim_forward is judged
against (tests/test_forward.py), pinned on the observations the oracle's own reset and step write.  CPU only."""
import numpy as np
import pytest

import forward_util as fu
import solve_util as su
from rui_b200 import abi
from rui_b200.env import packed_model

SCENES = ["soft", "rigid", "cylinder", "ur5e"]


def _oracle(O, name, seed=5):
    params, cc = su.scene(name)
    return O.OracleEnv(packed_model(params.soft_torso, params), abi.make_config(1, cc, seed=seed, **su.KW), 0), cc


def _action(rng, orc, cc):
    return rng.uniform(0, 1, size=orc.adim) if cc["impedance_mode"] == "tracking" else rng.uniform(-1, 1, size=orc.adim)


@pytest.mark.parametrize("name", SCENES)
def test_observation_after_reset_is_the_reset_observation(O, name):
    """a reset ends with sim.forward() at ctrl = 0: forwarding again at the reset state gives the reset's observation, and the
    state is left as it was"""
    orc, _ = _oracle(O, name)
    obs0 = orc.reset()
    state = orc.get_state()
    orc.forward(np.zeros(7))
    np.testing.assert_allclose(fu.oracle_observation(O, orc), obs0, rtol=0, atol=1e-12)
    for a, b in zip(orc.get_state(), state):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name", SCENES)
def test_observation_reproduces_the_step_observation(O, name):
    """Mid-episode (one physics substep per step).  A step's observation carries the hand velocity of the step's kinematics, at the
    joint positions q0 before it, times the velocity v1 after it; its task channels are the record t0 before the step, and its pose
    channels the grip site at q0.  A forward at (q0, v1, t0) gives exactly those channels (6-18), so the hand Jacobian, derived from
    the grip-site Jacobian, is the oracle's own.  Channels 0-5 are the forward's probe wrench and F/T torque; the forward leaves the
    state unchanged."""
    orc, cc = _oracle(O, name)
    orc.reset()
    rng = np.random.default_rng(1)
    for _ in range(12):
        orc.step(_action(rng, orc, cc))
    q0, _, w0, t0 = orc.get_state()
    obs1, _, _ = orc.step(_action(rng, orc, cc))
    _, v1, _, _ = orc.get_state()
    assert np.abs(v1[:7]).max() > 1e-3, "the arm is at rest: the hand velocity would not be checked"
    orc.set_state(q0, v1, w0, t0)
    orc.forward(rng.uniform(-1, 1, size=7) * np.asarray(orc.packed.model.g_ctrl_range))
    obs = fu.oracle_observation(O, orc)
    np.testing.assert_allclose(obs[6:19], obs1[6:19], rtol=0, atol=1e-12)
    np.testing.assert_allclose(obs[0:6], orc.diag()[0:6], rtol=0, atol=0)
    for a, b in zip(orc.get_state(), (q0, v1, w0, t0)):
        assert np.array_equal(a, b)
