"""Contact-record parity against the float64 oracle on identical states (usim_get_contact_forces vs oracle_contacts).

Used by tests/test_contact_forces.py (asserts the stated tolerances) and scripts/contact_force_report.py (measures the maxima the
tolerances are derived from).
"""
from __future__ import annotations

import numpy as np
import torch

from conftest import CC_FIXED, CC_TRACK
from parity_util import make_oracles

PROBE_GEOM, TABLE_GEOM = 2, 1


def pair_friction(packed, g1, g2):
    """Friction coefficient of each contact (geom id arrays): the larger of the two geoms' (MuJoCo's pair rule), as the kernel uses."""
    m = packed.struct
    g1, g2 = np.asarray(g1), np.asarray(g2)
    table_probe = (g1 == TABLE_GEOM) & (g2 == PROBE_GEOM)
    part_probe = (g1 >= 4) & (g2 == PROBE_GEOM)
    return np.where(table_probe, max(m.table_friction, m.probe_friction),
                    np.where(part_probe, max(m.probe_friction, m.particle_friction), max(m.table_friction, m.particle_friction)))


def contact_parity(O, soft: bool, n: int = 4):
    """Both sides evaluate the SAME float32-representable states taken along oracle trajectories; the oracle's
    forward pass is given the device's joint torques (diag[:, 13:20]) so that both solve the same problem.  Where the contact pair
    lists agree, contact by contact: max |dpos|, max |dframe| and, per env-step, the largest |df_c| over max(1 N, sum_c f_n,c)
    (f: the frame-coordinate force on geom2, the oracle's f_n).  Soft scene: box torso, tracking OSC, 40 steps of random actions,
    every 4th checked; rigid scene: fixed-gain OSC, 250 steps pressing the probe down onto the table, then 50 random ones, every step
    checked from step 150 (one or two probe-table contacts per env)."""
    from rui_b200.env import BatchedUltrasound
    cc = CC_TRACK if soft else CC_FIXED
    kw = dict(torso_solref_randomization=True, initial_probe_pos_randomization=True, seed=5, control_freq=500, horizon=1000)
    env = BatchedUltrasound(n, device=0, soft_torso=soft, controller_configs=cc, record_contacts=True, **kw)
    env.reset()
    orcs = make_oracles(O, env, cc, soft=soft, **kw)
    rng = np.random.default_rng(3)
    steps, first, every = (40, 0, 4) if soft else (300, 150, 1)
    res = dict(pos=0.0, frame=0.0, force_rel=0.0, contacts=0, env_steps=0, list_mismatch=0, force_rel_at=None)
    for s in range(steps):
        if soft:
            a = rng.uniform(0, 1, size=(n, 6))
        else:
            a = np.zeros((n, 6)) if s < 250 else rng.uniform(-1, 1, size=(n, 6))
            if s < 250:
                a[:, 2] = -1
        for i in range(n):
            orcs[i].step(a[i])
        if s < first or s % every:
            continue
        st = [orcs[i].get_state() for i in range(n)]
        q32, v32, w32, t32 = [np.array([x[k] for x in st], dtype=np.float32) for k in range(4)]
        env.set_state(q32, v32, w32, t32)
        env.step(torch.as_tensor(a, dtype=torch.float32), auto_reset=False)  # the record belongs to the pre-step state's forward pass
        ncon, g1, g2, _ = env.contacts()
        pos, frame, force = [x.cpu().numpy().astype(np.float64) for x in env.contact_forces()]
        tau = env.diag()[:, 13:20].cpu().numpy().astype(np.float64)
        for i in range(n):
            orcs[i].set_state(q32[i].astype(np.float64), v32[i].astype(np.float64), w32[i].astype(np.float64), t32[i].astype(np.float64))
            orcs[i].forward(tau[i])
            c = orcs[i].contacts()
            k = int(ncon[i])
            res["env_steps"] += 1
            got = list(zip(g1[i, :k].tolist(), g2[i, :k].tolist()))
            want = list(zip(c["geom1"].tolist(), c["geom2"].tolist()))
            if got != want:  # a pair on the detection threshold: the solve differs, nothing to compare contact by contact
                res["list_mismatch"] += 1
                continue
            res["contacts"] += k
            if k == 0:
                continue
            res["pos"] = max(res["pos"], float(np.abs(pos[i, :k] - c["pos"]).max()))
            res["frame"] = max(res["frame"], float(np.abs(frame[i, :k] - c["frame"]).max()))
            rel = float(np.linalg.norm(force[i, :k] - c["force"], axis=1).max() / max(1.0, c["force"][:, 0].sum()))
            if rel > res["force_rel"]:
                res["force_rel"], res["force_rel_at"] = rel, (s, i)
    env.close()
    return res
