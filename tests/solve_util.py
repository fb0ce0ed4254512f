"""The device's constraint solve on identical inputs, judged by the float64 oracle evaluated AT the device's qacc.

Both sides get the same float32-representable states, taken along oracle trajectories (as contact_util.contact_parity does); the
device runs one step (auto_reset off, contact record on), the oracle runs the forward pass of that state with the device's joint
torques (diag[13:20]) and evaluates its problem at the device's qacc (the warm-start row the kernel stores, oracle_evaluate).  What
does not depend on convergence -- gradient, cost, forces, probe wrench, F/T torque -- is then compared at the same qacc, so only
fp32 evaluation error remains; convergence is judged by the device's own stopping rule, |grad| <= tol (1 + |rhs| + |Hx|), restated
in float64.

Used by tests/test_solve_identical_inputs.py (asserts the bounds) and scripts/solve_parity_report.py (measures the maxima the
bounds come from; profiles/solve_parity.json).
"""
from __future__ import annotations

import dataclasses
import functools

import numpy as np
import torch

from conftest import CC_FIXED, CC_TRACK
from rui_b200 import abi

KW = dict(torso_solref_randomization=True, initial_probe_pos_randomization=True, control_freq=500, horizon=1000)
DEFAULT = dict(solver_iterations=40, solver_tolerance=3e-5, precond_rebuilds=8)  # the library's defaults (precond_rebuilds 0 = 8)
CAPS = (1, 2, 3, 5)
# solver knobs of the knob test, by name; "default" is the shipped configuration
KNOBS = {"default": {}, **{f"cap{k}": dict(solver_iterations=k) for k in CAPS},
         "tol3e-5": dict(solver_iterations=200, solver_tolerance=3e-5), "tol3e-6": dict(solver_iterations=200, solver_tolerance=3e-6),
         "rebuilds1": dict(precond_rebuilds=1), "rebuilds40": dict(precond_rebuilds=40)}
PROBE_GEOM = 2


def scene(name):
    """(scene parameters, controller) of a named scene"""
    from rui_b200.model import SceneParams, cylinder_torso_params, ur5e_params
    return {"soft": (SceneParams(), CC_TRACK), "rigid": (SceneParams(soft_torso=False), CC_FIXED),
            "cylinder": (cylinder_torso_params(), CC_TRACK), "ur5e": (ur5e_params(), CC_TRACK),
            "rigid_ur5e": (ur5e_params(SceneParams(soft_torso=False)), CC_FIXED)}[name]


def knob_values(knobs):
    return {**DEFAULT, **knobs}


def make_env(params, cc, n, seed, knobs=None):
    from rui_b200.env import BatchedUltrasound
    return BatchedUltrasound(n, device=0, soft_torso=params.soft_torso, controller_configs=cc, scene_params=params, record_contacts=True,
                             seed=seed, **KW, **(knobs or {}))


def make_oracle(O, pk, cc, seed, i):
    e = O.OracleEnv(pk, abi.make_config(1, cc, seed=seed, **KW), i)
    e.reset()
    return e


@functools.lru_cache(maxsize=None)
def trajectory_batches(O, name, n=4, seed=5):
    """float32 states (q, v, w, t) and the actions of the next step, along n oracle trajectories started from the device's reset.
    Tracking scenes: 40 steps of random gains, every 4th state.  Rigid: fixed gains pressing the probe onto the table for 250 steps,
    then random deltas; every 10th state from step 150 (the probe reaches the table near step 220)."""
    params, cc = scene(name)
    env = make_env(params, cc, n, seed)
    env.reset()
    q, v, w, t = [x.cpu().numpy().astype(np.float64) for x in env.get_state()]
    orcs = [make_oracle(O, env.packed, cc, seed, i) for i in range(n)]
    for i in range(n):
        orcs[i].set_state(q[i], v[i], w[i], t[i])
    env.close()
    rng = np.random.default_rng(3)
    rigid = not params.soft_torso
    steps, first, every = (300, 150, 10) if rigid else (40, 0, 4)
    out = []
    for s in range(steps):
        if rigid:
            a = np.zeros((n, 6)) if s < 250 else rng.uniform(-1, 1, size=(n, 6))
            if s < 250:
                a[:, 2] = -1
        else:
            a = rng.uniform(0, 1, size=(n, 6))
        if s >= first and s % every == 0:
            st = [o.get_state() for o in orcs]
            out.append(tuple(np.array([x[k] for x in st], dtype=np.float32) for k in range(4)) + (a.astype(np.float32),))
        for i in range(n):
            orcs[i].step(a[i])
    return out


def device_step(env, batch):
    """set the batch's state, run one step; returns what the comparison needs, as float64 numpy"""
    q, v, w, t, a = batch
    env.set_state(q, v, w, t)
    env.step(torch.as_tensor(a), auto_reset=False)
    ncon, g1, g2, _ = [x.cpu().numpy() for x in env.contacts()]
    _, frame, force = [x.cpu().numpy().astype(np.float64) for x in env.contact_forces()]
    return dict(qacc=env.get_state()[2].cpu().numpy().astype(np.float64), diag=env.diag().cpu().numpy().astype(np.float64),
                ncon=ncon, g1=g1, g2=g2, force=force)


def compare(orc, dev, i, knobs, opt):
    """One env of one device step against the oracle (forward already run on the same state): a flat record of the metrics."""
    kv = knob_values(knobs)
    d = dev["diag"][i]
    x = dev["qacc"][i]
    ev = orc.evaluate(x)
    c = orc.contacts()
    k = int(dev["ncon"][i])
    got = list(zip(dev["g1"][i, :k].tolist(), dev["g2"][i, :k].tolist()))
    list_ok = got == list(zip(c["geom1"].tolist(), c["geom2"].tolist()))
    scale = 1.0 + ev["rhs_norm"] + ev["hx_norm"]
    fsum = max(1.0, float(c["force"][:, 0].sum()) if k else 0.0)
    xo = opt["qacc"]
    rec = dict(iters=int(d[20]), cap=kv["solver_iterations"], tol=kv["solver_tolerance"], rebuilds=int(d[24]),
               max_rebuilds=kv["precond_rebuilds"], list_ok=list_ok, ncon=k, nefc_dev=int(d[23]), nefc=ev["nefc"],
               nlim=int((ev["efc_type"] == 1).sum()), finite=bool(np.isfinite(x).all() and np.isfinite(d).all()),
               gnorm=ev["gnorm"], scale=scale, diag_gnorm=float(d[21]), rule_dev=float(d[21]) / (kv["solver_tolerance"] * scale),
               # |diag[21] - |grad|_64| and how far |grad|_64 is past the stopping rule, both in units of the rule's scale
               gnorm_err=abs(float(d[21]) - ev["gnorm"]) / scale, rule_excess=(ev["gnorm"] - kv["solver_tolerance"] * scale) / scale,
               cost=ev["cost"], cost_opt=opt["cost"], gap_rel=(ev["cost"] - opt["cost"]) / (1.0 + abs(opt["cost"])),
               qacc_dist=float(np.abs(x - xo).max() / (1.0 + np.abs(xo).max())),
               cfrc_rel=float(np.abs(d[0:3] - ev["cfrc"]).max() / fsum),
               ft_rel=float(np.abs(d[3:6] - ev["ft_torque"]).max() / max(0.1, float(np.abs(ev["ft_torque"]).max()))),
               force_rel=0.0, x=x, grad=ev["grad"])
    if list_ok and k:
        rec["force_rel"] = float(np.linalg.norm(dev["force"][i, :k] - ev["contact_force"], axis=1).max() / fsum)
    return rec


def run(O, params, cc, batches, knob_names, seed=5):
    """Every batch through one fresh handle per knob set (identical histories, so the warm starts agree), every env against the
    oracle; returns {knob name: [record per (batch, env)]}."""
    n = batches[0][0].shape[0]
    envs = {kn: make_env(params, cc, n, seed, KNOBS[kn]) for kn in knob_names}
    for e in envs.values():
        e.reset()
    pk = next(iter(envs.values())).packed
    orcs = [make_oracle(O, pk, cc, seed, i) for i in range(n)]
    out = {kn: [] for kn in knob_names}
    for b in batches:
        devs = {kn: device_step(e, b) for kn, e in envs.items()}
        tau = next(iter(devs.values()))["diag"][:, 13:20]
        for kn, dv in devs.items():
            assert np.array_equal(dv["diag"][:, 13:20], tau), "the knobs changed the joint torques"
        for i in range(n):
            orcs[i].set_state(*(x[i].astype(np.float64) for x in b[:4]))
            orcs[i].forward(tau[i])
            opt = orcs[i].evaluate(orcs[i].qacc)
            opt["qacc"] = orcs[i].qacc
            for kn, dv in devs.items():
                out[kn].append(compare(orcs[i], dv, i, KNOBS[kn], opt))
    for e in envs.values():
        e.close()
    return out


def line_search_ratios(recs_k, recs_k1):
    """Cap k and cap k + 1 from the same state: x_{k+1} - x_k is the step of line search k + 1, which stops where the directional
    derivative has dropped below LS_TOL = 0.03 of its value at the start.  Returns |grad(x_{k+1}) . d| / |grad(x_k) . d| for every
    env where both runs hit their cap (the step exists)."""
    out = []
    for a, b in zip(recs_k, recs_k1):
        if a["iters"] != a["cap"] or b["iters"] != b["cap"]:
            continue
        dx = b["x"] - a["x"]
        g0 = abs(float(a["grad"] @ dx))
        if g0 > 0:
            out.append(abs(float(b["grad"] @ dx)) / g0)
    return out


def limit_cases(nj):
    """(joints, side, delta, direction) of the joint-limit cases: each real joint past its lower (side 0) and upper (side 1) limit by
    1e-4 and 2e-2 rad, moving into (+1) or out of (-1) the limit; and joints 1 and 3 both past their lower limits."""
    cases = [((j,), side, dl, dr) for j in range(nj) for side in (0, 1) for dl in (1e-4, 2e-2) for dr in (1, -1)]
    return cases + [((1, 3), 0, 2e-2, dr) for dr in (1, -1)]


def _put_past(q, v, jr, case, move_limit):
    """state (and joint ranges) of one case: q_j past the limit by delta, qdot_j = 0.5 rad/s into or out of it.  move_limit: the limit
    moves to the joint (the probe stays where it is) instead of the joint to the limit"""
    joints, side, dl, dr = case
    q, v, jr = q.copy(), v.copy(), [list(r) for r in jr]
    sg = 1.0 if side == 0 else -1.0  # lower limit: q = lo - delta, into it = negative velocity
    for j in joints:
        if move_limit:
            jr[j][side] = q[j] + sg * dl
        else:
            q[j] = jr[j][side] - sg * dl
        v[j] = -sg * 0.5 * dr
    return q, v, tuple(tuple(r) for r in jr)


def _soft_limit_groups(q, v, joint_range, nj):
    """Soft-scene limit cases, grouped by model (the limits move, the probe stays in contact): (joint ranges, [(q, v, case)]).
    delta 1e-4: one model per side with every limit 1e-4 past its joint; the env of joint j moves the other joints 2e-4 rad back
    inside (a tenth of a millimetre at the probe).  delta 2e-2: one model per joint, the side alternating with the joint; and joints 1
    and 3 both past their lower limits.  Both directions of every case."""
    groups = []
    for side in (0, 1):
        sg = 1.0 if side == 0 else -1.0
        jr = tuple(tuple(q[j] + sg * 1e-4 if s == side else r[s] for s in (0, 1)) if j < nj else tuple(r)
                   for j, r in enumerate(joint_range))
        cases = []
        for j in range(nj):
            for dr in (1, -1):
                qq, vv = q.copy(), v.copy()
                for k in range(nj):
                    if k != j:
                        qq[k] += sg * 2e-4
                vv[j] = -sg * 0.5 * dr
                cases.append((qq, vv, ((j,), side, 1e-4, dr)))
        groups.append((jr, cases))
    for joints, side in [((j,), j % 2) for j in range(nj)] + [((1, 3), 0)]:
        cases = []
        for dr in (1, -1):
            qq, vv, jr = _put_past(q, v, joint_range, (joints, side, 2e-2, dr), move_limit=True)
            cases.append((qq, vv, (joints, side, 2e-2, dr)))
        groups.append((jr, cases))
    return groups


def limit_records(O, robot):
    """Joint-limit rows, for robot "panda" or "ur5e".
    Soft box torso, probe pressing on it: the state of the env with the most probe contacts at the end of a tracking trajectory; the
    LIMITS move past the joints (_soft_limit_groups), so the contacts stay.  Rigid scene, probe in the
    air (no contacts, so the rebuild-every-iteration rule of the rigid scene stays off): the state after a reset with every case in one
    batch, the joint moved past the limit; run at the default knobs and at caps 1, 2, 3.
    Returns {"soft": [records], "rigid": {knob: [records]}}; every record carries its case."""
    name = "ur5e" if robot == "ur5e" else "soft"
    params, cc = scene(name)
    nj = len(params.joint_range)
    batches = trajectory_batches(O, name)
    q, v, w, t, _ = batches[-1]
    ref = make_env(params, cc, 4, 5)
    ref.reset()
    dev = device_step(ref, batches[-1])
    ref.close()
    best = int(np.argmax([(dev["g2"][i, :dev["ncon"][i]] == PROBE_GEOM).sum() for i in range(4)]))
    base = [x[best].astype(np.float64) for x in (q, v, w, t)]
    out = {"soft": [], "rigid": {}}
    for jr, group in _soft_limit_groups(base[0], base[1], params.joint_range, nj):
        qs, vs, cases = zip(*group)
        m = len(cases)
        bt = (np.array(qs, np.float32), np.array(vs, np.float32), np.array([base[2]] * m, np.float32),
              np.array([base[3]] * m, np.float32), np.full((m, 6), 0.5, np.float32))
        recs = run(O, dataclasses.replace(params, joint_range=jr), cc, [bt], ["default"])["default"]
        for r, c in zip(recs, cases):
            r["case"] = c
        out["soft"] += recs
    # rigid, probe in the air
    rparams, rcc = scene("rigid_ur5e" if robot == "ur5e" else "rigid")
    env = make_env(rparams, rcc, 1, 5)
    env.reset()
    q0, v0, w0, t0 = [x[0].cpu().numpy().astype(np.float64) for x in env.get_state()]
    env.close()
    cases = limit_cases(nj)
    qs, vs = zip(*[_put_past(q0, v0, rparams.joint_range, c, move_limit=False)[:2] for c in cases])
    m = len(cases)
    b = (np.array(qs, np.float32), np.array(vs, np.float32), np.array([w0] * m, np.float32), np.array([t0] * m, np.float32),
         np.zeros((m, 6), np.float32))
    out["rigid"] = run(O, rparams, rcc, [b], ["default", "cap1", "cap2", "cap3"])
    for recs in out["rigid"].values():
        for r, c in zip(recs, cases):
            r["case"] = c
    return out


def cap_increase(by_knob):
    """largest relative increase of the float64 cost at the device qacc from one cap to the next (caps 1, 2, 3, 5, then the default)"""
    names = [f"cap{k}" for k in CAPS if f"cap{k}" in by_knob] + ["default"]
    worst = -np.inf
    for lo, hi in zip(names, names[1:]):
        for a, b in zip(by_knob[lo], by_knob[hi]):
            worst = max(worst, (b["cost"] - a["cost"]) / (1.0 + abs(a["cost"])))
    return float(worst)


def stats(recs):
    """Maxima of the metrics over records.  Env-steps whose contact lists differ (a pair on the detection threshold: the two sides
    solve different problems) are counted and left out; the stopping rule is checked where the solve stopped before its cap."""
    ok = [r for r in recs if r["list_ok"]]
    conv = [r for r in ok if r["iters"] < r["cap"]]
    mx = lambda k, rs=ok: float(max((r[k] for r in rs), default=0.0))
    return dict(env_steps=len(recs), list_mismatch=len(recs) - len(ok), contacts=sum(r["ncon"] for r in ok),
                capped=sum(r["iters"] >= r["cap"] for r in ok), nefc_mismatch=sum(r["nefc_dev"] != r["nefc"] for r in ok),
                finite=all(r["finite"] for r in recs), over_cap=sum(r["iters"] > r["cap"] for r in recs),
                over_rebuilds=sum(r["rebuilds"] > r["max_rebuilds"] for r in recs),
                gnorm_err=mx("gnorm_err"), rule_excess=mx("rule_excess", conv) if conv else None,
                rule_dev=mx("rule_dev", conv) if conv else None, gap_rel=mx("gap_rel", conv) if conv else None,
                cost_below=float(min((r["gap_rel"] for r in ok), default=0.0)), force_rel=mx("force_rel"), cfrc_rel=mx("cfrc_rel"),
                ft_rel=mx("ft_rel"), qacc_dist_median=float(np.median([r["qacc_dist"] for r in ok])) if ok else 0.0,
                qacc_dist=mx("qacc_dist"), mean_iters=float(np.mean([r["iters"] for r in ok])) if ok else 0.0,
                worst=_brief(max(conv, key=lambda r: r["rule_excess"])) if conv else None)


def _brief(r):
    return {k: (list(v) if isinstance(v, tuple) else v) for k, v in r.items() if k not in ("x", "grad")}


def knob_stats(by_knob):
    """the knob comparisons of one scene: cost against the cap, the line searches, tolerance and rebuild settings"""
    out = dict(cap_increase=cap_increase(by_knob))
    ls = line_search_ratios(by_knob["cap1"], by_knob["cap2"]) + line_search_ratios(by_knob["cap2"], by_knob["cap3"])
    out["line_search_ratio"] = float(max(ls, default=0.0))
    out["line_search_ratio_p90"] = float(np.quantile(ls, 0.9)) if ls else 0.0
    out["line_search_n"] = len(ls)
    if "tol3e-5" in by_knob:
        for kn in ("tol3e-5", "tol3e-6"):
            out[kn + "_median_dist"] = stats(by_knob[kn])["qacc_dist_median"]
        out["rebuilds_dist"] = float(max(abs(a["x"] - b["x"]).max() / (1.0 + abs(a["x"]).max())
                                         for a, b in zip(by_knob["rebuilds1"], by_knob["rebuilds40"])))
    return out
