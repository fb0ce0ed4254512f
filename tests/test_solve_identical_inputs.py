"""The constraint solve (solve_kernel) on identical inputs, judged by the float64 oracle evaluated at the device's own qacc.

tests/solve_util.py sets the same float32 states on both sides, runs one device step and evaluates the oracle's problem of that state
at the qacc the device returned.  Gradient, cost, forces, probe wrench and F/T torque are thus compared at the SAME qacc: only fp32
evaluation error remains, however far the solve stopped from the optimum.  Convergence is judged by the device's own stopping rule,
|grad| <= tol (1 + |rhs| + |Hx|), restated in float64.

Every bound is <= 4x the maximum measured on a B200 by scripts/solve_parity_report.py (profiles/solve_parity.json); the measured
maximum is named beside each.
"""
import numpy as np
import pytest

import solve_util as su

pytestmark = pytest.mark.gpu

# Bounds per group of runs (profiles/solve_parity.json "groups"; the measured maximum in the comment, the bound <= 4x it):
#  gnorm_err  |diag[21] - |grad|_64| / (1 + |rhs| + |Hx|): the fp32 evaluation error of the gradient, in units of the stopping rule's
#             scale.  The float64 gradient of a converged solve may pass tol * scale by at most this.  It is largest where fp32 input
#             data set the problem: in the rigid scene the probe-table depth (a few mm, from metre-scale fp32 positions) times a stiff
#             contact, and at the UR5e's +-2 pi joint limits the fp32 spacing of q and of the limit (5e-7 rad) times the limit stiffness.
#  gap_rel    (cost(device qacc) - cost(oracle optimum)) / (1 + |cost|), float64, solves that stopped before their cap.
#  force_rel  per contact |df| / max(1 N, sum f_n);  cfrc_rel: diag[0:3] likewise;  ft_rel: diag[3:6] over max(0.1 N m, |T|).
#             Zero where the probe touches nothing.
BOUNDS = {  # gnorm_err, gap_rel, force_rel, cfrc_rel, ft_rel
    "soft": (2.2e-4, 1.3e-8, 3.5e-5, 1.0e-4, 6.8e-4),             # 5.7e-5, 3.3e-9, 8.8e-6, 2.7e-5, 1.7e-4
    "rigid": (1.8e-3, 1.5e-7, 7.6e-3, 5.4e-3, 5.4e-3),            # 4.7e-4, 3.8e-8, 1.9e-3, 1.35e-3, 1.35e-3
    "cylinder": (1.6e-4, 5.0e-8, 7.3e-5, 1.3e-4, 7.2e-4),         # 4.0e-5, 1.26e-8, 1.85e-5, 3.3e-5, 1.8e-4
    "ur5e": (8.5e-5, 2.8e-8, 2.7e-5, 7.5e-5, 3.8e-4),             # 2.15e-5, 7.2e-9, 6.9e-6, 1.9e-5, 9.7e-5
    "limit_panda_soft": (1.1e-4, 1.2e-7, 4.6e-5, 9.6e-5, 3.7e-4),  # 2.8e-5, 3.0e-8, 1.17e-5, 2.4e-5, 9.4e-5
    "limit_panda_rigid": (9.6e-5, 3.6e-8, 0.0, 0.0, 6.1e-5),      # 2.4e-5, 9.0e-9, 0, 0, 1.54e-5
    "limit_ur5e_soft": (1.1e-4, 2.8e-8, 4.3e-5, 1.0e-4, 3.2e-4),   # 3.0e-5, 7.2e-9, 1.1e-5, 2.5e-5, 8.2e-5
    "limit_ur5e_rigid": (1.0e-2, 5.6e-6, 0.0, 0.0, 2.6e-5),        # 2.6e-3, 1.4e-6, 0, 0, 6.6e-6
}
# diag[21] / (tol (1 + |rhs| + |Hx|)_64) of a converged solve: the device's own rule, with the norms of its scale in float64 instead
# of fp32; measured max 0.997
RULE_DEV = 1.01
# float64 round-off of a cost difference, relative (not measured: the measured cost gaps are all >= 2.5e-14 and the cost never rose
# from one cap to the next)
COST_ROUNDOFF = 1e-12
# line search k+1 stops where |phi'| has dropped to LS_TOL = 0.03 of its value at the start: the 90th percentile of
# |grad(x_k+1).d| / |grad(x_k).d| over caps 1->2 and 2->3 (profiles/solve_parity.json "knobs" and "limits": line_search_ratio_p90)
LS_P90 = {"soft": 0.058, "rigid": 0.098, "panda": 1.3e-4, "ur5e": 9.5e-4}  # 0.0145, 0.0247, 3.5e-5, 2.4e-4
# median qacc distance to the oracle's optimum, relative: the fp32 floor, the smallest median at tolerance 3e-6 (rigid, 2.75e-6)
DIST_FLOOR = 1.1e-5
# max qacc distance between precond_rebuilds 1 and 40, relative (the rigid scene rebuilds every iteration either way); 2.4e-4, 0
REBUILD_DIST = {"soft": 9.6e-4, "rigid": 0.0}
MIN_CONTACTS = {"soft": 1000, "rigid": 10, "cylinder": 1000, "ur5e": 1000}

_CACHE = {}


def _records(O, name):
    if name not in _CACHE:
        params, cc = su.scene(name)
        knobs = list(su.KNOBS) if name in ("soft", "rigid") else ["default"]
        _CACHE[name] = su.run(O, params, cc, su.trajectory_batches(O, name), knobs)
    return _CACHE[name]


def _limits(O, robot):
    key = "limits_" + robot
    if key not in _CACHE:
        _CACHE[key] = su.limit_records(O, robot)
    return _CACHE[key]


def _ctx(what, r):
    return what, {k: v for k, v in r.items() if k not in ("x", "grad")}


def _check_residual(recs, what, group):
    """every env-step has the oracle's contact list, nefc and a finite solution within the cap; where the solve stopped before its
    cap, the device's rule held and the float64 gradient meets it up to the fp32 evaluation error; diag[21] is |grad|_64 up to that
    error; the cost is never below the optimum and, for a converged solve, above it by at most what the tolerance leaves"""
    gn, gap = BOUNDS[group][:2]
    for r in recs:
        ctx = _ctx(what, r)
        assert r["list_ok"] and r["nefc_dev"] == r["nefc"], ctx
        assert r["finite"] and r["iters"] <= r["cap"], ctx
        assert r["gnorm_err"] <= gn and r["gap_rel"] >= -COST_ROUNDOFF, ctx
        if r["iters"] < r["cap"]:
            assert r["rule_dev"] <= RULE_DEV and r["gnorm"] <= (r["tol"] + gn) * r["scale"] and r["gap_rel"] <= gap, ctx


def _check_forces(recs, what, group):
    f, cf, ft = BOUNDS[group][2:]
    for r in recs:
        assert r["force_rel"] <= f and r["cfrc_rel"] <= cf and r["ft_rel"] <= ft, _ctx(what, r)


def _line_search_p90(by):
    ls = su.line_search_ratios(by["cap1"], by["cap2"]) + su.line_search_ratios(by["cap2"], by["cap3"])
    return len(ls), float(np.quantile(ls, 0.9)) if ls else 0.0


@pytest.mark.parametrize("name", ["soft", "rigid", "cylinder", "ur5e"])
def test_residual_at_device_qacc(O, name):
    recs = _records(O, name)["default"]
    _check_residual(recs, name, name)
    assert sum(r["ncon"] for r in recs) >= MIN_CONTACTS[name]
    assert all(r["iters"] < r["cap"] for r in recs), "a solve at the default knobs hit the iteration cap (none did, measured)"


@pytest.mark.parametrize("name", ["soft", "rigid", "cylinder", "ur5e"])
def test_forces_and_probe_wrench_at_device_qacc(O, name):
    _check_forces(_records(O, name)["default"], name, name)


@pytest.mark.parametrize("robot", ["panda", "ur5e"])
def test_arm_joint_limit_rows(O, robot):
    """each real joint past its lower and upper limit by 1e-4 and 2e-2 rad, moving into and out of it, and two joints at once: soft box
    torso with the probe pressing on it, rigid scene with the probe in the air (no contacts: no rebuild every iteration), the latter
    also at caps 1, 2, 3.  The oracle has one limit row per joint past its limit (the UR5e's inert seventh slot never has one) and the
    device the same nefc; no solve hits the default cap (none did, measured)."""
    lr = _limits(O, robot)
    for part, by in (("soft", {"default": lr["soft"]}), ("rigid", lr["rigid"])):
        group = f"limit_{robot}_{part}"
        for kn, recs in by.items():
            _check_residual(recs, (robot, part, kn), group)
            _check_forces(recs, (robot, part, kn), group)
            for r in recs:
                assert r["nlim"] == len(r["case"][0]), _ctx((robot, part, kn), r)
        assert all(r["iters"] < r["cap"] for r in by["default"]), (robot, part, "hit the iteration cap")
    assert sum(r["ncon"] for r in lr["soft"]) >= 20 * len(lr["soft"])
    assert all(r["ncon"] == 0 for r in lr["rigid"]["default"])
    assert su.cap_increase(lr["rigid"]) <= COST_ROUNDOFF
    n, p90 = _line_search_p90(lr["rigid"])
    assert n >= 10 and p90 <= LS_P90[robot], (n, p90)


@pytest.mark.parametrize("name", ["soft", "rigid"])
def test_iteration_cap_and_solver_knobs(O, name):
    by = _records(O, name)
    # caps 1, 2, 3, 5: the cap holds, the outputs are finite, the cost does not rise with the cap, and forces, wrench and F/T torque
    # belong to the unconverged qacc (every exit of the CG loop follows a gradient evaluation of the returned iterate)
    for k in su.CAPS:
        _check_residual(by[f"cap{k}"], (name, k), name)
        _check_forces(by[f"cap{k}"], (name, k), name)
    assert su.cap_increase(by) <= COST_ROUNDOFF
    n, p90 = _line_search_p90(by)
    assert n >= 10 and p90 <= LS_P90[name], (n, p90)
    # tolerance 3e-5 and 3e-6, cap 200: the rule holds in float64; the solution moves toward the optimum or sits on the fp32 floor
    for kn in ("tol3e-5", "tol3e-6"):
        _check_residual(by[kn], (name, kn), name)
        assert all(r["iters"] < r["cap"] for r in by[kn]), (name, kn)
    d5, d6 = (su.stats(by[kn])["qacc_dist_median"] for kn in ("tol3e-5", "tol3e-6"))
    assert d6 < d5 or d6 <= DIST_FLOOR, (d5, d6)
    # preconditioner rebuilds 1 and 40: the knob caps diag[24] (the rigid scene rebuilds on every iteration with contacts: Newton);
    # both stop by the rule near the same solution
    for kn in ("rebuilds1", "rebuilds40"):
        _check_residual(by[kn], (name, kn), name)
        for r in by[kn]:
            assert r["rebuilds"] <= (r["max_rebuilds"] if name == "soft" else max(r["max_rebuilds"], r["iters"])), _ctx((name, kn), r)
    dist = max(np.abs(a["x"] - b["x"]).max() / (1 + np.abs(a["x"]).max()) for a, b in zip(by["rebuilds1"], by["rebuilds40"]))
    assert dist <= REBUILD_DIST[name], dist
