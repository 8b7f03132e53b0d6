"""GPU: the device Levenberg-Marquardt solver, step by step, against the float64 restatement of tests/lm_reference.py
built on the CPU oracle's normal equations.

  A  one step, backward error of delta = x1 - x0 against the model's damped system (independent of conditioning);
  B  one step, forward error against the model's step (bound max(1e-11, 1e-12 kappa_s)), trial cost, lambda after the
     step, and exact zeros for fixed and unobserved parameters;
  C  trajectories of max_iter = 1..6 from the same start: iterations, status, lambda, cost, both evaluation counters and
     the iterates; across a rejected step the point does not move and the next step is the model's step from the SAME
     linearisation with twice the damping;
  D  termination by gtol, ftol and xtol (with |x| the norm of the free vector).

Each fixture is a distinct path of the solver: template chain with pose elimination (small and padded, partial masks,
goldens, the sparse Schur plan and its dense alternative, more cameras than the Z kernel's window with the chunked
Cholesky); self-calibration with the points eliminated, with the poses eliminated and on the dense fallback."""
import functools

import numpy as np
import pytest

from tests import lm_reference as R
from tests.helpers import solver_env

pytestmark = pytest.mark.gpu
LAMBDAS = (1e-6, 1e-3, 1.0, 1e2)


@functools.lru_cache(maxsize=None)
def fixture(name):
    return R.FIXTURES[name]()


@functools.lru_cache(maxsize=None)
def model(name, path="block"):
    return fixture(name).model(path)


def device_runs(name, runs, env=None):
    """[(x, stats, parameter string)] of lm_solve(x0, **run) for each run, every run from the fixture's start.
    env: solver switches (PCS_LM_*), read when the problem's solver workspace is built."""
    env = env or {}
    fx = fixture(name)
    out = []
    with solver_env(**env), fx.problem() as p:
        if name == "ring32_template":
            frac = p.lm_schur_fraction()
            if "PCS_LM_SCHUR" in env:
                assert frac == 1.0
            else:
                assert 0.2 < frac < 0.85, frac
        for r in runs:
            p.set_param_string(fx.params0)
            x, st = p.lm_solve(fx.x0, **r)
            out.append((x, st, p.get_param_string()))
    return out


def _path_label(name, env):
    return f"{name} [{', '.join(f'{k}={v}' for k, v in env.items()) or 'library default'}]"


# ---- A + B: one step ---------------------------------------------------------------------------------------------------
ONE_STEP = [
    ("rig4_template", {}, LAMBDAS),
    ("rig4_template_masks", {}, LAMBDAS),
    ("ring5_fixedcam_template", {}, LAMBDAS),
    ("ccube_template", {}, LAMBDAS),
    ("ring32_template", {}, LAMBDAS),
    ("ring32_template", {"PCS_LM_SCHUR": "dense"}, (1e-3, 1.0)),
    ("dome128_template", {}, (1e-3, 1.0)),
    ("rig4_selfcal_point_masks", {}, (1e-3, 1.0, 1e2)),
    ("ccube_selfcal", {}, (1e-3, 1.0)),
    ("ring5_fixedcam_selfcal", {"PCS_LM_SELFCAL": "poses"}, (1e-3, 1.0)),
    ("ring5_fixedcam_selfcal", {"PCS_LM_SELFCAL": "dense"}, (1e-3, 1.0)),
    ("ccube_selfcal", {"PCS_LM_SELFCAL": "poses"}, (1e-3,)),
    ("ccube_selfcal", {"PCS_LM_SELFCAL": "dense"}, (1e-3,)),
]


@pytest.mark.parametrize("name,env,lambdas", ONE_STEP, ids=[f"{n}-{'-'.join(e.values()) or 'default'}" for n, e, _ in ONE_STEP])
def test_one_step_matches_the_model(name, env, lambdas):
    fx = fixture(name)
    path = "dense" if env.get("PCS_LM_SELFCAL") == "dense" else "block"
    m = model(name, path)
    x0 = fx.x0
    runs = device_runs(name, [dict(max_iter=1, lambda0=lam, ftol=0.0, xtol=0.0, gtol=0.0) for lam in lambdas], env)
    H0, _, c0 = m.linearise(x0)
    unobserved_free = np.diag(H0) == 0.0
    n_checked = 0
    for lam, (x1, st, pstr) in zip(lambdas, runs):
        delta_ref, pred, A, D, g, kappa = m.step(x0, lam)
        c1 = m.cost(x0 + delta_ref)
        rho = (c0 - c1) / pred if pred > 0.0 else -1.0
        lam1 = max(R.LAMBDA_MIN, lam * max(1.0 / 3.0, 1.0 - (2.0 * rho - 1.0) ** 3)) if rho > 0 else 2.0 * lam
        label = f"{_path_label(name, env)} lambda={lam:g}"
        assert st["iterations"] == 1 and st["status"] == 0, (label, st)
        assert np.all(np.isfinite(x1))
        # fixed entries of the parameter string never move; an unobserved free parameter has a zero step
        assert np.array_equal(pstr[~fx.unfixed], fx.params0[~fx.unfixed]), label
        assert np.array_equal(x1[unobserved_free], x0[unobserved_free]), label
        if rho <= 0.0:
            # a rejected step leaves the start point and doubles the damping
            print(f"[lm-step] {label}: model rejects (rho={rho:.3g}); device x1 == x0: {np.array_equal(x1, x0)}")
            assert np.array_equal(x1, x0), label
            assert abs(st["lambda_final"] - lam1) <= 1e-12 * lam1, (label, st["lambda_final"], lam1)
            continue
        n_checked += 1
        d_gpu = x1 - x0
        s = np.sqrt(np.diag(A))
        eta = R.backward_error(A, g, d_gpu)
        eta_floor, fwd_floor = R.subtraction_floor(A, g, d_gpu, x0, x1)
        fwd = np.linalg.norm(s * (d_gpu - delta_ref)) / np.linalg.norm(s * delta_ref)
        fwd_bound = max(1e-11, 1e-12 * kappa) + fwd_floor / np.linalg.norm(s * delta_ref)
        print(f"[lm-step] {label}: eta={eta:.2e} (bound 1e-11 + subtraction floor {eta_floor:.2e}); forward error "
              f"{fwd:.2e}, kappa_s={kappa:.2e}, ratio to 1e-12 kappa_s {fwd / (1e-12 * kappa):.3g}; rho={rho:.4f}")
        assert eta <= 1e-11 + eta_floor, (label, eta)
        assert fwd <= fwd_bound, (f"{label}: forward error {fwd:.3e} > {fwd_bound:.3e} while the backward error {eta:.2e} "
                                  "is small: the device's normal-equation blocks, not the solve, differ from the oracle's")
        assert abs(st["cost_final"] - 0.5 * c1) <= 1e-9 * 0.5 * c1, (label, st["cost_final"], 0.5 * c1)
        if abs(c0 - c1) >= 1e-6 * c0:
            assert abs(st["lambda_final"] - lam1) <= 1e-8 * lam1, (label, st["lambda_final"], lam1)
        # block path: start + trial point (full kernel); dense path: start + re-linearisation, one cost-only trial pass
        assert (st["n_eval_normal"], st["n_eval_cost"]) == ((2, 0) if path == "block" else (2, 1)), (label, st)
    assert n_checked >= 1, "every damping was rejected: the fixture checks nothing"


# ---- C: trajectories ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,lam0", R.TRAJECTORIES)
def test_trajectory_matches_the_model(name, lam0):
    fx = fixture(name)
    m = model(name)
    x0 = fx.x0
    tol = dict(ftol=0.0, xtol=0.0, gtol=0.0)
    ks = list(range(1, R.N_TRAJ + 1))
    refs = {k: m.run(x0, k, lambda0=lam0, condition=False, **tol) for k in ks}
    ref = refs[ks[-1]]
    runs = device_runs(name, [dict(max_iter=k, lambda0=lam0, **tol) for k in ks])
    # a second run of the step before each rejection tells whether the device iterates are reproducible bitwise
    rej = [i for i, s in enumerate(ref["steps"]) if not s.accepted]
    again = device_runs(name, [dict(max_iter=i, lambda0=lam0, **tol) for i in rej if i >= 1]) if rej else []
    s = np.sqrt(np.diag(m.linearise(x0)[0]))
    s[s == 0.0] = 1.0
    xs = {0: x0}
    for k, (xk, st, _) in zip(ks, runs):
        rk = refs[k]
        xs[k] = xk
        xr = rk["x"]
        err = np.linalg.norm(s * (xk - xr)) / max(np.linalg.norm(s * (xr - x0)), 1e-300)
        print(f"[lm-traj] {name} k={k}: rho={ref['steps'][k - 1].rho:.4f} accepted={ref['steps'][k - 1].accepted} "
              f"lambda {st['lambda_final']:.6e}/{rk['lambda_final']:.6e} cost {st['cost_final']:.12e}/{rk['cost_final']:.12e} "
              f"x err {err:.2e} evals {st['n_eval_normal']}/{rk['n_eval_normal']} {st['n_eval_cost']}/{rk['n_eval_cost']}")
        assert st["iterations"] == k and st["status"] == rk["status"] == 0, (k, st)
        assert abs(st["lambda_final"] - rk["lambda_final"]) <= 1e-6 * rk["lambda_final"], (k, st["lambda_final"], rk["lambda_final"])
        assert abs(st["cost_final"] - rk["cost_final"]) <= 1e-9 * rk["cost_final"], (k, st["cost_final"], rk["cost_final"])
        assert (st["n_eval_normal"], st["n_eval_cost"]) == (rk["n_eval_normal"], rk["n_eval_cost"]), (k, st)
        assert err <= 1e-7, (k, err)
    for j, i in enumerate(i for i in rej if i >= 1):
        # step i + 1 (1-based) is rejected: the device point stays x_i; step i + 2 is the model's step from x_i with 2 lambda
        reproducible = np.array_equal(again[j][0], xs[i])
        print(f"[lm-traj] {name}: step {i + 1} rejected; iterates reproducible bitwise: {reproducible}")
        if reproducible:
            assert np.array_equal(xs[i + 1], xs[i])
        else:   # FP64 atomics: separate runs agree to ~1e-10 of the path, a taken step would move the point by ~1e-1 of it
            assert np.linalg.norm(s * (xs[i + 1] - xs[i])) <= 1e-8 * np.linalg.norm(s * (xs[i] - x0))
        if i + 2 in xs:
            st_next = ref["steps"][i + 1]
            assert st_next.lam == 2.0 * ref["steps"][i].lam and np.array_equal(st_next.x, ref["steps"][i].x)
            d_dev = xs[i + 2] - xs[i + 1]
            err = np.linalg.norm(s * (d_dev - st_next.delta)) / np.linalg.norm(s * st_next.delta)
            print(f"[lm-traj] {name}: step {i + 2} after the rejection, error against the model's step {err:.2e}")
            assert err <= 1e-6, err


# ---- D: termination ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", range(len(R.TERMINATIONS)), ids=[f"{t[0]}-status{t[3]}" for t in R.TERMINATIONS])
def test_termination_matches_the_model(case):
    name, lam0, tol, status, its = R.TERMINATIONS[case]
    fx = fixture(name)
    ref = model(name).run(fx.x0, 20, lambda0=lam0, condition=False, **tol)
    assert (ref["status"], ref["iterations"]) == (status, its)
    (x, st, _), = device_runs(name, [dict(max_iter=20, lambda0=lam0, **tol)])
    print(f"[lm-term] {name} {tol}: device status {st['status']} after {st['iterations']}, model {status} after {its}")
    assert (st["status"], st["iterations"]) == (status, its), st
    assert (st["n_eval_normal"], st["n_eval_cost"]) == (ref["n_eval_normal"], ref["n_eval_cost"]), st
    assert abs(st["cost_final"] - ref["cost_final"]) <= 1e-9 * ref["cost_final"]
    assert abs(st["lambda_final"] - ref["lambda_final"]) <= 1e-6 * ref["lambda_final"]
    s = np.sqrt(np.diag(model(name).linearise(fx.x0)[0]))
    s[s == 0.0] = 1.0
    assert np.linalg.norm(s * (x - ref["x"])) <= 1e-7 * np.linalg.norm(s * (ref["x"] - fx.x0))
