"""CPU: the properties of the LM step fixtures (tests/lm_reference.py) that the device step tests rely on.

A change to the synthetic rigs, the goldens or the model must not quietly empty a device test: the trajectory fixture
keeps a rejected step with a meaningful gain ratio, the lambda comparisons keep gain ratios away from 0, every
termination fixture stops by its own criterion with a 10x margin, and the model's own steps solve their systems."""
import numpy as np
import pytest

from tests import lm_reference as R


def _run(name, lam0, n, **tol):
    fx = R.FIXTURES[name]()
    m = fx.model()
    return fx, m, m.run(fx.x0, n, lambda0=lam0, **({"ftol": 0.0, "xtol": 0.0, "gtol": 0.0} | tol))


@pytest.mark.parametrize("name", R.REJECTING)
def test_trajectory_fixture_has_a_meaningful_rejected_step(name):
    lam0 = dict(R.TRAJECTORIES)[name]
    _, _, res = _run(name, lam0, R.N_TRAJ)
    rejected = [s for s in res["steps"] if not s.accepted]
    assert rejected, "no rejected step"
    assert any(abs(s.rho) > 0.1 for s in rejected)
    # the rejected step is followed by an accepted one from the same linearisation with twice the damping
    k = next(i for i, s in enumerate(res["steps"]) if not s.accepted)
    assert k + 1 < len(res["steps"]) and res["steps"][k + 1].accepted
    assert np.array_equal(res["steps"][k + 1].x, res["steps"][k].x)
    assert res["steps"][k + 1].lam == 2.0 * res["steps"][k].lam


@pytest.mark.parametrize("name,lam0", [t for t in R.TRAJECTORIES if t[0].startswith("rig4")])
def test_accepted_gain_ratios_are_away_from_zero(name, lam0):
    _, _, res = _run(name, lam0, R.N_TRAJ)
    assert res["iterations"] == R.N_TRAJ and res["status"] == 0
    for s in res["steps"]:
        assert s.accepted == (s.rho > 0.0)
        if s.accepted:
            assert s.rho >= 1e-3
        assert abs(s.cost - s.cost_trial) >= 1e-6 * s.cost     # the gain ratio is not rounding noise


def test_trajectory_fixture_exercises_the_lambda_floor():
    """One of the accepted steps of the trajectory fixtures has rho > 0.94, where the 1/3 floor of the Nielsen update is
    the active branch: a wrong floor changes lambda_final."""
    hits = 0
    for name, lam0 in R.TRAJECTORIES[:2]:
        _, _, res = _run(name, lam0, R.N_TRAJ)
        hits += sum(1 for s in res["steps"] if s.accepted and 1.0 - (2.0 * s.rho - 1.0) ** 3 < 1.0 / 3.0 - 1e-3)
    assert hits >= 1


@pytest.mark.parametrize("case", range(len(R.TERMINATIONS)))
def test_termination_fixture_margins(case):
    name, lam0, tol, status, its = R.TERMINATIONS[case]
    _, _, res = _run(name, lam0, 20, **tol)
    assert res["status"] == status and res["iterations"] == its
    steps = res["steps"]
    if status == 1:
        vals, thr = [s.ginf for s in steps], [tol["gtol"]] * len(steps)
    elif status == 3:
        vals, thr = [s.dx for s in steps], [tol["xtol"] * (tol["xtol"] + s.xn) for s in steps]
    else:
        pairs = [(s.rel, tol["ftol"]) for s in steps if s.accepted]
        vals, thr = [p[0] for p in pairs], [p[1] for p in pairs]
    assert vals[-1] <= 0.1 * thr[-1]
    assert all(v >= 10.0 * t for v, t in zip(vals[:-1], thr[:-1]))


def test_xtol_fixture_separates_the_free_vector_from_the_parameter_string():
    """With the norm of the whole parameter string in place of the free vector's, the xtol test stops earlier."""
    name, lam0, tol, status, its = R.TERMINATIONS[2]
    fx, _, res = _run(name, lam0, 20, **tol)
    full = float(np.linalg.norm(fx.params0))
    assert full > 100.0 * res["steps"][0].xn
    early = [i for i, s in enumerate(res["steps"]) if s.dx < tol["xtol"] * (tol["xtol"] + full)]
    assert early and early[0] + 1 < its


@pytest.mark.parametrize("name,lam", [("rig4_template", 1e-6), ("rig4_template_masks", 1.0), ("rig4_selfcal_point_masks", 1e-3),
                                      ("ccube_template", 1e2)])
def test_model_step_backward_error(name, lam):
    fx = R.FIXTURES[name]()
    m = fx.model()
    delta, pred, A, D, g, kappa = m.step(fx.x0, lam)
    assert R.backward_error(A, g, delta) <= 1e-14
    assert np.isfinite(kappa) and kappa >= 1.0
    unobserved = np.diag(m.linearise(fx.x0)[0]) == 0.0
    assert np.all(delta[unobserved] == 0.0)


def test_fixtures_cover_fixed_and_unobserved_parameters():
    fx = R.FIXTURES["rig4_template_masks"]()
    obs = fx.observed()
    assert np.any(fx.unfixed & ~obs)                    # free but never observed (camera 4, pose 6)
    assert np.any(~fx.unfixed & obs)                    # fixed and observed
    C = fx.C
    pose4 = fx.unfixed[15 * C + 24:15 * C + 30]
    assert not pose4[:3].any() and pose4[3:].all()      # a partly fixed pose block
    sc = R.FIXTURES["rig4_selfcal_point_masks"]()
    pts = slice(15 * sc.C + 6 * sc.M, None)
    assert np.any(sc.unfixed[pts] & ~sc.observed()[pts])
    assert np.any(~sc.unfixed[pts])
    assert 3 * sc.K > 6 * sc.M                          # the point-elimination path
