"""GPU: the parameter covariance of pcs_covariance against the float64 CPU reference of tests/cov_reference.py.

Every fixture is checked at its start and at the device LM solution: each returned entry within
max(1e-11, 1e-12 kappa_s) sqrt(Sigma_aa Sigma_bb) of the reference, fixed entries exactly 0, unobserved ones NaN, s2 and
dof exact, the camera block symmetric and every diagonal block positive definite.  The fixtures cover the template chain
(small and padded, partial masks, goldens, the sparse Schur plan and its dense alternative, the 128-camera dome) and the
self-calibration chain with the points and with the poses eliminated.  The 32-camera ring is compared with its
intrinsics fixed, and the ccube self-calibration golden not at all: undamped, both are singular to working precision
(tests/test_covariance_reference.py).  Further: an LM solve after a
covariance call behaves as without it, mixed precision is overridden and kept, the unsupported configurations are
refused, the scale s2 has its statistical meaning, and run_bundle_adjustment(covariance=True) returns the standard
deviations in x order."""
import functools

import numpy as np
import pytest

from tests import cov_reference as CR
from tests import lm_reference as R
from tests.helpers import solver_env

pytestmark = pytest.mark.gpu

CASES = [
    ("rig4_template", {}),
    ("rig4_template_masks", {}),
    ("ring5_fixedcam_template", {}),
    ("ccube_template", {}),
    ("ring32_template_intr_fixed", {}),
    ("ring32_template_intr_fixed", {"PCS_LM_SCHUR": "dense"}),
    ("dome128_template", {}),
    ("rig4_selfcal_point_masks", {}),
    ("ring5_fixedcam_selfcal", {"PCS_LM_SELFCAL": "poses"}),
]


@functools.lru_cache(maxsize=None)
def fixture(name):
    return CR.FIXTURES[name]()


def check_against_reference(fx, dev, x, label):
    """Asserts the contract at x; returns the largest ratio |error| / bound."""
    ref = CR.reference(fx, x)
    tol = max(1e-11, 1e-12 * ref["kappa"])
    exp = CR.blocks(ref["Sigma"], fx.C, fx.M, fx.K, fx.chain)
    fixed = CR.blocks(np.logical_or.outer(~fx.unfixed, ~fx.unfixed).astype(float), fx.C, fx.M, fx.K, fx.chain)
    worst = 0.0
    assert set(exp) == {k for k in ("cam", "pose", "point") if k in dev}, label
    for part, e in exp.items():
        d = dev[part]
        assert d.shape == e.shape, (label, part)
        fx_mask = fixed[part] > 0
        nan_mask = np.isnan(e) & ~fx_mask
        assert np.all(d[fx_mask] == 0.0), (label, part, "fixed entries are not exactly 0")
        assert np.array_equal(np.isnan(d), nan_mask), (label, part, "NaN pattern differs from the unobserved parameters")
        ok = ~fx_mask & ~nan_mask
        diag = np.diagonal(e, axis1=-2, axis2=-1)
        scale = np.sqrt(np.abs(diag[..., :, None] * diag[..., None, :]))
        err = np.abs(d - e)[ok] / (tol * scale[ok])
        if err.size:
            worst = max(worst, float(err.max()))
    assert worst <= 1.0, (label, worst)
    assert dev["dof"] == ref["dof"], (label, dev["dof"], ref["dof"])
    r = fx.oracle().residual(fx.model().full(x))
    s2 = float(r @ r) / ref["dof"]
    assert abs(dev["s2"] - s2) <= 1e-12 * s2, (label, dev["s2"], s2)
    assert np.array_equal(dev["cam"], dev["cam"].T, equal_nan=True), label
    # every diagonal block is positive definite over its free, observed parameters
    C = fx.C
    cam_blocks = [dev["cam"][15 * c:15 * c + 15, 15 * c:15 * c + 15] for c in range(C)]
    for blk in cam_blocks + list(dev["pose"]) + list(dev.get("point", [])):
        live = np.isfinite(np.diag(blk)) & (np.diag(blk) != 0.0)
        if live.any():
            assert np.linalg.eigvalsh(blk[np.ix_(live, live)]).min() > 0.0, label
    print(f"[cov] {label}: kappa_s={ref['kappa']:.2e} worst |error| / bound = {worst:.3g} (bound {tol:.1e} sqrt(S_aa S_bb)); "
          f"dof={dev['dof']} s2={dev['s2']:.6e}")
    return worst


@pytest.mark.parametrize("name,env", CASES, ids=[f"{n}-{'-'.join(e.values()) or 'default'}" for n, e in CASES])
def test_covariance_matches_the_reference(name, env):
    fx = fixture(name)
    with solver_env(**env), fx.problem() as p:
        if name.startswith("ring32_template"):
            frac = p.lm_schur_fraction()
            assert (frac == 1.0) if "PCS_LM_SCHUR" in env else (0.2 < frac < 0.85), frac
        dev0 = p.covariance(fx.x0)
        x, st = p.lm_solve(fx.x0, max_iter=50)
        assert st["status"] > 0, st
        dev1 = p.covariance(x)
        # side effect: the parameters are x
        assert np.array_equal(p.get_param_string()[fx.unfixed], x)
    label = f"{name} [{', '.join(f'{k}={v}' for k, v in env.items()) or 'library default'}]"
    check_against_reference(fx, dev0, fx.x0, label + " at x0")
    check_against_reference(fx, dev1, x, label + " at the LM solution")


@pytest.mark.parametrize("name", ["ring32_template_intr_fixed", "rig4_selfcal_point_masks"])
def test_lm_solve_after_covariance_is_unchanged(name):
    fx = fixture(name)
    with fx.problem() as p:
        x_a, st_a = p.lm_solve(fx.x0, max_iter=30)
        p.covariance(x_a)
        x_b, st_b = p.lm_solve(fx.x0, max_iter=30)
    assert (st_b["iterations"], st_b["status"]) == (st_a["iterations"], st_a["status"]), (st_a, st_b)
    s = np.sqrt(np.diag(fx.model().linearise(fx.x0)[0]))
    s[s == 0.0] = 1.0
    err = np.linalg.norm(s * (x_b - x_a)) / np.linalg.norm(s * (x_a - fx.x0))
    print(f"[cov] {name}: lm_solve after covariance differs from the first solve by {err:.2e} of the path length")
    assert err <= 1e-10, err


def test_mixed_precision_is_overridden_and_kept():
    fx = fixture("ring32_template_intr_fixed")
    with fx.problem() as p:
        U64 = p.normal_equations(fx.x0, with_W=False)["U"]
        ref = p.covariance(fx.x0)
        p.set_normal_precision(True)
        dev = p.covariance(fx.x0)
        Umx = p.normal_equations(fx.x0, with_W=False)["U"]
    # an FP64 evaluation: the result agrees with the FP64 one (and the CPU reference) to the reference bound
    check_against_reference(fx, dev, fx.x0, "ring32_template_intr_fixed mixed precision")
    tol = max(1e-11, 1e-12 * CR.reference(fx, fx.x0)["kappa"])
    for k in ("cam", "pose"):
        d = np.sqrt(np.abs(np.diagonal(ref[k], axis1=-2, axis2=-1)))
        bound = tol * d[..., :, None] * d[..., None, :]
        ok = np.isfinite(bound)
        assert np.array_equal(np.isnan(dev[k]), np.isnan(ref[k])), k
        assert np.all(np.abs(dev[k] - ref[k])[ok] <= bound[ok]), k
    # still mixed afterwards: the blocks come from the BF16-split path again
    assert np.max(np.abs(Umx - U64)) > 1e-9 * np.max(np.abs(U64))


def test_multi_rank_is_refused():
    from pycamset_b200 import _lib as L
    fx = fixture("rig4_template")
    with fx.problem() as p:
        p.set_allreduce(lambda ptr, n, op, stream: None, 0, 2)
        with pytest.raises(L.PcsError) as e:
            p.covariance(fx.x0)
        assert e.value.code == L.PCS_ERR_UNSUPPORTED


def test_dense_selfcal_fallback_is_refused():
    from pycamset_b200 import _lib as L
    fx = R.FIXTURES["ring5_fixedcam_selfcal"]()
    with solver_env(PCS_LM_SELFCAL="dense"), fx.problem() as p:
        with pytest.raises(L.PcsError) as e:
            p.covariance(fx.x0)
        assert e.value.code == L.PCS_ERR_UNSUPPORTED


def test_scale_has_its_statistical_meaning():
    """200 seeded draws of sigma = 0.5 px noise on a noise-free 4-camera ring x 12 poses, each solved by the device LM
    from the truth: the mean of s2 is sigma^2, and the spread of the estimates matches sigma^2 Sigma (unit-weight
    covariance at the truth) and the mean of s2 Sigma at the solutions.  The watched parameters are well determined, so
    that the linearisation holds across the draws: camera 0 (972 observations) and two poses.  Cameras 1 and 3 see the
    board in a few poses only; their intrinsics move far enough between draws that the covariance at the solution varies
    with them (camera 2 never sees the board's front face)."""
    from pycamset_b200 import synthetic as syn
    from pycamset_b200.problem import BundleProblem
    sigma, n_draws = 0.5, 200
    C, M = 4, 12
    rig = syn.make_rig(C, M, distortion=True, seed=21, noise_px=0.0)
    cam, pose, key = (np.ascontiguousarray(a.numpy()) for a in (rig.cam, rig.pose, rig.key))
    uv0 = rig.uv.numpy()
    truth = rig.param_string()
    unfixed = np.ones(truth.shape[0], bool)
    unfixed[15 * C:15 * C + 6] = False
    xt = truth[unfixed]
    # parameters watched: focal lengths and principal point of camera 0, one extrinsic, the translations of poses 1 and 2
    fm = -np.ones(truth.shape[0], int)
    fm[unfixed] = np.arange(unfixed.sum())
    watch_str = [0, 1, 2, 3, 9 * C + 3] + [15 * C + 6 * m + a for m in (1, 2) for a in (3, 4, 5)]
    watch = fm[watch_str]
    assert np.all(watch >= 0)
    rng = np.random.default_rng(1234)
    xs, s2s, s2sig = [], [], []
    sig_truth = None
    for i in range(n_draws):
        uv = uv0 + sigma * rng.normal(size=uv0.shape)
        with BundleProblem(0, cam, pose, key, uv, C, M, rig.n_keys, template=rig.template, unfixed=unfixed) as p:
            p.set_param_string(truth)
            if sig_truth is None:
                sig_truth = p.covariance(xt)
            x, st = p.lm_solve(xt, max_iter=100)
            assert st["status"] >= 0, st
            cov = p.covariance(x)
        var = np.zeros(truth.shape[0])
        d = np.diagonal(cov["cam"]).reshape(C, 15)
        var[:9 * C], var[9 * C:15 * C] = d[:, :9].ravel(), d[:, 9:].ravel()
        var[15 * C:15 * C + 6 * M] = np.diagonal(cov["pose"], axis1=1, axis2=2).ravel()
        xs.append(x)
        s2s.append(cov["s2"])
        s2sig.append(cov["s2"] * var[unfixed][watch])
    xs, s2s = np.array(xs), np.array(s2s)
    var_t = np.zeros(truth.shape[0])
    d = np.diagonal(sig_truth["cam"]).reshape(C, 15)
    var_t[:9 * C], var_t[9 * C:15 * C] = d[:, :9].ravel(), d[:, 9:].ravel()
    var_t[15 * C:15 * C + 6 * M] = np.diagonal(sig_truth["pose"], axis1=1, axis2=2).ravel()
    emp = xs[:, watch].var(axis=0, ddof=1)
    pred_truth = sigma ** 2 * var_t[unfixed][watch]
    pred_sol = np.mean(s2sig, axis=0)
    print(f"[cov-stat] mean s2 / sigma^2 = {s2s.mean() / sigma ** 2:.4f}; empirical / predicted variance at the truth: "
          f"{np.round(emp / pred_truth, 3)}; against mean s2 Sigma: {np.round(emp / pred_sol, 3)}")
    assert 0.9 <= s2s.mean() / sigma ** 2 <= 1.1
    assert np.all((0.7 <= emp / pred_truth) & (emp / pred_truth <= 1.4))
    assert np.all((0.7 <= emp / pred_sol) & (emp / pred_sol <= 1.4))


def test_run_bundle_adjustment_returns_parameter_std():
    from pycamset_b200.handler import run_bundle_adjustment
    from tests import fake_reference as fr
    from tests.helpers import load_case
    g = load_case("ring4_template")
    h = fr.TemplateBundleHandler(g)
    h.problem_opts["max_nfev"] = 20
    res, _ = run_bundle_adjustment(h, solver="lm", jac=False, covariance=True)
    cov = res["covariance"]
    n_free = int(np.asarray(g["unfixed"], bool).sum())
    assert cov["param_std"].shape == (n_free,)
    C, M, K = int(g["n_cams"]), int(g["n_poses"]), g["template"].shape[0]
    # param_std = sqrt(diag(s2 Sigma)) scattered to x order
    var = np.zeros(15 * C + 6 * M)
    d = np.diagonal(cov["cam"]).reshape(C, 15)
    var[:9 * C], var[9 * C:15 * C] = d[:, :9].ravel(), d[:, 9:].ravel()
    var[15 * C:] = np.diagonal(cov["pose"], axis1=1, axis2=2).ravel()
    unfixed = np.asarray(g["unfixed"], bool)
    assert np.array_equal(cov["param_std"], np.sqrt(var[unfixed]), equal_nan=True)
    # against the oracle at the solution
    fx = R.golden_fixture("ring4_template")
    ref = CR.reference(fx, res.x)
    std_ref = np.sqrt(ref["s2"] * np.diag(ref["Sigma"])[unfixed])
    tol = max(1e-11, 1e-12 * ref["kappa"])
    assert np.array_equal(np.isnan(cov["param_std"]), np.isnan(std_ref))
    ok = np.isfinite(std_ref)
    rel = np.abs(cov["param_std"][ok] / std_ref[ok] - 1.0)
    print(f"[cov] run_bundle_adjustment param_std: largest relative difference from the oracle {rel.max():.2e} (bound {tol:.1e})")
    assert np.all(rel <= tol), rel.max()
    # the scipy path carries the same dict
    h2 = fr.TemplateBundleHandler(g)
    h2.problem_opts["max_nfev"] = 8
    res2, _ = run_bundle_adjustment(h2, solver="scipy", covariance=True)
    assert res2["covariance"]["param_std"].shape == (n_free,)
