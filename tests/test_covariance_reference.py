"""CPU: the properties of the covariance fixtures (tests/cov_reference.py) that the device covariance test relies on.

The device result is compared with a tolerance max(1e-11, 1e-12 kappa_s) sqrt(Sigma_aa Sigma_bb): that bound only means
something while the undamped systems stay well enough conditioned, at the start and at the solution.  The masked
fixtures must really contain fixed and unobserved free parameters, and every fixture must have residual degrees of
freedom."""
import functools

import numpy as np
import pytest

from tests import cov_reference as CR
from tests import lm_reference as R

# every fixture of tests/test_gpu_covariance.py (the environment switches do not change the normal equations)
NAMES = ["rig4_template", "rig4_template_masks", "ring5_fixedcam_template", "ccube_template", "ring32_template_intr_fixed",
         "dome128_template", "rig4_selfcal_point_masks", "ring5_fixedcam_selfcal"]


@functools.lru_cache(maxsize=None)
def fixture(name):
    return CR.FIXTURES[name]()


@functools.lru_cache(maxsize=None)
def solution(name):
    """The model's LM solution, a stand-in for the device's (they agree to ~1e-10 of the path length)."""
    fx = fixture(name)
    return fx.model().run(fx.x0, 30, condition=False)["x"]


@pytest.mark.parametrize("name", NAMES)
def test_fixture_is_well_posed_at_start_and_solution(name):
    fx = fixture(name)
    for where, x in (("x0", fx.x0), ("solution", solution(name))):
        ref = CR.reference(fx, x)
        print(f"[cov-ref] {name} at {where}: kappa_s={ref['kappa']:.3e} dof={ref['dof']} s2={ref['s2']:.4e}")
        assert ref["kappa"] < 1e12, (where, ref["kappa"])
        assert ref["dof"] > 0
        assert np.all(np.isfinite(np.diag(ref["Sigma"])[fx.unfixed & fx.observed()]))


@pytest.mark.parametrize("name", ["ring32_template", "ccube_selfcal"])
def test_singular_fixtures_are_left_out(name):
    """The 32-camera ring with free intrinsics (a camera that sees few poses trades focal length / principal point for
    translation) and the ccube self-calibration golden are singular to working precision without damping: the device
    comparison uses the ring with its intrinsics fixed and leaves the golden out."""
    fx = fixture(name)
    H = fx.model().linearise(fx.x0)[0]
    obs = np.diag(H) > 0.0
    assert not 0.0 < R.LmModel.scaled_condition(H[np.ix_(obs, obs)]) < 1e12


@pytest.mark.parametrize("name", ["rig4_template_masks", "rig4_selfcal_point_masks"])
def test_masked_fixtures_have_fixed_and_unobserved_free_parameters(name):
    fx = fixture(name)
    ref = CR.reference(fx, fx.x0)
    assert (~fx.unfixed).any()
    assert ref["n_unobserved_free"] > 0
    assert ((~fx.observed()) & fx.unfixed).sum() == ref["n_unobserved_free"]
    # every returned part holds fixed (0) and unobserved (NaN) entries
    b = CR.blocks(ref["Sigma"], fx.C, fx.M, fx.K, fx.chain)
    assert any(np.isnan(v).any() for v in b.values())
    assert any((v == 0.0).any() for v in b.values())
