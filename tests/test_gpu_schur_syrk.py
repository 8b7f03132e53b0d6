"""GPU: the stream-K FP64 tensor-path SYRK of the reduced camera system (csrc/pcs_schur.cu) against numpy.

Shapes cover ragged tiles (n not a multiple of 96), odd n (8-byte copy path), k not a multiple of the 16-column slab,
fewer work units than SMs, and the bench shape (480 x 12000).  Tolerance: |dS| <= 1e-12 * sum_k |Z_ik||Z_jk| + tiny
(FP64 accumulation in a different order)."""
import numpy as np
import pytest

from tests.helpers import solver_env

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,k", [(1, 1), (15, 6), (45, 30), (96, 16), (97, 50), (120, 594), (480, 1200), (495, 333), (480, 12000)])
def test_syrk_matches_numpy(n, k):
    from pycamset_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(n * 131 + k)
    Z = rng.standard_normal((n, k))
    S0 = rng.standard_normal((n, n))
    S0 = S0 + S0.T
    Zf = np.asfortranarray(Z)          # column-major [k][n]: column index slowest
    S = np.asfortranarray(S0.copy())
    rc = lib.pcs_syrk_sub(0, n, k, Zf.ctypes.data, S.ctypes.data)
    assert rc == 0, lib.pcs_last_error()
    ref = S0 - Z @ Z.T
    bound = 1e-12 * (np.abs(Z) @ np.abs(Z).T) + 1e-13
    lo = np.tril_indices(n)
    assert np.all(np.abs(S[lo] - ref[lo]) <= bound[lo])
    up = np.triu_indices(n, 1)
    assert np.array_equal(S[up], S0[up])   # the strict upper triangle is not touched


def _ring_lm(max_iter, dense):
    """LM iterates of a 32-camera ring (every pose seen by about half of the cameras) with / without the sparsity plan."""
    from pycamset_b200 import synthetic as syn
    from pycamset_b200.problem import BundleProblem
    rig = syn.make_rig(32, 300, distortion=True, seed=3, detect_prob=0.9)
    intr, extr, poses = rig.perturbed(np.random.default_rng(5), 2e-3)
    params = rig.param_string(intr, extr, poses)
    unfixed = np.ones(params.shape[0], bool)
    unfixed[15 * 32:15 * 32 + 6] = False
    with solver_env(**({"PCS_LM_SCHUR": "dense"} if dense else {})), \
            BundleProblem(0, rig.cam.numpy(), rig.pose.numpy(), rig.key.numpy(), rig.uv.numpy(), 32, 300, 81, template=rig.template,
                          unfixed=unfixed) as p:
        p.set_param_string(params)
        frac = p.lm_schur_fraction()
        x, st = p.lm_solve(params[unfixed], max_iter=max_iter, ftol=0, xtol=0, gtol=0)
    return frac, x, st


def test_block_sparse_pose_elimination_equals_the_dense_one():
    """The unit list skips only (tile pair, slab) units whose product is exactly zero and the permuted pose columns are
    summed in a different order: same LM iterates up to FP64 summation order."""
    f_sparse, x_s, st_s = _ring_lm(6, dense=False)
    f_dense, x_d, st_d = _ring_lm(6, dense=True)
    assert f_dense == 1.0
    assert 0.2 < f_sparse < 0.85, f_sparse          # the plan is active and skips a substantial part of the units
    assert st_s["iterations"] == st_d["iterations"]
    assert abs(st_s["cost_final"] - st_d["cost_final"]) <= 1e-9 * st_d["cost_final"]
    assert np.max(np.abs(x_s - x_d)) <= 1e-7 * max(1.0, np.max(np.abs(x_d)))
