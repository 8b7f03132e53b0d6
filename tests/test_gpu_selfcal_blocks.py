"""GPU: block normal equations and the Schur LM of the SELF-CALIBRATION chain (projection + extrinsic3D + rigidTform3d +
free_point; BASELINE.json config 3, standard_bundle_handler.py:129-226).

  * every block -- U, V, W, g_c, g_m, r.r and the point blocks Pk, gk, Xck (camera x point), Ymk (pose x point) -- against
    the corresponding block of the oracle's dense J^T J / J^T r with no parameter fixed (tolerance 1e-9 sqrt(d_a d_b));
  * the device LM on the block path, in both elimination orders (points eliminated, cameras + poses in the reduced system
    -- the library's choice when 3 K > 6 M; or poses eliminated, cameras + points in the reduced system), own SYRK +
    Cholesky kernels, against the dense n_free x n_free path, which stays as the comparator: same cost trajectory."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests.helpers import available, load_case, oracle_problem, solver_env

pytestmark = pytest.mark.gpu
CASES = available(["ring4_selfcal", "ring5_fixedcam_selfcal", "ccube_selfcal"])


def _problem(g):
    from pycamset_b200.problem import BundleProblem
    dd = g["dd"]
    return BundleProblem(1, dd[:, 0], dd[:, 1], dd[:, 2], dd[:, 3:5], int(g["n_cams"]), int(g["n_poses"]), g["template"].shape[0],
                         unfixed=g["unfixed"])


@pytest.mark.parametrize("case", CASES)
def test_selfcal_blocks_against_the_oracle(case):
    g = load_case(case)
    o = oracle_problem(g)
    C, M, K, L = o.C, o.M, o.K, o.L
    with _problem(g) as p:
        p.set_param_string(g["param0"])
        ne = p.normal_equations(g["x"])
        sc, sp, sl = p.segments()
    JtJ, Jtr, cost = o.normal_dense(g["param0"], np.arange(L, dtype=np.int32))
    d = np.sqrt(np.maximum(np.diag(JtJ), 1e-300))
    cam_idx = np.stack([np.r_[9 * c:9 * c + 9, 9 * C + 6 * c:9 * C + 6 * c + 6] for c in range(C)])
    pose_idx = 15 * C + 6 * np.arange(M)[:, None] + np.arange(6)[None, :]
    pt_idx = 15 * C + 6 * M + 3 * np.arange(K)[:, None] + np.arange(3)[None, :]

    def close(a, rows, cols):
        ref = JtJ[rows[..., :, None], cols[..., None, :]]
        scale = d[rows][..., :, None] * d[cols][..., None, :]
        return float(np.max(np.abs(a - ref) / scale))

    assert abs(ne["cost"] - cost) <= 1e-11 * cost
    assert close(ne["U"], cam_idx, cam_idx) < 1e-9
    assert close(ne["V"], pose_idx, pose_idx) < 1e-9
    assert close(ne["W"], cam_idx[sc], pose_idx[sp]) < 1e-9
    assert close(ne["Pk"], pt_idx, pt_idx) < 1e-9
    assert close(ne["Xck"], np.broadcast_to(cam_idx[:, None, :], (C, K, 15)), np.broadcast_to(pt_idx[None, :, :], (C, K, 3))) < 1e-9
    assert close(ne["Ymk"], np.broadcast_to(pose_idx[:, None, :], (M, K, 6)), np.broadcast_to(pt_idx[None, :, :], (M, K, 3))) < 1e-9
    for got, idx in ((ne["gc"], cam_idx), (ne["gp"], pose_idx), (ne["gk"], pt_idx)):
        assert np.max(np.abs(got - Jtr[idx]) / (d[idx] * np.sqrt(cost))) < 1e-9
    # every camera x pose pair without a segment has a zero block in the dense matrix
    seen = np.zeros((C, M), bool); seen[sc, sp] = True
    for c, m in zip(*np.nonzero(~seen)):
        assert not JtJ[np.ix_(cam_idx[c], pose_idx[m])].any()


def _lm_runs(case, mode):
    """Four LM solves (max_iter 1, 2, 5, 100) from the golden start on a fresh problem.  mode: None = the library's choice
    (the larger of the pose / point block sets is eliminated), "poses" = pose elimination forced (cameras + points in the
    reduced system), "dense" = the dense n_free x n_free comparator."""
    g = load_case(case)
    out = []
    with solver_env(**({"PCS_LM_SELFCAL": mode} if mode else {})), _problem(g) as p:
        for it in (1, 2, 5, 100):
            p.set_param_string(g["param0"])
            x, st = p.lm_solve(g["x"], max_iter=it, ftol=1e-12, xtol=1e-12, gtol=1e-12)
            r = p.residual(x)
            out.append(dict(it=st["iterations"], cost=st["cost_final"], true_cost=0.5 * float(r @ r), seconds=st["seconds"],
                            px=float(np.mean(np.linalg.norm(r.reshape(-1, 2), axis=1)))))
    return out


@pytest.mark.parametrize("case", CASES)
def test_selfcal_block_lm_matches_the_dense_path(case):
    dns = _lm_runs(case, "dense")
    for mode in (None, "poses"):             # both elimination orders of the block path: the same Newton systems, solved differently
        blk = _lm_runs(case, mode)
        for b, d in zip(blk[:3], dns[:3]):   # the first iterations: same linear systems, solved two ways
            assert b["it"] == d["it"]
            assert abs(b["cost"] - d["cost"]) <= 1e-8 * d["cost"], (mode, b, d)
        for b in blk:
            assert abs(b["cost"] - b["true_cost"]) <= 1e-9 * b["true_cost"]
        assert abs(blk[-1]["cost"] - dns[-1]["cost"]) <= 1e-3 * dns[-1]["cost"], (mode, blk[-1], dns[-1])
        if case == "ccube_selfcal":
            assert blk[-1]["px"] < 0.2184    # the reference's own final error on this fixture (0.21834 px, max_nfev = 100)
