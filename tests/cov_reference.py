"""A float64 CPU reference of the parameter covariance (pcs_covariance, pycamset_b200/csrc/pcs_cov.cu).

TEST INFRASTRUCTURE ONLY.  H = J^T J, c = r.r come from the CPU oracle (oracle.Problem.normal_dense) over the free
parameters; Sigma = H^-1 over the observed ones (diag H > 0) by Cholesky with two rounds of extended-precision
refinement (LmModel.spd_solve).  Sigma is returned over the whole parameter string: 0 where a parameter is fixed, NaN
where a free parameter is unobserved.  kappa_s is the condition number of the Jacobi-scaled H over the observed
parameters."""
from __future__ import annotations

import dataclasses

import numpy as np

from tests import lm_reference as R


def reference(fx, x):
    """dict(Sigma [L][L] over the parameter string, kappa, s2, dof) at the free vector x of fixture fx."""
    H, _, c = fx.model().linearise(np.asarray(x, np.float64))
    obs = np.diag(H) > 0.0
    Hs = H[np.ix_(obs, obs)]
    inv = R.LmModel.spd_solve(Hs, np.eye(Hs.shape[0]))
    inv = 0.5 * (inv + inv.T)
    full = np.full(H.shape, np.nan)
    full[np.ix_(obs, obs)] = inv
    idx = np.flatnonzero(fx.unfixed)
    sigma = np.zeros((fx.params0.shape[0],) * 2)
    sigma[np.ix_(idx, idx)] = full
    dof = 2 * int(fx.cam.shape[0]) - int(obs.sum())
    return dict(Sigma=sigma, kappa=R.LmModel.scaled_condition(Hs), s2=c / dof if dof > 0 else float("nan"), dof=dof,
                n_unobserved_free=int((~obs).sum()))


def layout(C, M, K, chain):
    """Parameter-string index of every entry the ABI returns: cam [15 C] (camera-major, 9 intrinsics then 6 extrinsics),
    pose [M][6], point [K][3] (self-calibration chain, else None)."""
    cam = np.array([9 * c + a if a < 9 else 9 * C + 6 * c + a - 9 for c in range(C) for a in range(15)])
    pose = 15 * C + np.arange(6 * M).reshape(M, 6)
    point = 15 * C + 6 * M + np.arange(3 * K).reshape(K, 3) if chain == 1 else None
    return cam, pose, point


def blocks(S, C, M, K, chain):
    """The parts of a parameter-string matrix S in the ABI's layout: dict(cam, pose[, point])."""
    cam, pose, point = layout(C, M, K, chain)
    out = dict(cam=S[np.ix_(cam, cam)], pose=S[pose[:, :, None], pose[:, None, :]])
    if point is not None:
        out["point"] = S[point[:, :, None], point[:, None, :]]
    return out


def intrinsics_fixed(fx):
    """The fixture with every camera's intrinsics fixed.  On the 32-camera ring a camera that sees few poses leaves its
    focal length / principal point and its translation nearly interchangeable: undamped, the system is singular to
    working precision (kappa_s ~ 1e16), so the covariance is compared on this variant."""
    unfixed = fx.unfixed.copy()
    unfixed[:9 * fx.C] = False
    return dataclasses.replace(fx, name=fx.name + "_intr_fixed", unfixed=unfixed)


FIXTURES = dict(R.FIXTURES) | {
    "ring32_template_intr_fixed": lambda: intrinsics_fixed(R.ring32_template()),
}
