"""A float64 CPU restatement of the device Levenberg-Marquardt solver (lm_solve_impl, pycamset_b200/csrc/pcs_solver.cu).

TEST INFRASTRUCTURE ONLY.  Every linearisation comes from the CPU oracle (oracle.Problem.normal_dense: H = J^T J,
g = J^T r, c = r.r over the free parameters); the damping, the step, the gain ratio, the lambda schedule, the
termination tests and the evaluation counters follow the rules of the device solver:

  * damping      D = diag(H), A = H + lambda diag(D).  Block path (both chains, the library's default): a free parameter
                 with D == 0 (never observed) is an identity row with a zero step.  Dense self-calibration fallback:
                 D -> max(D, 1e-12).
  * step         delta = -A^-1 g: Cholesky plus two rounds of iterative refinement with the residual accumulated in
                 np.longdouble.  kappa_s = condition number of the Jacobi-scaled A.
  * acceptance   pred = delta . (lambda D delta - g), rho = (c - c') / pred (-1 if pred <= 0 or c' is not finite);
                 rho > 0: lambda <- max(lambda_min, lambda max(1/3, 1 - (2 rho - 1)^3)), nu = 2;
                 otherwise lambda <- min(lambda_max, lambda nu), nu <- 2 nu.
  * termination  gtol (|g|_inf), then xtol (|dx| < xtol (xtol + |x|), x the FREE vector) before the trial point is used;
                 ftol after an accepted step (relative decrease of r.r).
  * counters     the block path evaluates the trial point with the full normal-equation kernel; a rejected step (and a
                 gtol / xtol exit) turns that evaluation into a cost-only one.  The dense path evaluates the trial cost
                 alone and re-linearises after an accepted step.

`Fixture` bundles the problems the step tests run: each is a distinct path of the device solver.
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np
import scipy.linalg as sla

from oracle import oracle as orc

LAMBDA_MIN, LAMBDA_MAX = 1e-12, 1e12


@dataclasses.dataclass
class Step:
    """One iteration of the model: the system solved at linearisation `x` (free vector) with damping `lam`."""
    x: np.ndarray
    lam: float
    cost: float              # r.r at x
    delta: np.ndarray
    pred: float
    cost_trial: float        # r.r at x + delta (nan when a gtol / xtol exit came first)
    rho: float
    accepted: bool
    kappa_s: float
    ginf: float
    dx: float
    xn: float
    rel: float               # (c - c') / c


class LmModel:
    """path: "block" (identity rows for unobserved free parameters) or "dense" (D floored at 1e-12)."""

    def __init__(self, oproblem: orc.Problem, unfixed, params0, path: str = "block"):
        assert path in ("block", "dense")
        self.o = oproblem
        self.unfixed = np.asarray(unfixed, bool)
        self.fm = orc.free_map_from_mask(self.unfixed)
        self.params0 = np.array(params0, np.float64)
        self.path = path
        self._lin = {}

    # ---- linear algebra --------------------------------------------------------------------------
    def full(self, x):
        p = self.params0.copy()
        p[self.unfixed] = x
        return p

    def linearise(self, x):
        key = np.asarray(x, np.float64).tobytes()
        if key not in self._lin:
            if len(self._lin) > 8:
                self._lin.clear()
            self._lin[key] = self.o.normal_dense(self.full(x), self.fm)
        return self._lin[key]

    def cost(self, x):
        r = self.o.residual(self.full(x))
        return float(r @ r)

    def damped(self, H, lam):
        """(A, D, identity-row mask) of the damped system."""
        d = np.diag(H).copy()
        if self.path == "dense":
            D = np.maximum(d, 1e-12)
            ident = np.zeros(d.shape, bool)
        else:
            ident = d == 0.0
            D = np.where(ident, 0.0, d)
        A = H + lam * np.diag(D)
        A[ident, :] = 0.0
        A[:, ident] = 0.0
        A[ident, ident] = 1.0
        return A, D, ident

    @staticmethod
    def spd_solve(A, b):
        """Cholesky + two rounds of iterative refinement with the residual in extended precision."""
        cf = sla.cho_factor(A, lower=True)
        x = sla.cho_solve(cf, b)
        Al = A.astype(np.longdouble)
        bl = b.astype(np.longdouble)
        for _ in range(2):
            r = (bl - Al @ x.astype(np.longdouble)).astype(np.float64)
            x = x + sla.cho_solve(cf, r)
        return x

    @staticmethod
    def scaled_condition(A):
        s = 1.0 / np.sqrt(np.diag(A))
        ev = np.linalg.eigvalsh(A * s[:, None] * s[None, :])
        return float(ev[-1] / ev[0])

    def step(self, x, lam, condition=True):
        """(delta, pred, A, D, g, kappa_s) of the damped system at x."""
        H, g, c = self.linearise(x)
        A, D, ident = self.damped(H, lam)
        rhs = -g.copy()
        rhs[ident] = 0.0
        delta = self.spd_solve(A, rhs)
        delta[ident] = 0.0
        pred = float(delta @ (lam * D * delta - g))
        kappa = self.scaled_condition(A) if condition else float("nan")
        return delta, pred, A, D, g, kappa

    # ---- the solver ------------------------------------------------------------------------------
    def run(self, x0, max_iter, lambda0=1e-3, ftol=1e-8, xtol=1e-8, gtol=1e-8, lambda_min=LAMBDA_MIN,
            lambda_max=LAMBDA_MAX, condition=True):
        """Returns dict(x, iterations, status, cost_initial, cost_final, lambda_final, n_eval_normal, n_eval_cost,
        steps=[Step], iterates=[x after each iteration])."""
        block = self.path == "block"
        x = np.array(x0, np.float64)
        lam, nu = float(lambda0), 2.0
        n_normal, n_cost, it, status = 1, 0, 0, 0
        cost = cost0 = self.linearise(x)[2]
        steps, iterates = [], []
        while it < max_iter:
            it += 1
            delta, pred, A, D, g, kappa = self.step(x, lam, condition)
            if block:
                n_normal += 1                      # the trial point is evaluated with the full kernel
            ginf = float(np.max(np.abs(g))) if g.size else 0.0
            dx, xn = float(np.linalg.norm(delta)), float(np.linalg.norm(x))
            st = Step(x=x.copy(), lam=lam, cost=cost, delta=delta, pred=pred, cost_trial=float("nan"), rho=float("nan"),
                      accepted=False, kappa_s=kappa, ginf=ginf, dx=dx, xn=xn, rel=float("nan"))
            steps.append(st)
            if ginf < gtol or dx < xtol * (xtol + xn):
                status = 1 if ginf < gtol else 3
                if block:
                    n_normal -= 1
                    n_cost += 1
                iterates.append(x.copy())
                break
            if not block:
                n_cost += 1
            c_new = self.cost(x + delta)
            actual = cost - c_new
            rho = actual / pred if (pred > 0.0 and math.isfinite(c_new)) else -1.0
            st.cost_trial, st.rho = c_new, rho
            if rho > 0.0:
                st.accepted = True
                rel = actual / max(cost, 1e-300)
                st.rel = rel
                cost = c_new
                lam = max(lambda_min, lam * max(1.0 / 3.0, 1.0 - (2.0 * rho - 1.0) ** 3))
                nu = 2.0
                x = x + delta
                if not block:
                    n_normal += 1
                iterates.append(x.copy())
                if rel < ftol:
                    status = 2
                    break
            else:
                if block:
                    n_normal -= 1
                    n_cost += 1
                lam = min(lambda_max, lam * nu)
                nu *= 2.0
                iterates.append(x.copy())
                if lam >= lambda_max:
                    status = -1
                    break
        return dict(x=x, iterations=it, status=status, cost_initial=0.5 * cost0, cost_final=0.5 * cost, lambda_final=lam,
                    n_eval_normal=n_normal, n_eval_cost=n_cost, steps=steps, iterates=iterates)


# ---- fixtures ----------------------------------------------------------------------------------------
@dataclasses.dataclass
class Fixture:
    name: str
    chain: int
    cam: np.ndarray
    pose: np.ndarray
    key: np.ndarray
    uv: np.ndarray
    C: int
    M: int
    K: int
    template: np.ndarray | None
    unfixed: np.ndarray
    params0: np.ndarray
    path: str = "block"

    @property
    def x0(self):
        return self.params0[self.unfixed]

    def oracle(self):
        return orc.Problem(self.chain, self.cam, self.pose, self.key, self.uv, self.C, self.M, self.K,
                           self.template if self.chain == 0 else None)

    def model(self, path=None):
        return LmModel(self.oracle(), self.unfixed, self.params0, path or self.path)

    def problem(self):
        from pycamset_b200.problem import BundleProblem
        p = BundleProblem(self.chain, self.cam, self.pose, self.key, self.uv, self.C, self.M, self.K,
                          template=self.template if self.chain == 0 else None, unfixed=self.unfixed)
        p.set_param_string(self.params0)
        return p

    def observed(self):
        """Boolean mask over the parameter string: does any observation depend on the entry?"""
        C, M = self.C, self.M
        seen = np.zeros(self.params0.shape[0], bool)
        for c in np.unique(self.cam):
            seen[9 * c:9 * c + 9] = True
            seen[9 * C + 6 * c:9 * C + 6 * c + 6] = True
        for m in np.unique(self.pose):
            seen[15 * C + 6 * m:15 * C + 6 * m + 6] = True
        if self.chain == 1:
            for k in np.unique(self.key):
                seen[15 * C + 6 * M + 3 * k:15 * C + 6 * M + 3 * k + 3] = True
        return seen


def _idx_intr(C, c, a):
    return 9 * c + a


def _idx_extr(C, c, a):
    return 9 * C + 6 * c + a


def _idx_pose(C, m, a):
    return 15 * C + 6 * m + a


def _rig_arrays(rig, drop=None):
    cam, pose, key, uv = rig.cam.numpy(), rig.pose.numpy(), rig.key.numpy(), rig.uv.numpy()
    if drop is not None:
        keep = ~drop(cam, pose, key)
        cam, pose, key, uv = cam[keep], pose[keep], key[keep], uv[keep]
    return (np.ascontiguousarray(cam), np.ascontiguousarray(pose), np.ascontiguousarray(key), np.ascontiguousarray(uv))


def small_template_rig(masks=False):
    """Template chain, pose elimination: a 4-camera ring x 6 poses, plus a fifth
    camera and a seventh pose that are free but never observed (identity rows; 15 C = 75 is padded to 96 in the reduced
    system).  Pose 0 is fixed.
    masks: partial masks as well -- k3, p1, p2 fixed on every camera, camera 1's intrinsics fixed, pose 4's rotation fixed
    and its translation free.
    """
    from pycamset_b200 import synthetic as syn
    C0, M0 = 4, 6
    rig = syn.make_rig(C0, M0, distortion=True, seed=2, detect_prob=0.7)
    intr, extr, poses = rig.perturbed(np.random.default_rng(2), 1e-2)
    C, M = C0 + 1, M0 + 1
    intr = np.vstack([intr, intr[:1]])
    extr = np.vstack([extr, 1.01 * extr[:1]])
    poses = np.vstack([poses, poses[1:2]])
    params = rig.param_string(intr, extr, poses)
    unfixed = np.ones(params.shape[0], bool)
    unfixed[_idx_pose(C, 0, 0):_idx_pose(C, 0, 6)] = False
    if masks:
        for c in range(C):
            unfixed[_idx_intr(C, c, 6):_idx_intr(C, c, 9)] = False      # p1, p2, k3
        unfixed[_idx_intr(C, 1, 0):_idx_intr(C, 1, 9)] = False
        unfixed[_idx_pose(C, 4, 0):_idx_pose(C, 4, 3)] = False
    return Fixture("rig4_template_masks" if masks else "rig4_template", 0, *_rig_arrays(rig), C, M, 81, rig.template, unfixed, params)


def intrinsics_fixed_rig():
    """The 4-camera ring with every intrinsic fixed at its true value and pose 0 fixed: the free vector (extrinsics and
    poses) is ~6 in size, the whole parameter string ~3e3 (focal lengths and principal points)."""
    from pycamset_b200 import synthetic as syn
    C, M = 4, 6
    rig = syn.make_rig(C, M, distortion=True, seed=2, detect_prob=0.7)
    _, extr, poses = rig.perturbed(np.random.default_rng(2), 1e-2)
    params = rig.param_string(rig.intr, extr, poses)
    unfixed = np.ones(params.shape[0], bool)
    unfixed[:9 * C] = False
    unfixed[_idx_pose(C, 0, 0):_idx_pose(C, 0, 6)] = False
    return Fixture("rig4_template_intr_fixed", 0, *_rig_arrays(rig), C, M, 81, rig.template, unfixed, params)


def golden_fixture(case):
    from tests.helpers import load_case
    g = load_case(case)
    dd = g["dd"]
    chain = g["chain"]
    return Fixture(case, chain, np.ascontiguousarray(dd[:, 0], np.int32), np.ascontiguousarray(dd[:, 1], np.int32),
                   np.ascontiguousarray(dd[:, 2], np.int32), np.ascontiguousarray(dd[:, 3:5]), int(g["n_cams"]),
                   int(g["n_poses"]), g["template"].shape[0], g["template"] if chain == 0 else None,
                   np.asarray(g["unfixed"], bool), np.asarray(g["param0"], np.float64))


def ring32_template():
    """The 32-camera ring x 300 poses of the sparse Schur plan test (every pose seen by about half of the cameras)."""
    from pycamset_b200 import synthetic as syn
    rig = syn.make_rig(32, 300, distortion=True, seed=3, detect_prob=0.9)
    intr, extr, poses = rig.perturbed(np.random.default_rng(5), 2e-3)
    params = rig.param_string(intr, extr, poses)
    unfixed = np.ones(params.shape[0], bool)
    unfixed[15 * 32:15 * 32 + 6] = False
    return Fixture("ring32_template", 0, *_rig_arrays(rig), 32, 300, 81, rig.template, unfixed, params)


def dome128_template():
    """128-camera dome, M = 40: more cameras than the Z kernel's camera window, n = 1920 (chunked Cholesky)."""
    from pycamset_b200 import synthetic as syn
    rig = syn.make_rig(128, 40, layout="dome", distortion=True, seed=7, detect_prob=0.9)
    intr, extr, poses = rig.perturbed(np.random.default_rng(7), 2e-3)
    params = rig.param_string(intr, extr, poses)
    unfixed = np.ones(params.shape[0], bool)
    unfixed[15 * 128:15 * 128 + 6] = False
    return Fixture("dome128_template", 0, *_rig_arrays(rig), 128, 40, 81, rig.template, unfixed, params)


def small_selfcal_rig():
    """Self-calibration chain, C = 4, M = 6, K = 81 (3 K > 6 M: points eliminated).  Gauge: pose 0 and camera 0's
    extrinsics fixed.  Partial point masks: the z coordinate of every fifth point and the whole of point 7 fixed;
    point 80 free but never observed."""
    from pycamset_b200 import synthetic as syn
    C, M, K = 4, 6, 81
    rig = syn.make_rig(C, M, distortion=True, seed=11, detect_prob=0.8)
    rng = np.random.default_rng(11)
    intr, extr, poses = rig.perturbed(rng, 3e-3)
    pts = rig.template + 2e-5 * rng.normal(size=rig.template.shape)
    params = rig.param_string(intr, extr, poses, points=pts)
    cam, pose, key, uv = _rig_arrays(rig, drop=lambda c, m, k: k == 80)
    unfixed = np.ones(params.shape[0], bool)
    unfixed[_idx_pose(C, 0, 0):_idx_pose(C, 0, 6)] = False
    unfixed[_idx_extr(C, 0, 0):_idx_extr(C, 0, 6)] = False
    p0 = 15 * C + 6 * M
    for k in range(0, K, 5):
        unfixed[p0 + 3 * k + 2] = False
    unfixed[p0 + 21:p0 + 24] = False
    return Fixture("rig4_selfcal_point_masks", 1, cam, pose, key, uv, C, M, K, None, unfixed, params)


# ---- error measures shared by the CPU and GPU tests ------------------------------------------------------------------
def backward_error(A, g, delta):
    """eta = |S (A d + g)| / (|S A S| |S^-1 d| + |S g|), S = diag(A)^-1/2."""
    s = 1.0 / np.sqrt(np.diag(A))
    As = A * s[:, None] * s[None, :]
    num = np.linalg.norm(s * (A @ delta + g))
    den = np.linalg.norm(As, 2) * np.linalg.norm(delta / s) + np.linalg.norm(s * g)
    return float(num / den)


def subtraction_floor(A, g, delta, x0, x1):
    """Backward error that the rounding of delta = x1 - x0 alone can cause: entries eps (|x0| + |x1|) through S A."""
    eps = np.finfo(np.float64).eps
    e = eps * (np.abs(x0) + np.abs(x1))
    s = 1.0 / np.sqrt(np.diag(A))
    As = A * s[:, None] * s[None, :]
    num = np.linalg.norm(s * (np.abs(A) @ e))
    den = np.linalg.norm(As, 2) * np.linalg.norm(delta / s) + np.linalg.norm(s * g)
    return float(num / den), float(np.linalg.norm(e * np.sqrt(np.diag(A))))


FIXTURES = {
    "rig4_template": lambda: small_template_rig(False),
    "rig4_template_masks": lambda: small_template_rig(True),
    "rig4_template_intr_fixed": intrinsics_fixed_rig,
    "ring5_fixedcam_template": lambda: golden_fixture("ring5_fixedcam_template"),
    "ccube_template": lambda: golden_fixture("ccube_template"),
    "ring32_template": ring32_template,
    "dome128_template": dome128_template,
    "rig4_selfcal_point_masks": small_selfcal_rig,
    "ring5_fixedcam_selfcal": lambda: golden_fixture("ring5_fixedcam_selfcal"),
    "ccube_selfcal": lambda: golden_fixture("ccube_selfcal"),
}

# Trajectory fixtures: (fixture, lambda0).  The first one has a rejected step with a meaningful gain ratio.
TRAJECTORIES = [("rig4_template", 1e-6), ("rig4_template_masks", 1e-6), ("ring5_fixedcam_template", 1e-3),
                ("ccube_template", 1e-3), ("rig4_selfcal_point_masks", 1e-3)]
REJECTING = ["rig4_template"]
N_TRAJ = 6

# Termination fixtures: (fixture, lambda0, dict(ftol, xtol, gtol), expected status, expected iterations).  Each tolerance
# lies between two consecutive values of its measure along the model's trajectory with a margin >= 10x on both sides.
TERMINATIONS = [
    ("rig4_template", 1e-6, dict(gtol=2.06e6, ftol=0.0, xtol=0.0), 1, 2),
    ("rig4_template", 1e-6, dict(ftol=2.8e-2, xtol=0.0, gtol=0.0), 2, 4),
    ("rig4_template_intr_fixed", 1e-6, dict(xtol=2.9e-6, ftol=0.0, gtol=0.0), 3, 3),
]
