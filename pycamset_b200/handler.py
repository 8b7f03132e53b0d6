"""Host-side mirror of the reference's optimiser interface for the bundle-adjustment hot path.

The reference asks a parameter handler for two closures and hands them to scipy
(pyCamSet/optimisation/optimisation_handling.py:24-49, :52-117):

    loss_fun(x) -> float64[2N]           (template_handler.py:157-170, standard_bundle_handler.py:184-198)
    jac_fn(x)   -> csr_array (2N, n_free) (template_handler.py:172-193, standard_bundle_handler.py:200-226)

`GpuBundleHandler` wraps ANY reference handler instance (TemplateBundleHandler, SelfBundleHandler or a user
subclass: the extensibility hook of examples/extend_param_handler.py) and returns closures with exactly those
signatures, evaluated by the CUDA library.  Everything the handler owns stays the handler's: its `op_fun` chain
names the kernels, its `bundlePrimitive` masks give the fixed parameters, `get_detection_data` /
`return_flattened_keys` gives the observation table, `get_bundle_adjustment_inputs` + `op_fun.build_param_list`
turn x into the parameter string.  The module never imports pyCamSet: handlers are used through those attributes
only, so the same code runs where the reference is not installed (tests use a duck-typed handler).

    from pycamset_b200.handler import run_bundle_adjustment          # same name, same return contract
    result, camset = run_bundle_adjustment(param_handler, threads=16)

Unknown function-block chains raise UnknownChainError: there is no CPU fallback.
"""
from __future__ import annotations

import logging
import time

import numpy as np

from . import _lib as L
from .problem import BundleProblem, chain_id_from_blocks

_STOCK_INPUTS = ("TemplateBundleHandler.get_bundle_adjustment_inputs", "SelfBundleHandler.get_bundle_adjustment_inputs")


class OptimizeResult(dict):
    """Attribute + item access like scipy.optimize.OptimizeResult (camera_set.py:700-702 reads it dict-style)."""

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as e:
            raise AttributeError(name) from e

    __setattr__ = dict.__setitem__


def chain_block_names(op_fun):
    """Tuple of block class names, the key the reference uses for its generated kernels
    (abstract_function_blocks.py:297, :504)."""
    return tuple(type(b).__name__ for b in op_fun.function_blocks)


def unfixed_mask(bundle_primitive) -> np.ndarray:
    """Boolean mask over the parameter string: the reference builds the same array in make_loss_jac
    (template_handler.py:176-183; standard_bundle_handler.py:209-217)."""
    parts = [np.repeat(np.asarray(bundle_primitive.intr_unfixed, bool), 9),
             np.repeat(np.asarray(bundle_primitive.extr_unfixed, bool), 6),
             np.repeat(np.asarray(bundle_primitive.poses_unfixed, bool), 6)]
    if hasattr(bundle_primitive, "bdpt_unfixed"):
        parts.append(np.asarray(bundle_primitive.bdpt_unfixed, bool))
    return np.concatenate(parts)


def detection_table(handler) -> np.ndarray:
    """The flattened observation table `dd` (N x 5: cam, image, flat key, u, v) exactly as the reference's closures
    build it: `self.detection.return_flattened_keys(target_shape[:-1]).get_data()` -- UNFILTERED, i.e. rows of
    `missing_poses` are kept (template_handler.py:160-163, :175; target_detections.py:333-351), so residual length and
    row order equal those of the closures this module replaces.  `get_detection_data(flatten=True)` (which deletes the
    rows of missing poses, :398-403) is only the fallback for handlers that expose no `detection` object."""
    det = getattr(handler, "detection", None)
    if det is not None and hasattr(det, "return_flattened_keys"):
        shape = handler.target.point_data.shape
        return np.asarray(det.return_flattened_keys(shape[:-1]).get_data(), np.float64)
    return np.asarray(handler.get_detection_data(flatten=True), np.float64)


def export_problem(handler) -> dict:
    """Everything the device needs from a reference handler, as plain host arrays (no CUDA involved): the block
    names of the chain, the observation table, the template, the fixed-parameter mask and the problem sizes."""
    bp = handler.bundlePrimitive
    template = np.ascontiguousarray(handler.target.point_data, np.float64).reshape(-1, 3)
    fn = getattr(handler.get_bundle_adjustment_inputs, "__func__", None)
    return dict(blocks=chain_block_names(handler.op_fun), dd=detection_table(handler), template=template,
                unfixed=unfixed_mask(bp), n_cams=int(bp.intr.shape[0]), n_poses=int(bp.poses.shape[0]),
                n_keys=int(template.shape[0]), stock_mapping=getattr(fn, "__qualname__", "") in _STOCK_INPUTS)


class GpuBundleHandler:
    """CUDA-backed closures for one reference parameter handler."""

    def __init__(self, handler, device: int = 0, stream=None):
        self.handler = handler
        e = export_problem(handler)
        self.blocks = e["blocks"]
        self.chain = chain_id_from_blocks(self.blocks)          # raises UnknownChainError for unknown chains
        dd = self.dd = e["dd"]
        self.n_cams, self.n_poses, self.n_keys, self.unfixed = e["n_cams"], e["n_poses"], e["n_keys"], e["unfixed"]
        # the handler maps x -> arrays itself when a subclass overrides get_bundle_adjustment_inputs; the stock
        # mapping (fill_flat of the free rows, compiled_helpers.py:155-177) is done on the device instead
        self.stock_mapping = e["stock_mapping"]
        self.problem = BundleProblem(self.chain, dd[:, 0], dd[:, 1], dd[:, 2], dd[:, 3:5], self.n_cams, self.n_poses,
                                     self.n_keys, template=e["template"] if self.chain == L.CHAIN_TEMPLATE else None,
                                     unfixed=self.unfixed, device=device, stream=stream)
        self._have_fixed = False

    # ---- x -> device parameters -------------------------------------------------------------------
    def param_string(self, x) -> np.ndarray:
        """x -> full parameter string through the handler's own mapping (abstract_function_blocks.py:669-681)."""
        inps = self.handler.get_bundle_adjustment_inputs(np.asarray(x, np.float64))
        return self.handler.op_fun.build_param_list(*inps)

    def _load(self, x):
        """Returns the x to pass to the device call (None = parameters already loaded as a full string)."""
        x = np.ascontiguousarray(x, np.float64)
        if not self.stock_mapping:
            self.problem.set_param_string(self.param_string(x))
            return None
        if not self._have_fixed:      # fixed entries (and anything a subclass pre-populated) are uploaded once
            self.problem.set_param_string(self.param_string(x))
            self._have_fixed = True
        return x

    # ---- the two closures of make_optimisation_function ---------------------------------------------
    def make_loss_fun(self, threads: int = 1):
        """`threads` is accepted for signature compatibility; the device ignores it."""
        def loss_fun(params):
            return self.problem.residual(self._load(params))
        return loss_fun

    def make_loss_jac(self, threads: int = 1):
        from scipy.sparse import csr_array
        col, rp = self.problem.csr_structure()
        shape = (2 * self.problem.n_obs, self.problem.n_free)

        def jac_fn(params):
            return csr_array((self.problem.jacobian_values(self._load(params)), col, rp), shape=shape)
        return jac_fn

    def can_make_jac(self) -> bool:
        return True

    def get_initial_params(self):
        return self.handler.get_initial_params()

    # ---- beyond the reference: normal equations and the LM solve on the device ------------------------
    def normal_equations(self, params):
        return self.problem.normal_equations(self._load(params))

    def solve(self, x0=None, max_nfev=None, ftol=1e-8, xtol=1e-8, gtol=1e-8, verbose=0):
        if x0 is None:
            x0 = self.handler.get_initial_params()
        if max_nfev is None:
            max_nfev = int(getattr(self.handler, "problem_opts", {}).get("max_nfev", 100))
        if not self.stock_mapping:
            raise L.PcsError(L.PCS_ERR_UNSUPPORTED,
                             "the device LM solver updates the reference's free vector directly; handlers that "
                             "override get_bundle_adjustment_inputs must use the loss_fun / jac_fn closures")
        x = self._load(x0)
        return self.problem.lm_solve(x, max_iter=max_nfev, ftol=ftol, xtol=xtol, gtol=gtol, verbose=verbose)

    def covariance(self, x):
        """Covariance of the least-squares estimate at x (the reference's free vector): the unit-weight blocks of
        BundleProblem.covariance scaled by s2 = r.r / dof -- cam (15 C, 15 C), pose (M, 6, 6), point (K, 3, 3;
        self-calibration chain) -- with s2, dof and `param_std`, the standard deviation of every entry of x in x order
        (NaN for a parameter no observation depends on)."""
        cov = self.problem.covariance(self._load(x))
        s2 = cov["s2"]
        out = {k: s2 * cov[k] for k in ("cam", "pose", "point") if k in cov}
        C, M = self.n_cams, self.n_poses
        var = np.zeros(self.problem.n_params)
        d = np.diagonal(cov["cam"]).reshape(C, 15)
        var[:9 * C] = d[:, :9].ravel()
        var[9 * C:15 * C] = d[:, 9:].ravel()
        var[15 * C:15 * C + 6 * M] = np.diagonal(cov["pose"], axis1=1, axis2=2).ravel()
        if "point" in cov:
            var[15 * C + 6 * M:] = np.diagonal(cov["point"], axis1=1, axis2=2).ravel()
        out.update(s2=s2, dof=cov["dof"], param_std=np.sqrt(s2 * var[self.unfixed]))
        return out

    def get_camset(self, x):
        """The reference handler's own get_camset(x) (camera objects are the reference's).  For the self-calibration
        handler its post-solve gauge transform (standard_bundle_handler.py:339-410) is routed through
        pycamset_b200.gauge for the duration of the call -- same arithmetic, the O(K^2) pair search on the GPU."""
        h = self.handler
        if not hasattr(h, "get_camset"):
            return None
        if not (hasattr(h, "apply_gauge_transform") and hasattr(h, "visible_feature_mask")):
            return h.get_camset(x)
        from . import gauge
        device = self.problem.device
        h.apply_gauge_transform = lambda proj, extr, poses, pts: gauge.apply_gauge_transform_for(h, proj, extr, poses, pts, device)
        try:
            return h.get_camset(x)
        finally:
            del h.apply_gauge_transform          # back to the class's method

    def close(self):
        self.problem.close()


def make_optimisation_function(param_handler, threads: int = 1, device: int = 0):
    """Same contract as optimisation_handling.make_optimisation_function (:24-49): (loss_fun, jac_fn, x0)."""
    gpu = param_handler if isinstance(param_handler, GpuBundleHandler) else GpuBundleHandler(param_handler, device=device)
    init_params = gpu.get_initial_params()
    return gpu.make_loss_fun(threads), gpu.make_loss_jac(threads), init_params


JAC_AUTO_LIMIT_BYTES = 2 << 30   # jac="auto": the explicit CSR Jacobian is formed at the solution only below this size


def run_bundle_adjustment(param_handler, threads: int = 1, device: int = 0, solver: str = "lm", ftol=1e-8, xtol=1e-8,
                          gtol=1e-8, jac="auto", covariance=False):
    """Drop-in for optimisation_handling.run_bundle_adjustment (:52-117): returns (result, camset).

    solver="lm"    Levenberg-Marquardt on the device (block normal equations + Schur complement).
    solver="scipy" scipy.optimize.least_squares driven by the CUDA closures, i.e. the reference's own solver
                   (TRF + LSMR, x_scale='jac', max_nfev from the handler) with only the callbacks replaced.
    `result` carries x, fun, jac, cost, nfev, status like scipy's OptimizeResult.

    jac (solver="lm"): the device solver never forms the Jacobian; `result.jac` is evaluated once at the solution because
    the reference stores it with the camera set (camera_set.py:700-703) and writes it to the .camset file
    (utils/saving.py:143-147).  At 10^8 observations that matrix is tens of GB (SURVEY.md 8f rank 4), so: True = always,
    False = never, "auto" = only below JAC_AUTO_LIMIT_BYTES of CSR values.  When it is skipped `result.jac` is None (the
    reference's save_camset then omits it, as it does for any result without a usable Jacobian) and
    `result.normal_blocks` holds the block diagonal of J^T J at the solution instead -- U [C][15][15], V [M][6][6], gc,
    gp, cost: O(C + M) numbers.

    covariance=True: `result["covariance"]` holds GpuBundleHandler.covariance(result.x) -- the scaled covariance blocks,
    s2, dof and the standard deviation of every free parameter -- for either solver."""
    gpu = param_handler if isinstance(param_handler, GpuBundleHandler) else GpuBundleHandler(param_handler, device=device)
    handler = gpu.handler
    loss_fn, jac_fn = gpu.make_loss_fun(threads), gpu.make_loss_jac(threads)
    x0 = np.asarray(gpu.get_initial_params(), np.float64)
    init_err = loss_fn(x0)
    init_euclid = float(np.mean(np.linalg.norm(init_err.reshape(-1, 2), axis=1)))
    logging.info(f"found {len(x0):.2e} parameters")
    logging.info(f"found {len(init_err):.2e} control points")
    logging.info(f"Initial Euclidean error: {init_euclid:.2f} px")
    if init_euclid > 150 or np.isnan(init_euclid):
        logging.critical("Found worryingly high/NaN initial error: check that the initial parametisation is sensible")
    opts = getattr(handler, "problem_opts", {})
    max_nfev = int(opts.get("max_nfev", 100))
    start = time.time()
    if solver == "scipy":
        from scipy.optimize import least_squares
        result = least_squares(loss_fn, x0, verbose=opts.get("verbosity", 0), jac=jac_fn, max_nfev=max_nfev, x_scale="jac")
    elif solver == "lm":
        x, st = gpu.solve(x0, max_nfev=max_nfev, ftol=ftol, xtol=xtol, gtol=gtol, verbose=1 if opts.get("verbosity", 0) > 1 else 0)
        fun = loss_fn(x)
        want_jac = bool(jac) if jac != "auto" else 8 * int(gpu.problem.nnz) <= JAC_AUTO_LIMIT_BYTES
        result = OptimizeResult(x=x, fun=fun, jac=jac_fn(x) if want_jac else None, cost=0.5 * float(fun @ fun),
                                nfev=st["n_eval_normal"] + st["n_eval_cost"], njev=st["n_eval_normal"], status=st["status"],
                                success=st["status"] > 0, optimality=st["grad_norm_inf"], message="device Levenberg-Marquardt", lm=st)
        if not want_jac:
            ne = gpu.problem.normal_equations(x, with_W=False)
            result["normal_blocks"] = {k: ne[k] for k in ("U", "gc", "V", "gp", "cost")}
    else:
        raise ValueError("solver must be 'lm' or 'scipy'")
    if covariance:
        result["covariance"] = gpu.covariance(result.x)
    end = time.time()
    final_euclid = float(np.mean(np.linalg.norm(np.reshape(result.fun, (-1, 2)), axis=1)))
    logging.info(f"Final Euclidean error: {final_euclid:.2f} px")
    logging.info(f"Optimisation took {end - start: .2f} seconds.")
    if final_euclid > 5:
        logging.critical("Remaining error is very large: please check the output results")
    camset = gpu.get_camset(result.x)
    if camset is not None and hasattr(camset, "set_calibration_history"):
        camset.set_calibration_history(result, handler)
    return result, camset


def run_bundle_adjustment_sharded(param_handler, device=None, group=None, ftol=1e-8, xtol=1e-8, gtol=1e-8):
    """run_bundle_adjustment over the ranks of a torch.distributed process group, one process per GPU (template chain).

    Every rank calls this with the same handler.  The observations are sharded by target pose, every rank eliminates its
    own poses, the Schur-reduced camera system is all-reduced over NCCL (SURVEY.md 8e) and the pose blocks of the
    solution are all-gathered, so `result.x` is the FULL free vector on every rank -- the same return contract as
    run_bundle_adjustment: (result, camset)."""
    import torch
    from . import distributed as pdist
    e = export_problem(param_handler)
    if chain_id_from_blocks(e["blocks"]) != L.CHAIN_TEMPLATE:
        raise L.PcsError(L.PCS_ERR_UNSUPPORTED, "the sharded entry point covers the template chain")
    if not e["stock_mapping"]:
        raise L.PcsError(L.PCS_ERR_UNSUPPORTED, "handlers that override get_bundle_adjustment_inputs must use the closures")
    x0 = np.asarray(param_handler.get_initial_params(), np.float64)
    params = np.asarray(param_handler.op_fun.build_param_list(*param_handler.get_bundle_adjustment_inputs(x0)), np.float64)
    dd = e["dd"]
    opts = getattr(param_handler, "problem_opts", {})
    start = time.time()
    full, st = pdist.lm_solve_sharded(dd[:, 0].astype(np.int32), dd[:, 1].astype(np.int32), dd[:, 2].astype(np.int32), dd[:, 3:5],
                                      e["n_cams"], e["n_poses"], e["n_keys"], e["template"], params, e["unfixed"],
                                      device=torch.cuda.current_device() if device is None else device, group=group,
                                      max_iter=int(opts.get("max_nfev", 100)), ftol=ftol, xtol=xtol, gtol=gtol)
    x = full[e["unfixed"]]
    result = OptimizeResult(x=x, cost=st["cost_final"], nfev=st["n_eval_normal"] + st["n_eval_cost"], njev=st["n_eval_normal"],
                            status=st["status"], success=st["status"] > 0, optimality=st["grad_norm_inf"],
                            message="device Levenberg-Marquardt, pose-sharded", lm=st, seconds=time.time() - start)
    camset = param_handler.get_camset(x) if hasattr(param_handler, "get_camset") else None
    return result, camset


class GpuCostFn:
    """Drop-in for compiled_helpers.bundle_adjustment_costfn as estimate_camera_relative_poses uses it
    (template_handler.py:510-593): the observation table is uploaded once, every call scores one or many candidate
    pose tables.

        cost = GpuCostFn(dd, n_cams, n_poses, n_keys)
        errors = cost(imlocs, proj, ints, dists)                        # (2N,) like the reference
        errors, per_image = cost.batch(tables, proj, ints, dists)       # all candidates at once, per-image sums on the GPU
    """

    def __init__(self, dd, n_cams, n_poses, n_keys, device: int = 0):
        dd = np.asarray(dd, np.float64)
        self.problem = BundleProblem(L.CHAIN_TEMPLATE, dd[:, 0], dd[:, 1], dd[:, 2], dd[:, 3:5], n_cams, n_poses, n_keys,
                                     template=np.zeros((n_keys, 3)), device=device)

    def __call__(self, im_points, projection_matrixes, intrinsics, dists):
        e, _ = self.problem.costfn(np.asarray(im_points).reshape(self.problem.n_poses, self.problem.n_keys, 3),
                                   projection_matrixes, intrinsics, dists, errors=True, per_image=False)
        return e[0]

    def batch(self, tables, projection_matrixes, intrinsics, dists, errors=True):
        return self.problem.costfn(tables, projection_matrixes, intrinsics, dists, errors=errors, per_image=True)

    def close(self):
        self.problem.close()
