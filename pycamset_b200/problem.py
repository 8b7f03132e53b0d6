"""BundleProblem: Python handle on one device-resident bundle-adjustment problem (thin over the C ABI).

Holds what the reference's compiled closures capture at build time (the observation table `dd`, the template
points, the gather / CSR structure: abstract_function_blocks.py:656-667) and exposes the per-call operations:
residual, CSR Jacobian, fused normal equations, LM solve.
"""
from __future__ import annotations

import ctypes as ct

import numpy as np

from . import _lib as L

CHAIN_NAMES = {
    L.CHAIN_TEMPLATE: "projection_extrinsic3D_template_points",
    L.CHAIN_SELFCAL: "projection_extrinsic3D_rigidTform3d_free_point",
}


def chain_id_from_blocks(block_names) -> int:
    """Tuple of function-block class names -> chain id.  The reference keys its generated kernels the same way
    (abstract_function_blocks.py:297).  Unknown chains raise UnknownChainError: there is no CPU fallback."""
    name = "_".join(block_names)
    rc = L.load().pcs_chain_from_name(name.encode())
    if rc < 0:
        L.check(rc)
    return rc


def free_map_from_mask(unfixed) -> np.ndarray:
    """Boolean mask over the parameter string -> free column index or -1 (the `conversion` renumbering of
    make_jac_CSR_columns_row_pointers, abstract_function_blocks.py:482-485)."""
    unfixed = np.asarray(unfixed, bool)
    fm = np.full(unfixed.shape[0], -1, np.int32)
    fm[unfixed] = np.arange(int(unfixed.sum()), dtype=np.int32)
    return fm


def _ptr(a):
    return None if a is None else ct.c_void_p(a.ctypes.data)


class BundleProblem:
    def __init__(self, chain, cam, pose, key, uv, n_cams, n_poses, n_keys, template=None, unfixed=None,
                 device=0, stream=None):
        """cam/pose/key/uv: numpy arrays (host) or torch CUDA tensors on `device` (int32 / float64).
        template: (K, 3) float64 host array (template chain).  unfixed: boolean mask over the parameter string."""
        lib = L.load()
        self._lib = lib
        self._h = ct.c_void_p()
        self.chain = int(chain)
        on_device = hasattr(cam, "data_ptr")
        keep = []
        if on_device:
            import torch
            def prep(t, dt):
                t = t.to(dtype=dt).contiguous()
                assert t.is_cuda and t.device.index == device, "device tensors must live on the problem's device"
                keep.append(t)
                return ct.c_void_p(t.data_ptr())
            n_obs = int(cam.shape[0])
            if not (int(pose.shape[0]) == n_obs and int(key.shape[0]) == n_obs and int(uv.numel()) == 2 * n_obs):
                raise ValueError("cam / pose / key / uv disagree on the number of observations")
            pc, pp, pk = prep(cam, torch.int32), prep(pose, torch.int32), prep(key, torch.int32)
            pu = prep(uv.reshape(-1), torch.float64)
            torch.cuda.synchronize(device)
        else:
            cam = np.ascontiguousarray(cam, np.int32); pose = np.ascontiguousarray(pose, np.int32)
            key = np.ascontiguousarray(key, np.int32); uv = np.ascontiguousarray(uv, np.float64).reshape(-1)
            keep += [cam, pose, key, uv]
            n_obs = int(cam.shape[0])
            if not (pose.shape[0] == n_obs and key.shape[0] == n_obs and uv.shape[0] == 2 * n_obs):
                raise ValueError("cam / pose / key / uv disagree on the number of observations")
            pc, pp, pk, pu = _ptr(cam), _ptr(pose), _ptr(key), _ptr(uv)
        n_params = 15 * n_cams + 6 * n_poses + (3 * n_keys if self.chain == L.CHAIN_SELFCAL else 0)
        fm = None
        if unfixed is not None:
            unfixed = np.asarray(unfixed, bool)
            if unfixed.shape[0] != n_params:
                raise ValueError(f"unfixed mask has length {unfixed.shape[0]}, parameter string has {n_params}")
            fm = free_map_from_mask(unfixed)
            keep.append(fm)
        tmpl = None
        if template is not None:
            tmpl = np.ascontiguousarray(template, np.float64).reshape(-1, 3)
            if tmpl.shape[0] != n_keys:
                raise ValueError("template must have n_keys rows")
            keep.append(tmpl)
        desc = L.ProblemDesc(chain=self.chain, device=device, n_obs=n_obs, n_cams=n_cams, n_poses=n_poses,
                             n_keys=n_keys, inputs_on_device=1 if on_device else 0, cam=pc, pose=pp, key=pk, uv=pu,
                             template_xyz=_ptr(tmpl), free_map=_ptr(fm),
                             stream=ct.c_void_p(stream) if stream else None)
        L.check(lib.pcs_problem_create(ct.byref(desc), ct.byref(self._h)))
        info = L.ProblemInfo()
        L.check(lib.pcs_problem_get_info(self._h, ct.byref(info)))
        self.n_obs, self.n_params, self.n_free, self.nnz = info.n_obs, info.n_params, info.n_free, info.nnz
        self.n_segments, self.cols_per_row = info.n_segments, info.cols_per_row
        self.n_cams, self.n_poses, self.n_keys, self.device = info.n_cams, info.n_poses, info.n_keys, info.device
        self._csr = None
        self._cb = None

    # ---- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.pcs_problem_destroy(self._h)
            self._h = ct.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- parameters ---------------------------------------------------------------------------------
    def set_param_string(self, params):
        params = np.ascontiguousarray(params, np.float64)
        if params.shape[0] != self.n_params:
            raise ValueError(f"parameter string has length {params.shape[0]}, expected {self.n_params}")
        L.check(self._lib.pcs_set_param_string(self._h, _ptr(params)))

    def get_param_string(self):
        out = np.empty(self.n_params)
        L.check(self._lib.pcs_get_param_string(self._h, _ptr(out)))
        return out

    def _x(self, x):
        if x is None:
            return None, None
        x = np.ascontiguousarray(x, np.float64)
        if x.shape[0] != self.n_free:
            raise ValueError(f"x has length {x.shape[0]}, expected n_free = {self.n_free}")
        return x, _ptr(x)

    # ---- per-call operations -----------------------------------------------------------------------------
    def residual(self, x=None, out=None):
        """(2N,) residuals, interleaved (x, y), dd row order; x=None evaluates at the current parameters."""
        xk, xp = self._x(x)
        r = np.empty(2 * self.n_obs) if out is None else out
        L.check(self._lib.pcs_residual(self._h, xp, _ptr(r)))
        return r

    def csr_structure(self):
        if self._csr is None:
            col = np.empty(self.nnz, np.int64)
            rp = np.empty(2 * self.n_obs + 1, np.int64)
            L.check(self._lib.pcs_csr_structure(self._h, _ptr(col), _ptr(rp)))
            self._csr = (col, rp)
        return self._csr

    def jacobian_values(self, x=None, out=None):
        xk, xp = self._x(x)
        v = np.empty(self.nnz) if out is None else out
        L.check(self._lib.pcs_jacobian_values(self._h, xp, _ptr(v)))
        return v

    def jacobian(self, x=None):
        """scipy csr_array (2N, n_free) like the reference's jac_fn (template_handler.py:188-193)."""
        from scipy.sparse import csr_array
        col, rp = self.csr_structure()
        return csr_array((self.jacobian_values(x), col, rp), shape=(2 * self.n_obs, self.n_free))

    def segments(self):
        S = self.n_segments
        sc = np.empty(S, np.int32); sp = np.empty(S, np.int32); sl = np.empty(S, np.int64)
        L.check(self._lib.pcs_segments(self._h, _ptr(sc), _ptr(sp), _ptr(sl)))
        return sc, sp, sl

    def normal_equations(self, x=None, with_W=True, out=None):
        """Fused residual + Jacobian + J^T J / J^T r blocks (both chains; the self-calibration chain adds the point blocks
        Pk, gk, Xck, Ymk).  Returns dict of host arrays.
        `out` may hold preallocated (e.g. pinned) arrays U, gc, V, gp, W, cost_buf to receive the copies."""
        xk, xp = self._x(x)
        C, M, S = self.n_cams, self.n_poses, self.n_segments
        out = out or {}
        U = out.get("U", None); gc = out.get("gc", None); V = out.get("V", None); gp = out.get("gp", None)
        U = np.empty((C, 15, 15)) if U is None else U
        gc = np.empty((C, 15)) if gc is None else gc
        V = np.empty((M, 6, 6)) if V is None else V
        gp = np.empty((M, 6)) if gp is None else gp
        W = out.get("W", None)
        if W is None and with_W:
            W = np.empty((S, 15, 6))
        cost = out.get("cost_buf", None)
        cost = np.empty(1) if cost is None else cost
        L.check(self._lib.pcs_normal_equations(self._h, xp, _ptr(U), _ptr(gc), _ptr(V), _ptr(gp), _ptr(W), _ptr(cost)))
        res = dict(U=U, gc=gc, V=V, gp=gp, W=W, cost=float(cost[0]))
        if self.chain == L.CHAIN_SELFCAL:
            K = self.n_keys
            res.update(Pk=np.empty((K, 3, 3)), gk=np.empty((K, 3)), Xck=np.empty((C, K, 15, 3)), Ymk=np.empty((M, K, 6, 3)))
            L.check(self._lib.pcs_point_blocks(self._h, _ptr(res["Pk"]), _ptr(res["gk"]), _ptr(res["Xck"]), _ptr(res["Ymk"])))
        return res

    def set_normal_precision(self, mixed: bool):
        """False (default): FP64 blocks.  True: gradients / cost / residual stay FP64, the J^T J blocks come from the
        BF16-split tensor path (they only precondition the LM step; include/pcs_b200.h)."""
        L.check(self._lib.pcs_set_normal_precision(self._h, L.PRECISION_MIXED if mixed else L.PRECISION_FP64))

    def normal_equations_device(self, x_dev_ptr=None):
        """Evaluate into the device-resident block buffers (no host copies, no synchronisation)."""
        L.check(self._lib.pcs_normal_equations_dev(self._h, ct.c_void_p(x_dev_ptr) if x_dev_ptr else None))

    def residual_device(self, r_dev_ptr, x_dev_ptr=None):
        L.check(self._lib.pcs_residual_dev(self._h, ct.c_void_p(x_dev_ptr) if x_dev_ptr else None, ct.c_void_p(r_dev_ptr)))

    def jacobian_values_device(self, vals_dev_ptr, x_dev_ptr=None):
        L.check(self._lib.pcs_jacobian_values_dev(self._h, ct.c_void_p(x_dev_ptr) if x_dev_ptr else None,
                                                  ct.c_void_p(vals_dev_ptr)))

    def normal_dense(self, x=None):
        xk, xp = self._x(x)
        n = self.n_free
        JtJ = np.empty((n, n)); Jtr = np.empty(n); cost = np.empty(1)
        L.check(self._lib.pcs_normal_dense(self._h, xp, _ptr(JtJ), _ptr(Jtr), _ptr(cost)))
        return JtJ, Jtr, float(cost[0])

    def device_buffers(self) -> L.DeviceBuffers:
        b = L.DeviceBuffers()
        L.check(self._lib.pcs_device_buffers_get(self._h, ct.byref(b)))
        return b

    def lm_schur_fraction(self) -> float:
        """Fraction of the (tile pair, slab) units the block-sparse pose elimination of lm_solve visits (1.0 = dense)."""
        f = ct.c_double()
        L.check(self._lib.pcs_lm_schur_fraction(self._h, ct.byref(f)))
        return f.value

    def timing_enable(self, on=True):
        L.check(self._lib.pcs_timing_enable(self._h, 1 if on else 0))

    def timing_normal_kernel_ms(self) -> float:
        ms = ct.c_double()
        L.check(self._lib.pcs_timing_get(self._h, ct.byref(ms)))
        return ms.value

    def timing_all_ms(self, capacity=1024) -> np.ndarray:
        """Durations (ms) of the normal-equation kernel launches since timing_enable(True), oldest first."""
        out = np.empty(capacity)
        n = ct.c_int64()
        L.check(self._lib.pcs_timing_get_all(self._h, _ptr(out), capacity, ct.byref(n)))
        return out[:n.value].copy()

    def launch_count(self) -> int:
        n = ct.c_int64()
        L.check(self._lib.pcs_launch_count(self._h, ct.byref(n)))
        return n.value

    def costfn(self, im_points, proj, ints, dists, errors=True, per_image=True):
        """Initialiser cost evaluation over all candidate tables at once (pcs_costfn).
        im_points: (B, M, K, 3) or (M, K, 3).  Returns (errors (B, 2N) or None, per_image (B, M) or None)."""
        im_points = np.ascontiguousarray(im_points, np.float64)
        if im_points.ndim == 3:
            im_points = im_points[None]
        B = im_points.shape[0]
        if im_points.shape[1:] != (self.n_poses, self.n_keys, 3):
            raise ValueError(f"im_points must be (B, {self.n_poses}, {self.n_keys}, 3), got {im_points.shape}")
        proj = np.ascontiguousarray(proj, np.float64); ints = np.ascontiguousarray(ints, np.float64)
        dists = np.ascontiguousarray(np.asarray(dists, np.float64).reshape(-1, 5))
        if proj.shape != (self.n_cams, 3, 4) or ints.shape != (self.n_cams, 3, 3) or dists.shape[0] != self.n_cams:
            raise ValueError("proj / ints / dists must be (C, 3, 4) / (C, 3, 3) / (C, 5)")
        e = np.empty((B, 2 * self.n_obs)) if errors else None
        pi = np.empty((B, self.n_poses)) if per_image else None
        L.check(self._lib.pcs_costfn(self._h, B, _ptr(im_points), _ptr(proj), _ptr(ints), _ptr(dists), _ptr(e), _ptr(pi)))
        return e, pi

    def p2p_buffer_bytes(self, world_size) -> int:
        return int(self._lib.pcs_p2p_buffer_bytes(self._h, int(world_size)))

    def p2p_setup(self, rank, world_size, peer_ptrs, buffer_bytes):
        arr = (ct.c_void_p * world_size)(*[ct.c_void_p(int(q)) for q in peer_ptrs])
        L.check(self._lib.pcs_p2p_allreduce_setup(self._h, int(rank), int(world_size), arr, int(buffer_bytes)))

    def p2p_allreduce_camera_blocks(self):
        L.check(self._lib.pcs_p2p_allreduce_camera_blocks(self._h))

    def p2p_timed_out(self) -> bool:
        """True if a poll of the peer-memory exchange ever gave up waiting for a peer (synchronises the stream)."""
        f = ct.c_int()
        L.check(self._lib.pcs_p2p_status(self._h, ct.byref(f)))
        return bool(f.value)

    def set_allreduce(self, fn, rank, world_size):
        """fn(ptr:int, n:int, op:int, stream:int) -> None; installed as the multi-GPU combine hook of the LM solver."""
        def _cb(user, buf, n, op, stream):
            try:
                fn(int(buf), int(n), int(op), int(stream or 0))
                return 0
            except Exception:  # never let an exception cross the C boundary
                import traceback
                traceback.print_exc()
                return 1
        self._cb = L.ALLREDUCE_FN(_cb)
        L.check(self._lib.pcs_set_allreduce(self._h, self._cb, None, int(rank), int(world_size)))

    def covariance(self, x=None):
        """Unit-weight covariance H^-1 (H = J^T J over the free parameters) at x (None: the current parameters), in the
        parts pcs_covariance returns: cam (15 C, 15 C), pose (M, 6, 6), point (K, 3, 3; self-calibration chain), the
        residual variance s2 = r.r / dof and dof.  Entries of fixed parameters are 0, of unobserved ones NaN."""
        xk, xp = self._x(x)
        C, M, K = self.n_cams, self.n_poses, self.n_keys
        cam, pose = np.empty((15 * C, 15 * C)), np.empty((M, 6, 6))
        point = np.empty((K, 3, 3)) if self.chain == L.CHAIN_SELFCAL else None
        s2, dof = ct.c_double(), ct.c_int64()
        L.check(self._lib.pcs_covariance(self._h, xp, _ptr(cam), _ptr(pose), _ptr(point), ct.byref(s2), ct.byref(dof)))
        res = dict(cam=cam, pose=pose, s2=s2.value, dof=dof.value)
        if point is not None:
            res["point"] = point
        return res

    def lm_solve(self, x0, max_iter=100, ftol=1e-8, xtol=1e-8, gtol=1e-8, lambda0=1e-3, verbose=0):
        x0k, x0p = self._x(x0)
        opts = L.LmOptions()
        self._lib.pcs_lm_default_options(ct.byref(opts))
        opts.max_iter, opts.ftol, opts.xtol, opts.gtol, opts.lambda0, opts.verbose = max_iter, ftol, xtol, gtol, lambda0, verbose
        stats = L.LmStats()
        x = np.empty(self.n_free)
        L.check(self._lib.pcs_lm_solve(self._h, x0p, ct.byref(opts), _ptr(x), ct.byref(stats)))
        return x, {f[0]: getattr(stats, f[0]) for f in L.LmStats._fields_}
