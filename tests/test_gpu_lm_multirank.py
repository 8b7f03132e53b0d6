"""GPU: multi-rank LM == single-rank LM.

The pose-sharded solve (every rank eliminates its own poses, the Schur-reduced camera system and the step scalars are
summed across ranks through the `pcs_set_allreduce` hook, SURVEY.md 8e) must walk through the same iterates as the
unsharded solve.  Two emulations of world_size = 2:

  * one GPU: two BundleProblems (pose halves) driven from two host threads, the hook being a HOST-side sum (stream
    synchronise, copy out, thread barrier, add, copy back) -- no kernel ever waits on another kernel, so the ranks
    need not be co-resident (B200_PROFILING.md);
  * two GPUs (skipped below 2 devices): torchrun + NCCL through `install_nccl_allreduce`.

Tolerances: cost after k iterations rel <= 1e-10; x after k iterations |dx| <= 1e-9 max(1, |x|) for k <= 3 (only the
summation order of the reduced system differs) and rel <= 1e-6 at convergence."""
import os
import subprocess
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

C, M, K = 8, 40, 81


def _rig():
    from pycamset_b200 import synthetic as syn
    rig = syn.make_rig(C, M, layout="dome", distortion=True, seed=13, detect_prob=0.8)
    intr, extr, poses = rig.perturbed(np.random.default_rng(14), 1e-3)
    return rig, rig.param_string(intr, extr, poses)


def _single(rig, params, iters, tol):
    from pycamset_b200.problem import BundleProblem
    unfixed = np.ones(params.shape[0], bool)
    unfixed[15 * C:15 * C + 6] = False
    with BundleProblem(0, rig.cam.numpy(), rig.pose.numpy(), rig.key.numpy(), rig.uv.numpy(), C, M, K,
                       template=rig.template, unfixed=unfixed) as p:
        p.set_param_string(params)
        return p.lm_solve(params[unfixed], max_iter=iters, ftol=tol, xtol=tol, gtol=tol)


class _HostSum:
    """world-size-2 all-reduce on the host for two problems living on ONE device."""

    def __init__(self, world, device=0):
        import torch
        self.torch, self.world, self.device = torch, world, device
        self.barrier = threading.Barrier(world)
        self.slots = [None] * world

    def hook(self, rank):
        from pycamset_b200.distributed import tensor_from_ptr
        torch = self.torch

        def fn(ptr, n, op, stream):
            ext = torch.cuda.ExternalStream(stream, device=self.device)
            t = tensor_from_ptr(ptr, n, self.device)
            with torch.cuda.stream(ext):
                ext.synchronize()
                self.slots[rank] = t.cpu().numpy().copy()
                self.barrier.wait()
                parts = list(self.slots)
                self.barrier.wait()                       # everybody has read the slots before anyone overwrites
                tot = np.maximum.reduce(parts) if op == 1 else np.sum(parts, axis=0)   # rank order: identical on all ranks
                t.copy_(torch.from_numpy(tot))
                ext.synchronize()
        return fn


def _sharded_one_gpu(rig, params, iters, tol):
    from pycamset_b200 import distributed as pdist
    from pycamset_b200.problem import BundleProblem
    cam, pose, key, uv = rig.cam.numpy(), rig.pose.numpy(), rig.key.numpy(), rig.uv.numpy()
    ranges = pdist.balanced_pose_ranges(np.bincount(pose, minlength=M), 2)
    hs = _HostSum(2)
    out, err = [None, None], []

    def worker(r):
        try:
            c_s, p_s, k_s, uv_s = pdist.shard_observations(cam, pose, key, uv, ranges[r])
            par = pdist.shard_param_string(params, C, M, ranges[r])
            unfixed = np.ones(par.shape[0], bool)
            if ranges[r][0] == 0:
                unfixed[15 * C:15 * C + 6] = False
            with BundleProblem(0, c_s, p_s, k_s, uv_s, C, ranges[r][1] - ranges[r][0], K, template=rig.template,
                               unfixed=unfixed) as p:
                p.set_param_string(par)
                p.set_allreduce(hs.hook(r), r, 2)
                out[r] = p.lm_solve(par[unfixed], max_iter=iters, ftol=tol, xtol=tol, gtol=tol)
        except Exception as e:  # pragma: no cover
            err.append(e)
            hs.barrier.abort()

    ts = [threading.Thread(target=worker, args=(r,)) for r in range(2)]
    [t.start() for t in ts]
    [t.join(timeout=600) for t in ts]
    assert not err, err
    (x0, st0), (x1, st1) = out
    # gather the full free vector: cameras (replicated) + rank 0's free poses + rank 1's poses
    assert np.array_equal(x0[:15 * C], x1[:15 * C])      # the reduced system is bitwise identical on both ranks
    return np.concatenate([x0, x1[15 * C:]]), st0, st1


@pytest.mark.parametrize("iters", [1, 2, 3])
def test_two_ranks_walk_through_the_same_iterates(iters):
    rig, params = _rig()
    x_s, st_s = _single(rig, params, iters, 0.0)
    x_m, st0, st1 = _sharded_one_gpu(rig, params, iters, 0.0)
    assert st0["iterations"] == st1["iterations"] == st_s["iterations"] == iters
    for st in (st0, st1):
        assert abs(st["cost_final"] - st_s["cost_final"]) <= 1e-10 * st_s["cost_final"], (st, st_s)
        assert abs(st["cost_initial"] - st_s["cost_initial"]) <= 1e-12 * st_s["cost_initial"]
    assert x_m.shape == x_s.shape
    assert np.max(np.abs(x_m - x_s) / np.maximum(1.0, np.abs(x_s))) <= 1e-9


def test_two_ranks_converge_to_the_single_rank_optimum():
    rig, params = _rig()
    x_s, st_s = _single(rig, params, 60, 1e-13)
    x_m, st0, st1 = _sharded_one_gpu(rig, params, 60, 1e-13)
    assert st0["status"] == st1["status"] and st0["iterations"] == st1["iterations"]
    assert abs(st0["cost_final"] - st_s["cost_final"]) <= 1e-9 * st_s["cost_final"]
    assert np.max(np.abs(x_m - x_s) / np.maximum(1e-3, np.abs(x_s))) <= 1e-6


def test_two_gpus_nccl_match_single_rank(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    rig, params = _rig()
    x_s, st_s = _single(rig, params, 3, 0.0)
    out = tmp_path / "mp_lm_out.npz"
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29731", str(ROOT / "tests" / "mp_lm_worker.py"), str(out), "3"]
    subprocess.run(cmd, check=True, env=env, timeout=600)
    g = np.load(out)
    assert abs(float(g["cost_final"]) - st_s["cost_final"]) <= 1e-10 * st_s["cost_final"]
    assert np.max(np.abs(g["x"] - x_s) / np.maximum(1.0, np.abs(x_s))) <= 1e-9


def test_two_ranks_self_calibration_chain():
    """The self-calibration chain on the block path, pose-sharded: the target points are replicated like the cameras (their
    blocks are partial sums that enter the all-reduced system), the poses are local.  Same iterates as the single-rank
    solve.  (The dense fallback refuses world_size > 1; ADVICE round 1.)"""
    from pycamset_b200 import distributed as pdist
    from pycamset_b200.problem import BundleProblem
    from tests.helpers import load_case
    g = load_case("ring5_fixedcam_selfcal")
    dd = g["dd"]
    Cn, Mn, Kn = int(g["n_cams"]), int(g["n_poses"]), g["template"].shape[0]
    cam, pose, key, uv = dd[:, 0].astype(np.int32), dd[:, 1].astype(np.int32), dd[:, 2].astype(np.int32), dd[:, 3:5].copy()
    params, unfixed = g["param0"], np.asarray(g["unfixed"], bool)

    def solve_single(iters):
        with BundleProblem(1, cam, pose, key, uv, Cn, Mn, Kn, unfixed=unfixed) as p:
            p.set_param_string(params)
            x, st = p.lm_solve(g["x"], max_iter=iters, ftol=0.0, xtol=0.0, gtol=0.0)
            return p.get_param_string(), st

    ranges = pdist.balanced_pose_ranges(np.bincount(pose, minlength=Mn), 2)

    def solve_sharded(iters):
        hs = _HostSum(2)
        out, err = [None, None], []

        def worker(r):
            try:
                c_s, p_s, k_s, uv_s = pdist.shard_observations(cam, pose, key, uv, ranges[r])
                par = pdist.shard_param_string(params, Cn, Mn, ranges[r], n_keys=Kn)
                unf = pdist.shard_param_string(unfixed, Cn, Mn, ranges[r], n_keys=Kn).astype(bool)
                with BundleProblem(1, c_s, p_s, k_s, uv_s, Cn, ranges[r][1] - ranges[r][0], Kn, unfixed=unf) as p:
                    p.set_param_string(par)
                    # builds the solver workspace while the problem is still single-rank (it then plans to eliminate the
                    # points); installing the hook for two ranks frees it, and the solve rebuilds it for the pose elimination
                    assert p.lm_schur_fraction() == 1.0
                    p.set_allreduce(hs.hook(r), r, 2)
                    _, st = p.lm_solve(par[unf], max_iter=iters, ftol=0.0, xtol=0.0, gtol=0.0)
                    out[r] = (p.get_param_string(), st)
            except Exception as e:  # pragma: no cover
                err.append(e)
                hs.barrier.abort()

        ts = [threading.Thread(target=worker, args=(r,)) for r in range(2)]
        [t.start() for t in ts]
        [t.join(timeout=600) for t in ts]
        assert not err, err
        (p0, st0), (p1, st1) = out
        C15 = 15 * Cn
        full = np.concatenate([p0[:C15], p0[C15:C15 + 6 * (ranges[0][1] - ranges[0][0])], p1[C15:C15 + 6 * (ranges[1][1] - ranges[1][0])],
                               p0[C15 + 6 * (ranges[0][1] - ranges[0][0]):]])
        assert np.array_equal(p0[:C15], p1[:C15])                                    # cameras replicated
        assert np.array_equal(p0[-3 * Kn:], p1[-3 * Kn:])                            # points replicated
        return full, st0, st1

    for iters in (1, 3):
        ref, st = solve_single(iters)
        full, st0, st1 = solve_sharded(iters)
        assert st0["iterations"] == st1["iterations"] == st["iterations"]
        assert abs(st0["cost_final"] - st["cost_final"]) <= 1e-9 * st["cost_final"], (st0, st)
        assert np.max(np.abs(full - ref) / np.maximum(1.0, np.abs(ref))) <= 1e-8


def test_forced_dense_fallback_refuses_two_ranks():
    """The dense self-calibration fallback does not combine the ranks' normal equations, so a solve on it with world_size
    > 1 is refused -- also when PCS_LM_SELFCAL=dense forces it on a problem that has the block path."""
    from pycamset_b200 import _lib as L
    from tests import lm_reference as R
    from tests.helpers import solver_env
    fx = R.FIXTURES["ring5_fixedcam_selfcal"]()
    with solver_env(PCS_LM_SELFCAL="dense"), fx.problem() as p:
        p.set_allreduce(lambda ptr, n, op, stream: None, 0, 2)
        with pytest.raises(L.PcsError) as e:
            p.lm_solve(fx.x0, max_iter=1)
        assert e.value.code == L.PCS_ERR_UNSUPPORTED
