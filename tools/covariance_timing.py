"""Time of the covariance call (pcs_covariance, pycamset_b200/csrc/pcs_cov.cu) on one GPU, next to the LM iteration time
of the same problem.

Workloads: config 4 (32-camera ring x 2000 poses) and config 5 (128-camera dome x 20 000 poses, detect_prob 0.5), built as
bench.py builds them (pose 0 is the gauge).  For each: the whole call (host clock around a call that ends in a device
synchronisation, best of --reps after a warm-up), its split into evaluate + factor / forward substitution / Gram + assembly
(device timestamps of one call under torch.profiler), and the forward substitution's FLOP count nc^2 (n_elim + nc) from the
shapes with its rate over the k_cov_forward kernel time.  The card's name and power limit are read in the same run.

    python tools/covariance_timing.py --out result.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

WORKLOADS = {"config4_ring32x2000": ("ring", 32, 2000, 1.0), "config5_dome128x20000": ("dome", 128, 20000, 0.5)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def build(layout, n_cams, n_poses, detect_prob, seed):
    from pycamset_b200 import synthetic as syn
    from pycamset_b200.problem import BundleProblem
    rig = syn.make_rig(n_cams, n_poses, layout=layout, distortion=True, seed=seed, detect_prob=detect_prob, device="cuda")
    intr, extr, poses = rig.perturbed(np.random.default_rng(seed + 1), 1e-3)
    params = np.concatenate([intr.ravel(), extr.ravel(), poses.ravel()])
    unfixed = np.ones(params.shape[0], bool)
    unfixed[15 * n_cams:15 * n_cams + 6] = False
    p = BundleProblem(0, rig.cam, rig.pose, rig.key, rig.uv, n_cams, n_poses, rig.n_keys, template=rig.template, unfixed=unfixed)
    p.set_param_string(params)
    return p, params[unfixed]


def phases(prof):
    """Device intervals of one call: [first kernel, k_cov_tile_inverse) / [k_cov_tile_inverse, end of k_cov_forward] /
    (end of k_cov_forward, last kernel or copy]."""
    ev = [e for e in prof.events() if e.device_type.name == "CUDA"]
    ev.sort(key=lambda e: e.time_range.start)
    t0, t1 = ev[0].time_range.start, max(e.time_range.end for e in ev)
    inv = next(e for e in ev if "k_cov_tile_inverse" in e.name)
    fwd = next(e for e in ev if "k_cov_forward" in e.name)
    us = lambda a, b: (b - a) * 1e-3   # noqa: E731
    return dict(evaluate_factor_ms=us(t0, inv.time_range.start), forward_substitution_ms=us(inv.time_range.start, fwd.time_range.end),
                gram_assembly_ms=us(fwd.time_range.end, t1), device_total_ms=us(t0, t1),
                k_cov_forward_ms=(fwd.time_range.end - fwd.time_range.start) * 1e-3)


def measure(name, seed, reps, lm_iters):
    import torch
    from torch.profiler import ProfilerActivity, profile
    layout, C, M, dp = WORKLOADS[name]
    p, x0 = build(layout, C, M, dp, seed)
    try:
        _, st = p.lm_solve(x0, max_iter=2, ftol=0.0, xtol=0.0, gtol=0.0)        # warm-up
        _, st = p.lm_solve(x0, max_iter=lm_iters, ftol=0.0, xtol=0.0, gtol=0.0)
        lm_ms = 1e3 * st["seconds"] / max(st["iterations"], 1)
        cov = p.covariance(x0)                                                 # warm-up (allocations, opt-ins)
        walls = []
        for _ in range(reps):
            t = time.perf_counter()
            cov = p.covariance(x0)
            walls.append(1e3 * (time.perf_counter() - t))
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            p.covariance(x0)
            torch.cuda.synchronize()
        ph = phases(prof)
    finally:
        p.close()
    nc = (15 * C + 31) // 32 * 32
    n_elim = 6 * M
    flops = float(nc) ** 2 * (n_elim + nc)
    return dict(n_cams=C, n_poses=M, n_obs=p.n_obs, nc=nc, n_elim=n_elim, call_ms_best=min(walls), call_ms_all=walls, **ph,
                forward_flop=flops, forward_tflops=flops / (ph["k_cov_forward_ms"] * 1e-3) / 1e12,
                lm_iteration_ms=lm_ms, lm_iterations=st["iterations"], call_over_lm_iteration=min(walls) / lm_ms,
                s2=cov["s2"], dof=cov["dof"])


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="JSON file to write (printed to stdout as well)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lm-iters", type=int, default=10)
    ap.add_argument("--workloads", nargs="*", default=list(WORKLOADS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("covariance_timing: no CUDA device")
    from pycamset_b200.build import build_library
    build_library()
    res = dict(card=card(), device=torch.cuda.get_device_name(0))
    for name in args.workloads:
        res[name] = measure(name, args.seed, args.reps, args.lm_iters)
        print(name, json.dumps(res[name]), flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
