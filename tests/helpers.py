"""Shared helpers for the parity tests (oracle side only; test infrastructure)."""
from __future__ import annotations

import contextlib
import os
from pathlib import Path

import numpy as np

from oracle import oracle as orc

GOLDEN = Path(__file__).resolve().parent / "golden"

SYNTH_CASES = ["ring4_template", "ring4_selfcal", "ring5_fixedcam_template", "ring5_fixedcam_selfcal"]
CCUBE_CASES = ["ccube_template", "ccube_selfcal"]


def available(cases):
    return [c for c in cases if (GOLDEN / f"{c}.npz").exists()]


def load_case(name):
    g = dict(np.load(GOLDEN / f"{name}.npz"))
    g["chain"] = int(g["chain"])
    return g


def oracle_problem(g):
    """oracle.Problem sized like the handler arrays (C, M from the golden, not from data maxima)."""
    chain = g["chain"]
    K = g["template"].shape[0]
    return orc.Problem.from_dd(chain, g["dd"], template=g["template"] if chain == 0 else None,
                               C=int(g["n_cams"]), M=int(g["n_poses"]), K=K)


def rel_err(a, b, floor=1e-12):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)) if a.size else 0.0


@contextlib.contextmanager
def solver_env(**switches):
    """Exactly the given PCS_LM_* solver switches inside the block (the library reads them when it builds a problem's
    solver workspace), the caller's environment restored on exit."""
    saved = {k: os.environ.pop(k) for k in list(os.environ) if k.startswith("PCS_LM_")}
    os.environ.update(switches)
    try:
        yield
    finally:
        for k in switches:
            os.environ.pop(k, None)
        os.environ.update(saved)
