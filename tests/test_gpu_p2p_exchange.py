"""2 GPUs (skipped below 2 devices): the one-shot peer-memory all-reduce of the camera blocks
(csrc/pcs_p2p.cu: "the data is the signal" with sentinel-initialised slots) against an NCCL all-reduce of the same data,
nine exchanges so that both slot sets are reused several times.
Bitwise identical on every rank, equal to NCCL to rounding (different summation order for world > 2 only)."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def test_peer_memory_exchange_matches_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "mp_p2p_out.json"
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29741", str(ROOT / "tests" / "mp_p2p_worker.py"), str(out)]
    subprocess.run(cmd, check=True, env=env, timeout=600)
    r = json.loads(out.read_text())
    assert r["world"] == 2 and not r["timed_out"]
    assert r["rel_err"] <= 1e-14, r
