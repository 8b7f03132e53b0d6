"""torchrun worker of tests/test_gpu_p2p_exchange.py (one rank per GPU): the peer-memory camera-block exchange against NCCL."""
import json
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))


def main():
    out = sys.argv[1]
    from pycamset_b200 import distributed as pdist, synthetic as syn
    from pycamset_b200.problem import BundleProblem
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    rank, world = dist.get_rank(), dist.get_world_size()
    C, M = 8, 24
    # every rank evaluates its own observations (a different rig per rank: only the sum over ranks matters here)
    rig = syn.make_rig(C, M, distortion=True, seed=2 + rank)
    stream = torch.cuda.Stream(device=local)
    prob = BundleProblem(0, rig.cam.numpy(), rig.pose.numpy(), rig.key.numpy(), rig.uv.numpy(), C, M, 81, template=rig.template, device=local,
                         stream=stream.cuda_stream)
    prob.set_param_string(rig.param_string())
    p2p = pdist.P2PCameraAllReduce(prob)
    n = C * 240 + 1
    head = pdist.tensor_from_ptr(prob.device_buffers().U, n, local)
    worst = 0.0
    with torch.cuda.stream(stream):
        for it in range(9):                       # both data slots, several rounds of reuse
            prob.normal_equations_device()
            ref = head.clone()
            dist.all_reduce(ref)
            p2p()
            worst = max(worst, float(((head - ref).abs().max() / ref.abs().max()).item()))
            gathered = [torch.empty_like(head) for _ in range(world)]
            dist.all_gather(gathered, head)
            assert all(torch.equal(g, gathered[0]) for g in gathered), "ranks disagree bitwise"
    torch.cuda.synchronize(local)
    timed_out = prob.p2p_timed_out()
    if rank == 0:
        with open(out, "w") as f:
            json.dump({"rel_err": worst, "timed_out": bool(timed_out), "world": world}, f)
    prob.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
