"""Kernel time of the fused normal-equation kernel on config 4 (device-resident, L2 flushed between calls), for A/B runs
of build variants.
Usage: [KNE_MIXED=1] [KNE_RIG=C,M,layout,detect_prob] python tools/kne_ab.py"""
import sys, os, json
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pycamset_b200 import synthetic as syn
from pycamset_b200.problem import BundleProblem

spec = os.environ.get("KNE_RIG", "32,2000,ring,1.0").split(",")
C, M, layout, dp = int(spec[0]), int(spec[1]), spec[2], float(spec[3])
rig = syn.make_rig(C, M, distortion=True, seed=0, device="cuda:0", layout=layout, detect_prob=dp)
rng = np.random.default_rng(1)
intr, extr, poses = rig.perturbed(rng, 1e-3)
params = rig.param_string(intr, extr, poses)
unfixed = np.ones(params.shape[0], bool); unfixed[15 * C:15 * C + 6] = False
stream = torch.cuda.Stream()
prob = BundleProblem(0, rig.cam, rig.pose, rig.key, rig.uv, C, M, 81, template=rig.template, unfixed=unfixed, stream=stream.cuda_stream)
prob.set_param_string(params)
if os.environ.get("KNE_MIXED"):
    prob.set_normal_precision(int(os.environ["KNE_MIXED"]))
N = prob.n_obs
x = torch.from_numpy(params[unfixed]).cuda()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
with torch.cuda.stream(stream):
    for _ in range(5): prob.normal_equations_device(x.data_ptr())
    torch.cuda.synchronize()
    prob.timing_enable(True)
    for _ in range(30):
        flush.zero_()
        prob.normal_equations_device(x.data_ptr())
    torch.cuda.synchronize()
ms = float(np.median(prob.timing_all_ms()))
b = prob.device_buffers()
print(json.dumps({"mixed": os.environ.get("KNE_MIXED"), "rig": spec, "n_obs": N, "kernel_ms": ms,
                  "Gobs_per_s": N / ms / 1e6, "frac_hbm_28B": 28.0 * N / ms / 1e6 / 6544.7}))
