"""Time the fp32 observation raster: python tools/time_observe.py <k> [B]

k = "base" times the package's libwrsn_b200.so; any other k times multi_agent_rl_wrsn_b200/csrc/libwrsn_b200_obs<k>.so, another
build of the library, such as the parent commit's, for an A/B comparison in one process:

  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false -std=c++17 -Xcompiler -fPIC -shared -I include \
       -o multi_agent_rl_wrsn_b200/csrc/libwrsn_b200_obs<k>.so <other tree>/multi_agent_rl_wrsn_b200/csrc/wrsn_kernels.cu
"""
import ctypes, os, sys
import numpy as np, torch
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from multi_agent_rl_wrsn_b200 import _lib, BatchedWRSN, synthetic
k = sys.argv[1]
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
if k != "base":
    _lib._lib = _lib._bind(ctypes.CDLL(os.path.join(REPO, "multi_agent_rl_wrsn_b200", "csrc", "libwrsn_b200_obs%s.so" % k)))
dev = torch.device("cuda:0")
if os.environ.get("WRSN_SCENARIO"):                  # a shipped scenario of the reference, from its committed fixture
    from tests import parity_cases as pc
    from tests.helpers import golden
    scs = [pc.sc_from_golden(golden(os.environ["WRSN_SCENARIO"]))]
else:
    scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + s) for s in range(64)]
env = BatchedWRSN(scs, num_agent=3, num_envs=B, device=dev)
env.reset()
g = torch.Generator(device=dev); g.manual_seed(0)
for _ in range(40):
    a = torch.rand((B, 3), dtype=torch.float64, device=dev, generator=g); a[:, 2] *= 0.05
    env.rollout_step(a)
obs = [torch.zeros((B, 4, 100, 100), dtype=torch.float32, device=dev) for _ in range(2)]
for o in obs: env.get_state(out=o)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 20
e0.record()
for i in range(n): env.get_state(out=obs[i % 2])
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / n
ref = env.get_state(dtype=torch.float64)
err = float(((obs[0].double() - ref).abs().amax((2, 3)) / ref.abs().amax((2, 3)).clamp_min(1e-3)).max())
print("variant %s: %.3f ms per %d maps, %.0f GB/s written, max err / channel max %.2e, checksum %.9e" % (k, ms, B, B * 160e3 / ms / 1e6, err, float(obs[0].double().sum())), flush=True)
