"""Launch every kernel of the library a few times on realistic states, for `ncu --set full` (one capture per kernel, see
profiles/r02_kernels.md): python tools/ncu_kernels.py [B].  Kernels: k_env<STEP> (rollout), k_env<RESTORE_RESET>, k_decode_map,
k_decode_locate, k_observe (chunked, synthetic fields) / k_observe_win (hanoi1000n100: narrow sources), k_observe<double>,
k_charge, k_record_transitions, the per-tick kernels k_env<K_BFS / K_DRAIN / K_BOOK / K_REWARD>, k_env<FITNESS>, k_step_order
and gany::k_env<STEP> on 1000-node environments (256 threads)."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_agent_rl_wrsn_b200 import BatchedWRSN, synthetic
from multi_agent_rl_wrsn_b200.controllers import IPPORollout
from tests import parity_cases as pc
from tests.helpers import golden
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev = torch.device("cuda:0")
scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + k) for k in range(64)]
env = BatchedWRSN(scs, num_agent=3, num_envs=B, device=dev, step_budget=100)
obs = torch.zeros((B, 4, 100, 100), dtype=torch.float32, device=dev)
env.reset(); env.get_state(out=obs)
for k in range(120):
    env.rollout_step(env.linear_controller_action(obs, (1.0, 1.0, -10.0, 1.0)), obs)
torch.cuda.synchronize()
torch.cuda.profiler.start()                               # ncu --profile-from-start off: only what follows is captured
a = env.linear_controller_action(obs, (1.0, 1.0, -10.0, 1.0))
env.rollout_step(a, obs)
env.get_state(dtype=torch.float64)                        # k_observe<double>
env.charge_rates()                                        # k_charge
env.get_network_fitness()                                 # k_env<FITNESS>
for name in ("drain", "reward", "bookkeep", "bfs"):       # the per-tick kernels on the rolled-out states (copies: the state moves)
    env.kernel(name)
ro = IPPORollout(env, 2, with_obs=False, action_shape=(3,))
ro.collect(lambda a, o: (torch.rand((B, 3), device=dev) * torch.tensor([1.0, 1.0, 0.05], device=dev), torch.zeros(B, device=dev)))   # k_record_transitions
torch.cuda.synchronize()
torch.cuda.profiler.stop()
hn = BatchedWRSN(pc.sc_from_golden(golden("net_hanoi1000n100")), num_agent=3, num_envs=B, device=dev, step_budget=100)
o2 = torch.zeros((B, 4, 100, 100), dtype=torch.float32, device=dev)
hn.reset(); hn.get_state(out=o2)
for k in range(30):
    hn.rollout_step(hn.linear_controller_action(o2, (1.0, 1.0, -10.0, 1.0)), o2)
torch.cuda.synchronize()
torch.cuda.profiler.start()
hn.get_state(out=o2)                                      # k_observe_win
torch.cuda.synchronize()
torch.cuda.profiler.stop()
# BASELINE.json configs[4]: 1000 nodes / 10 chargers, 256 threads per environment (gany::k_env)
if os.environ.get("WRSN_NCU_C5", "1") == "1":
    big = [synthetic(num_nodes=1000, num_targets=1000, seed=1000 + k, num_gateways=25) for k in range(4)]
    e5 = BatchedWRSN(big, num_agent=10, num_envs=512, device=dev, step_budget=100)
    o5 = torch.zeros((512, 4, 100, 100), dtype=torch.float32, device=dev)
    e5.reset(); e5.get_state(out=o5)
    for k in range(60):
        e5.rollout_step(e5.linear_controller_action(o5, (1.0, 1.0, -10.0, 1.0)), o5)
    torch.cuda.synchronize()
    torch.cuda.profiler.start()
    e5.rollout_step(e5.linear_controller_action(o5, (1.0, 1.0, -10.0, 1.0)), o5)  # gany::k_env<STEP>, 256 threads, 512 environments
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
torch.cuda.synchronize()
print("ok", env.counters())
