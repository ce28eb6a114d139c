"""B200-native batched WRSN simulator — drop-in for the hot path of ``rl_env/WRSN.py``.

``BatchedWRSN`` advances thousands of independent network + mobile-charger instances per launch;
``WRSN`` is the single-environment façade with the reference's constructor and request dict.
"""
from .scenario import Scenario, build_static, load_mc_type, synthetic  # noqa: F401
from .batched import BatchedWRSN, Requests  # noqa: F401
from .snapshot import EnvSnapshot  # noqa: F401
from .wrsn import WRSN  # noqa: F401
from .ippo import BatchedIPPO  # noqa: F401
from .controllers import (BatchedRandomController, HeuristicController, IPPORollout, LookaheadController, PerAgentPolicy, allreduce_gradients,  # noqa: F401
                          evaluate, ppo_update, rollout, select_batch)  # noqa: F401

__all__ = ["Scenario", "build_static", "load_mc_type", "synthetic", "BatchedWRSN", "Requests", "EnvSnapshot", "WRSN", "BatchedIPPO",
           "BatchedRandomController", "HeuristicController", "IPPORollout", "LookaheadController", "PerAgentPolicy", "allreduce_gradients", "evaluate", "ppo_update", "rollout", "select_batch"]
