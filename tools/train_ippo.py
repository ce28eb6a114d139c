"""The reference's ``runner/IPPO.py`` / ``runner/PPO.py`` on the batched simulator: the reference's scenario / charger /
``alg_args`` YAML schemas, B environments per GPU instead of one.  Runs without a checkout of the reference: the networks are
``nets.UNetActor`` / ``nets.CNNCritic`` (same shapes and parameter names as the reference's), the scenario defaults to a
synthetic 100-node network and ``alg_args`` to the values of ``alg_args/ippo.yaml``; with ``--reference-root`` the reference's own
YAML files (and, with ``--reference-networks``, its own network classes) are used.

    python tools/train_ippo.py --envs 2048 --iterations 10
    python tools/train_ippo.py --reference-root /path/to/multi_agent_rl_wrsn --envs 2048 --iterations 1000
    python tools/train_ippo.py --reference-root /path/to/multi_agent_rl_wrsn --scenario physical_env/network/network_scenarios/hanoi1000n{50,100,150,200}.yaml
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/train_ippo.py --envs 16384

Under torchrun the ``--envs`` environments are split into contiguous blocks, one per rank / GPU (``sharding.shard_range``); the
simulation has no collective, the update averages its gradients once per minibatch over NCCL.
"""
import argparse
import os
import random
import sys

import numpy as np
import torch
import yaml

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_agent_rl_wrsn_b200 import BatchedIPPO, BatchedWRSN  # noqa: E402
from multi_agent_rl_wrsn_b200.sharding import shard_range  # noqa: E402


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--reference-root", default=None, help="checkout of the reference (its YAML files; its networks with --reference-networks)")
    p.add_argument("--reference-networks", action="store_true")
    p.add_argument("--step-budget", type=int, default=100)
    p.add_argument("--scenario", nargs="+", default=["physical_env/network/network_scenarios/hanoi1000n50.yaml"],   # runner/IPPO.py:19
                   help="with --reference-root: one or several scenario files, of any sizes, assigned to the environments round robin")
    p.add_argument("--agent-type", default="physical_env/mc/mc_types/default.yaml")
    p.add_argument("--alg-args", default="alg_args/ippo.yaml")
    p.add_argument("--num-agent", type=int, default=3)
    p.add_argument("--envs", type=int, default=2048, help="environments of the whole job")
    p.add_argument("--window", type=int, default=8, help="rollout steps per collection window")
    p.add_argument("--iterations", type=int, default=1000)
    p.add_argument("--save-folder", default="save_model/ippo")
    p.add_argument("--model-path", default=None)
    p.add_argument("--ppo", action="store_true", help="one shared network pair (controller/ppo/PPO.py) instead of one per agent")
    a = p.parse_args()

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    random.seed(0); np.random.seed(0); torch.manual_seed(0)                 # runner/IPPO.py:12-15 (identical replicas on every rank)
    torch.backends.cudnn.deterministic = True

    lo, hi = shard_range(a.envs, rank, world)
    factories = {}
    if a.reference_root:
        ref = lambda rel: rel if os.path.isabs(rel) else os.path.join(a.reference_root, rel)
        with open(ref(a.alg_args)) as f:
            args = yaml.safe_load(f)["alg_args"]
        scenarios, mc = [ref(s) for s in a.scenario], ref(a.agent_type)
        if a.reference_networks:
            sys.path.insert(0, a.reference_root)
            from controller.ppo.actor.UnetActor import UNet                # the reference's networks, unmodified
            from controller.ppo.critic.CNNCritic import CNNCritic
            factories = dict(actor_factory=UNet, critic_factory=CNNCritic)
    else:
        from multi_agent_rl_wrsn_b200 import synthetic
        args = dict(seed=0, lr=3.0e-4, gamma=0.99, clip=0.2, batch_size=512, n_updates_per_iteration=5, save_freq=5, gae=True,
                    norm_adv=True, minibatch_size=64, ent_coef=0.0, vf_coef=0.5, gae_lambda=0.95, max_grad_norm=0.5, clip_vloss=True)
        scenarios, mc = [synthetic(num_nodes=100, num_targets=100, seed=1000 + k) for k in range(16)], None
    env = BatchedWRSN(scenarios, num_agent=a.num_agent, mc_type=mc, num_envs=hi - lo, device=dev, step_budget=a.step_budget)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1 + rank)                                               # different action samples on every shard
    trainer = BatchedIPPO(args, env, device=dev, model_path=a.model_path, window=a.window, shared=a.ppo, generator=gen, **factories)
    trainer.train(a.iterations, a.save_folder)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
