"""What a batch of mixed field sizes costs: decisions/s of one mixed BatchedWRSN against one batch per size.

    python tools/time_mixed.py [--envs 4096] [--steps 300] [--repeats 3]

The environments are those of the five golden episode fixtures (82 / 82 / 82 / 98 / 132 nodes, 50 / 50 / 50 / 100 / 200 targets,
three default chargers, 100 x 100 maps), environment b on fixture b % 5, under the reference's RandomController law decoded on the
device (``BatchedWRSN.linear_controller_action``, then ``rollout_step``: the loop of ``controllers.rollout``).  Two arms:

  mixed     one mixed batch, split into --groups groups on as many CUDA streams, as bench.py runs its environments; every row runs on
            the thread count of the largest scenario (132 nodes: 64 threads);
  per-size  the same environments as one batch per node count, each on its own stream (82 and 98 nodes on one warp, 132 on 64).

Each arm is pre-rolled (--preroll steps, so that the episodes' phases spread out), then timed over --steps steps with CUDA events;
the arms alternate --repeats times.  One JSON line per timed run, then a summary line with the card and its power limit.  Both arms
simulate the same environments, bit for bit, so they hand out the same number of decisions in every window."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_agent_rl_wrsn_b200 import BatchedWRSN  # noqa: E402
from multi_agent_rl_wrsn_b200.controllers import BatchedRandomController  # noqa: E402
from tests import parity_cases as pc  # noqa: E402
from tests.helpers import golden, mc_dict_of  # noqa: E402

FIXTURES = ("ep_basic_n50", "ep_edge_n50", "ep_longcharge_n50", "ep_full_n100", "ep_full_n200")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class Arm:
    """Batches of one arm, each on its own stream, stepped under the RandomController law."""

    def __init__(self, name, batches, mc, budget, dev):
        """``batches``: (scenarios, scenario index of every row) of each batch"""
        self.name, self.dev = name, dev
        self.envs = [BatchedWRSN(scs, num_agent=3, mc_type=mc, num_envs=len(sid), scenario_index=sid, device=dev, step_budget=budget)
                     for scs, sid in batches]
        self.streams = [torch.cuda.Stream(device=dev) for _ in self.envs]
        self.obs = [torch.zeros((e.B, 4, e.S, e.S), dtype=torch.float32, device=dev) for e in self.envs]
        self.act = [torch.zeros((e.B, 3), dtype=torch.float64, device=dev) for e in self.envs]
        for e, o in zip(self.envs, self.obs):
            e.reset()
            e.get_state(out=o)
        torch.cuda.synchronize(dev)

    def step(self):
        for e, s, o, a in zip(self.envs, self.streams, self.obs, self.act):
            with torch.cuda.stream(s):
                e.linear_controller_action(o, BatchedRandomController.weights, out=a)
                e.rollout_step(a, o)

    def decisions(self):
        return float(torch.stack([e.req.stats[:, 0].sum() for e in self.envs]).sum().item())

    def timed(self, steps):
        torch.cuda.synchronize(self.dev)
        d0 = self.decisions()
        cur = torch.cuda.current_stream(self.dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for s in self.streams:
            s.wait_stream(cur)
        for _ in range(steps):
            self.step()
        for s in self.streams:
            cur.wait_stream(s)
        e1.record(cur)
        torch.cuda.synchronize(self.dev)
        for e in self.envs:
            e.raise_on_error()
        ms = e0.elapsed_time(e1)
        return ms, self.decisions() - d0


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--envs", type=int, default=4096)
    p.add_argument("--groups", type=int, default=4, help="streams of the mixed arm")
    p.add_argument("--steps", type=int, default=300, help="timed steps per run (300: about half a second)")
    p.add_argument("--preroll", type=int, default=200)
    p.add_argument("--repeats", type=int, default=3)
    p.add_argument("--budget", type=int, default=100, help="wrsn_dims.step_budget (bench.py's default)")
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_mixed.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    gs = [golden(n) for n in FIXTURES]
    scs, mc = [pc.sc_from_golden(g) for g in gs], mc_dict_of(gs[0])
    sid = np.arange(a.envs) % len(scs)
    Bg = a.envs // a.groups
    mixed = Arm("mixed", [(scs, sid[g * Bg:(g + 1) * Bg]) for g in range(a.groups)], mc, a.budget, dev)
    per_size = []
    for n in sorted({sc.N for sc in scs}):          # one batch per node count, holding the same environments
        keep = [k for k, sc in enumerate(scs) if sc.N == n]
        rows = sid[np.isin(sid, keep)]
        per_size.append(([scs[k] for k in keep], np.searchsorted(keep, rows)))
    arms = (mixed, Arm("per-size", per_size, mc, a.budget, dev))
    for arm in arms:
        for _ in range(a.preroll):
            arm.step()
    torch.cuda.synchronize(dev)
    res = {arm.name: [] for arm in arms}
    decisions = {arm.name: [] for arm in arms}
    for r in range(a.repeats):
        for arm in arms:
            ms, dec = arm.timed(a.steps)
            rate = dec / (ms / 1e3)
            res[arm.name].append(rate)
            decisions[arm.name].append(dec)
            print(json.dumps(dict(arm=arm.name, repeat=r, ms=round(ms, 3), decisions=dec, decisions_per_s=round(rate, 1),
                                  batches=[dict(rows=e.B, nodes=e.N, threads=e.dims.threads) for e in arm.envs])), flush=True)
    summary = dict(card=card(), envs=a.envs, steps=a.steps, budget=a.budget)
    for name, v in res.items():
        summary[name] = dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)))
    summary["mixed_over_per_size"] = summary["mixed"]["median"] / summary["per-size"]["median"]
    summary["same_decisions"] = decisions["mixed"] == decisions["per-size"]   # both arms simulate the same environments identically
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
