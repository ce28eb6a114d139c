"""What the lookahead planner costs and what it achieves: k_heuristic_candidates beside k_heuristic, one planning call
(LookaheadController.plan) on the headline workload, and controllers.evaluate lifetimes of the planner beside the two rules
and the reference's RandomController.

    python tools/time_lookahead.py [--reps 200] [--plans 10] [--eval-envs 1024] [--max-decisions 3000]

1. Kernel time per call, CUDA events over --reps launches after 20 warm-up launches (arguments prepared once), and the kernel's
   own device time from torch.profiler, at 4096 rows of 100 nodes (synthetic seeds 1000..1003) and 2048 rows of 1000 nodes,
   pre-rolled 20 steps under min_lifetime, 3 chargers: wrsn_heuristic_action (k_heuristic) and wrsn_heuristic_candidates
   (k_heuristic_candidates) at K = 8 and 32.
2. LookaheadController(width=K, horizon=H).plan on the headline workload (4096 rows, step budget 100, pre-rolled 20 steps):
   wall time per call over --plans calls after 2 warm-up calls (the first builds the branch batch of 4096 K rows), each ending in
   a device synchronisation, for (K, H) = (4, 2), (8, 4), (16, 4).  Every call plans from the same state: lookahead leaves
   the source rows unchanged.
3. controllers.evaluate on --eval-envs rows of the same scenarios, 1 episode, max_decisions = --max-decisions, as
   profiles/r07_heuristics.md §3: the two rules, the RandomController and the planner
   LookaheadController("min_lifetime", width=4, horizon=4, charge_levels=(1.0,)) (8 candidates: the rule's 4 best nodes, each
   at the rule's charge fraction and at a full charge).
Prints one JSON line per measurement, after a line with the card's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_agent_rl_wrsn_b200 import BatchedWRSN, synthetic  # noqa: E402
from multi_agent_rl_wrsn_b200.controllers import (BatchedRandomController, HeuristicController, LookaheadController,  # noqa: E402
                                                  evaluate, rollout)

KINDS = ("min_lifetime", "nearest_urgent")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def emit(**kw):
    print(json.dumps(kw), flush=True)


def headline(B, budget=100):
    return BatchedWRSN([synthetic(100, 100, seed=1000 + k) for k in range(4)], num_agent=3, num_envs=B, device="cuda:0",
                       step_budget=budget)


def kernel_time(call, name, reps):
    for _ in range(20):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    torch.cuda.synchronize()
    ev_us = e0.elapsed_time(e1) * 1e3 / reps
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    dev = [e for e in prof.key_averages() if e.key.startswith(name + "(") or e.key == name]
    prof_us = dev[0].device_time_total / dev[0].count if dev else float("nan")
    return ev_us, prof_us


def checked(L, fn, *args):
    def call():
        if fn(*args) != 0:
            raise RuntimeError(L.wrsn_last_error().decode())
    return call


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--reps", type=int, default=200)
    p.add_argument("--plans", type=int, default=10)
    p.add_argument("--eval-envs", type=int, default=1024)
    p.add_argument("--max-decisions", type=int, default=3000)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_lookahead.py measures on a CUDA device; none is visible")
    emit(card=card(), torch=torch.__version__)

    # 1. the kernels
    for B, N, topo in ((4096, 100, 4), (2048, 1000, 2)):
        env = BatchedWRSN([synthetic(N, N, seed=1000 + k) for k in range(topo)], num_agent=3, num_envs=B, device="cuda:0",
                          step_budget=100)
        env.reset()
        rollout(env, HeuristicController("min_lifetime"), 20)
        aid = env.req.agent_id.clone()
        L = env.L
        base = (C.byref(env.dims), env.scen.data_ptr(), env.scen_id.data_ptr(), env.state.data_ptr(), aid.data_ptr())
        for kind in KINDS:
            k = KINDS.index(kind)
            out = torch.zeros((B, 3), dtype=torch.float64, device="cuda:0")
            ev, pr = kernel_time(checked(L, L.wrsn_heuristic_action, *base, k, out.data_ptr(), env._stream()), "k_heuristic", a.reps)
            emit(what="kernel", kernel="k_heuristic", kind=kind, rows=B, nodes=N, deciding_rows=int((aid >= 0).sum()),
                 events_us_per_call=round(ev, 2), profiler_kernel_us=round(pr, 2))
            for K in (8, 32):
                act = torch.zeros((B, K, 3), dtype=torch.float64, device="cuda:0")
                node = torch.zeros((B, K), dtype=torch.int32, device="cuda:0")
                ev, pr = kernel_time(checked(L, L.wrsn_heuristic_candidates, *base, k, K, act.data_ptr(), node.data_ptr(), env._stream()),
                                     "k_heuristic_candidates", a.reps)
                emit(what="kernel", kernel="k_heuristic_candidates", kind=kind, K=K, rows=B, nodes=N, deciding_rows=int((aid >= 0).sum()),
                     events_us_per_call=round(ev, 2), profiler_kernel_us=round(pr, 2))
        del env
        torch.cuda.empty_cache()

    # 2. one planning call on the headline workload
    env = headline(4096)
    env.reset()
    rollout(env, HeuristicController("min_lifetime"), 20)
    out = torch.zeros((4096, 3), dtype=torch.float64, device="cuda:0")
    for K, H in ((4, 2), (8, 4), (16, 4)):
        ctl = LookaheadController("min_lifetime", width=K, horizon=H)
        for _ in range(2):
            ctl.plan(env, out)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.plans):
            ctl.plan(env, out)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / a.plans
        values, best = ctl.last
        deciding = ~torch.isnan(values[:, 0])
        emit(what="plan", K=K, H=H, rows=4096, branch_rows=4096 * K, deciding_rows=int(deciding.sum()), ms_per_call=round(dt * 1e3, 2),
             not_slot0=int((best[deciding] != 0).sum()))
        env._branches.clear()
        torch.cuda.empty_cache()
    del env
    torch.cuda.empty_cache()

    # 3. lifetimes
    for name, ctl in (("min_lifetime", HeuristicController("min_lifetime")), ("nearest_urgent", HeuristicController("nearest_urgent")),
                      ("random", BatchedRandomController()),
                      ("lookahead_min_lifetime_w4_h4_full", LookaheadController("min_lifetime", width=4, horizon=4, charge_levels=(1.0,)))):
        env = headline(a.eval_envs)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = evaluate(env, ctl, episodes=1, max_decisions=a.max_decisions)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        life, ended = r["lifetime"][:, 0], ~r["truncated"][:, 0]
        per_topology = [round(float(life[k::4].mean()), 1) for k in range(4)]   # row b runs topology b % 4
        emit(what="evaluate", controller=name, rows=a.eval_envs, max_decisions=a.max_decisions, seconds=round(dt, 2),
             lifetime_mean=round(float(life.mean()), 2), lifetime_min=round(float(life.min()), 2), lifetime_max=round(float(life.max()), 2),
             lifetime_mean_per_topology=per_topology, truncated_rows=int(r["truncated"].sum()),
             ended_network_dead=int((ended & (env.req.terminal != 0)).sum()),
             ended_every_charger_dead=int((ended & (env.req.terminal == 0) & ((env.req.flags & 1) != 0)).sum()),
             decisions_mean=round(float(r["decisions"].double().mean()), 1), return_mean=round(float(r["return"].mean()), 4))
        del env
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
