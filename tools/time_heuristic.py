"""What the hand-written charging rules cost and what they achieve: k_heuristic, rollouts under HeuristicController, and
controllers.evaluate lifetimes against the reference's RandomController.

    python tools/time_heuristic.py [--reps 200] [--steps 100] [--eval-envs 1024] [--max-decisions 3000]

1. k_heuristic per call, CUDA events over --reps launches of wrsn_heuristic_action after a warm-up (arguments prepared once), at
   4096 rows of 100 nodes (synthetic seeds 1000..1003, the headline workload) and 2048 rows of 1000 nodes, both pre-rolled 20
   steps under min_lifetime so the records hold mid-episode state, 3 chargers.  The same launches are also read from
   torch.profiler (the kernel's own device time), which shows whether the events figure is set by the kernel or by the launch.
   Bytes: what the rule reads once per row (energy, energyCS, status: 17 B/node of state; node x / y: 16 B/node of scenario; the
   chargers' position, status and destination; agent_id) and the 24 B action it writes.  Every working set here fits the 126 MB
   L2, so the share of 7.7 TB/s is bytes / time / 7.7 TB/s and nothing more.
2. controllers.rollout decisions/s on the headline workload (4096 rows, step budget 100) under each heuristic and under
   BatchedRandomController (its map decoded on the device, the bench.py law), --steps timed after 20 warm-up steps.
3. controllers.evaluate on --eval-envs rows of the same scenarios, 1 episode, max_decisions = --max-decisions: network lifetime
   (simulated seconds after the warm-up) mean / min / max over rows and mean per topology, how many rows were cut by the cap
   (their lifetime is a lower bound), and how the others ended: the network dead (terminal) or every charger dead.
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
from multi_agent_rl_wrsn_b200.controllers import BatchedRandomController, HeuristicController, evaluate, rollout  # noqa: E402

HBM_TBS = 7.7                                        # HGX B200 data sheet, one GPU
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


def kernel_time(env, kind, reps):
    out = torch.zeros((env.B, 3), dtype=torch.float64, device=env.device)
    aid = env.req.agent_id.clone()
    k = KINDS.index(kind)
    L, args = env.L, (C.byref(env.dims), env.scen.data_ptr(), env.scen_id.data_ptr(), env.state.data_ptr(), aid.data_ptr(), k,
                      out.data_ptr(), env._stream())

    def call():
        if L.wrsn_heuristic_action(*args) != 0:
            raise RuntimeError(L.wrsn_last_error().decode())

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
    dev = [e for e in prof.key_averages() if "k_heuristic" in e.key]
    prof_us = dev[0].device_time_total / dev[0].count if dev else float("nan")
    return ev_us, prof_us, int((aid >= 0).sum())


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--reps", type=int, default=200)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--eval-envs", type=int, default=1024)
    p.add_argument("--max-decisions", type=int, default=3000)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_heuristic.py measures on a CUDA device; none is visible")
    emit(card=card(), torch=torch.__version__)

    # 1. the kernel
    for B, N, topo in ((4096, 100, 4), (2048, 1000, 2)):
        env = BatchedWRSN([synthetic(N, N, seed=1000 + k) for k in range(topo)], num_agent=3, num_envs=B, device="cuda:0",
                          step_budget=100)
        env.reset()
        rollout(env, HeuristicController("min_lifetime"), 20)
        nbytes = B * (N * (17 + 16) + env.M * 5 * 8 + 4 + 24)
        for kind in KINDS:
            ev_us, prof_us, deciding = kernel_time(env, kind, a.reps)
            emit(what="k_heuristic", kind=kind, rows=B, nodes=N, chargers=env.M, deciding_rows=deciding, events_us_per_call=round(ev_us, 2),
                 profiler_kernel_us=round(prof_us, 2), bytes=nbytes, rate_TBs_events=round(nbytes / ev_us / 1e6, 3),
                 share_of_hbm_bound_events=round(nbytes / ev_us / 1e6 / HBM_TBS, 4))
        del env
        torch.cuda.empty_cache()

    # 2. rollouts on the headline workload
    for name, ctl in (("min_lifetime", HeuristicController("min_lifetime")), ("nearest_urgent", HeuristicController("nearest_urgent")),
                      ("random", BatchedRandomController())):
        env = headline(4096)
        env.reset()
        rollout(env, ctl, 20)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, st = rollout(env, ctl, a.steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        emit(what="rollout", controller=name, rows=4096, steps=a.steps, seconds=round(dt, 4), decisions=st["decisions"],
             decisions_per_s=round(st["decisions"] / dt), ms_per_step=round(dt / a.steps * 1e3, 3), episodes=st["episodes"])
        del env
        torch.cuda.empty_cache()

    # 3. lifetimes
    for name, ctl in (("min_lifetime", HeuristicController("min_lifetime")), ("nearest_urgent", HeuristicController("nearest_urgent")),
                      ("random", BatchedRandomController())):
        env = headline(a.eval_envs)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = evaluate(env, ctl, episodes=1, max_decisions=a.max_decisions)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        life, ended = r["lifetime"][:, 0], ~r["truncated"][:, 0]
        per_topology = [round(float(life[k::4].mean()), 1) for k in range(4)]   # row b runs topology b % 4
        # how the episodes that were not cut ended: the last request of each row is still in place (no reset after it)
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
