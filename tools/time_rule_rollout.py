"""What rule rollouts on the device (BatchedWRSN.rule_rollout, wrsn_rule_rollout) save against driving the rule from the host,
request by request, in the same run.

    python tools/time_rule_rollout.py [--reps 5] [--eval-envs 1024] [--max-decisions 3000]

1. Rule rollouts of H decisions (H = 4, 16, 64) on the headline workload (4096 rows, synthetic seeds 1000..1003, 100 nodes,
   3 chargers, pre-rolled 10 steps under min_lifetime), step budgets 0 and 100: `host` is the loop lookahead ran before
   (heuristic_action + episode_step per request, one host synchronisation per request once the first H + 1 are done), `fused`
   is rule_rollout.  Every repeat restores the same rows first; the two alternate.  Both must give the same returns bit for bit.
2. LookaheadController(width=K, horizon=H).plan at (K, H) = (4, 2), (8, 4), (16, 4), (8, 32) on the same workload at budget 100:
   `host` runs the branches with the loop of 1., `fused` with lookahead (rule_rollout); values must be equal bit for bit.
3. controllers.evaluate on --eval-envs rows, 1 episode, max_decisions = --max-decisions: HeuristicController (rule_rollout per
   episode) against the same rule as a generic controller (make_action), which runs evaluate's per-request loop.
Wall times end in a device synchronisation; median, min and max over --reps repeats.  One JSON line per measurement, after a
line with the card's name and power limit read in the same run."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_agent_rl_wrsn_b200 import BatchedWRSN, synthetic  # noqa: E402
from multi_agent_rl_wrsn_b200.batched import episode_ends, episode_step  # noqa: E402
from multi_agent_rl_wrsn_b200.controllers import HeuristicController, LookaheadController, evaluate  # noqa: E402

KINDS = ("min_lifetime", "nearest_urgent")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def emit(**kw):
    print(json.dumps(kw), flush=True)


def spread(ts):
    return dict(median_ms=round(1e3 * statistics.median(ts), 3), min_ms=round(1e3 * min(ts), 3), max_ms=round(1e3 * max(ts), 3))


def headline(B, budget):
    env = BatchedWRSN([synthetic(100, 100, seed=1000 + k) for k in range(4)], num_agent=3, num_envs=B, device="cuda:0",
                      step_budget=budget)
    env.reset()
    act = torch.zeros((B, 3), dtype=torch.float64, device="cuda:0")
    for _ in range(10):
        env.heuristic_action("min_lifetime", out=act)
        env.rollout_step(act)
    return env


def host_rollout(env, kind, limit, first=None, running=None):
    """The per-request loop lookahead used to run its branches with."""
    B, dev = env.B, env.device
    run = (env.req.agent_id >= 0) if running is None else running.clone()
    dec = torch.zeros(B, dtype=torch.int64, device=dev)
    ret = torch.zeros(B, dtype=torch.float64, device=dev)
    action = torch.zeros((B, 3), dtype=torch.float64, device=dev) if first is None else first.clone()
    k = 0
    while True:
        _, ended = episode_ends(env.req, run, dec, limit)
        run &= ~ended
        if k >= limit and not bool(run.any()):
            break
        if k > 0 or first is None:
            env.heuristic_action(kind, out=action)
        episode_step(env, run, action, dec, ret)
        k += 1
    env.raise_on_error()
    return ret


def host_lookahead(env, cand, H, kind, valid):
    """BatchedWRSN.lookahead with the branch loop of host_rollout."""
    import ctypes as C
    B, K = env.B, cand.shape[1]
    br = env._branch(K)
    aid = env.req.agent_id
    decider = (aid >= 0) & (aid < env.M)
    running = (decider[:, None] & valid).reshape(B * K)
    rows = torch.arange(B * K, dtype=torch.int32, device=env.device)
    src = torch.where(running, rows // K, torch.full_like(rows, -1))
    env._call(env.L.wrsn_copy_rows, C.byref(env.dims), B * K, env.state.data_ptr(), C.byref(env.req.c), env.scen_id.data_ptr(),
              src.data_ptr(), B, br.state.data_ptr(), C.byref(br.req.c), br.scen_id.data_ptr(), rows.data_ptr(), B * K, env._stream())
    br._refresh_counts()
    ret = host_rollout(br, kind, H + 1, first=cand.reshape(B * K, 3), running=running)
    val = torch.where(valid, ret.view(B, K), torch.full_like(ret.view(B, K), -math.inf))
    return torch.where(decider[:, None], val, torch.full_like(val, math.nan))


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--eval-envs", type=int, default=1024)
    p.add_argument("--max-decisions", type=int, default=3000)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    emit(card=card())
    for budget in (0, 100):
        env = headline(4096, budget)
        snap = env.snapshot()
        for H in (4, 16, 64):
            ts = {"host": [], "fused": []}
            res = {}
            for rep in range(a.reps + 1):                   # repeat 0 warms up
                for name in ("host", "fused") if rep % 2 == 0 else ("fused", "host"):
                    env.restore(snap)
                    fn = (lambda: host_rollout(env, "min_lifetime", H)) if name == "host" else \
                        (lambda: env.rule_rollout("min_lifetime", H)[0])
                    t, out = timed(fn)
                    res[name] = out
                    if rep:
                        ts[name].append(t)
            same = bool(torch.equal(res["host"].view(torch.int64), res["fused"].view(torch.int64)))
            emit(what="rule_rollout", rows=4096, budget=budget, H=H, same_returns=same,
                 host=spread(ts["host"]), fused=spread(ts["fused"]), speedup=round(statistics.median(ts["host"]) / statistics.median(ts["fused"]), 2))
    env = headline(4096, 100)
    for K, H in ((4, 2), (8, 4), (16, 4), (8, 32)):
        ctl = LookaheadController("min_lifetime", width=K, horizon=H)
        cand, valid = ctl.candidates(env)
        ts = {"host": [], "fused": []}
        res = {}
        for rep in range(a.reps + 1):
            for name in ("host", "fused") if rep % 2 == 0 else ("fused", "host"):
                fn = (lambda: host_lookahead(env, cand, H, "min_lifetime", valid)) if name == "host" else \
                    (lambda: env.lookahead(cand, H, "min_lifetime", valid))
                t, out = timed(fn)
                res[name] = out
                if rep:
                    ts[name].append(t)
        same = bool(torch.equal(torch.nan_to_num(res["host"], nan=0.0).view(torch.int64), torch.nan_to_num(res["fused"], nan=0.0).view(torch.int64)))
        emit(what="plan", rows=4096, K=K, H=H, same_values=same, host=spread(ts["host"]), fused=spread(ts["fused"]),
             speedup=round(statistics.median(ts["host"]) / statistics.median(ts["fused"]), 2))

    class Generic:
        def __init__(self, kind):
            self.kind = kind

        def make_action(self, agent_id, state, info=None, wrsn=None):
            return self.env.heuristic_action(self.kind, agent_id=agent_id)

    for kind in KINDS:
        ts = {"host": [], "fused": []}
        res = {}
        for rep in range(2):
            for name in ("host", "fused") if rep % 2 == 0 else ("fused", "host"):
                env = BatchedWRSN([synthetic(100, 100, seed=1000 + k) for k in range(4)], num_agent=3, num_envs=a.eval_envs,
                                  device="cuda:0")
                ctl = HeuristicController(kind) if name == "fused" else Generic(kind)
                ctl.env = env
                t, out = timed(lambda: evaluate(env, ctl, episodes=1, max_decisions=a.max_decisions))
                res[name] = out
                ts[name].append(t)
        same = all(torch.equal(res["host"][k].cpu(), res["fused"][k].cpu()) for k in res["host"])
        emit(what="evaluate", kind=kind, rows=a.eval_envs, max_decisions=a.max_decisions, same=same,
             mean_lifetime_s=round(float(res["fused"]["lifetime"].mean()), 1), host=spread(ts["host"]), fused=spread(ts["fused"]),
             speedup=round(statistics.median(ts["host"]) / statistics.median(ts["fused"]), 2))


if __name__ == "__main__":
    main()
