#!/usr/bin/env python
"""bench.py — agent-decisions/s of the batched WRSN hot path (reset / step / observation / reward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs B] [--nodes 100] [--chargers 3] [--actions controller|uniform]
    python bench.py --impl reference ...        # the CPU restatement of the reference on the host cores, same law
    python bench.py ... --dump-outputs DIR      # also write the outputs of the last timed step as DIR/<name>.npy

One *step* = one pass of the hot path over the batch: the controller's action for every environment that holds a request,
``WRSN.step`` (advance to the next charger decision — at most ``--budget`` work units per launch, a longer step continues
at the next pass), the reset of every environment whose episode ended, and the observation raster of every deciding
charger.  Workload at N = 1: BASELINE.json configs[1] — 100 nodes / 3 chargers / 4096 environments, **random
controller** (``controller/random/RandomController.py:12-15``: density map ``s0 + s1 - 10 s2 + s3`` of the observation,
decoded by ``WRSN.density_map_to_action`` ``rl_env/WRSN.py:229-287`` — here on the device).  ``--actions uniform`` is the
decode-free law of SURVEY 8d(ii) (a ~ U[0,1]^3, a[2] *= 0.05), reported as a side figure by the default run.
Environments shard across ranks by index with no data-path collective (weak scaling: B per GPU is fixed).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "agent-decisions/sec"
UNIT = "decisions/s"


def parse(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=None, help="timed steps (default 60); --workload ippo: timed training iterations")
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--envs", type=int, default=4096, help="environments per GPU")
    p.add_argument("--nodes", type=int, default=100)
    p.add_argument("--targets", type=int, default=None)
    p.add_argument("--chargers", type=int, default=3)
    p.add_argument("--topologies", type=int, default=64, help="distinct synthetic scenarios per GPU")
    p.add_argument("--scenario", default=None,
                   help="a shipped scenario of the reference, replicated in every environment: name of a committed fixture "
                        "that carries it (e.g. net_hanoi1000n100; the reference's YAML files do not travel to the GPU box)")
    p.add_argument("--actions", default="controller", choices=["controller", "uniform"],
                   help="controller: the reference's RandomController density map, decoded on the device (configs[1]); "
                        "uniform: 3-vector actions a ~ U[0,1]^3, a[2] *= 0.05")
    p.add_argument("--threads", type=int, default=0)
    p.add_argument("--budget", type=int, default=DEFAULT_BUDGET, help="work units per launch and environment (wrsn_dims.step_budget; 0 = unlimited)")
    p.add_argument("--rounds", type=int, default=DEFAULT_ROUNDS, help="wrsn_dims.step_rounds: rounds of (events kernel, batch kernel) per step; 0 = one kernel")
    p.add_argument("--preroll", type=int, default=200, help="untimed steps before warm-up that desynchronise the episodes")
    p.add_argument("--groups", type=int, default=DEFAULT_GROUPS, help="asynchronous environment groups (CUDA streams) per GPU")
    p.add_argument("--workload", default="rollout", choices=["rollout", "ippo"],
                   help="rollout: the simulator's hot path under the configured controller (the headline); ippo: BASELINE.json "
                        "configs[2], the IPPO training loop (alg_args/ippo.yaml) on the batched simulator — roll_out + clipped-PPO "
                        "update with the gradient all-reduce, U-Net actors / CNN critics per charger (SURVEY 8 f2)")
    p.add_argument("--iterations", type=int, default=3, help="--workload ippo: timed training iterations when --steps is not given")
    p.add_argument("--window", type=int, default=4, help="--workload ippo: rollout steps per collection window")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-extras", action="store_true", help="skip the side figures (uniform actions, standalone kernels)")
    p.add_argument("--engine-switch", type=int, default=0, help="diagnostic: hdr[OPT_NOBATCH] of every environment (see include/wrsn_b200.h)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step handed its caller to DIR/<name>.npy (rank 0's environments; see dump_outputs)")
    a = p.parse_args(argv)
    if a.workload == "ippo":                         # one timed step of the IPPO workload is one training iteration
        a.iterations = a.iterations if a.steps is None else a.steps
        a.steps = a.iterations
    elif a.steps is None:
        a.steps = 60
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload != "rollout"):
        p.error("--dump-outputs covers the rollout workload of --impl b200")
    return a


DEFAULT_BUDGET = 100
DEFAULT_GROUPS = 4
DEFAULT_ROUNDS = 0


def workload_name(a):
    law = ("RandomController density maps (s0 + s1 - 10 s2 + s3) decoded by density_map_to_action"
           if getattr(a, "actions", "controller") == "controller" else "uniform 3-vector actions")
    if a.scenario:
        return "%s of the reference replicated, %d chargers, %d envs per GPU, %s" % (
            a.scenario.replace("net_", ""), a.chargers, a.envs, law)
    return "%d-node/%d-charger synthetic WRSN, %d envs per GPU, %s" % (a.nodes, a.chargers, a.envs, law)


def scenarios_for(a, rank):
    from multi_agent_rl_wrsn_b200 import Scenario, synthetic
    if a.scenario:                                   # the arrays of the reference's YAML as stored in the golden fixture
        g = np.load(os.path.join(REPO, "tests", "golden", a.scenario + ".npz"), allow_pickle=False)
        q = g["sc_par"]
        spe = dict(capacity=q[0], threshold=q[1], com_range=q[2], sen_range=q[3], prob_gp=q[4], package_size=q[5],
                   er=q[6], et=q[7], efs=q[8], emp=q[9])
        return [Scenario(nodes=g["sc_nodes"].reshape(-1, 2), targets=g["sc_targets"].reshape(-1, 2),
                         base_station=g["sc_bs"], node_phy_spe=spe, max_time=float(q[10]), name=a.scenario)]
    T = a.nodes if a.targets is None else a.targets
    kw = dict(num_gateways=max(3, a.nodes // 40)) if a.nodes > 100 else {}
    return [synthetic(num_nodes=a.nodes, num_targets=T, seed=1000 + rank * a.topologies + k, **kw) for k in range(a.topologies)]


CONTROLLER_WEIGHTS = (1.0, 1.0, -10.0, 1.0)          # RandomController: state[0] + state[1] - 10 * state[2] + state[3]


def controller_map(obs):
    """``RandomController.make_action`` (controller/random/RandomController.py:12-15) for a batch of observations."""
    return obs[:, 0] + obs[:, 1] - 10.0 * obs[:, 2] + obs[:, 3]


# ----------------------------------------------------------------------------------------------- CPU side
def _cpu_worker(args):
    """One host core: an oracle environment (C restatement of the reference) driven by the same action law — for the
    controller law the RandomController map of the returned state, normalised and decoded by the reference's own
    statements (oracle/decode_oracle.py: numpy argmax / percentile, scipy L-BFGS-B)."""
    sc_dict, M, seed, budget_s, actions = args
    from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict, DEFAULT_MC
    from oracle import decode_oracle as do
    rng = np.random.default_rng(seed)
    o = OracleWRSN(scenario_from_dict(sc_dict), num_agent=M)
    xy = np.asarray(o.sc["nodes"], np.float64)
    thr = float(o.sc["par"][1])
    frame = None
    t0 = time.perf_counter()
    r = o.reset(want_state=True)
    n = 1
    ticks = 0.0
    t_decode = 0.0
    while time.perf_counter() - t0 < budget_s:
        if r["raw_agent_id"] < 0:
            ticks += o.now
            r = o.reset(want_state=True)
            n += 1
            continue
        if actions == "controller":
            td = time.perf_counter()
            if frame is None:
                frame = o.consts()["frame"]
            s = r["state"]
            nd = o.nodes()
            act = do.density_map_to_action(do.normalise_map(s[0] + s[1] - 10.0 * s[2] + s[3]), frame, xy, nd["status"], nd["energy"],
                                           nd["cs"], thr, DEFAULT_MC["charging_range"], DEFAULT_MC["alpha"], DEFAULT_MC["beta"], o.S)
            t_decode += time.perf_counter() - td
        else:
            act = rng.uniform(0, 1, 3)
            act[2] *= 0.05
        r = o.step(r["raw_agent_id"], act, want_state=True)
        if r["raw_agent_id"] >= 0:
            n += 1
    ticks += o.now
    return n, time.perf_counter() - t0, ticks, t_decode


def cpu_baseline(a, cores, budget_s):
    import multiprocessing as mp
    scs = scenarios_for(a, 0)
    law = getattr(a, "actions", "controller")
    jobs = [(scs[k % len(scs)].to_dict(), a.chargers, k, budget_s, law) for k in range(cores)]
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(cores) as pool:
            res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    n = sum(r[0] for r in res)
    per = sum(r[0] / r[1] for r in res)
    dec_share = sum(r[3] for r in res) / max(sum(r[1] for r in res), 1e-9)
    return dict(value=per, unit=UNIT, cores=cores, kind="port",
                sample="%d oracle envs (C restatement of rl_env/WRSN.py, one per core), %.0f s each, reset+step+get_state%s, "
                       "%d decisions, %.0f simulated s" % (
                           cores, budget_s,
                           " + RandomController map decoded by the reference's numpy/scipy statements (%.0f %% of the time)" % (100 * dec_share)
                           if law == "controller" else "", n, sum(r[2] for r in res)),
                wall_s=wall)


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = max(2.0, min(20.0, 120.0 / max(1, a.steps + a.warmup)))
    vals = []
    for k in range(a.warmup + a.steps):
        cb = cpu_baseline(a, cores, per_step)
        if k >= a.warmup:
            vals.append(cb)
    v = float(np.mean([c["value"] for c in vals]))
    ms = 1e3 * float(np.mean([c["wall_s"] for c in vals]))
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup, ms_per_step=ms,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=config_common(a), run=dict(note="each step = a %.0f s sample on every host core" % per_step),
                impl="reference",
                cpu_baseline=dict(value=v, unit=UNIT, cores=cores, kind="port", sample=vals[-1]["sample"]),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


def config_common(a, **extra):
    """`config` of the JSON line: the workload, described identically by both arms (the driver compares the two dicts).  What is specific
    to an arm or measured in a run (groups, budget, simulated seconds per decision ...) goes into the line's `run` object instead."""
    T = a.nodes if a.targets is None else a.targets
    c = dict(workload=workload_name(a), nodes=a.nodes, targets=T, chargers=a.chargers, envs_per_gpu=a.envs, map_size=100,
             actions=a.actions, topologies_per_gpu=a.topologies, observation="float32 [B,4,100,100]",
             l2="per GPU the environment records (22 KB each at 100 nodes) and the observations (160 KB per environment) are several times "
                "the 126 MB L2; no explicit flush")
    c.update(extra)
    return c


# ----------------------------------------------------------------------------------------------- GPU side
DUMP_OBS_ROWS = 64                                   # observation rows kept by --dump-outputs (160 KB each at S = 100)
DUMP_MAX_ENVS = 1 << 18                              # environments kept by --dump-outputs: 136 B each, 36 MB at most


def dump_outputs(out_dir, groups, act, obs):
    """``--dump-outputs``: what the last timed step handed its caller, one ``<name>.npy`` per array, so that two builds run with
    the same arguments (hence the same scenarios, seeds and step count) can be compared output for output.  The request record
    (``request_*``, float64; ``request_stats`` holds the running totals of the whole run, ``request_flags`` the engine's error
    bits) and the actions the step applied (``action``) of every environment, or of a fixed, seeded sample of ``DUMP_MAX_ENVS``
    of them (their indices in ``env_rows``); the float32 observations of a fixed, seeded sample of ``DUMP_OBS_ROWS`` environments
    (``observation``, their indices in ``observation_rows``): all of them would be 655 MB at 4096 environments.  A row without a
    request (``request_agent_id < 0``) has no reward, detail or action (the reference's None, NaN in the record): written as 0."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    B, Bg = sum(env.B for env in groups), obs[0].shape[0]
    env_rows = np.arange(B) if B <= DUMP_MAX_ENVS else np.sort(np.random.default_rng(1).choice(B, size=DUMP_MAX_ENVS, replace=False))
    rows = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_OBS_ROWS), replace=False))
    out = {"request_" + name: torch.cat([getattr(env.req, name) for env in groups]).to(torch.float64).cpu().numpy()[env_rows]
           for name in ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "stats")}
    none = out["request_agent_id"] < 0
    for name in ("reward", "detail", "action"):
        out["request_" + name][none] = 0.0
    out["action"] = torch.cat(act).cpu().numpy()[env_rows]
    out["env_rows"] = env_rows.astype(np.float64)
    out["observation"] = np.stack([obs[r // Bg][r % Bg].cpu().numpy() for r in rows])
    out["observation_rows"] = rows.astype(np.float64)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def run_b200(a):
    import torch
    import torch.distributed as dist
    from multi_agent_rl_wrsn_b200 import BatchedWRSN
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, M, S, G = a.envs, a.chargers, 100, max(1, a.groups)
    if B % G:
        raise SystemExit("--envs must be a multiple of --groups")
    Bg = B // G
    scs = scenarios_for(a, rank)
    # G asynchronous groups of environments, one CUDA stream each: one group's kernels (decode | step | reset | observe) overlap
    # with the other groups'.  Inside a launch the step budget bounds what one environment can do, so a launch lasts about as
    # long as the budget, not as long as its slowest environment (environments are independent; no collective).
    groups = [BatchedWRSN(scs, num_agent=M, num_envs=Bg, device=dev, threads=a.threads, map_size=S, step_budget=a.budget, step_rounds=a.rounds,
                          scenario_index=(np.arange(Bg) + g * Bg) % len(scs)) for g in range(G)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(G)]
    if a.engine_switch:
        for env in groups:
            env.hdr("OPT_NOBATCH")[:] = float(a.engine_switch)
            env.view("hdr", env._snap)[:, env.E["WRSN_H_OPT_NOBATCH"]] = float(a.engine_switch)
    N, T = groups[0].N, groups[0].T
    obs = [torch.zeros((Bg, 4, S, S), dtype=torch.float32, device=dev) for _ in range(G)]
    act = [torch.zeros((Bg, 3), dtype=torch.float64, device=dev) for _ in range(G)]
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    scale = torch.tensor([1.0, 1.0, 0.05], dtype=torch.float64, device=dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for g in range(G):
        groups[g].reset()
        groups[g].get_state(out=obs[g])
    sync_all()

    def group_step(g, law):
        """one pass of the hot path over group g: 4 launches of this library (decode | step | reset | observe) for the
        controller law, 3 for uniform actions (the map itself is three elementwise torch kernels: the controller's arithmetic)"""
        with torch.cuda.stream(streams[g]):
            if law == "controller":
                groups[g].linear_controller_action(obs[g], CONTROLLER_WEIGHTS, out=act[g])   # == density_map_to_action(controller_map(obs))
            else:
                torch.mul(torch.rand((Bg, 3), generator=gen, dtype=torch.float64, device=dev), scale, out=act[g])
            groups[g].rollout_step(act[g], obs[g])

    def totals():
        """(decisions, simulated seconds, resets) so far, from the kernels' own running totals"""
        st = torch.stack([env.req.stats.sum(0) for env in groups]).sum(0)
        return float(st[0].item()), float(st[1].item()), float(st[2].item())

    def timed(law, steps):
        sync_all()
        d0 = totals()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream(dev)
        t0 = time.perf_counter()
        e0.record(cur)
        for st in streams:
            st.wait_stream(cur)
        for k in range(steps):
            for g in range(G):
                group_step(g, law)
        for st in streams:
            cur.wait_stream(st)
        e1.record(cur)
        sync_all()
        d1 = totals()
        return e0.elapsed_time(e1), [y - x for x, y in zip(d0, d1)], t0, time.perf_counter()

    # untimed pre-roll: all episodes start at the same instant; run long enough for their phases to spread out, so the
    # timed window sees the steady state of a rollout (resets, death ticks and charging phases mixed) whatever K is
    for k in range(a.preroll + a.warmup):
        for g in range(G):
            group_step(g, a.actions)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    elapsed_ms, (decisions, ticks, episodes), t_wall0, t_wall1 = timed(a.actions, a.steps)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if a.dump_outputs and rank == 0:                 # before the legs below advance the same environments
        dump_outputs(a.dump_outputs, groups, act, obs)
    # per group and step: [k_decode_map, k_decode_locate,] [k_step_order (launches of >= 2048 rows),] k_env<STEP>, k_env<RESTORE_RESET>, k_observe
    launches_per_step = ((6 if a.actions == "controller" else 4) - (0 if 2048 <= Bg <= 16384 else 1)) * G
    n_launch = launches_per_step * a.steps
    inflight = float(sum((env.req.agent_id == -4).sum().item() for env in groups)) / B

    # ---- end to end through the reference's contract with HOST buffers (rl_env/WRSN.py:289-330: the request's `state` is a host
    # array, the controller runs on the host and hands `step` a density map).  Per step and group: the request record goes to
    # pinned host memory; the observations of the rows that CARRY a request (a row whose step is still in flight has no request
    # and no `state` to hand out) are packed on the device and copied to pinned host memory; the RandomController map of those rows
    # is formed ON THE HOST from that copy (torch CPU ops), copied back, scattered to its rows, decoded, stepped and rasterised on
    # the device.  The groups pipeline: while the host forms one group's maps the other groups' kernels and copies run.  The byte
    # counts are those of the tensors actually copied.  For uniform actions: actions from pinned host memory, request record back.
    ctl = a.actions == "controller"
    host_obs = [torch.zeros((Bg, 4, S, S), dtype=torch.float32).pin_memory() for _ in range(G)] if ctl else None
    host_map = [torch.zeros((Bg, S, S), dtype=torch.float32).pin_memory() for _ in range(G)] if ctl else None
    dev_map = [torch.zeros((Bg, S, S), dtype=torch.float32, device=dev) for _ in range(G)] if ctl else None
    dev_map_c = [torch.zeros((Bg, S, S), dtype=torch.float32, device=dev) for _ in range(G)] if ctl else None
    obs_c = [torch.zeros((Bg, 4, S, S), dtype=torch.float32, device=dev) for _ in range(G)] if ctl else None
    order = [torch.zeros(Bg, dtype=torch.int64, device=dev) for _ in range(G)]
    host_act = [(torch.rand((a.steps, Bg, 3), dtype=torch.float64) * scale.cpu()).pin_memory() for _ in range(G)]
    host_req = [dict(agent_id=torch.zeros(Bg, dtype=torch.int32).pin_memory(), reward=torch.zeros(Bg, dtype=torch.float64).pin_memory(),
                     terminal=torch.zeros(Bg, dtype=torch.uint8).pin_memory(), now=torch.zeros(Bg, dtype=torch.float64).pin_memory())
                for _ in range(G)]
    # many callers on few cores (several ranks per host): a waiting thread yields its core instead of spinning
    ev_blocking = G * int(os.environ.get("LOCAL_WORLD_SIZE", world)) * 2 > (os.cpu_count() or 1)
    rec_ev = [torch.cuda.Event(blocking=ev_blocking) for _ in range(G)]
    CH = 4                                                   # chunks per group and step of the state copy
    obs_ev = [[torch.cuda.Event(blocking=ev_blocking) for _ in range(CH)] for _ in range(G)]
    map_ev = [torch.cuda.Event() for _ in range(G)]
    copy_streams = [torch.cuda.Stream(device=dev) for _ in range(G)]
    req_bytes = sum(v.numel() * v.element_size() for v in host_req[0].values())
    row_obs, row_map = 4 * S * S * 4, S * S * 4
    h2d = d2h = 0

    def read_record(g):
        """request record to the host; the rows with a request first in `order`, their observations packed behind that order"""
        for name, v in host_req[g].items():
            v.copy_(getattr(groups[g].req, name), non_blocking=True)
        if ctl:
            has = groups[g].req.agent_id >= 0
            order[g].copy_(torch.argsort(has.to(torch.uint8), descending=True, stable=True))
            torch.index_select(obs[g], 0, order[g], out=obs_c[g])
        rec_ev[g].record(streams[g])

    sync_all()
    for g in range(G):
        with torch.cuda.stream(streams[g]):
            read_record(g)
    # one host thread per group (the groups are independent callers: each waits for ITS request records, asks for ITS states,
    # runs ITS controller and issues ITS next step; torch's CPU kernels, the CUDA synchronisations and the C-ABI calls release
    # the GIL), so that one group's host arithmetic overlaps the other groups' copies and kernels
    import threading
    counts = [[0, 0, 0] for _ in range(G)]                  # per group: decisions, h2d bytes, d2h bytes
    diag = [[0.0, 0.0, 0.0] for _ in range(G)]              # per group: seconds waiting for the records / for the states / in the controller
    errors = []
    cpu_threads = torch.get_num_threads()
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    e2e_threads = int(os.environ.get("WRSN_E2E_THREADS", "0")) or max(1, (os.cpu_count() or cpu_threads) // (G * max(1, local_world)))
    torch.set_num_threads(e2e_threads)
    host_w = torch.tensor(CONTROLLER_WEIGHTS, dtype=torch.float32).view(1, 1, 4)

    def caller(g, n_steps):
        try:
            torch.cuda.set_device(dev)
            cnt = counts[g]
            tm = diag[g]
            for k in range(n_steps + 1):
                t_a = time.perf_counter()
                rec_ev[g].synchronize()                    # the caller holds the request records of this group's last step
                tm[0] += time.perf_counter() - t_a
                n = int((host_req[g]["agent_id"] >= 0).sum())
                if k > 0:
                    cnt[0] += n
                    cnt[2] += req_bytes
                if k == n_steps:
                    break
                if ctl:
                    # ... and asks for the `state` of every request: copied in CHUNKS, so that the controller works on one chunk
                    # while the next one crosses PCIe, and its maps go back chunk by chunk
                    edges = [n * c // CH for c in range(CH + 1)]
                    with torch.cuda.stream(streams[g]):
                        for c in range(CH):
                            host_obs[g][edges[c]:edges[c + 1]].copy_(obs_c[g][edges[c]:edges[c + 1]], non_blocking=True)
                            obs_ev[g][c].record(streams[g])
                    cnt[2] += n * row_obs
                    for c in range(CH):
                        lo, hi = edges[c], edges[c + 1]
                        t_a = time.perf_counter()
                        obs_ev[g][c].synchronize()
                        t_b = time.perf_counter()
                        # RandomController.make_action on the host: the channel combination as ONE pass over the states (a [1 x 4]
                        # by [4 x S^2] product per request; elementwise adds on channel slices are strided and 20 x slower)
                        torch.matmul(host_w, host_obs[g][lo:hi].view(hi - lo, 4, S * S), out=host_map[g][lo:hi].view(hi - lo, 1, S * S))
                        tm[1] += t_b - t_a; tm[2] += time.perf_counter() - t_b
                        with torch.cuda.stream(copy_streams[g]):       # (the maps go back on a second stream: the state copies of
                            dev_map_c[g][lo:hi].copy_(host_map[g][lo:hi], non_blocking=True)   # the later chunks are still queued on the first)
                    map_ev[g].record(copy_streams[g])
                with torch.cuda.stream(streams[g]):
                    if ctl:
                        streams[g].wait_event(map_ev[g])
                        dev_map[g].index_copy_(0, order[g][:n], dev_map_c[g][:n])
                        groups[g].density_map_to_action(dev_map[g], out=act[g])
                        cnt[1] += n * row_map
                    else:
                        act[g].copy_(host_act[g][k % a.steps], non_blocking=True)
                        cnt[1] += host_act[g][0].numel() * 8
                    groups[g].rollout_step(act[g], obs[g])
                    read_record(g)
        except Exception as ex:                              # noqa: BLE001 - re-raised on the main thread
            errors.append(ex)

    def run_callers(n_steps):
        workers = [threading.Thread(target=caller, args=(g, n_steps)) for g in range(G)]
        for w in workers:
            w.start()
        for w in workers:
            w.join()

    run_callers(a.warmup)                                    # untimed: thread pools, first-touch of the pinned buffers, pipeline fill
    for c, d in zip(counts, diag):
        c[:] = [0, 0, 0]
        d[:] = [0.0, 0.0, 0.0]
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cur = torch.cuda.current_stream(dev)
    sync_all()
    f0.record(cur)
    for st in streams:
        st.wait_stream(cur)
    run_callers(a.steps)
    for st in streams:
        cur.wait_stream(st)
    f1.record(cur)
    sync_all()
    torch.set_num_threads(cpu_threads)
    if errors:
        raise errors[0]
    e2e_ms = f0.elapsed_time(f1)
    if os.environ.get("WRSN_E2E_DIAG") == "1" and rank == 0:
        print("e2e host threads, ms per step [wait records, wait states, controller]: " +
              ", ".join("[%.2f %.2f %.2f]" % tuple(1e3 * x / a.steps for x in d) for d in diag), file=sys.stderr)
    e2e_dec = sum(c[0] for c in counts)
    h2d, d2h = sum(c[1] for c in counts), sum(c[2] for c in counts)
    h2d, d2h = h2d // a.steps, d2h // a.steps              # per step, averaged over the timed steps
    del host_obs, host_map, dev_map, dev_map_c, obs_c

    # ---- roofline pass: the same hot path issued serially on ONE stream through the separate entry points, a pair of CUDA
    # events around every launch (concurrent groups time-share the SMs and blur per-launch durations).  The row masks are
    # computed before the events are recorded, so that an interval holds this library's launches and nothing else.
    R = min(a.steps, 16)
    names = ("decode", "step", "reset", "observe")
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in names] for _ in range(R * G)]
    u8 = lambda t: t.to(torch.uint8)
    sync_all()
    rd0 = totals()
    for k in range(R):
        for g in range(G):
            env = groups[g]
            e = ev[k * G + g]
            aid = env.req.agent_id
            m_step = u8((aid >= 0) | (aid == -4))
            e[0][0].record()
            if a.actions == "controller":
                env.linear_controller_action(obs[g], CONTROLLER_WEIGHTS, out=act[g])     # k_decode_map + k_decode_locate
            else:
                torch.mul(torch.rand((Bg, 3), generator=gen, dtype=torch.float64, device=dev), scale, out=act[g])
            e[0][1].record()
            e[1][0].record()
            env.step(aid, act[g], mask=m_step)
            e[1][1].record()
            m_done = u8((env.req.agent_id < 0) & (env.req.agent_id != -4))
            e[2][0].record()
            env.reset(mask=m_done)
            e[2][1].record()
            e[3][0].record()
            env.get_state(out=obs[g])
            e[3][1].record()
    sync_all()
    k_ms = {n: sum(x[i][0].elapsed_time(x[i][1]) for x in ev) for i, n in enumerate(names)}
    rd1 = totals()
    r_decisions, r_ticks = rd1[0] - rd0[0], rd1[1] - rd0[1]
    n_l = R * G

    extras = {}
    if not a.no_extras:
        # ---- side figure: the other action law on the same environments (device-resident, short)
        other = "uniform" if a.actions == "controller" else "controller"
        K2 = min(a.steps, 30)
        for k in range(20):
            for g in range(G):
                group_step(g, other)
        o_ms, (o_dec, o_sim, _), _, _ = timed(other, K2)
        extras["other_law"] = (other, o_ms, o_dec, o_sim, K2)
        # ---- standalone kernels, timed alone behind a spin kernel (a launch lasts ~10 us, less than the host needs to issue it)
        maps = [torch.rand((Bg, S, S), generator=gen, dtype=torch.float32, device=dev) for _ in range(max(G, 1 + (B * S * S * 4 < 2e8) * (int(2e8 // (Bg * S * S * 4)))))]
        dec_out = torch.zeros((Bg, 3), dtype=torch.float64, device=dev)
        all_agents = torch.zeros(Bg, dtype=torch.int32, device=dev)
        for m in maps:
            groups[0].density_map_to_action(m, agent_id=all_agents, out=dec_out)
        n_dec = 6 * len(maps)
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        torch.cuda._sleep(int(2e7))
        d0.record()
        for k in range(n_dec):
            groups[0].density_map_to_action(maps[k % len(maps)], agent_id=all_agents, out=dec_out)
        d1.record()
        sync_all()
        extras["decode_alone"] = (d0.elapsed_time(d1) / n_dec, Bg * (S * S * 4 + 24), len(maps) * Bg * S * S * 4)
        del maps
        try:
            node_rate, mc_rate = groups[0].charge_rates()
            n_chg = 48
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sync_all()
            torch.cuda._sleep(int(2e7))
            c0.record()
            for k in range(n_chg):
                groups[k % G].charge_rates(out=(node_rate, mc_rate))
            c1.record()
            sync_all()
            extras["charge_alone"] = (c0.elapsed_time(c1) / n_chg, Bg * (17 * N + 8 * N + 8 * M))
        except Exception as ex:                              # noqa: BLE001 - diagnostic figure only
            extras["charge_error"] = str(ex)[:200]

    # ---- reduce over ranks: max time, summed work
    t = torch.tensor([elapsed_ms, e2e_ms], dtype=torch.float64, device=dev)
    w = torch.tensor([decisions, ticks, float(e2e_dec), episodes], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    elapsed_ms, e2e_ms = [float(x) for x in t.tolist()]
    decisions_all, ticks_all, e2e_dec_all, episodes_all = [float(x) for x in w.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = decisions_all / (elapsed_ms * 1e-3)
    peaks = {}
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    # algorithmic bytes per SURVEY §8(d): 82 N + T per environment and simulated second, 16 T + 88 per decision in the
    # step kernel, 4 S^2 float32 per decision in the observation kernel, S^2 float32 + 24 per decision in the decoder
    alg = dict(step=(r_ticks * (82 * N + T) + r_decisions * (16 * T + 88)) / n_l, observe=r_decisions * (4 * S * S * 4) / n_l,
               decode=r_decisions * (4 * S * S * 4 + 24) / n_l if a.actions == "controller" else 0.0, reset=0.0)   # (decode: the four channels it reads)
    pass_ms = sum(k_ms.values())
    kern_name = dict(step="k_env<MODE_STEP>", observe="k_observe<float>", decode="k_decode_map<float,4> + k_decode_locate",
                     reset="k_env<MODE_RESTORE_RESET>")
    kernels = {}
    for n in names:
        ms = k_ms[n] / n_l
        kernels[kern_name[n]] = dict(ms_per_launch=ms, algorithmic_bytes=alg[n], gbs=alg[n] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0,
                                     share=k_ms[n] / pass_ms)
    dom = max(names, key=lambda n: k_ms[n])
    ach = kernels[kern_name[dom]]["gbs"]
    # in situ: the whole timed region's algorithmic bytes over its duration (all kernels, concurrent groups)
    insitu_bytes = ticks_all * (82 * N + T) + decisions_all * (16 * T + 88 + 4 * S * S * 4 + (4 * S * S * 4 + 24 if a.actions == "controller" else 0))
    insitu_gbs = insitu_bytes / world / (elapsed_ms * 1e-3) / 1e9
    traffic, issue = None, None
    try:                                                 # numbers of the committed ncu capture of this launch shape (profiles/)
        with open(os.path.join(REPO, "profiles", "traffic_r02.json")) as f:
            tj = json.load(f)
        if tj.get("nodes") == N and tj.get("chargers") == M:
            traffic = tj.get("dram_bytes_per_env_launch", 0.0) * Bg
            wi = tj.get("warp_instructions_per_sim_second", 0.0) * (r_ticks / n_l) + tj.get("warp_instructions_per_launch_fixed", 0.0) * Bg
            sm_hz = (clocks or {}).get("sm_mhz") or 1965.0
            peak_issue = 148 * 4 * sm_hz * 1e6
            issue = dict(warp_instructions_per_launch=wi, achieved=wi / (k_ms["step"] / n_l * 1e-3), peak=peak_issue,
                         frac=wi / (k_ms["step"] / n_l * 1e-3) / peak_issue, unit="warp-instructions/s",
                         note="instruction-issue roofline of the step kernel (148 SMs x 4 schedulers x SM clock): DRAM traffic is far "
                              "below the algorithmic bytes (the record lives in shared memory), the issue slots are what it spends; "
                              "instruction counts from " + str(tj.get("source")))
    except Exception:
        pass
    line = dict(
        metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup,
        ms_per_step=elapsed_ms / a.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
        data="synthetic",
        config=config_common(a),
        run=dict(
            groups="%d asynchronous groups of %d environments, one CUDA stream each" % (G, Bg),
            step_budget=a.budget, step_rounds=a.rounds, threads_per_env=int(groups[0].dims.threads),
            working_set="state %.0f MB + observations %.0f MB per GPU" % (B * groups[0].dims.state_bytes / 1e6, B * 4 * S * S * 4 / 1e6),
            sim_seconds_per_decision=ticks_all / max(decisions_all, 1.0),
            decisions_per_env_step=decisions_all / (a.steps * B * world),
            steps_in_flight_at_end=inflight,
            env_ticks_per_s=ticks_all / (elapsed_ms * 1e-3),
            episodes_per_s=episodes_all / (elapsed_ms * 1e-3),
            resets="finished episodes are reset inside the timed step (wrsn_rollout_step: step | reset | observe)"),
        clocks=clocks,
        e2e=dict(value=e2e_dec_all / (e2e_ms * 1e-3), unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                 ms_per_step=e2e_ms / a.steps,
                 note=("the reference's contract with host buffers: per step the request record AND the observations of the rows that "
                       "carry a request (the request's `state`; a row whose step is still in flight has none) go to pinned host memory, "
                       "the RandomController map is formed on the host from them, copied to the device, decoded, stepped, rasterised; "
                       "one host thread per group (PCIe- and host-bound); bytes = per-step mean of the tensors actually copied") if a.actions == "controller" else
                      "per step: actions from pinned host memory, rollout_step, request record read back on the host"),
        gpu_launches=n_launch,
        roofline=dict(bound="hbm", kernel=kern_name[dom], achieved=ach, peak=peak, unit="GB/s", frac=ach / peak,
                      traffic=traffic, peak_source=peak_src,
                      how="serialized pass of %d launches per kernel on one stream right after the timed region, CUDA events around "
                          "every launch; achieved = algorithmic bytes (SURVEY 8d) / launch duration" % n_l,
                      in_situ=dict(achieved=insitu_gbs, frac=insitu_gbs / peak,
                                   note="all kernels of the timed region together: its algorithmic bytes / its device time"),
                      issue=issue, kernels=kernels))
    if "other_law" in extras:
        other, o_ms, o_dec, o_sim, K2 = extras["other_law"]
        line["run"]["other_action_law"] = dict(actions=other, value=o_dec / (o_ms * 1e-3), unit=UNIT, steps=K2,
                                                  sim_seconds_per_decision=o_sim / max(o_dec, 1.0),
                                                  note="same environments, device-resident, not the headline workload")
    if "decode_alone" in extras:
        ms, by, ws = extras["decode_alone"]
        line["roofline"]["kernels"]["k_decode_map<float> alone"] = dict(
            ms_per_launch=ms, algorithmic_bytes=by, gbs=by / (ms * 1e-3) / 1e9, frac=by / (ms * 1e-3) / 1e9 / peak,
            note="every environment decodes; %d MB of maps cycled (more than the 126 MB L2)" % (ws / 1e6))
    if "charge_alone" in extras:
        ms, by = extras["charge_alone"]
        line["roofline"]["kernels"]["k_charge"] = dict(
            ms_per_launch=ms, algorithmic_bytes=by, gbs=by / (ms * 1e-3) / 1e9, frac=by / (ms * 1e-3) / 1e9 / peak, share=0.0,
            note="dense node x charger charging model, standalone (unit parity / profiling); the rollout applies the model "
                 "incrementally inside the step kernel")
    if world == 1 and not a.no_cpu_baseline:
        line["cpu_baseline"] = {k: v for k, v in cpu_baseline(a, 1, a.cpu_seconds).items() if k != "wall_s"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------- configs[2]: IPPO training
IPPO_ARGS = dict(seed=0, lr=3.0e-4, gamma=0.99, clip=0.2, batch_size=512, n_updates_per_iteration=5, save_freq=10 ** 9, gae=True,
                 norm_adv=True, minibatch_size=64, ent_coef=0.0, vf_coef=0.5, gae_lambda=0.95, max_grad_norm=0.5,
                 clip_vloss=True)                                    # alg_args/ippo.yaml (save_freq: no checkpoints while timing)


def run_ippo(a):
    """One training iteration = IPPO.train's loop body (controller/ippo/IPPO.py:212-310): roll_out until every charger's
    network has batch_size transitions (batched: every environment of the shard advances together, the record stays in HBM),
    then n_updates_per_iteration x (batch_size / minibatch_size) clipped-PPO minibatch steps per charger with ONE gradient
    all-reduce per minibatch (NCCL over NVLink: 8.3 MB per actor + critic pair).  Reports agent-decisions/s of the whole loop
    and where the time goes: simulator kernels vs actor inference in roll_out, update compute vs all-reduce."""
    import torch
    import torch.distributed as dist
    from multi_agent_rl_wrsn_b200 import BatchedWRSN
    from multi_agent_rl_wrsn_b200 import controllers as ctl
    from multi_agent_rl_wrsn_b200.ippo import BatchedIPPO
    from multi_agent_rl_wrsn_b200.nets import CNNCritic, UNetActor, num_parameters
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(1234 + rank)                           # (different seeds on purpose: the constructor broadcasts rank 0's weights)
    B, M, S = a.envs, a.chargers, 100
    env = BatchedWRSN(scenarios_for(a, rank), num_agent=M, num_envs=B, device=dev, threads=a.threads, map_size=S,
                      step_budget=a.budget, step_rounds=a.rounds)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(99 + rank)
    tr = BatchedIPPO(IPPO_ARGS, env, device=dev, window=a.window, generator=gen)
    n_params = num_parameters(tr.actors[0]) + num_parameters(tr.critics[0])
    timers = []
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def iteration(timed):
        e = [ev() for _ in range(3)]
        e[0].record()
        batches = tr.roll_out()
        e[1].record()
        for i in range(M):
            ctl.ppo_update(tr.actors[i], tr.critics[i], tr.optimizers[i], batches[i], IPPO_ARGS, group=None, generator=gen,
                           timers=timers if timed else None)
        e[2].record()
        return e, dict(tr.last_rollout)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(max(1, a.warmup // 3)):
        iteration(False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    sync_all()
    t0w = time.perf_counter()
    g0, g1 = ev(), ev()
    g0.record()
    recs = [iteration(True) for _ in range(a.iterations)]
    g1.record()
    sync_all()
    t1w = time.perf_counter()
    clocks = sampler.stop(t0w, t1w) if rank == 0 else None
    total_ms = g0.elapsed_time(g1)
    roll_ms = sum(e[0].elapsed_time(e[1]) for e, _ in recs)
    upd_ms = sum(e[1].elapsed_time(e[2]) for e, _ in recs)
    ar_ms = sum(x.elapsed_time(y) for x, y in timers)
    decisions = sum(r["decisions"] for _, r in recs)         # (already summed over ranks by roll_out)
    sim_s = sum(r["simulated_seconds"] for _, r in recs)
    # the simulator's own share of roll_out: the same number of rollout steps without any network (RandomController law)
    t = torch.tensor([total_ms, roll_ms, upd_ms, ar_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, roll_ms, upd_ms, ar_ms = [float(x) for x in t.tolist()]
    if rank == 0:
        cfg = config_common(a, envs_per_gpu=B, step_budget=a.budget, window=a.window, alg_args="alg_args/ippo.yaml",
                            networks="U-Net actor (%d parameters) + CNN critic per charger, cuDNN convolutions (TF32), written from "
                                     "the reference's shapes (multi_agent_rl_wrsn_b200/nets.py); %d parameters = %.1f MB per all-reduce"
                                     % (num_parameters(tr.actors[0]), n_params, n_params * 4 / 1e6),
                            iterations=a.iterations, minibatch_steps_per_iteration=len(timers) // max(a.iterations, 1),
                            sim_seconds_per_decision=sim_s / max(decisions, 1.0))
        cfg["workload"] = "IPPO training loop (alg_args/ippo.yaml), %d-node/%d-charger synthetic WRSN, %d envs per GPU" % (a.nodes, M, B)
        line = dict(metric=METRIC, value=decisions / (total_ms * 1e-3), unit=UNIT, n_gpus=world, steps=a.iterations, warmup=a.warmup,
                    ms_per_step=total_ms / a.iterations, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64 simulator / tf32 networks",
                    data="synthetic", config=cfg, clocks=clocks,
                    breakdown=dict(roll_out_ms=roll_ms / a.iterations, update_ms=upd_ms / a.iterations, allreduce_ms=ar_ms / a.iterations,
                                   allreduce_share_of_update=ar_ms / max(upd_ms, 1e-9),
                                   limiter="update" if upd_ms > roll_ms else "roll_out",
                                   note="roll_out = simulator kernels + actor inference (U-Net forward on every request) + critic "
                                        "values for the advantages; update = forward / backward of actor + critic on %d minibatches "
                                        "per charger; all-reduce = one flat %.1f MB bucket per minibatch" % (
                                            IPPO_ARGS["n_updates_per_iteration"] * IPPO_ARGS["batch_size"] // IPPO_ARGS["minibatch_size"],
                                            n_params * 4 / 1e6)))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "ippo":
        run_ippo(args)
    else:
        run_b200(args)
