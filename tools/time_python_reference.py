#!/usr/bin/env python
"""Time the UNMODIFIED Python reference (a checkout found through $WRSN_REFERENCE_ROOT, run under the oracle shims: oracle/ref_runner.py) on the host cores,
as BASELINE.md §4 plans it: one `WRSN` per process on all cores, the reference's own loop (runner/checkRL.py:33-36) —
`RandomController.make_action` -> `WRSN.step` with `density_map=True` (default), or uniform 3-vector actions with
`--actions uniform` — for a fixed wall budget after `reset()`.  Prints one JSON line (`kind: "python-reference"`).

BUILD CONTAINER ONLY: the reference does not travel to the GPU box; the committed line lives in profiles/.
    python tools/time_python_reference.py [--scenario hanoi1000n100] [--seconds 120] [--cores N] [--actions controller|uniform]
"""
import argparse, json, multiprocessing as mp, os, sys, time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(args):
    scenario, seconds, actions, seed = args
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    from ref_runner import load_reference
    import numpy as np
    R = load_reference()
    os.chdir(R.root)                                                 # SURVEY Q11: the reference resolves paths from its root
    t0 = time.perf_counter()
    env = R.WRSN(scenario_path=os.path.join(R.scenario_dir, scenario + ".yaml"), agent_type_path=R.mc_type, num_agent=3,
                 map_size=100, density_map=(actions == "controller"))
    request = env.reset()
    t_reset = time.perf_counter() - t0
    rng = np.random.default_rng(seed)
    n, resets, sim = 0, 0, 0.0
    t1 = time.perf_counter()
    while time.perf_counter() - t1 < seconds:
        if request is None or request["terminal"]:
            sim += env.env.now - 100.0
            request = env.reset(); resets += 1
            continue
        if actions == "controller":                                  # controller/random/RandomController.py:12-15
            s = request["state"]
            a = np.copy(s[0] + s[1] - 10 * s[2] + s[3])
        else:
            a = rng.uniform(0, 1, 3); a[2] *= 0.05
        request = env.step(request["agent_id"], a)
        if request is not None and request["agent_id"] is not None:
            n += 1
    sim += env.env.now - 100.0
    return n, time.perf_counter() - t1, t_reset, sim, resets


if __name__ == "__main__":
    p = argparse.ArgumentParser()
    p.add_argument("--scenario", default="hanoi1000n100")
    p.add_argument("--seconds", type=float, default=120.0)
    p.add_argument("--cores", type=int, default=os.cpu_count() or 1)
    p.add_argument("--actions", default="controller", choices=["controller", "uniform"])
    a = p.parse_args()
    with mp.get_context("spawn").Pool(a.cores) as pool:
        res = pool.map(worker, [(a.scenario, a.seconds, a.actions, k) for k in range(a.cores)])
    per = sum(r[0] / r[1] for r in res)
    n = sum(r[0] for r in res)
    print(json.dumps(dict(metric="agent-decisions/sec", value=per, unit="decisions/s", cores=a.cores, kind="python-reference",
                          per_core=per / a.cores, decisions=n, seconds_per_worker=a.seconds,
                          reset_seconds=sum(r[2] for r in res) / len(res), simulated_seconds=sum(r[3] for r in res),
                          sim_seconds_per_decision=sum(r[3] for r in res) / max(n, 1),
                          sample="unmodified reference under oracle/shims (SimPy-4.0.1-semantics shim), %s.yaml, 3 chargers, "
                                 "map 100, %s, one WRSN per process x %d processes, %.0f s each after reset()" % (
                                     a.scenario, "RandomController density maps (density_map=True)" if a.actions == "controller"
                                     else "uniform 3-vector actions (density_map=False)", a.cores, a.seconds),
                          host="%d-core build container" % (os.cpu_count() or 1))), flush=True)
