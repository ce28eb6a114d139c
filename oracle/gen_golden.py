#!/usr/bin/env python
"""Generate the committed golden fixtures under ``tests/golden/`` by running the
UNMODIFIED reference (a checkout: set ``WRSN_REFERENCE_ROOT``) under the oracle shims.

TEST INFRASTRUCTURE (oracle side).  Run from the repo root in the build container:

    python oracle/gen_golden.py            # everything (≈15 min of CPU)
    python oracle/gen_golden.py net:hanoi1000n50 ep:basic_n50   # selected cases

The reference has no tests or golden vectors of its own (SURVEY.md §4), so these
outputs of the reference itself are what pins the C restatement
(``oracle/wrsn_oracle.c``) and, through it and directly, the CUDA path.

Fixtures:
  net_<scenario>.npz   pure network, no chargers (``runner/test_network.py`` logic,
                       Network.py:69-81): death list, `alive` flip time, end time,
                       energy snapshots, levels / targets_active before and after.
  ep_<case>.npz        ``WRSN.reset/step`` episodes with injected 3-vector actions
                       (``density_map=False``; rl_env/WRSN.py:41-83,289-330):
                       per-decision agent id, env.now, terminal, reward, action, node
                       energy / status / energyCS / level, targets_active, charger
                       records, observation channel sums and a few full observations.
"""
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, HERE)
from ref_runner import load_reference  # noqa: E402

OUT = os.environ.get("WRSN_GOLDEN_OUT") or os.path.join(REPO, "tests", "golden")
MAX_EVENTS_PER_STEP = 3_000_000      # the reference never returns if every charger is dead (Q1)


class Budget(Exception):
    pass


def _net_snapshot(net):
    return dict(
        energy=np.array([float(n.energy) for n in net.listNodes], np.float64),
        status=np.array([n.status for n in net.listNodes], np.uint8),
        cs=np.array([float(n.energyCS) for n in net.listNodes], np.float64),
        rr=np.array([float(n.energyRR) for n in net.listNodes], np.float64),
        level=np.array([(-1 if n.level is None else n.level) for n in net.listNodes], np.int32),
        log_energy=np.array([float(n.log_energy) for n in net.listNodes], np.float64),
        targets_active=np.array(net.targets_active, np.uint8),
        alive=np.uint8(net.alive),
    )


def pure_network(R, scn, snap_times=(0.25, 0.75, 1.25, 10.75, 11.25, 100.0 - 0.25)):
    """Network only, until ``net.operate`` finishes (Network.py:69-81)."""
    io = R.NetworkIO(os.path.join(R.scenario_dir, scn + ".yaml"))
    env, net = io.makeNetwork()
    proc = env.process(net.operate())
    N = len(net.listNodes)
    deaths = []          # (tick time k+0.5, node id) in id order inside a tick
    alive_flip = -1.0
    snaps = {}
    prev_status = np.ones(N, np.uint8)
    k = 0
    snap_times = set(snap_times)
    post_death_snaps = 0
    t0 = time.time()
    while True:
        # poll at k+0.25 (after setLevels at k+0.1) and k+0.75 (after the drain tick at k+0.5)
        for frac in (0.25, 0.75):
            t = k + frac
            if proc.callbacks is None:
                break
            env.run(until=t)
            if frac == 0.25 and alive_flip < 0 and net.alive == 0:
                alive_flip = k + 0.1
            if frac == 0.75:
                st = np.array([n.status for n in net.listNodes], np.uint8)
                died = np.nonzero((prev_status == 1) & (st == 0))[0]
                for d in died:
                    deaths.append((k + 0.5, int(d)))
                if len(died):
                    snaps["t%.2f" % t] = _net_snapshot(net)
                    post_death_snaps = 2
                prev_status = st
            elif post_death_snaps > 0:
                snaps["t%.2f" % t] = _net_snapshot(net)
                post_death_snaps -= 1
            if t in snap_times or (k % 500 == 0 and frac == 0.75):
                snaps["t%.2f" % t] = _net_snapshot(net)
        if proc.callbacks is None:
            break
        k += 1
    # drain whatever is left at the final timestamp (nodes' k+1.0 bookkeeping follows the exit check)
    end_time = float(np.floor(env.now))      # Network.operate leaves its loop at an integer second
    env.run(until=float(env.now) + 0.5)
    final = _net_snapshot(net)
    out = dict(
        scenario=scn, N=N, T=len(net.listTargets),
        deaths_t=np.array([d[0] for d in deaths], np.float64),
        deaths_node=np.array([d[1] for d in deaths], np.int32),
        alive_flip=np.float64(alive_flip), end_time=np.float64(end_time),
        inactive_targets=np.int32(int(np.sum(final["targets_active"] == 0))),
        sum_energy_end=np.float64(sum(float(n.energy) for n in net.listNodes)),
        frame=np.array(net.frame, np.float64),
        direct=np.array([n.id for n in net.baseStation.direct_nodes], np.int32),
        snap_keys=np.array(sorted(snaps.keys(), key=lambda s: float(s[1:]))),
    )
    out.update(_scenario_arrays(os.path.join(R.scenario_dir, scn + ".yaml")))
    for key, s in snaps.items():
        for f, v in s.items():
            out["%s_%s" % (key, f)] = v
    for f, v in final.items():
        out["final_%s" % f] = v
    print("net:%s N=%d T=%d first death %s end %.1f inactive %d sumE %.10f  (%.0fs)" % (
        scn, N, out["T"], deaths[0] if deaths else None, end_time, out["inactive_targets"],
        out["sum_energy_end"], time.time() - t0), flush=True)
    np.savez_compressed(os.path.join(OUT, "net_%s.npz" % scn), **out)


def _scenario_arrays(io_or_path):
    """The scenario as plain arrays, so tests need neither a checkout of the reference nor its YAML files."""
    import yaml
    with open(io_or_path) as f:
        d = yaml.safe_load(f)
    spe = d["node_phy_spe"]
    par = np.array([spe["capacity"], spe["threshold"], spe["com_range"], spe["sen_range"], spe["prob_gp"],
                    spe["package_size"], spe["er"], spe["et"], spe["efs"], spe["emp"], d["max_time"]], np.float64)
    return dict(sc_nodes=np.array(d["nodes"], np.float64), sc_targets=np.array(d["targets"], np.float64),
                sc_bs=np.array(d["base_station"], np.float64), sc_par=par, sc_seed=np.int64(d["seed"]))


def _mc_record(w):
    ag = w.agents
    M = len(ag)
    rec = dict(
        mc_loc=np.array([[float(a.location[0]), float(a.location[1])] for a in ag], np.float64),
        mc_energy=np.array([float(a.energy) for a in ag], np.float64),
        mc_status=np.array([a.status for a in ag], np.uint8),
        mc_cpa=np.array([[float(a.cur_phy_action[0]), float(a.cur_phy_action[1]),
                          float(a.cur_phy_action[2])] for a in ag], np.float64),
        mc_type=np.array([1 if a.cur_action_type == "charging" else 0 for a in ag], np.uint8),
        mc_nconn=np.array([len(a.connected_nodes) for a in ag], np.int32),
        excl=np.array([float(x) for x in w.agents_exclusive_reward], np.float64),
    )
    assert rec["mc_loc"].shape == (M, 2)
    return rec


def episode(R, case, scn, actions, num_agent=3, mc_yaml=None, max_decisions=10**9,
            full_state_every=20, map_size=100, event_budget=MAX_EVENTS_PER_STEP):
    """reset() then step() with the injected action list (cycled) until terminal,
    `max_decisions`, a ``None`` request (Q7) or the event budget (all chargers dead, Q1)."""
    mc_path = R.mc_type
    if mc_yaml is not None:
        mc_path = os.path.join(OUT, "mc_%s.yaml" % case)
        with open(mc_path, "w") as f:
            f.write(mc_yaml)
    t0 = time.time()
    w = R.WRSN(os.path.join(R.scenario_dir, scn + ".yaml"), mc_path, num_agent,
               map_size=map_size, density_map=False)
    req = w.reset()
    recs = []
    full_states = {}

    def record(req, fed_agent, fed_action):
        i = len(recs)
        r = dict(fed_agent=-1 if fed_agent is None else fed_agent,
                 fed_action=np.array(fed_action if fed_action is not None else [np.nan] * 3, np.float64),
                 now=float(w.env.now))
        if req is None:      # Q7: implicit None
            r.update(agent_id=-2, terminal=0, reward=np.nan, action=np.full(3, np.nan), chan_sum=np.full(4, np.nan))
        else:
            aid = req["agent_id"]
            r.update(agent_id=-1 if aid is None else int(aid), terminal=int(bool(req["terminal"])),
                     reward=np.nan if req["reward"] is None else float(req["reward"]),
                     action=np.full(3, np.nan) if req["action"] is None else np.array(req["action"], np.float64))
            if req["state"] is not None:
                st = np.asarray(req["state"], np.float64)
                r["chan_sum"] = st.reshape(4, -1).sum(axis=1)
                if i % full_state_every == 0 or i < 4:
                    full_states[i] = st
                    if req["prev_state"] is not None and i in (3, full_state_every):
                        full_states[(i, "prev")] = np.asarray(req["prev_state"], np.float64)
            else:
                r["chan_sum"] = np.full(4, np.nan)
        r.update(_net_snapshot(w.net))
        r.update(_mc_record(w))
        r["fitness_min"] = float(np.min(w.get_network_fitness()))
        recs.append(r)

    record(req, None, None)
    nev = [0]

    def tr(now, prio, eid, ev):
        nev[0] += 1
        if nev[0] > event_budget:
            raise Budget()
    end = "max_decisions"
    i = 0
    while len(recs) <= max_decisions:
        if req is None:
            end = "none_request"
            break
        if req["terminal"]:
            end = "terminal"
            break
        a = actions[i % len(actions)]
        i += 1
        nev[0] = 0
        w.env._trace = tr
        try:
            req2 = w.step(req["agent_id"], a)
        except Budget:
            end = "hang_all_chargers_dead"
            break
        record(req2, req["agent_id"], a)
        req = req2
    keys = [k for k in recs[0].keys()]
    out = dict(case=case, scenario=scn, num_agent=num_agent, end=end, n=len(recs), map_size=map_size,
               mc_yaml="" if mc_yaml is None else mc_yaml,
               moving_time_max=float(w.moving_time_max), charging_time_max=float(w.charging_time_max),
               avg_nodes_agent=float(w.avg_nodes_agent), frame=np.array(w.net.frame, np.float64))
    out.update(_scenario_arrays(os.path.join(R.scenario_dir, scn + ".yaml")))
    import yaml
    with open(mc_path) as f:
        mcd = yaml.safe_load(f)
    out["mc_par"] = np.array([mcd["capacity"], mcd["threshold"], mcd["velocity"], mcd["pm"], mcd["charging_range"],
                              mcd["alpha"], mcd["beta"], mcd["epsilon"]], np.float64)
    if mc_yaml is not None:
        os.remove(mc_path)
    for k in keys:
        out[k] = np.stack([np.asarray(r[k]) for r in recs])
    idx = sorted(k for k in full_states if not isinstance(k, tuple))
    out["full_state_idx"] = np.array(idx, np.int32)
    out["full_state"] = np.stack([full_states[k] for k in idx]).astype(np.float64)
    pidx = sorted(k[0] for k in full_states if isinstance(k, tuple))
    out["full_prev_state_idx"] = np.array(pidx, np.int32)
    if pidx:
        out["full_prev_state"] = np.stack([full_states[(k, "prev")] for k in pidx]).astype(np.float64)
    np.savez_compressed(os.path.join(OUT, "ep_%s.npz" % case), **out)
    print("ep:%s %s decisions=%d end=%s now=%.6f (%.0fs)" % (case, scn, len(recs), end, w.env.now,
                                                             time.time() - t0), flush=True)


def episode_density(R, case, scn, n_dec, num_agent=3):
    """``density_map=True`` with the reference's RandomController rule (controller/random/RandomController.py:12-15:
    dmap = s0 + s1 - 10 s2 + s3), i.e. runner/checkRL.py's loop: records the decoded action of every decision."""
    t0 = time.time()
    w = R.WRSN(os.path.join(R.scenario_dir, scn + ".yaml"), R.mc_type, num_agent, map_size=100, density_map=True)
    req = w.reset()
    rows = []
    while len(rows) < n_dec and not req["terminal"]:
        st = req["state"]
        dmap = np.copy(st[0] + st[1] - 10 * st[2] + st[3])
        aid = req["agent_id"]
        req = w.step(aid, dmap)
        rows.append(dict(fed_agent=aid, agent_id=-1 if req["agent_id"] is None else req["agent_id"], now=float(w.env.now),
                         action=np.array(w.agents_action[aid], np.float64),
                         reward=np.nan if req["reward"] is None else float(req["reward"]),
                         energy=np.array([float(n.energy) for n in w.net.listNodes])))
    out = dict(case=case, scenario=scn, num_agent=num_agent, n=len(rows))
    out.update(_scenario_arrays(os.path.join(R.scenario_dir, scn + ".yaml")))
    for k in rows[0]:
        out[k] = np.stack([np.asarray(r[k]) for r in rows])
    np.savez_compressed(os.path.join(OUT, "dmap_%s.npz" % case), **out)
    print("dmap:%s decisions=%d now=%.4f (%.0fs)" % (case, len(rows), w.env.now, time.time() - t0), flush=True)


def rand_actions(seed, n, scale2=0.05):
    rng = np.random.default_rng(seed)
    a = rng.uniform(0.0, 1.0, size=(n, 3))
    a[:, 2] *= scale2
    return [list(map(float, x)) for x in a]


SMALL_MC = ('"capacity" : 2500\n"threshold" : 0\n"velocity" : 5\n"pm" : 1\n"charging_range" : 27\n'
            '"alpha" : 4500\n"beta" : 30\n"epsilon" : 0.0000000001\n')

TINY_MC = SMALL_MC.replace("2500", "700")

EDGE_ACTIONS = [
    [0.9, 0.9, 0.01], [0.1, 0.2, 0.02], [0.5, 0.1, 0.0],      # the SURVEY §8(c) known-answer opening
    [1.5, -0.2, 0.01],                                       # clipped to [1, 0, .01]  (Q14)
    [0.0, 0.0, 0.0], [1.0, 1.0, 0.0],                        # frame corners, zero charge
    [0.4881256, 0.52171893, 0.003],                          # ≈ base station
    [0.5, 0.1, 0.0],                                         # same destination again → zero-length move
    [0.3, 0.7, 0.0004873294346978558],                       # charge time 1.0000000000000002 s → span residue
    [0.62, 0.33, 0.0009746588693957114],                     # exactly 2 s of charging
    [0.25, 0.25, 1.0 / 2052.0],
    [0.77, 0.12, 0.02], [0.12, 0.77, 0.03], [0.5, 0.5, 0.05],
]

CASES = {
    # name: (scenario, actions, kwargs)
    "basic_n50": ("hanoi1000n50", rand_actions(0, 64), dict(max_decisions=45)),
    "edge_n50": ("hanoi1000n50", EDGE_ACTIONS, dict(max_decisions=30, full_state_every=10)),
    "full_n100": ("hanoi1000n100", rand_actions(1, 256), dict()),
    "full_n200": ("hanoi1000n200", rand_actions(2, 256), dict()),
    "longcharge_n50": ("hanoi1000n50", rand_actions(3, 64, scale2=0.6), dict(max_decisions=24)),
    "smallmc_n50": ("hanoi1000n50", rand_actions(4, 64, scale2=0.01), dict(mc_yaml=SMALL_MC, max_decisions=40)),
    "deadmc_n50": ("hanoi1000n50", rand_actions(8, 64, scale2=0.002), dict(mc_yaml=TINY_MC, max_decisions=60,
                                                                           event_budget=400_000)),
    "two_mc_sonla": ("sonla1000n50", rand_actions(5, 64), dict(num_agent=2, max_decisions=30)),
    "one_mc_n150": ("hanoi1000n150", rand_actions(6, 64), dict(num_agent=1, max_decisions=16)),
    "map32_n50": ("hanoi1000n50", rand_actions(7, 64), dict(max_decisions=12, map_size=32, full_state_every=3)),
}
NETS = ["hanoi1000n50", "hanoi1000n100", "hanoi1000n150", "hanoi1000n200", "sonla1000n50"]


def main(argv):
    os.makedirs(OUT, exist_ok=True)
    R = load_reference()
    todo = argv or (["net:" + s for s in NETS] + ["ep:" + c for c in CASES] + ["dmap:random_n50"])
    for item in todo:
        kind, name = item.split(":")
        if kind == "net":
            pure_network(R, name)
        elif kind == "dmap":
            episode_density(R, name, "hanoi1000n50", 8)
        else:
            scn, actions, kw = CASES[name]
            episode(R, name, scn, actions, **kw)


if __name__ == "__main__":
    main(sys.argv[1:])
